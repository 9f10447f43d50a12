#!/usr/bin/env python
"""bench.py — corrected bases/s of the features -> inference -> consensus hot path.

  python bench.py --gpus 1 --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      (the reference algorithm on the host cores)
  python bench.py ... --dump-outputs DIR                    (also writes the last timed step's corrected reads: dump_outputs)

Workload (BASELINE.json configs[2], "cfg3", the one the metric is quoted on; it fits one GPU): ONE synthetic
read set of 50k reads x 20 kb, R10 error profile, ~40x, `-b 128`, W = 4096.  The job is that set: its target
reads are cut into W + K steps of `--step-targets` (2000) consecutive targets — 5 + 20 steps cover all 50k.
With N GPUs the read store is replicated on every GPU and every step's targets are split by read id
(herro_b200/shard.py: contiguous ranges balanced by window count): no collective on the data path,
total work fixed, `scaling: strong`.  A rank builds only its own targets' alignments (the generator is
deterministic per read, so every rank sees the same read set).

Reported on ONE JSON line:
  value      corrected bases/s, whole job, device stages only, inputs already resident in HBM
             (hb_replay_last_launch of the rank's last step, K times; CUDA events on the launch stream)
  e2e        the same metric through the public C ABI with host buffers over the K timed steps:
             hb_submit_* from the feature threads -> hb_flush -> hb_poll_corrected, H2D/D2H inside the timed
             region (FASTQ/PAF ingest and the one-off read-store upload are the Rust host's job and are reported
             separately in `config`)
  roofline   the dominant kernel class, timed live with CUDA events inside the library
  cpu_baseline  the CPU oracle (a port: the reference is Rust and cannot be built here) + torch
             fp32 forward on a bounded sample of the same targets, and `parity_sample`: the CUDA path's segments
             for those targets compared with the oracle's
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "corrected_bases_per_sec"
UNIT = "bases/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=50000)
    ap.add_argument("--read-len", type=int, default=20000)
    ap.add_argument("--profile", default="r10")
    ap.add_argument("--window", type=int, default=4096)
    ap.add_argument("--batch-size", type=int, default=128, help="reference -b")
    ap.add_argument("--step-targets", type=int, default=2000, help="target reads per step, job-wide (split over the ranks)")
    ap.add_argument("--cpu-sample", type=int, default=16, help="targets in the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--feature-threads", type=int, default=8, help="reference -t: host threads submitting targets (4 threads stage ~40 targets/ms, about what one B200 consumes)")
    ap.add_argument("--e2e-launch-targets", type=int, default=2000, help="hb_options.launch_targets in the e2e regions (shared by the feature "
                    "threads: each hands over max(256, launch_targets / threads) targets per device launch; measured on cfg3 with 8 threads: "
                    "256-target launches 800-868 Mbases/s, 500: 785-796, 1000: 709, 2000: 584 - smaller launches overlap better across the lanes)")
    ap.add_argument("--host-windowing", action="store_true", help="e2e region submits host-computed OverlapWindows (hb_submit_target) instead of raw alignments")
    ap.add_argument("--cpu-threads", type=int, default=0, help="threads of the CPU legs (cpu_baseline / --impl reference); 0 = all host threads")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the corrected reads of the last timed step (rank 0's share) as .npy "
                    "files under DIR (see dump_outputs)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons of the job's GPUs DURING the timed region (B200_PROFILING.md).  One sampler for the whole
    job (rank 0), through NVML in-process: a poller per rank spawning nvidia-smi five times a second contends for the driver
    with the very launches being timed (measured at N=4).  Falls back to nvidia-smi when pynvml is unavailable."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, indices):
        super().__init__(daemon=True)
        self.indices = list(indices)
        self.stop_flag = threading.Event()
        self.sm, self.mx, self.reasons = [], [], set()
        self.n = 0

    def _nvml_loop(self):
        import pynvml
        pynvml.nvmlInit()
        hs = [pynvml.nvmlDeviceGetHandleByIndex(i) for i in self.indices]
        while not self.stop_flag.is_set():
            for h in hs:
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))
                r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.reasons |= {name for bit, name in self.REASONS.items() if r & bit}
            self.n += 1
            self.stop_flag.wait(0.1)

    def _smi_loop(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        ids = ",".join(str(i) for i in self.indices)
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={ids}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                for line in out.splitlines():
                    r = [x.strip() for x in line.split(",")]
                    if len(r) >= 6 and r[0].replace(".", "").isdigit():
                        self.sm.append(float(r[0])); self.mx.append(float(r[1]))
                        self.reasons |= {names[i] for i in range(4) if r[2 + i].lower().startswith("active")}
                self.n += 1
            except Exception:
                pass
            self.stop_flag.wait(0.5)

    def run(self):
        try:
            self._nvml_loop()
        except Exception:
            self._smi_loop()

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": self.n,
                "gpus": self.indices}


_CACHE = {}
_TUNED = {}  # host threads -> torch intra-op threads chosen by the probe in cpu_reference_run


def cpu_reference_run(rs, model, targets, window, batch_size, threads):
    """The reference algorithm on the host: C++ oracle (features, collate, consensus) on `threads`
    workers + torch fp32 forward exactly as src/inference.rs:147-175 would call the model on CPU."""
    import torch
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po, forward_ref
    from herro_b200 import weights as hbw
    if _CACHE.get("rs") is not rs:  # the oracle's read store and the torch module are built once per read set / model
        _CACHE.update(rs=rs, reads=po.Reads(rs.ids, [rs.seq(i) for i in range(rs.n)], [rs.qual(i) for i in range(rs.n)]))
    if _CACHE.get("model") != model:
        cfg, tensors = hbw.load_blob(model)
        _CACHE.update(model=model, net=forward_ref.from_weights(cfg, tensors))
    reads, net = _CACHE["reads"], _CACHE["net"]

    def feat(t):
        ovl, cigs = rs.target_alns(t)
        return t, (po.Target(reads, t, ovl, cigs, window, batch_size) if len(ovl) else None)

    # Intra-op threads of the torch forward: "all host threads" is not the fastest setting on a many-core box (the
    # per-batch tensors are small), so the CPU arm gets the best of a few settings, measured on one batch outside the
    # timed region.  The feature/consensus legs always use `threads` workers.
    fwd_threads = _TUNED.get(threads, threads)
    if threads > 16 and threads not in _TUNED:
        probe = next((tg for _, tg in map(feat, targets[:4]) if tg is not None and tg.n_batches), None)
        if probe is not None:
            B = probe.batch(0)
            best = None
            for nt in sorted({threads, 64, 32, 16} & set(range(1, threads + 1)), reverse=True):
                torch.set_num_threads(nt)
                forward_ref.run_batch(net, B.bases, B.quals, B.lens, B.indices)  # warm
                t = time.time()
                forward_ref.run_batch(net, B.bases, B.quals, B.lens, B.indices)
                t = time.time() - t
                if best is None or t < best[0]:
                    best = (t, nt)
            fwd_threads = best[1]
        _TUNED[threads] = fwd_threads
    torch.set_num_threads(fwd_threads)
    t0 = time.time()

    with ThreadPoolExecutor(threads) as ex:
        T = list(ex.map(feat, targets))
    t_feat = time.time() - t0
    t1 = time.time()
    for _, tg in T:
        if tg is None:
            continue
        for b in range(tg.n_batches):
            B = tg.batch(b)
            info, bl = forward_ref.run_batch(net, B.bases, B.quals, B.lens, B.indices)
            for k, wi in enumerate(B.win_index):
                tg.set_logits(int(wi), info[k], bl[k])
    t_fwd = time.time() - t1
    t2 = time.time()
    bases = 0
    segs = {}
    for t, tg in T:
        if tg is None:
            continue
        s = tg.consensus()
        segs[t] = s
        bases += sum(len(x) for x in (s or []))
    t_cons = time.time() - t2
    return dict(bases=bases, seconds=time.time() - t0, t_features=t_feat, t_forward=t_fwd, t_consensus=t_cons, segments=segs,
                torch_threads=fwd_threads)


def gpu_numa_cpus(local_rank):
    """CPUs of the NUMA node the rank's GPU hangs off (sysfs), or None."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        return (node, cpus) if cpus else None
    except Exception:
        return None


def workload_name(args):
    # BASELINE.json configs: cfg2 10k x 15 kb R10 -b 64; cfg3 50k x 20 kb R10 -b 128 (the default); cfg4 100 kb reads; cfg5 R9 profile 15 kb
    name = "cfg5" if args.profile == "r9" else ("cfg4" if args.read_len >= 50000 else ("cfg2" if args.read_len <= 15000 else "cfg3"))
    return (f"{name}: synthetic {args.reads} reads x {args.read_len} bp, {args.profile} profile, 40x, W={args.window}, "
            f"-b {args.batch_size}")


DUMP_SAMPLE_BASES = 8 << 20  # corrected bases written by dump_outputs: 32 MB as float32


def dump_outputs(d, segments):
    """What a caller of the timed path received for the last timed step, as float .npy files under `d`:
      target_ids           [T] f64  targets that produced a record, ascending
      segments_per_target  [T] f64  0 = the read is omitted from the output
      segment_lengths      [S] f64  every segment of those targets, in target order
      sample_target_ids    [k] f64  a fixed, seeded sample of target_ids whose bases fit DUMP_SAMPLE_BASES
      sample_bases         [B] f32  ASCII codes of the sampled targets' segments back to back, in sample order
    `segments`: {target id: list of bytes (empty or None = omitted)}."""
    os.makedirs(d, exist_ok=True)
    rids = sorted(segments)
    segs = [segments[t] or [] for t in rids]
    sample, bases, n = [], [], 0
    for i in np.random.default_rng(0).permutation(len(rids)):
        size = sum(len(x) for x in segs[i])
        if n + size <= DUMP_SAMPLE_BASES:
            sample.append(rids[i])
            bases += segs[i]
            n += size
    out = {"target_ids": np.array(rids, np.float64), "segments_per_target": np.array([len(s) for s in segs], np.float64),
           "segment_lengths": np.array([len(x) for s in segs for x in s], np.float64),
           "sample_target_ids": np.array(sample, np.float64),
           "sample_bases": np.frombuffer(b"".join(bases), np.uint8).astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)


def ensure_model():
    """The benchmark's model blob, written to a temporary file (the tree may be read-only); the caller removes it."""
    from herro_b200 import weights as hbw
    fd, p = tempfile.mkstemp(prefix="herro_bench_model_", suffix=".hbw")
    os.close(fd)
    cfg = hbw.NetConfig()
    hbw.save_blob(p, cfg, hbw.random_weights(cfg, seed=7))
    return p, cfg


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    threads = args.cpu_threads or os.cpu_count() or 1
    workload = workload_name(args)
    n_steps = args.warmup + args.steps
    from tools import synth

    # ------------------------------------------------------------------ reference arm (CPU only)
    if args.impl == "reference":
        if rank != 0:
            return
        model, cfg = ensure_model()
        # bounded sample: the torch fp32 forward over whole [B,L,31] batches costs seconds per target read on the host,
        # so a step is 2 target reads (1 when many steps are requested) and the whole run stays within a few minutes
        per = 2 if n_steps <= 14 else 1
        need = n_steps * per
        rs = synth.generate(args.reads, args.read_len, profile=args.profile, seed=args.seed, coverage=40.0, min_ovl=2048,
                            targets=(0, need))
        tg = list(range(need))
        times, bases = [], 0
        for s in range(n_steps):
            r = cpu_reference_run(rs, model, tg[s * per:(s + 1) * per], args.window, args.batch_size, threads)
            if s >= args.warmup:
                times.append(r["seconds"])
                bases += r["bases"]
        tot = sum(times)
        v = bases / tot
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
            "config": {"workload": workload, "sample": f"{per} target reads per step"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"{args.steps} steps x {per} target reads of the workload (CPU oracle on {threads} threads + torch fp32 "
                                       f"forward on {r['torch_threads']} intra-op threads, the fastest of a probe)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["segments"])
        os.remove(model)
        return

    # ------------------------------------------------------------------ our arm
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (herro_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa = gpu_numa_cpus(local_rank)
    if world > 1 and numa:  # keep this rank's generator / packing / harness threads and their memory on the GPU's socket
        os.sched_setaffinity(0, numa[1])
    my_cpus = len(os.sched_getaffinity(0))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    from herro_b200 import Context, api, shard
    model, cfg = ensure_model()
    # ---- the job: the first n_steps * S target reads of ONE read set, sharded by read id
    S = max(1, min(args.step_targets, args.reads // n_steps))
    n_job = n_steps * S
    t0 = time.time()
    gen = synth.Generator(args.reads, args.read_len, profile=args.profile, seed=args.seed, coverage=40.0, min_ovl=2048,
                          threads=my_cpus)
    lens_all = gen.read_lens()
    mine = shard.shard_targets(lens_all[:n_job], args.window, rank, world)
    lo, hi = (int(mine[0]), int(mine[-1]) + 1) if len(mine) else (0, 0)
    rs = gen.readset(targets=(lo, hi))
    gen.close()
    t_gen = time.time() - t0
    # this rank's slice of step s: [cut[s], cut[s+1])
    cut = [lo + (hi - lo) * s // n_steps for s in range(n_steps + 1)]
    t_w0, t_w1 = cut[0], cut[args.warmup]          # warm-up steps
    t_t0, t_t1 = cut[args.warmup], cut[n_steps]    # timed steps
    lt = max(1, max(cut[s + 1] - cut[s] for s in range(n_steps)))   # targets per launch = this rank's share of a step
    nthr = max(1, min(args.feature_threads, my_cpus))
    ctx = Context(model, local_rank, args.window, args.batch_size, launch_targets=lt)
    t0 = time.time()
    ctx.upload_reads(rs.seqs, rs.quals, rs.off)
    torch.cuda.synchronize()
    t_upload = time.time() - t0
    # The C++ host harness plays the Rust binary: `-t` feature threads submit targets through the C ABI,
    # one consumer thread polls corrected reads (herro_b200/host/harness.cpp).
    harness = api.HostHarness(ctx, rs.ovl9, rs.cigars, rs.cig_off, rs.aln_off, np.diff(rs.off).astype(np.uint32))
    # ---- host side that stays in the Rust binary: windowing (timed, outside the measured region)
    t0 = time.time()
    wthr = max(nthr, min(32, my_cpus))
    win_warm = harness.windowing(t_w0, t_w1, wthr)
    win_timed = harness.windowing(t_t0, t_t1, wthr)
    t_windowing = time.time() - t0

    ctx.set_launch_targets(max(lt, args.e2e_launch_targets))
    # warm-up: once from a single thread (hands over whole launches: every pinned / device pool reaches at least its steady-state
    # size whatever the length of the warm-up), then through the same multi-threaded path as the timed steps
    harness.run(t_w0, t_w1, 1, win_warm)
    harness.run(t_w0, t_w1, nthr, win_warm)
    harness.run(t_w0, min(t_w1, t_w0 + 2 * lt), nthr, None)
    ctx.replay_last_launch(1)
    ctx.reset_stats()
    sampler = ClockSampler(range(args.gpus) if rank == 0 else [])
    if rank == 0:
        sampler.start()
    # ---- region 1: end to end through the C ABI, host buffers, copies inside: hb_submit_target from the feature threads
    #      (OverlapWindows from the host's extract_windows, as the Rust host would pass them), hb_poll_corrected from the consumer
    barrier()
    t0 = time.perf_counter()
    r_e2e = harness.run(t_t0, t_t1, nthr, win_timed)
    barrier()
    t_e2e = time.perf_counter() - t0
    st = ctx.stats()
    # ---- region 1b: the same targets as raw alignments (hb_submit_alignments: windowing inside the library, inside the timed region)
    ctx.reset_stats()
    barrier()
    t0 = time.perf_counter()
    r_e2e_w = harness.run(t_t0, t_t1, nthr, None)
    barrier()
    t_e2e_w = time.perf_counter() - t0
    st_w = ctx.stats()
    assert r_e2e_w["checksum"] == r_e2e["checksum"], "hb_submit_alignments and hb_submit_target disagree"
    # one full-size launch (this rank's share of the last step), alone on the GPU: its per-kernel CUDA-event times feed the
    # roofline (in the pipelined region the lanes overlap, so per-kernel times there include the other lanes' kernels), and it
    # is the launch the HBM-resident replay re-runs; its corrected reads are what --dump-outputs writes
    ctx.reset_stats()
    ctx.set_launch_targets(lt)
    ctx.set_kernel_timing(True)
    r_full = harness.run(cut[n_steps - 1], cut[n_steps], 1, harness.windowing(cut[n_steps - 1], cut[n_steps], wthr),  # same entry as `e2e`
                         collect=bool(args.dump_outputs) and rank == 0)
    st_full = ctx.stats()
    # ---- region 2: device stages only, inputs resident in HBM (one launch's working set is GBs of matrices + activations,
    #      larger than the 126 MB L2, so no L2 flush is needed)
    last_launch_bases = st_full["last_launch_bases"]
    barrier()
    ms_dev = ctx.replay_last_launch(args.steps)
    barrier()
    sampler.stop_flag.set()
    if rank == 0:
        sampler.join(timeout=3)
    st2 = ctx.stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {c.rid: c.segments for c in r_full["results"]})
    t_dev = ms_dev / 1e3
    vals = torch.tensor([t_dev, t_e2e, float(last_launch_bases * args.steps), float(r_e2e["bases"]), t_e2e_w, t_upload, t_gen,
                         float(st["host_allocs"]), float(st["windows"]), float(hi - lo)], dtype=torch.float64, device="cuda")
    if dist is not None:
        gathered = [torch.zeros_like(vals) for _ in range(args.gpus)]
        dist.all_gather(gathered, vals)
    else:
        gathered = [vals]
    G = torch.stack(gathered).cpu().numpy()
    t_dev, t_e2e, t_e2e_w = float(G[:, 0].max()), float(G[:, 1].max()), float(G[:, 4].max())
    bases_dev, bases_e2e_all = float(G[:, 2].sum()), float(G[:, 3].sum())
    per_rank = {"ms_per_step": [round(1e3 * x / args.steps, 3) for x in G[:, 0]], "bases_per_step": [x / args.steps for x in G[:, 2]],
                "e2e_seconds": [round(x, 4) for x in G[:, 1]], "e2e_incl_windowing_seconds": [round(x, 4) for x in G[:, 4]],
                "read_store_upload_s": [round(x, 3) for x in G[:, 5]], "generate_s": [round(x, 2) for x in G[:, 6]],
                "host_allocs_in_e2e_region": [int(x) for x in G[:, 7]], "windows": [int(x) for x in G[:, 8]], "targets": [int(x) for x in G[:, 9]],
                "imbalance_windows": round(float(G[:, 8].max() / max(G[:, 8].mean(), 1.0) - 1.0), 4),
                "imbalance_e2e_seconds": round(float(G[:, 1].max() / max(G[:, 1].mean(), 1e-9) - 1.0), 4)}

    parity_failed = False
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tf_peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        mk, nk, cf = st_full["ms_kernel"], st_full["n_kernel"], st_full["class_flops"]
        # the dominant kernel of the step, by CUDA-event time of the isolated full-size launch
        KERNEL_OF = {"gemm": "k_gemm_ws", "ffn": "k_ffn_ws", "qkv_attn": "k_qkv_attn_ws", "stem": "k_stem_tc", "pileup": "k_pileup"}
        DESCR = {"gemm": "tcgen05 bf16x3 contractions: out-proj(+LN) and read-axis collapse",
                 "ffn": "fused FFN1 -> ReLU -> FFN2 + residual + LayerNorm on tcgen05, bf16x3",
                 "qkv_attn": "fused QKV projection (tcgen05) + read-axis attention (mma.sync), bf16x3",
                 "stem": "embedding+conv stem as a tcgen05 contraction (2 passes) + first LayerNorm",
                 "pileup": "pileup build (consume bitmaps, 4-row groups; second get_supported, majority vote)"}
        top = max((k for k in mk if k in KERNEL_OF), key=lambda k: mk[k])
        pile_gbs = st_full["pileup_algo_bytes"] / (mk["pileup"] * 1e-3) / 1e9 if mk["pileup"] > 0 else 0.0
        traffic, traffic_src = {}, None
        for name in ("r02_traffic.json", "r01d_traffic.json"):
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", name)))
                traffic_src = name
                break
            except Exception:
                pass
        import re
        traffic = {re.sub(r"^void |<.*", "", k): v for k, v in traffic.items()}   # "void k_ffn_ws<1>" -> "k_ffn_ws"
        t_top = traffic[KERNEL_OF[top]].get("dram_bytes_per_launch") if isinstance(traffic.get(KERNEL_OF[top]), dict) else None
        tnote = (f"from file profiles/{traffic_src} ({traffic.get('_note', 'ncu --set full capture of another run')}); not measured in this run"
                 ) if t_top is not None else None
        if top == "pileup":
            roof = {"kernel": "k_pileup (" + DESCR[top] + ")", "bound": "hbm", "achieved": pile_gbs, "peak": hbm_peak,
                    "unit": "GB/s", "frac": pile_gbs / hbm_peak, "traffic": t_top, "traffic_note": tnote, "peak_source": peak_src,
                    "launches_per_step": nk[top], "ms_per_launch": mk[top] / max(nk[top], 1)}
        else:
            tf = cf[top] / (mk[top] * 1e-3) / 1e12
            roof = {"kernel": KERNEL_OF[top] + " (" + DESCR[top] + "; algorithmic fp32 FLOPs over 31 read tokens per position, "
                    "each executed as 3 bf16 MMA passes)", "bound": "tensor", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s",
                    "frac": tf / tf_peak, "traffic": t_top, "traffic_note": tnote,
                    "peak_source": peak_src, "launches_per_step": nk[top], "ms_per_launch": mk[top] / max(nk[top], 1)}
        tensor_classes = {k: {"ms": mk[k], "launches": nk[k], "algorithmic_tflops": cf[k] / (mk[k] * 1e-3) / 1e12}
                          for k in ("stem", "qkv_attn", "gemm", "ffn") if nk.get(k) and mk[k] > 0}
        nl = max(st["device_launches"], 1)
        out = {
            "metric": METRIC, "value": bases_dev / t_dev, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8 pileup/consensus + f32 forward", "data": "synthetic",
            "config": {"workload": workload, "job_targets": n_job, "targets_per_step": S, "targets_per_step_per_rank": lt, "e2e_launch_targets": max(lt, args.e2e_launch_targets),
                       "windows_per_step_rank0": st_full["windows"], "supported_positions_per_step_rank0": st_full["supported"],
                       "sharding": (f"read-id shard of one read set over {world} GPUs (shard.shard_targets: contiguous, balanced by windows), "
                                    f"read store replicated, no collective") if world > 1 else "single GPU",
                       "l2": "inputs larger than L2 (per-launch working set >> 126 MB)",
                       "host_feature_threads": nthr, "numa_node": numa[0] if numa else None, "host_cpus_of_rank": my_cpus,
                       "host_worker_busy_ms_per_launch": st["ms_worker_busy"] / nl,
                       "host_worker_gpu_wait_ms_per_launch": st["ms_worker_gpu_wait"] / nl,
                       "launches_in_e2e_region": st["device_launches"], "host_allocs_in_e2e_region": st["host_allocs"],
                       "host_alloc_ms_in_e2e_region": st["ms_host_alloc"], "submit_backpressure_ms_sum": st["ms_submit_wait"],
                       "worker_phase_ms_per_launch": [round(x / nl, 3) for x in st["ms_worker_phase"][:7]],
                       "harness_seconds": r_e2e["seconds"], "submit_seconds_sum": r_e2e["submit_seconds_sum"],
                       "host_windowing_s": t_windowing, "host_windowing_threads": wthr, "read_store_upload_s": t_upload, "generate_s": t_gen,
                       "model": {"channels": cfg.channels, "heads": cfg.heads, "layers": cfg.layers, "ffn": cfg.ffn,
                                 "stem_k": cfg.stem_k, "collapse": cfg.collapse,
                                 "weights": "random init, architecture of north_star (the production TorchScript is not available offline)"}},
            "e2e": {"value": bases_e2e_all / t_e2e, "unit": UNIT, "seconds": t_e2e,
                    "h2d_bytes_per_step": st["h2d_bytes"] / args.steps, "d2h_bytes_per_step": st["d2h_bytes"] / args.steps,
                    "entry": "hb_submit_target (OverlapWindows from the host's extract_windows, computed outside the timed region)"},
            "e2e_incl_windowing": {"value": bases_e2e_all / t_e2e_w, "unit": UNIT, "seconds": t_e2e_w,
                                   "h2d_bytes_per_step": st_w["h2d_bytes"] / args.steps, "d2h_bytes_per_step": st_w["d2h_bytes"] / args.steps,
                                   "entry": "hb_submit_alignments (raw alignments; windowing inside the library, inside the timed region)"},
            "gpu_launches": int(st["kernel_launches"] + st_w["kernel_launches"] + st_full["kernel_launches"] + st2["kernel_launches"]),
            "roofline": roof,
            "kernels_ms_per_step": {k: mk[k] for k in mk if nk[k]},
            "tensor_kernels": tensor_classes,
            "pileup_roofline": {"bound": "hbm", "achieved": pile_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": pile_gbs / hbm_peak},
            "clocks": sampler.summary(),
            "per_rank": per_rank,
        }
        if not args.no_cpu_baseline and args.gpus == 1:
            tg = list(range(t_t0, t_t0 + args.cpu_sample))
            r = cpu_reference_run(rs, model, tg, args.window, args.batch_size, threads)
            # parity on the measured workload: the same targets through the CUDA path (a second context with the debug taps),
            # every matrix byte, SupportedPos, logits within 1e-3 and the corrected segments (tests/helpers.compare)
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import helpers
            ptg = tg[:max(1, min(len(tg), 8))]
            try:
                ora = helpers.run_oracle(rs, model, args.window, args.batch_size, targets=ptg)
                got = helpers.run_product(rs, model, args.window, args.batch_size, targets=ptg, keep_debug=True)
                pr = helpers.compare(ora, got, 1e-3)
                got["ctx"].close()
                out["parity_sample"] = {"targets": len(ptg), "identical": True, "windows": pr["windows"], "max_logit_abs_diff": pr["max_logit_diff"],
                                        "reads_differing_only_by_logit_near_ties": pr["tie_reads"],
                                        "checked": "tokens, quals, SupportedPos, logits <= 1e-3, corrected segments vs the CPU oracle"}
            except AssertionError as e:
                out["parity_sample"] = {"targets": len(ptg), "identical": False, "error": str(e)[:300]}
                parity_failed = True
            out["cpu_baseline"] = {"value": r["bases"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": "port",
                                   "sample": f"{len(tg)} target reads of the workload; features {r['t_features']:.1f}s, "
                                             f"forward {r['t_forward']:.1f}s ({r['torch_threads']} torch threads, fastest of a probe), "
                                             f"consensus {r['t_consensus']:.2f}s"}
        print(json.dumps(out))
    ctx.close()
    try:
        os.remove(model)
    except OSError:
        pass
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and parity_failed:
        raise SystemExit("parity_sample: the CUDA path and the CPU oracle disagree on the sampled targets")


if __name__ == "__main__":
    main()
