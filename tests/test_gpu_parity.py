"""Parity of the CUDA path (through the C ABI) with the CPU oracle: bit-exact pileup matrices,
supported positions and corrected segments; logits within 1e-3 (BASELINE.json north_star)."""
import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu

LOGITS_TOL = 1e-3  # absolute, fp32 (BASELINE.json: "per-base logits match within 1e-3 fp32")


@pytest.mark.parametrize("profile,seed", [("r10", 1), ("r9", 2)])
def test_end_to_end_parity_w4096(profile, seed):
    rs = helpers.small_readset(n_reads=40, mean_len=9000, seed=seed, profile=profile)
    model = helpers.model_path(seed=3)
    ora = helpers.run_oracle(rs, model, 4096, 64)
    got = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    helpers.compare(ora, got, LOGITS_TOL)
    assert got["stats"]["supported"] == sum(len(w.supported) for w in ora["windows"].values())


def test_small_window_many_windows():
    # -w is a runtime parameter (src/main.rs:69-74): W=512 gives ~20 windows per read, short last
    # windows, reads split by uncovered windows, and batch groups (-b 4) smaller than a read.
    rs = helpers.small_readset(n_reads=60, mean_len=6000, seed=5, coverage=12.0, min_ovl=600)
    model = helpers.model_path(seed=4)
    ora = helpers.run_oracle(rs, model, 512, 4)
    got = helpers.run_product(rs, model, 512, 4, keep_debug=True)
    helpers.compare(ora, got, LOGITS_TOL)


def test_submit_target_equals_submit_alignments():
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=7)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64)
    b = helpers.run_product(rs, model, 4096, 64, use_submit_target=True)
    assert a["segments"] == b["segments"]


def test_launch_batching_invariance():
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=8)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64, launch_targets=1 << 20)
    b = helpers.run_product(rs, model, 4096, 64, launch_targets=3)
    assert a["segments"] == b["segments"]
    assert a["stats"]["device_launches"] == 1 and b["stats"]["device_launches"] > 1


def test_host_harness_matches_python_path():
    """C++ harness (feature threads + consumer over the C ABI) == single-threaded ctypes path."""
    from herro_b200 import Context, api
    rs = helpers.small_readset(n_reads=40, mean_len=8000, seed=9)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64)
    want_bases = sum(len(x) for v in a["segments"].values() for x in (v or []))
    want_targets = sum(1 for v in a["segments"].values() if v)
    ctx = Context(model, 0, 4096, 64, launch_targets=7)
    ctx.upload_reads(rs.seqs, rs.quals, rs.off)
    h = api.HostHarness(ctx, rs.ovl9, rs.cigars, rs.cig_off, rs.aln_off, np.diff(rs.off).astype(np.uint32))
    r1 = h.run(0, rs.n, 4)                                   # library does the windowing
    r2 = h.run(0, rs.n, 3, h.windowing(0, rs.n, 2))          # host-computed windows
    r3 = h.run(0, rs.n, 2, h.windowing(0, rs.n, 2), collect=True)  # the records the consumer polled, kept
    for r in (r1, r2, r3):
        assert r["bases"] == want_bases and r["targets"] == want_targets
    assert r1["checksum"] == r2["checksum"] == r3["checksum"]
    assert {c.rid: c.segments or None for c in r3["results"]} == a["segments"]


def test_cli_fastq_oec_to_fasta(tmp_path):
    """configs[0]-style plumbing: FASTQ + *.oec.zst batches -> FASTA, record set identical to the oracle's."""
    from herro_b200 import cli
    from tools import synth
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=13, min_len=4200)  # reads < W are never loaded (src/haec_io.rs:48)
    descs = [None if i % 3 else f"ch={i} run=x" for i in range(rs.n)]
    fq = str(tmp_path / "reads.fastq")
    synth.write_fastq(rs, fq, descs)
    synth.write_oec_batches(rs, str(tmp_path / "alns"), batch_size=11)
    model = helpers.model_path(seed=3)
    out = str(tmp_path / "out.fasta")
    cli.main(["inference", "--read-alns", str(tmp_path / "alns"), "-m", model, "-b", "64", fq, out])
    got = sorted(open(out, "rb").read().split(b">")[1:])
    ora = helpers.run_oracle(rs, model, 4096, 64)
    from herro_b200.api import fasta_records
    want = []
    for rid, segs in ora["segments"].items():
        if segs:
            d = descs[rid].encode() if descs[rid] is not None else None
            want += fasta_records(rs.ids[rid].encode(), d, segs).split(b">")[1:]
    assert got == sorted(want) and len(got) > 0


def test_forward_chunking_invariance(monkeypatch):
    """The forward pass over the supported positions is split into passes of HERRO_B200_CHUNK_POS positions
    (one pass per launch by default); the split must not change a single emitted base or logit."""
    rs = helpers.small_readset(n_reads=40, mean_len=9000, seed=11)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    monkeypatch.setenv("HERRO_B200_CHUNK_POS", "200")   # not a multiple of the 128-position GEMM tile; ragged last pass
    b = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    assert a["stats"]["supported"] > 3 * 200
    assert b["stats"]["kernel_launches"] > a["stats"]["kernel_launches"]
    assert a["segments"] == b["segments"]
    for key, wa in a["windows"].items():
        wb = b["windows"][key]
        assert np.array_equal(wa["bases_logits"], wb["bases_logits"]), key
        assert np.array_equal(wa["info_logits"], wb["info_logits"]), key


def test_lane_count_invariance(monkeypatch):
    """One launch lane or four: same records (HERRO_B200_LANES only changes how launches overlap)."""
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=12)
    model = helpers.model_path(seed=3)
    monkeypatch.setenv("HERRO_B200_LANES", "1")
    a = helpers.run_product(rs, model, 4096, 64, launch_targets=4)
    monkeypatch.setenv("HERRO_B200_LANES", "4")
    b = helpers.run_product(rs, model, 4096, 64, launch_targets=4)
    assert a["segments"] == b["segments"]
    assert b["stats"]["device_launches"] >= 4


def test_fused_qkv_attention_equals_unfused(monkeypatch):
    """k_qkv_attn_ws (QKV projection + attention on chip; scores and P·V as bf16x3 mma.sync) against the separate
    contraction + fp32 SIMT k_attention kernels: same emitted bases, logits equal to fp32 rounding noise."""
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=13)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    monkeypatch.setenv("HERRO_B200_NO_FUSE_ATTN", "1")
    b = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    assert b["stats"]["kernel_launches"] > a["stats"]["kernel_launches"]
    assert a["segments"] == b["segments"]
    worst = 0.0
    for key, wa in a["windows"].items():
        wb = b["windows"][key]
        worst = max(worst, float(np.abs(wa["bases_logits"] - wb["bases_logits"]).max(initial=0.0)))
    assert worst <= 1e-4, worst


@pytest.mark.parametrize("env", ["HERRO_B200_NO_FUSE_OPROJ", "HERRO_B200_NO_FUSE_FFN", "HERRO_B200_NO_FUSE_LN"])
def test_fused_ffn_and_layernorm_equal_unfused(monkeypatch, env):
    """k_ffn_ws (attention out-projection + residual + LayerNorm in front, hidden activations on chip, LayerNorm in the
    epilogue) / the LayerNorm-fused epilogues against the chain of separate contraction and LayerNorm kernels: same emitted
    bases, logits equal to fp32 rounding noise."""
    rs = helpers.small_readset(n_reads=30, mean_len=7000, seed=14)
    model = helpers.model_path(seed=3)
    a = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    monkeypatch.setenv(env, "1")
    b = helpers.run_product(rs, model, 4096, 64, keep_debug=True)
    assert b["stats"]["kernel_launches"] > a["stats"]["kernel_launches"]
    assert a["segments"] == b["segments"]
    worst = 0.0
    for key, wa in a["windows"].items():
        wb = b["windows"][key]
        worst = max(worst, float(np.abs(wa["bases_logits"] - wb["bases_logits"]).max(initial=0.0)))
    assert worst <= 1e-4, worst


def test_cli_features_reproduces_the_golden_dump(tmp_path):
    """`herro features` end to end (FASTQ + *.oec.zst -> per-window feature files) from the inputs committed with the fixture:
    native ingest (host/io.cpp), device windowing, pileup, hb_dump_features — byte-identical to the oracle-generated files."""
    import glob
    import os
    from herro_b200 import cli
    golden = os.path.join(helpers.ROOT, "tests", "golden", "features_dump")
    model = helpers.model_path(seed=3)
    out = str(tmp_path / "feats")
    cli.main(["features", "--read-alns", os.path.join(golden, "alns"), "-w", "256", "-m", model, "--targets-per-launch", "5",
              os.path.join(golden, "reads.fastq"), out])
    n = 0
    for d in sorted(glob.glob(os.path.join(golden, "read_*"))):
        for a in sorted(glob.glob(os.path.join(d, "*"))):
            b = os.path.join(out, os.path.basename(d), os.path.basename(a))
            assert open(a, "rb").read() == open(b, "rb").read(), b
            n += 1
    assert n >= 30


def test_native_pipeline_multithreaded_equals_single_threaded(tmp_path):
    """hbh_inference with `-t 4` (feature threads racing for targets, results in completion order) writes the same record set."""
    from herro_b200 import cli
    from tools import synth
    rs = helpers.small_readset(n_reads=40, mean_len=7000, seed=14, min_len=4200)
    fq = str(tmp_path / "reads.fastq")
    synth.write_fastq(rs, fq)
    synth.write_oec_batches(rs, str(tmp_path / "alns"), batch_size=7)
    model = helpers.model_path(seed=3)
    outs = []
    for t in ("1", "4"):
        out = str(tmp_path / f"out{t}.fasta")
        r = cli.main(["inference", "--read-alns", str(tmp_path / "alns"), "-m", model, "-b", "64", "-t", t, fq, out])
        assert r["failed_targets"] == 0 and r["records"] > 0
        outs.append(sorted(open(out, "rb").read().split(b">")[1:]))
    assert outs[0] == outs[1]


def test_torchscript_archive_as_model(tmp_path):
    """`-m model.pt` (src/inference.rs:185): a TorchScript archive of the stand-in graph is read natively by hb_create
    (torchscript.cpp) and corrects exactly like the HB200W1 blob holding the same weights."""
    torch = pytest.importorskip("torch")
    from oracle import forward_ref
    from herro_b200 import weights as hbw
    rs = helpers.small_readset(n_reads=20, mean_len=6000, seed=31)
    blob = helpers.model_path(seed=3)
    cfg, T = hbw.load_blob(blob)
    pt = str(tmp_path / "model.pt")
    torch.jit.script(forward_ref.from_weights(cfg, T)).save(pt)
    a = helpers.run_product(rs, blob, 4096, 64)
    b = helpers.run_product(rs, pt, 4096, 64)
    assert a["segments"] == b["segments"] and any(a["segments"].values())
