"""Host-side mirror of the reference's hot-path interface over the C ABI (include/herro_b200.h).

The deployed host is the reference's Rust binary (INTEGRATION.md); there is no Rust toolchain
offline, so this ctypes layer is the harness that plays `lib.rs::error_correction`
(src/lib.rs:113-206) for tests and benchmarks: it keeps the reference's vocabulary — reads,
alignments grouped by target (`(tid, Vec<Alignment>)`, src/overlaps.rs:371-373), windows,
corrected segments — and calls exactly the entry points the Rust `mod ffi` would bind.

Everything compute-related happens inside libherro_b200.so (CUDA, sm_100a).  There is no CPU
fallback: constructing a Context without a CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libherro_b200.so")

HB_FLAG_KEEP_DEBUG = 1

OVERLAP_DTYPE = np.dtype(
    {"names": ["qid", "qlen", "qstart", "qend", "strand", "tid", "tlen", "tstart", "tend", "cigar", "cigar_len"],
     "formats": ["<u4"] * 9 + ["<u8", "<u4"],
     "offsets": [0, 4, 8, 12, 16, 20, 24, 28, 32, 40, 48],
     "itemsize": 56})
OVERLAP_WINDOW_DTYPE = np.dtype([(n, "<u4") for n in (
    "overlap_idx", "window_idx", "tstart", "qstart", "qend", "cigar_start_idx", "cigar_start_offset", "cigar_end_idx",
    "cigar_end_offset")])


class HbOptions(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("window_size", C.c_uint32), ("batch_size", C.c_uint32),
                ("launch_targets", C.c_uint32), ("flags", C.c_uint32)]


KERNEL_CLASSES = ["tokenize", "pass1", "scores", "pass2a", "scan", "pileup", "lists", "stem", "layernorm", "gemm",
                  "attention", "heads", "consensus", "ffn", "qkv_attn"]


class HbStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("targets", "windows", "overlap_windows", "rows", "supported",
                                          "corrected_bases", "h2d_bytes", "d2h_bytes", "kernel_launches",
                                          "device_launches", "pileup_algo_bytes", "gemm_flops", "forward_flops")] + \
               [(n, C.c_double) for n in ("ms_features", "ms_forward", "ms_consensus")] + \
               [("ms_kernel", C.c_double * 16), ("n_kernel", C.c_uint64 * 16)] + \
               [(n, C.c_uint64) for n in ("last_launch_targets", "last_launch_windows", "last_launch_bases")] + \
               [("ms_worker_busy", C.c_double), ("ms_worker_gpu_wait", C.c_double)] + \
               [("host_allocs", C.c_uint64), ("ms_host_alloc", C.c_double), ("ms_submit_wait", C.c_double),
                ("class_flops", C.c_uint64 * 16), ("ms_worker_phase", C.c_double * 8)]


HOST_LIB_PATH = os.path.join(_HERE, "libherro_host.so")


class HerroError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"herro_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """dlopen the in-tree CUDA library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HerroError(-2, f"{LIB_PATH} not built - run `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(herro_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u32, u32p = C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)
    L.hb_last_error.restype = C.c_char_p
    L.hb_last_error.argtypes = [vp]
    L.hb_create.argtypes = [C.POINTER(vp), C.c_int, C.c_char_p, C.POINTER(HbOptions)]
    L.hb_destroy.argtypes = [vp]
    L.hb_destroy.restype = None
    L.hb_upload_reads.argtypes = [vp, u32, vp, vp, vp]
    L.hb_submit_target.argtypes = [vp, u32, u32, vp, u32, vp, u32]
    L.hb_submit_alignments.argtypes = [vp, u32, vp, u32]
    L.hb_extract_windows.argtypes = [vp, u32, u32, u32, vp, u32, u32p]
    L.hb_window_range.argtypes = [vp, u32, u32, u32p, u32p]
    L.hb_flush.argtypes = [vp]
    L.hb_set_launch_targets.argtypes = [vp, u32]
    L.hb_set_kernel_timing.argtypes = [vp, C.c_int]
    L.hb_poll_corrected.argtypes = [vp, u32p, C.POINTER(vp), C.POINTER(vp), u32p]
    L.hb_release_result.argtypes = [vp, vp]
    L.hb_release_result.restype = None
    L.hb_bind_calling_thread.argtypes = [vp]
    L.hb_get_stats.argtypes = [vp, C.POINTER(HbStats)]
    L.hb_reset_stats.argtypes = [vp]
    L.hb_debug_window_shape.argtypes = [vp, u32, u32, u32p]
    L.hb_debug_dump_window.argtypes = [vp, u32, u32, vp, vp, vp, vp, vp, vp]
    L.hb_replay_last_launch.argtypes = [vp, u32, C.POINTER(C.c_float)]
    L.hb_dump_features.argtypes = [vp, u32, C.c_char_p, vp]
    L.hb_inspect_model.argtypes = [C.c_char_p, u32p, C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]
    fp = C.POINTER(C.c_float)
    L.hb_selftest_gemm.argtypes = [C.c_int, u32, u32, u32, C.c_int, C.c_int, u32, fp, fp, fp, fp]
    _lib = L
    return L


EXPORTED_SYMBOLS = ["hb_inspect_model", "hb_dump_features", "hb_window_range", "hb_bind_calling_thread", "hb_set_launch_targets", "hb_set_kernel_timing", "hb_extract_windows", "hb_create", "hb_destroy", "hb_upload_reads", "hb_submit_target", "hb_submit_alignments", "hb_flush",
                    "hb_poll_corrected", "hb_release_result", "hb_last_error", "hb_get_stats", "hb_reset_stats",
                    "hb_debug_window_shape", "hb_debug_dump_window", "hb_replay_last_launch", "hb_selftest_gemm"]


def selftest_gemm(M, N, K, act=0, res=0, lda_extra=0, device=0):
    """-> dict(max_abs_err, max_abs_ref, ms_tc, ms_simt): tcgen05 bf16x3 contraction vs fp32 SIMT."""
    L = load_library()
    v = [C.c_float() for _ in range(4)]
    rc = L.hb_selftest_gemm(device, M, N, K, act, res, lda_extra, *[C.byref(x) for x in v])
    if rc != 0:
        raise HerroError(rc, L.hb_last_error(None).decode())
    return dict(max_abs_err=v[0].value, max_abs_ref=v[1].value, ms_tc=v[2].value, ms_simt=v[3].value)


# ------------------------------------------------------------------------------------------
# haec_io.rs host side: 2-bit packing (src/haec_io.rs:121-136).  Host data plane — stays in the
# Rust binary in deployment; needed here only because the harness replaces that binary.
# ------------------------------------------------------------------------------------------
_ENC = np.full(256, 255, dtype=np.uint64)
for _i, _ch in enumerate(b"ACGT"):
    _ENC[_ch] = _i
    _ENC[_ch + 32] = _i


def pack_2bit(seq: np.ndarray) -> np.ndarray:
    """ASCII u8 array -> u64 words, 32 bases per word, A0 C1 G2 T3, little-endian in the word."""
    n = int(seq.shape[0])
    codes = _ENC[seq]
    if n and int(codes.max()) > 3:
        raise ValueError("non-ACGT base: the reference's 2-bit packing is undefined for it (SURVEY.md H12)")
    nw = (n + 31) // 32
    pad = np.zeros(nw * 32, dtype=np.uint64)
    pad[:n] = codes
    shifts = (np.arange(32, dtype=np.uint64) * np.uint64(2))[None, :]
    return np.bitwise_or.reduce(pad.reshape(nw, 32) << shifts, axis=1)


def extract_windows(overlaps: np.ndarray, window_size: int, n_windows: int) -> np.ndarray:
    """Host-only windowing of all alignments of one target (hb_extract_windows) -> OVERLAP_WINDOW_DTYPE array."""
    L = load_library()
    cap = len(overlaps) * (n_windows + 1) + 1
    out = np.zeros(cap, dtype=OVERLAP_WINDOW_DTYPE)
    n = C.c_uint32()
    rc = L.hb_extract_windows(overlaps.ctypes.data, len(overlaps), window_size, n_windows, out.ctypes.data, cap,
                              C.byref(n))
    if rc != 0:
        raise HerroError(rc, "alignment on which the reference would panic")
    return out[:n.value]


def inspect_model(path: str):
    """Architecture and parameter hash of a model file (HB200W1 blob or TorchScript archive), host only (hb_inspect_model)."""
    L = load_library()
    dims = (C.c_uint32 * 6)()
    h = C.c_uint64()
    err = C.create_string_buffer(512)
    rc = L.hb_inspect_model(path.encode(), dims, C.byref(h), err, len(err))
    if rc != 0:
        raise HerroError(rc, err.value.decode(errors="replace"))
    return dict(zip(("stem_k", "channels", "heads", "layers", "ffn", "collapse"), [int(x) for x in dims])), int(h.value)


def window_range(overlap: np.ndarray, window_size: int, n_windows: int):
    """(first, end) of the windows one alignment (a 1-element OVERLAP_DTYPE array) contributes to (hb_window_range)."""
    L = load_library()
    a, b = C.c_uint32(), C.c_uint32()
    rc = L.hb_window_range(overlap.ctypes.data, window_size, n_windows, C.byref(a), C.byref(b))
    if rc != 0:
        raise HerroError(rc, "alignment on which the reference would panic")
    return a.value, b.value


@dataclass
class Corrected:
    rid: int
    segments: list  # list[bytes]; empty = read omitted from the output (consensus() returned None)


class Context:
    """One per GPU — the per-device worker group of src/lib.rs:154-200."""

    def __init__(self, model_path: str, device: int = 0, window_size: int = 4096, batch_size: int = 64,
                 launch_targets: int = 0, keep_debug: bool = False):
        self._L = load_library()
        self._h = C.c_void_p()
        opt = HbOptions(C.sizeof(HbOptions), window_size, batch_size, launch_targets,
                        HB_FLAG_KEEP_DEBUG if keep_debug else 0)
        rc = self._L.hb_create(C.byref(self._h), device, model_path.encode(), C.byref(opt))
        if rc != 0:
            raise HerroError(rc, self._L.hb_last_error(None).decode())
        self.window_size = window_size
        self._keep = []
        self.read_len = None
        self.failed = []

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.hb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise HerroError(rc, self._L.hb_last_error(self._h).decode())
        return rc

    # -- read store ---------------------------------------------------------------------
    def upload_reads(self, seqs: np.ndarray, quals: np.ndarray, off: np.ndarray):
        """seqs/quals: concatenated ASCII / Phred+33 bytes, off[n+1].  Packs to the HAECSeq
        layout on the host (as get_reads does, src/haec_io.rs:56) and replicates it on the GPU."""
        n = len(off) - 1
        lens = np.diff(off).astype(np.uint32)
        woff = np.zeros(n + 1, dtype=np.uint64)
        woff[1:] = np.cumsum((lens.astype(np.uint64) + 31) // 32)
        words = np.zeros(int(woff[-1]) + 1, dtype=np.uint64)
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        off64 = np.ascontiguousarray(off, dtype=np.uint64)
        if _host_lib().hbh_pack_2bit(seqs.ctypes.data, off64.ctypes.data, n, words.ctypes.data, woff.ctypes.data,
                                     min(os.cpu_count() or 1, 32)) != 0:
            raise ValueError("non-ACGT base: the reference's 2-bit packing is undefined for it (SURVEY.md H12)")
        quals = np.ascontiguousarray(quals, dtype=np.uint8)
        wp = (words.ctypes.data + woff[:-1] * 8).astype(np.uint64)
        qp = (quals.ctypes.data + off[:-1].astype(np.uint64)).astype(np.uint64)
        self._check(self._L.hb_upload_reads(self._h, n, wp.ctypes.data, lens.ctypes.data, qp.ctypes.data))
        self.read_len = lens
        self.packed_words, self.packed_word_off = words, woff

    # -- submission ---------------------------------------------------------------------
    @staticmethod
    def make_overlaps(ovl9: np.ndarray, cigars: np.ndarray, cig_off: np.ndarray) -> np.ndarray:
        """hb_overlap[] whose cigar pointers reference `cigars` (must stay alive until submit returns)."""
        ovl9 = np.asarray(ovl9, dtype=np.uint32).reshape(-1, 9)
        n = ovl9.shape[0]
        o = np.zeros(n, dtype=OVERLAP_DTYPE)
        for k, name in enumerate(OVERLAP_DTYPE.names[:9]):
            o[name] = ovl9[:, k]
        cig_off = np.asarray(cig_off, dtype=np.uint64)
        o["cigar"] = cigars.ctypes.data + cig_off[:-1]
        o["cigar_len"] = (cig_off[1:] - cig_off[:-1]).astype(np.uint32)
        return o

    def submit_alignments(self, rid: int, overlaps: np.ndarray):
        """`(tid, Vec<Alignment>)` as alignment_reader sends it (src/overlaps.rs:371-373)."""
        self._check(self._L.hb_submit_alignments(self._h, rid, overlaps.ctypes.data, len(overlaps)))

    def submit_target(self, rid: int, n_windows: int, overlaps: np.ndarray, windows: np.ndarray):
        """Target with host-computed OverlapWindows (the Rust host keeps extract_windows)."""
        windows = np.ascontiguousarray(windows, dtype=OVERLAP_WINDOW_DTYPE)
        self._check(self._L.hb_submit_target(self._h, rid, n_windows, overlaps.ctypes.data, len(overlaps),
                                             windows.ctypes.data, len(windows)))

    def flush(self):
        self._check(self._L.hb_flush(self._h))

    def set_launch_targets(self, n: int):
        self._check(self._L.hb_set_launch_targets(self._h, n))

    def set_kernel_timing(self, on: bool):
        self._check(self._L.hb_set_kernel_timing(self._h, 1 if on else 0))

    def bind_calling_thread(self) -> bool:
        return self._check(self._L.hb_bind_calling_thread(self._h)) == 1

    def poll(self):
        """-> Corrected or None; raises HerroError (with .rid) for a target that failed (e.g. one the reference would
        have panicked on); the other targets are unaffected and polling can continue."""
        rid = C.c_uint32()
        seqs, seg_len = C.c_void_p(), C.c_void_p()
        n = C.c_uint32()
        rc = self._L.hb_poll_corrected(self._h, C.byref(rid), C.byref(seqs), C.byref(seg_len), C.byref(n))
        if rc == 0:
            return None
        try:
            if rc < 0:
                e = HerroError(rc, self._L.hb_last_error(self._h).decode())
                e.rid = rid.value
                raise e
            lens = np.ctypeslib.as_array(C.cast(seg_len, C.POINTER(C.c_uint32)), (max(n.value, 1),))[:n.value].copy()
            segs, o = [], 0
            for l in lens:
                segs.append(C.string_at(seqs.value + o, int(l)))
                o += int(l)
            return Corrected(rid.value, segs)
        finally:
            if seqs.value:
                self._L.hb_release_result(self._h, seqs)

    def drain(self, skip_failed: bool = False):
        """All queued results.  skip_failed: a failed target is recorded in `self.failed` as (rid, code, message) and the
        drain goes on (one bad read must not truncate the output of a whole run)."""
        out = []
        while True:
            try:
                r = self.poll()
            except HerroError as e:
                if not skip_failed:
                    raise
                self.failed.append((getattr(e, "rid", None), e.code, str(e)))
                continue
            if r is None:
                return out
            out.append(r)

    # -- counters / taps ----------------------------------------------------------------
    def stats(self) -> dict:
        s = HbStats()
        self._check(self._L.hb_get_stats(self._h, C.byref(s)))
        d = {n: getattr(s, n) for n, _ in HbStats._fields_ if n not in ("ms_kernel", "n_kernel", "ms_worker_phase", "class_flops")}
        d["class_flops"] = {k: int(s.class_flops[i]) for i, k in enumerate(KERNEL_CLASSES)}
        d["ms_worker_phase"] = [float(x) for x in s.ms_worker_phase]
        d["ms_kernel"] = {k: s.ms_kernel[i] for i, k in enumerate(KERNEL_CLASSES)}
        d["n_kernel"] = {k: int(s.n_kernel[i]) for i, k in enumerate(KERNEL_CLASSES)}
        return d

    def reset_stats(self):
        self._check(self._L.hb_reset_stats(self._h))

    def debug_window(self, rid: int, wid: int) -> dict:
        sh = (C.c_uint32 * 4)()
        self._check(self._L.hb_debug_window_shape(self._h, rid, wid, sh))
        L, n_alns, ns = int(sh[0]), int(sh[1]), int(sh[2])
        bases = np.zeros((L, 31), np.uint8)
        quals = np.zeros((L, 31), np.uint8)
        sup = np.zeros((max(ns, 1), 2), np.uint32)
        rows = np.zeros(max(ns, 1), np.uint32)
        info = np.zeros(max(ns, 1), np.float32)
        bl = np.zeros((max(ns, 1), 5), np.float32)
        self._check(self._L.hb_debug_dump_window(self._h, rid, wid, bases.ctypes.data, quals.ctypes.data,
                                                 sup.ctypes.data, rows.ctypes.data, info.ctypes.data, bl.ctypes.data))
        return dict(L=L, n_alns=n_alns, bases=bases, quals=quals, supported=sup[:ns], sup_rows=rows[:ns],
                    info_logits=info[:ns], bases_logits=bl[:ns])

    def dump_features(self, rid: int, out_dir: str, read_names: list):
        """`herro features` files of target `rid` (of the most recent launch; keep_debug) under out_dir/<read id>/."""
        if getattr(self, "_names_src", None) is not read_names:
            self._names_src = read_names
            self._names_buf = [n if isinstance(n, bytes) else str(n).encode() for n in read_names]
            self._names_arr = (C.c_char_p * len(read_names))(*self._names_buf)
        self._check(self._L.hb_dump_features(self._h, rid, out_dir.encode(), self._names_arr))

    def replay_last_launch(self, iters: int = 1) -> float:
        ms = C.c_float()
        self._check(self._L.hb_replay_last_launch(self._h, iters, C.byref(ms)))
        return float(ms.value)


# ------------------------------------------------------------------------------------------
# C++ host harness (herro_b200/host/harness.cpp): the Rust binary's thread topology over the C ABI
# ------------------------------------------------------------------------------------------
_host = None
# hbh_result_fn: (user, rid, seqs, seg_len, n_segs), called on the harness's consumer thread
_RESULT_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.c_uint32)


def _host_lib():
    global _host
    if _host is None:
        load_library()
        H = C.CDLL(HOST_LIB_PATH)
        vp, u32 = C.c_void_p, C.c_uint32
        H.hbh_pack_2bit.argtypes = [vp, vp, u32, vp, vp, C.c_int]
        H.hbh_windowing.argtypes = [vp, vp, vp, u32, u32, u32, C.c_int, vp, vp, C.c_uint64]
        H.hbh_run.argtypes = [vp, vp, vp, vp, u32, u32, u32, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]
        _host = H
    return _host


class HostHarness:
    """Feature threads + consumer thread over one Context, like src/lib.rs:154-200 for one device."""

    def __init__(self, ctx: "Context", ovl9: np.ndarray, cigars: np.ndarray, cig_off: np.ndarray, aln_off: np.ndarray,
                 read_len: np.ndarray):
        self.ctx = ctx
        self.cigars = cigars  # keep alive: hb_overlap.cigar points into it
        self.ovl = Context.make_overlaps(ovl9, cigars, cig_off)
        self.aln_off = np.ascontiguousarray(aln_off, dtype=np.uint64)
        self.read_len = np.ascontiguousarray(read_len, dtype=np.uint32)

    def windowing(self, t_begin: int, t_end: int, threads: int):
        H = _host_lib()
        off = np.zeros(t_end - t_begin + 1, dtype=np.uint64)
        rc = H.hbh_windowing(self.ovl.ctypes.data, self.aln_off.ctypes.data, self.read_len.ctypes.data, self.ctx.window_size,
                             t_begin, t_end, threads, off.ctypes.data, None, 0)
        if rc != 0:
            raise HerroError(rc, "windowing failed")
        ow = np.zeros(max(int(off[-1]), 1), dtype=OVERLAP_WINDOW_DTYPE)
        rc = H.hbh_windowing(self.ovl.ctypes.data, self.aln_off.ctypes.data, self.read_len.ctypes.data, self.ctx.window_size,
                             t_begin, t_end, threads, off.ctypes.data, ow.ctypes.data, len(ow))
        if rc != 0:
            raise HerroError(rc, "windowing failed")
        return ow, off

    def run(self, t_begin: int, t_end: int, threads: int, windows=None, collect: bool = False) -> dict:
        """collect: also return the corrected records the consumer polled, as `results` (list of Corrected)."""
        H = _host_lib()
        out3 = np.zeros(4, dtype=np.uint64)
        chk = C.c_uint64()
        sec = C.c_double()
        sub = C.c_double()
        ow_p = windows[0].ctypes.data if windows is not None else None
        off_p = windows[1].ctypes.data if windows is not None else None
        results = []

        def keep(_user, rid, seqs, seg_len, n):
            lens = [int(seg_len[k]) for k in range(n)]
            data = C.string_at(seqs, sum(lens)) if n else b""
            offs = np.cumsum([0] + lens)
            results.append(Corrected(int(rid), [data[offs[k]:offs[k + 1]] for k in range(n)]))

        cb = _RESULT_FN(keep) if collect else None  # alive until hbh_run returns
        rc = H.hbh_run(self.ctx._h, self.ovl.ctypes.data, self.aln_off.ctypes.data, self.read_len.ctypes.data,
                       self.ctx.window_size, t_begin, t_end, threads, ow_p, off_p, out3.ctypes.data, C.byref(chk), C.byref(sec), C.byref(sub),
                       C.cast(cb, C.c_void_p) if cb is not None else None, None)
        if rc != 0:
            raise HerroError(rc, self.ctx._L.hb_last_error(self.ctx._h).decode())
        r = dict(bases=int(out3[0]), records=int(out3[1]), targets=int(out3[2]), failed=int(out3[3]), checksum=int(chk.value),
                 seconds=sec.value, submit_seconds_sum=sub.value)
        if collect:
            r["results"] = results
        return r


# ------------------------------------------------------------------------------------------
# FASTA record format of correction_writer / write_sequence (src/lib.rs:267-317)
# ------------------------------------------------------------------------------------------
def fasta_records(read_id: bytes, description, segments: list) -> bytes:
    out = bytearray()
    for i, seg in enumerate(segments):
        out += b">" + read_id
        out += b" " if len(segments) == 1 else b":%d " % i
        if description is not None:
            out += description
        out += b"\n" + seg + b"\n"
    return bytes(out)
