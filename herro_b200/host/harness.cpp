// harness.cpp — C++ host harness that stands in for the Rust binary's thread topology
// (src/lib.rs:139-205) on top of the public C ABI only (include/herro_b200.h):
//
//   `threads` feature threads pull target ids from a shared counter (the MPMC alignment channel,
//   src/lib.rs:136,159-187) and call hb_submit_target / hb_submit_alignments;
//   one consumer thread polls hb_poll_corrected like consensus_worker -> correction_writer
//   (src/lib.rs:198-199,267-291) and, when the producers are done, hb_flush()es.
//
// There is no Rust toolchain in the build image; tests and bench.py drive this through ctypes.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/herro_b200.h"

extern "C" {

// 2-bit packing of the read store, HAECSeq layout (src/haec_io.rs:121-136: 32 bases per u64, A0 C1 G2 T3, base i of a word at
// bits [2i, 2i+2)); `threads` workers over reads.  words must hold woff[n] entries (woff[i] = sum of ceil(len/32) before read i).
// Returns 0, or -1 if a base is not one of ACGTacgt (the reference's packing is undefined for it, SURVEY.md H12).
int hbh_pack_2bit(const uint8_t* seqs, const uint64_t* off, uint32_t n_reads, uint64_t* words, const uint64_t* woff, int threads) {
    static const auto lut = [] {
        std::vector<uint8_t> t(256, 255);
        t['A'] = t['a'] = 0; t['C'] = t['c'] = 1; t['G'] = t['g'] = 2; t['T'] = t['t'] = 3;
        return t;
    }();
    std::atomic<uint32_t> next{0};
    std::atomic<int> bad{0};
    auto work = [&]() {
        for (;;) {
            const uint32_t i0 = next.fetch_add(64);
            if (i0 >= n_reads) break;
            for (uint32_t i = i0; i < std::min(n_reads, i0 + 64); i++) {
                const uint8_t* s = seqs + off[i];
                const uint64_t len = off[i + 1] - off[i];
                uint64_t* w = words + woff[i];
                for (uint64_t b = 0; b < len; b += 32) {
                    const uint64_t m = std::min<uint64_t>(32, len - b);
                    uint64_t v = 0;
                    uint8_t any = 0;
                    for (uint64_t k = 0; k < m; k++) { const uint8_t c = lut[s[b + k]]; any |= c; v |= (uint64_t)(c & 3) << (2 * k); }
                    if (any > 3) bad = 1;
                    w[b >> 5] = v;
                }
            }
        }
    };
    std::vector<std::thread> th;
    for (int i = 0; i < (threads > 0 ? threads : 1); i++) th.emplace_back(work);
    for (auto& t : th) t.join();
    return bad.load() ? -1 : 0;
}

// Parallel host windowing (what the Rust feature threads do before submitting): fills ow_off[n_t+1]
// and, if ow_out != NULL (cap records), the windows of targets [t_begin, t_end) back to back.
// Call once with ow_out == NULL to size, then again to fill.  Returns 0 or an hb_status.
int hbh_windowing(const hb_overlap* ovl_all, const uint64_t* aln_off, const uint32_t* read_len, uint32_t window,
                  uint32_t t_begin, uint32_t t_end, int threads, uint64_t* ow_off, hb_overlap_window* ow_out, uint64_t cap) {
    const uint32_t nt = t_end - t_begin;
    std::vector<std::vector<hb_overlap_window>> per(nt);
    std::atomic<uint32_t> next{0};
    std::atomic<int> rc{0};
    auto work = [&]() {
        for (;;) {
            const uint32_t k = next.fetch_add(1);
            if (k >= nt) break;
            const uint32_t t = t_begin + k;
            const uint32_t n_ovl = (uint32_t)(aln_off[t + 1] - aln_off[t]);
            const uint32_t nw = (read_len[t] + window - 1) / window;
            std::vector<hb_overlap_window>& v = per[k];
            v.resize((size_t)n_ovl * (nw + 1) + 1);
            uint32_t n = 0;
            const int r = hb_extract_windows(ovl_all + aln_off[t], n_ovl, window, nw, v.data(), (uint32_t)v.size(), &n);
            if (r != 0) { rc = r; n = 0; }
            v.resize(n);
        }
    };
    std::vector<std::thread> th;
    for (int i = 0; i < (threads > 0 ? threads : 1); i++) th.emplace_back(work);
    for (auto& t : th) t.join();
    ow_off[0] = 0;
    for (uint32_t k = 0; k < nt; k++) ow_off[k + 1] = ow_off[k] + per[k].size();
    if (ow_out) {
        if (ow_off[nt] > cap) return HB_ERR_CAPACITY;
        for (uint32_t k = 0; k < nt; k++)
            if (!per[k].empty()) memcpy(ow_out + ow_off[k], per[k].data(), per[k].size() * sizeof(hb_overlap_window));
    }
    return rc;
}

// Run targets [t_begin, t_end).  ow_all/ow_off: precomputed windows (hbh_windowing) or NULL to let the
// library window the alignments (hb_submit_alignments).  out4 = {corrected bases, records (segments),
// targets that produced output, targets that failed (skipped, the run goes on)}; checksum = order-independent
// hash of (rid, segment bytes).  Every thread binds itself to the NUMA node of the context's GPU.
// on_result (may be NULL) sees every corrected record as hb_poll_corrected returned it, on the consumer thread,
// before it is released.
typedef void (*hbh_result_fn)(void* user, uint32_t rid, const uint8_t* seqs, const uint32_t* seg_len, uint32_t n_segs);
int hbh_run(hb_ctx* ctx, const hb_overlap* ovl_all, const uint64_t* aln_off, const uint32_t* read_len, uint32_t window,
            uint32_t t_begin, uint32_t t_end, int threads, const hb_overlap_window* ow_all, const uint64_t* ow_off,
            uint64_t* out3, uint64_t* checksum, double* seconds, double* submit_seconds_sum, hbh_result_fn on_result,
            void* user) {
    if (!ctx || !ovl_all || !aln_off || !read_len || !out3 || !seconds) return HB_ERR_ARG;
    std::atomic<uint32_t> next{t_begin};
    std::atomic<int> rc{0};
    std::atomic<int> producers_left{threads > 0 ? threads : 1};
    const auto t0 = std::chrono::steady_clock::now();
    std::atomic<uint64_t> submit_ns{0};
    std::atomic<uint64_t> failed{0};
    auto feature_thread = [&]() {
        hb_bind_calling_thread(ctx);
        uint64_t my_ns = 0;
        for (;;) {
            const uint32_t t = next.fetch_add(1);
            if (t >= t_end || rc.load() != 0) break;
            const uint32_t n_ovl = (uint32_t)(aln_off[t + 1] - aln_off[t]);
            if (n_ovl == 0) continue;  // reads that never appear as a target (src/overlaps.rs:189-192)
            int r;
            const auto s0 = std::chrono::steady_clock::now();
            if (ow_all) {
                const uint32_t k = t - t_begin;
                r = hb_submit_target(ctx, t, (read_len[t] + window - 1) / window, ovl_all + aln_off[t], n_ovl, ow_all + ow_off[k],
                                     (uint32_t)(ow_off[k + 1] - ow_off[k]));
            } else {
                r = hb_submit_alignments(ctx, t, ovl_all + aln_off[t], n_ovl);
            }
            my_ns += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - s0).count();
            if (r != 0) rc = r;
        }
        submit_ns.fetch_add(my_ns);
        producers_left.fetch_sub(1);
    };
    uint64_t bases = 0, records = 0, targets = 0, sum = 0;
    auto consumer = [&]() {
        hb_bind_calling_thread(ctx);
        bool flushed = false;
        for (;;) {
            uint32_t rid = 0, n = 0;
            uint8_t* seqs = nullptr;
            uint32_t* lens = nullptr;
            const int r = hb_poll_corrected(ctx, &rid, &seqs, &lens, &n);
            if (r == 1) {
                uint64_t h = 1469598103934665603ull ^ rid;
                size_t off = 0;
                for (uint32_t k = 0; k < n; k++) {
                    bases += lens[k];
                    for (uint32_t i = 0; i < lens[k]; i++) h = (h ^ seqs[off + i]) * 1099511628211ull;
                    h = (h ^ 0xff) * 1099511628211ull;
                    off += lens[k];
                }
                records += n;
                targets += n ? 1 : 0;
                sum += h;
                if (on_result) on_result(user, rid, seqs, lens, n);
                hb_release_result(ctx, seqs);
            } else if (r == 0) {
                if (producers_left.load() == 0) {
                    if (flushed) break;
                    const int f = hb_flush(ctx);
                    if (f != 0 && f != HB_ERR_INPUT && f != HB_ERR_CAPACITY) rc = f;
                    flushed = true;
                } else {
                    std::this_thread::sleep_for(std::chrono::microseconds(100));
                }
            } else if (r == HB_ERR_INPUT || r == HB_ERR_CAPACITY) {
                failed.fetch_add(1);  // this target only: log-and-continue (hb_last_error names it)
            } else {
                rc = r;
                if (flushed) break;
            }
        }
    };
    std::vector<std::thread> th;
    for (int i = 0; i < (threads > 0 ? threads : 1); i++) th.emplace_back(feature_thread);
    std::thread cons(consumer);
    for (auto& t : th) t.join();
    cons.join();
    *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    out3[0] = bases; out3[1] = records; out3[2] = targets; out3[3] = failed.load();
    if (checksum) *checksum = sum;
    if (submit_seconds_sum) *submit_seconds_sum = (double)submit_ns.load() * 1e-9;
    return rc;
}

}  // extern "C"
