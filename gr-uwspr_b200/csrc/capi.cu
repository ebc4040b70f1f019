// C ABI of libuwspr_b200.so (include/uwspr_b200.h): context, constant tables, chunked
// submission with copy/compute overlap.  No CPU fallback exists for the ported stages:
// without a usable CUDA device uwspr_b200_create fails.
#include <limits.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <future>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "../host/wspr_tables.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

namespace {

const int kMaxChunks = 1024;
const int kCounterSets = 15;   // counter set q at 4 + 4q
const int kCounterInts = 4 + 4 * kCounterSets;   // [0] running total, [1] overflow, then the sets

// One submission unit: windows [w0, w0 + nw) of the call.  `set` selects the buffer set and the
// compute stream; `slot` is the chunk's first window slot inside that set, `xoff` its first
// staged sample (host input), `cset` its private {coarse ticket, fine ticket, end} counters,
// `group` the index of the full-size chunk it was cut from, `strm` its compute stream (the pieces
// of a cut chunk go to different streams so that they can overlap).
struct UwChunk {
    int w0, nw, set, slot, cset, group, strm;
    size_t xoff;
};

// Test / diagnosis knobs, read from the environment once, when the context is created
// (DESIGN.md section 3 lists them).
struct Knobs {
    int tail_groups = 2;        // UWSPR_B200_TAIL_GROUPS: chunk groups at the end of a host-fed call that are cut up
    int tail_piece = 0;         // UWSPR_B200_TAIL_PIECE: windows per piece (0: a quarter chunk)
    bool trace = false;         // UWSPR_B200_TRACE
    bool no_fine_reuse = false; // UWSPR_B200_NO_FINE_REUSE: stage E evaluates jiggle 0 again instead of taking it from the chain
    bool no_lag_share = false;  // UWSPR_B200_NO_LAG_SHARE: the lag searches (stages A, D) rotate one table set per point (R1)
};

Knobs read_knobs()
{
    Knobs k;
    auto geti = [](const char *name, int def) {
        const char *e = getenv(name);
        return e ? atoi(e) : def;
    };
    k.tail_groups = std::max(0, std::min(2, geti("UWSPR_B200_TAIL_GROUPS", k.tail_groups)));
    k.tail_piece = std::max(0, geti("UWSPR_B200_TAIL_PIECE", 0));
    k.trace = getenv("UWSPR_B200_TRACE") != nullptr;
    k.no_fine_reuse = getenv("UWSPR_B200_NO_FINE_REUSE") != nullptr;
    k.no_lag_share = getenv("UWSPR_B200_NO_LAG_SHARE") != nullptr;
    return k;
}

struct Buffers {
    // per chunk
    float2 *x_stage[3] = { nullptr, nullptr, nullptr };  // host-fed samples, three buffer sets
    size_t x_stage_elems = 0;
    float *amp = nullptr;
    float *ps_dbg = nullptr;
    float *psavg = nullptr;
    UwPeak *peaks = nullptr;
    // per call
    int *npk = nullptr;
    int *base = nullptr;
    size_t win_cap = 0;
    UwItem *items = nullptr;
    uwspr_b200_candidate_t *cands = nullptr;
    uwspr_b200_refined_t *refined = nullptr;
    uwspr_b200_jiggle_t *jig = nullptr;
    uint8_t *soft = nullptr;
    UwFineWork fine[3] = {};  // fine path workspaces, one per compute stream
    int *counters = nullptr;  // [0] running total, [1] overflow; set s at 4+4s: ticket coarse, ticket fine, end of chunk
    // tables
    float *window = nullptr;
    float2 *twiddle = nullptr;
    uint32_t *off4 = nullptr;
    short *hyp_unique = nullptr;
    // device decoder (uwspr_b200_decode_device), allocated by its first call for max_candidates
    int *dec_first_ok = nullptr;            // [cap]: smallest jiggle that decoded so far
    int *dec_tasks = nullptr;               // [cap * NJIG]: gated (candidate, jiggle) pairs
    uint32_t *dec_task_cycles = nullptr;    // [cap * NJIG]
    unsigned long long *dec_task_msg = nullptr;  // [cap * NJIG]: bytes 0..6 of a successful task's data
    int *dec_counters = nullptr;            // task count, task cursor
    uint8_t *dec_out = nullptr;             // decoded[cap], msg7[cap * 7], idt_used[cap], fano_cycles[cap]
    short *mettab = nullptr;                // WSPR_METTAB
    // raw decoder rows (uwspr_b200_fano_batch): symbols and outputs, grown on demand
    uint8_t *rows = nullptr;
    size_t rows_cap = 0;
};

}  // namespace

struct uwspr_b200_ctx {
    uwspr_b200_params_t prm;
    UwDims d;
    Buffers b;
    int device = 0, sm_count = 0;
    int chunk_windows = 0, max_windows = 0, max_candidates = 0;
    int grid_coarse = 0;
    UwFineLaunch fine_launch = {};
    cudaStream_t compute = nullptr, compute2 = nullptr, compute3 = nullptr, copy = nullptr, d2h = nullptr;
    int *h_ends = nullptr;  // pinned: end of every chunk's items (host-fed calls stream results back per chunk)
    bool own_compute = true;
    cudaEvent_t ev_h2d[3] = { nullptr, nullptr, nullptr }, ev_free[3] = { nullptr, nullptr, nullptr }, ev_wl[3] = { nullptr, nullptr, nullptr };
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join3 = nullptr;
    int last_cw = 0;
    std::vector<UwChunk> last_chunks;  // schedule of the last call
    Knobs knobs;
    int last_sets = 1;   // buffer sets the last call rotated through
    std::vector<cudaEvent_t> ev;  // 5 per chunk: start, after spec, after coarse, after fine
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    cudaEvent_t ev_cp0 = nullptr, ev_cp1 = nullptr, ev_kend = nullptr;  // UWSPR_B200_TRACE
    float ms[4] = { 0, 0, 0, 0 };
    int64_t launches = 0;
    std::string err;
    bool debug_ps = false;
    bool have_coarse = false;  // device candidate list valid for a following fine call
    bool have_fine = false;    // b.refined / b.jig / b.soft hold last_total candidates x last_jig_count jiggles
    int last_jig_count = 0;
    int fano_grid = 0;         // resident blocks of the decoder kernel
    int last_nwin = 0, last_total = 0;
    const float *last_samples = nullptr;
    int64_t last_stride = 0;
    std::future<int> pending;   // uwspr_b200_coarse_fine_submit: the submission running on its own thread
};

namespace {

int fail(uwspr_b200_ctx *c, int status, const std::string &msg)
{
    if (c) c->err = msg;
    return status;
}

#define CU(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess)                                                           \
            return fail(ctx, UWSPR_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// lib/slm.cc:36-73 restated for the host-side table build (double inside, fp32 result)
float slm_frequency_drift_host(double V1, double V2, int p1, int p2, float cf, float t)
{
    const double q1 = V1 * t + p1, q2 = V2 * t + p2;
    const float sign = (float)(((q1 * V1 + q2 * V2) > 0) * 2 - 1);
    const double num = fabs(V1 * q1 + V2 * q2);
    const double den = sqrt(q1 * q1 + q2 * q2);
    if (den == 0) return 0.0f;
    return (float)(-sign * num / den * cf / 1500.0f);
}

// Builds every table that depends only on the constructor arguments.
int build_tables(uwspr_b200_ctx *ctx, std::vector<uint32_t> &off4, std::vector<short> &hyp_unique)
{
    UwDims &d = ctx->d;
    const uwspr_b200_params_t &p = ctx->prm;
    d.fl = p.fl;
    d.size = 2 * p.spb;                                           // FDR_impl.cc:81
    d.df = (float)p.fs / (float)d.size;                           // :93
    d.m = d.size / 2;                                             // :95
    d.hpbm = (int)ceilf((float)(int)(float)p.halfbandwidth / d.df);  // :97
    d.finpb = 2 * d.hpbm;                                         // :265
    d.noiseidx = (int)floor(0.3 * (float)d.finpb);                // :283
    d.n_rows = (int)(floor(((float)p.fl / (float)p.spb) * 2.0) - 3);  // :109
    d.min_snr = (float)pow(10.0, -7.0 / 10.0);                    // :137
    d.floor_val = (float)(0.1 * d.min_snr);                       // :290
    d.threshold = (float)p.threshold;                             // :79
    d.maxfreqs = p.maxfreqs;
    d.maxdrift = p.maxdrift;
    d.cf = p.cf;
    d.nonlinear_intended_t = p.nonlinear_intended_t ? 1 : 0;
    for (int q = 0; q < 6; q++) d.sync_words[q] = WSPR_SYNC_WORDS[q];
    if (d.finpb < 3) return fail(ctx, UWSPR_B200_E_PARAM, "halfbandwidth too small: fewer than 3 pass-band bins");
    d.maxcand = std::min(p.maxfreqs, (d.finpb - 1) / 2);
    if (d.maxcand > 256) return fail(ctx, UWSPR_B200_E_PARAM, "more than 256 candidate slots per window");
    d.n_lin = 2 * p.maxdrift + 1;
    d.n_hyp = d.n_lin + UW_NTRAJ;

    // bins the coarse search can centre on: if0 in [m-hpbm+1, m+hpbm-2], ifr = if0-2..if0+2
    const int ifr_lo = d.m - d.hpbm - 1, ifr_hi = d.m + d.hpbm;
    if (ifr_lo < 0) return fail(ctx, UWSPR_B200_E_PARAM, "halfbandwidth reaches past the spectrum (reference reads out of bounds)");
    std::vector<std::vector<signed char>> seqs;
    hyp_unique.assign(d.n_hyp, 0);
    int off_min = 0, off_max = 0;
    for (int h = 0; h < d.n_hyp; h++) {
        std::vector<signed char> seq(UW_NSYM);
        for (int k = 0; k < UW_NSYM; k++) {
            int off_ref = 0;
            for (int ifr = ifr_lo; ifr <= ifr_hi; ifr++) {
                int ifd;
                if (h < d.n_lin) {
                    const int drift = h - p.maxdrift;
                    // FDR_impl.cc:353 (double expression, truncated)
                    ifd = (int)(ifr + ((float)k - 81.0) / 81.0 * ((float)drift) / (2.0 * d.df));
                } else {
                    const int t_idx = h - d.n_lin;  // slm.cc:76-116 order: p2 fastest, V1, V2
                    const double V1 = (double)((t_idx / 5) % 5) - 2.0, V2 = (double)(t_idx / 25) - 2.0;
                    const int p2 = (t_idx % 5) * 200 + 50;
                    const float t = (float)(k * 111 / 162);                       // :382
                    const float drift = slm_frequency_drift_host(V1, V2, 0, p2, (float)p.cf, t);
                    ifd = (int)(ifr + drift / d.df);                              // :384-385, fp32
                }
                const int off = ifd - ifr;
                if (ifr == ifr_lo)
                    off_ref = off;
                else if (off != off_ref)
                    return fail(ctx, UWSPR_B200_E_PARAM, "bin offsets depend on the bin (parameters outside the supported domain)");
            }
            if (off_ref < -100 || off_ref > 100) return fail(ctx, UWSPR_B200_E_PARAM, "drift hypotheses span too many bins");
            seq[k] = (signed char)off_ref;
            off_min = std::min(off_min, off_ref);
            off_max = std::max(off_max, off_ref);
        }
        int u = -1;
        for (size_t q = 0; q < seqs.size(); q++)
            if (seqs[q] == seq) {
                u = (int)q;
                break;
            }
        if (u < 0) {
            u = (int)seqs.size();
            seqs.push_back(seq);
        }
        hyp_unique[h] = (short)u;
    }
    d.n_unique = (int)seqs.size();
    d.off_min = off_min;
    d.off_max = off_max;
    d.tile_w = 11 + off_max - off_min;
    if (d.tile_w > UW_MAX_TILE_W || d.n_unique > UW_MAX_UNIQUE)
        return fail(ctx, UWSPR_B200_E_PARAM, "drift hypotheses span too many bins / sequences for one tile");
    // kept bins: everything the normalizer (:268-274) and powersum (:199-205) can index
    const int lo = std::min(d.m - d.hpbm - 3, (d.m - d.hpbm + 1) - 5 + off_min);
    const int hi = std::max(d.m + d.hpbm + 2, (d.m + d.hpbm - 2) + 5 + off_max);
    if (lo < 0 || hi > d.size - 1)
        return fail(ctx, UWSPR_B200_E_PARAM, "halfbandwidth too large: the reference would index outside the spectrum");
    d.bin_lo = lo;
    d.n_bins = hi - lo + 1;
    d.nbp = (d.n_bins + 3) & ~3;
    off4.assign((size_t)UW_NQUAD * d.n_unique, 0);
    for (int u = 0; u < d.n_unique; u++)
        for (int k = 0; k < UW_NSYM; k++)
            off4[(size_t)(k / 4) * d.n_unique + u] |= (uint32_t)(seqs[u][k] - off_min) << (8 * (k % 4));
    return UWSPR_B200_OK;
}

int ensure_window_capacity(uwspr_b200_ctx *ctx, int nwin)
{
    Buffers &b = ctx->b;
    if ((size_t)nwin + 1 <= b.win_cap) return UWSPR_B200_OK;
    if (b.npk) cudaFree(b.npk);
    if (b.base) cudaFree(b.base);
    b.npk = nullptr;
    b.base = nullptr;
    b.win_cap = 0;
    const size_t n = (size_t)nwin + 1;
    CU(cudaMalloc(&b.npk, n * sizeof(int)));
    CU(cudaMalloc(&b.base, n * sizeof(int)));
    b.win_cap = n;
    return UWSPR_B200_OK;
}

int ensure_stage(uwspr_b200_ctx *ctx, size_t elems)
{
    Buffers &b = ctx->b;
    if (elems <= b.x_stage_elems) return UWSPR_B200_OK;
    for (int q = 0; q < 3; q++) {
        if (b.x_stage[q]) cudaFree(b.x_stage[q]);
        b.x_stage[q] = nullptr;
    }
    b.x_stage_elems = 0;
    for (int q = 0; q < 3; q++) CU(cudaMalloc(&b.x_stage[q], elems * sizeof(float2)));
    b.x_stage_elems = elems;
    return UWSPR_B200_OK;
}

// The core: runs the requested stages over nwin windows in chunks.
//   do_coarse: spectrogram + normalizer + peaks + coarse search -> device candidate list
//   do_fine:   refinement + soft symbols for the device candidate list
// When !do_coarse the candidate list (npk + cands) is uploaded from the caller first.
int run_impl(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int wins_per_chan,
             int64_t chan_stride, int nwin, bool do_coarse, bool do_fine, const int32_t *npk_in, const uwspr_b200_candidate_t *cands_in, int total_in, int jig_first,
             int jig_count, int32_t *npk_out, uwspr_b200_candidate_t *cands_out, int cap_out, int32_t *total_out,
             uwspr_b200_refined_t *refined_out, uwspr_b200_jiggle_t *jig_out, uint8_t *soft_out)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (nwin < 0 || !samples || win_stride < 0) return fail(ctx, UWSPR_B200_E_PARAM, "bad sample arguments");
    if (nwin > ctx->max_windows) return fail(ctx, UWSPR_B200_E_PARAM, "nwin exceeds max_windows of the context");
    if (do_fine && (jig_first < 0 || jig_count < 0 || jig_first + jig_count > UWSPR_B200_NJIG))
        return fail(ctx, UWSPR_B200_E_PARAM, "jiggle range outside [0,17)");
    CU(cudaSetDevice(ctx->device));
    Buffers &b = ctx->b;
    const UwDims &d = ctx->d;
    cudaStream_t cs = ctx->compute;
    int rc = ensure_window_capacity(ctx, nwin);
    if (rc) return rc;
    for (int q = 0; q < 4; q++) ctx->ms[q] = 0.0f;
    if (nwin == 0) {
        if (total_out) *total_out = 0;
        ctx->last_total = 0;
        ctx->last_nwin = 0;
        ctx->have_fine = do_fine;
        ctx->last_jig_count = jig_count;
        return UWSPR_B200_OK;
    }
    // Device-resident input: one buffer set and one stream, chunks as large as the buffers allow (no tails between
    // chunks).  Host input: chunks rotate through three buffer sets and three compute streams, so that the H2D copies
    // run back to back while earlier chunks are in their kernels.  With two sets the copy of chunk c+2 waited for the
    // kernels of chunk c, which share the GPU with those of chunk c+1 and take longer than a copy when copy and
    // compute are balanced (a 100 000-window overlapped stream: 15.2 ms per 4 096-window chunk against 13.3 ms per
    // copy, trace in profiles/README.md).
    const bool host = space == UWSPR_B200_HOST;
    const Knobs &kn = ctx->knobs;
    const int nsets = host ? 3 : 1;
    // host-fed chunk: small enough that the first kernels start early and little is left after the last byte, large
    // enough that the fine path's launches are well filled (measured on a 100 000-window overlapped stream: 1024 /
    // 2048 / 4096 windows per chunk -> 235 / 248 / 251 k windows/s; a 10 000-window call does not care)
    const int host_chunk = std::min(4096, std::max(1024, nwin / 16));
    // a call that fits the chunk buffers is cut in three, so that every window's intermediate buffers survive the call
    const int set_cap = nwin <= ctx->chunk_windows ? std::max(ctx->chunk_windows / 3, (nwin + 2) / 3) : ctx->chunk_windows / 3;
    const int cw = host ? std::max(1, std::min(host_chunk, set_cap)) : ctx->chunk_windows;
    // Chunk schedule.  With host input the kernels of a chunk cannot start before its last byte
    // has crossed PCIe, so the end of the call is cut into small pieces (a quarter chunk by
    // default, UWSPR_B200_TAIL_PIECE) that use disjoint slices of their group's buffer set and
    // rotate over three streams: when the last byte arrives only one small piece is left to do.
    std::vector<UwChunk> &chunks = ctx->last_chunks;
    chunks.clear();
    {
        const int tail_groups = host ? kn.tail_groups : 0;
        const int piece = kn.tail_piece > 0 ? kn.tail_piece : std::max(1, cw / 4);
        const int ngroups = (nwin + cw - 1) / cw;
        int w = 0, cset = nsets, rr = 0;
        for (int group = 0; w < nwin; group++) {
            int gw = std::min(cw, nwin - w);
            const int set = group % nsets;
            if (!host) {
                // the fine path keeps window offsets from the chunk's first window in 32 bits (uw_window_offset)
                const UwGeom g{ (long long)win_stride, (long long)chan_stride, wins_per_chan, w };
                while (gw > 1 && uw_window_offset(g, gw - 1) - uw_window_offset(g, 0) > INT_MAX) gw = (gw + 1) / 2;
            }
            const bool cut = host && group > 0 && group >= ngroups - tail_groups && gw > piece;
            if (!cut) {
                chunks.push_back(UwChunk{ w, gw, set, 0, set, group, set, 0 });
                w += gw;
                continue;
            }
            int slot = 0;
            size_t xoff = 0;
            while (slot < gw) {
                // a last piece shorter than half a piece is merged into its predecessor
                int pw = std::min(piece, gw - slot);
                if (gw - slot - pw < (piece + 1) / 2) pw = gw - slot;
                const bool spare = cset < kCounterSets;
                chunks.push_back(UwChunk{ w, spare ? pw : gw - slot, set, slot, spare ? cset : set, group, rr % 3, xoff });
                if (!spare) pw = gw - slot;
                else cset++;
                rr++;
                w += pw;
                slot += pw;
                xoff += (size_t)(pw - 1) * (size_t)win_stride + (size_t)d.fl;
            }
        }
    }
    const int nchunks = (int)chunks.size();
    if (nchunks > kMaxChunks) return fail(ctx, UWSPR_B200_E_PARAM, "too many chunks: raise max_windows");
    while ((int)ctx->ev.size() < 4 * nchunks) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        ctx->ev.push_back(e);
    }
    cudaStream_t streams[3] = { cs, host && nchunks > 1 ? ctx->compute2 : cs, ctx->compute3 };
    bool use3 = false;
    for (const UwChunk &q : chunks) use3 = use3 || q.strm == 2;
    CU(cudaEventRecord(ctx->ev_begin, cs));
    CU(cudaMemsetAsync(b.counters, 0, kCounterInts * sizeof(int), cs));
    // caller's list: candidates before window w (the fine slices of a chunk cover exactly its own candidates)
    std::vector<long long> first_in;
    if (!do_coarse) {
        // candidate list comes from the caller (or stays from the previous coarse call)
        if (cands_in) {
            if (!npk_in) return fail(ctx, UWSPR_B200_E_PARAM, "cands given without npk");
            if (total_in < 0) return fail(ctx, UWSPR_B200_E_PARAM, "negative candidate total");
            if (total_in > ctx->max_candidates) return fail(ctx, UWSPR_B200_E_CAPACITY, "more candidates than max_candidates");
            first_in.assign((size_t)nwin + 1, 0);
            for (int w = 0; w < nwin; w++) {
                if (npk_in[w] < 0) return fail(ctx, UWSPR_B200_E_PARAM, "negative candidate count for a window");
                first_in[w + 1] = first_in[w] + npk_in[w];
            }
            if (first_in[nwin] != total_in) return fail(ctx, UWSPR_B200_E_PARAM, "sum of npk differs from total");
            CU(cudaMemcpyAsync(b.npk, npk_in, sizeof(int) * nwin, cudaMemcpyHostToDevice, cs));
            CU(cudaMemcpyAsync(b.cands, cands_in, sizeof(uwspr_b200_candidate_t) * (size_t)total_in,
                               cudaMemcpyHostToDevice, cs));
        } else if (!ctx->have_coarse || ctx->last_nwin != nwin) {
            return fail(ctx, UWSPR_B200_E_STATE, "no candidate list on the device for these windows");
        }
    }
    if (streams[1] != cs) {
        CU(cudaEventRecord(ctx->ev_fork, cs));
        CU(cudaStreamWaitEvent(streams[1], ctx->ev_fork, 0));
        if (use3) CU(cudaStreamWaitEvent(streams[2], ctx->ev_fork, 0));
    }
    const size_t span_max = (size_t)(cw - 1) * (size_t)win_stride + (size_t)d.fl;
    if (host) {
        rc = ensure_stage(ctx, span_max + (size_t)kCounterSets * (size_t)d.fl);  // pieces of a cut chunk are staged back to back
        if (rc) return rc;
    }
    // Host-fed calls return results chunk by chunk while later chunks are still copying in and
    // computing (PCIe is full duplex); only the last chunk's results are left for the end.
    const bool want_results = (cands_out && do_coarse) || (do_fine && (refined_out || jig_out || soft_out));
    const bool early = host && nchunks > 1 && want_results;
    for (int c = 0; c < nchunks; c++) {
        const UwChunk &ch = chunks[c];
        const int w0 = ch.w0, nw = ch.nw, s = ch.set;
        const bool first_of_group = c == 0 || chunks[c - 1].group != ch.group;
        cudaStream_t st = streams[ch.strm];
        // window w of the chunk is window ch.w0 + w of the call: staged host input holds only the chunk's windows
        // (one channel), device input is addressed from the call's first sample
        const float2 *xdev;
        UwGeom geom{ (long long)win_stride, (long long)chan_stride, wins_per_chan, w0 };
        if (host) {
            // copy stream: wait until the kernels of the chunk two groups back released this buffer
            // set, then copy
            if (first_of_group && ch.group >= nsets) CU(cudaStreamWaitEvent(ctx->copy, ctx->ev_free[s], 0));
            if (ctx->knobs.trace && c == 0) CU(cudaEventRecord(ctx->ev_cp0, ctx->copy));
            const size_t span = (size_t)(nw - 1) * (size_t)win_stride + (size_t)d.fl;
            CU(cudaMemcpyAsync(b.x_stage[s] + ch.xoff, samples + 2 * (size_t)w0 * (size_t)win_stride, span * sizeof(float2),
                               cudaMemcpyHostToDevice, ctx->copy));
            CU(cudaEventRecord(ctx->ev_h2d[s], ctx->copy));
            if (ctx->knobs.trace && c == nchunks - 1) CU(cudaEventRecord(ctx->ev_cp1, ctx->copy));
            CU(cudaStreamWaitEvent(st, ctx->ev_h2d[s], 0));
            xdev = b.x_stage[s] + ch.xoff;
            geom = UwGeom{ (long long)win_stride, 0, nw, 0 };
        } else {
            xdev = reinterpret_cast<const float2 *>(samples);
        }
        // the fine path addresses its windows from the chunk's first one (32-bit offsets)
        const float2 *xfine = xdev + uw_window_offset(geom, 0);
        // per-set slices of the chunk buffers
        const size_t so = (size_t)s * cw + (size_t)ch.slot;
        float *amp = b.amp + so * d.n_rows * d.nbp;
        float *psd = (ctx->debug_ps && b.ps_dbg) ? b.ps_dbg + so * d.n_rows * d.nbp : nullptr;
        float *psavg = b.psavg + so * d.nbp;
        UwPeak *peaks = b.peaks + so * d.maxcand;
        int *set = b.counters + 4 + 4 * ch.cset;
        cudaEvent_t *e = &ctx->ev[4 * c];
        CU(cudaEventRecord(e[0], st));
        if (do_coarse) {
            uw_launch_spectrogram(d, xdev, geom, nw, b.window, b.twiddle, amp, psd, psavg, peaks,
                                  b.npk + w0, st);
            ctx->launches++;
        }
        CU(cudaEventRecord(e[1], st));
        // the running total makes the work lists of consecutive chunks sequential
        if (c >= 1 && chunks[c - 1].strm != ch.strm) CU(cudaStreamWaitEvent(st, ctx->ev_wl[chunks[c - 1].strm], 0));
        uw_launch_worklist(b.npk + w0, nw, ctx->max_candidates, b.base + w0, b.items, b.counters, set, st);
        ctx->launches++;
        if (streams[1] != cs) CU(cudaEventRecord(ctx->ev_wl[ch.strm], st));
        if (early) CU(cudaMemcpyAsync(&ctx->h_ends[c], set + 2, sizeof(int), cudaMemcpyDeviceToHost, st));
        if (do_coarse) {
            uw_launch_coarse(d, amp, peaks, b.items, set + 2, ctx->max_candidates, b.off4, b.hyp_unique, b.cands, set,
                             ctx->grid_coarse, st);
            ctx->launches++;
        }
        CU(cudaEventRecord(e[2], st));
        if (do_fine) {
            // the stage sequence runs over slices of at most the workspace's slice of candidates.  A list from the
            // coarse search has at most maxcand candidates per window, but its length is a device value, so the
            // launches cover the most the chunk can hold; the caller's list may give a window any number of
            // candidates (the reference takes them all), and its chunk counts are known here
            const long long held = first_in.empty() ? (long long)nw * d.maxcand : first_in[w0 + nw] - first_in[w0];
            const long long most = std::min<long long>(ctx->max_candidates, held);
            const UwFineWork &fw = b.fine[ch.strm];
            for (long long s0 = 0; s0 < most; s0 += fw.slice)
                ctx->launches += uw_launch_fine(d, xfine, geom, b.items, set + 1, set + 2, ctx->max_candidates, b.cands,
                                                jig_first, jig_count, b.refined, b.jig, b.soft, (int)s0, fw,
                                                ctx->fine_launch, st);
        }
        CU(cudaEventRecord(e[3], st));
        if (host) CU(cudaEventRecord(ctx->ev_free[s], st));
    }
    if (streams[1] != cs) {
        CU(cudaEventRecord(ctx->ev_join, streams[1]));
        CU(cudaStreamWaitEvent(cs, ctx->ev_join, 0));
        if (use3) {
            CU(cudaEventRecord(ctx->ev_join3, streams[2]));
            CU(cudaStreamWaitEvent(cs, ctx->ev_join3, 0));
        }
    }
    ctx->last_cw = cw;
    ctx->last_sets = nsets;
    if (ctx->knobs.trace) CU(cudaEventRecord(ctx->ev_kend, cs));
    int done = 0;  // results [0, done) are already on their way to the caller
    auto fetch = [&](int lo, int hi, cudaStream_t q) -> cudaError_t {
        cudaError_t e = cudaSuccess;
        const size_t n = (size_t)(hi - lo);
        if (hi <= lo) return e;
        if (cands_out && do_coarse && e == cudaSuccess)
            e = cudaMemcpyAsync(cands_out + lo, b.cands + lo, sizeof(uwspr_b200_candidate_t) * n, cudaMemcpyDeviceToHost, q);
        if (do_fine && refined_out && e == cudaSuccess)
            e = cudaMemcpyAsync(refined_out + lo, b.refined + lo, sizeof(uwspr_b200_refined_t) * n, cudaMemcpyDeviceToHost, q);
        if (do_fine && jig_out && e == cudaSuccess)
            e = cudaMemcpyAsync(jig_out + (size_t)lo * jig_count, b.jig + (size_t)lo * jig_count,
                                sizeof(uwspr_b200_jiggle_t) * n * jig_count, cudaMemcpyDeviceToHost, q);
        if (do_fine && soft_out && e == cudaSuccess)
            e = cudaMemcpyAsync(soft_out + (size_t)lo * jig_count * UW_NSYM, b.soft + (size_t)lo * jig_count * UW_NSYM,
                                n * jig_count * UW_NSYM, cudaMemcpyDeviceToHost, q);
        return e;
    };
    if (early) {
        for (int c = 0; c + 1 < nchunks; c++) {
            CU(cudaEventSynchronize(ctx->ev[4 * c + 3]));   // chunk c's kernels are done
            const int end = ctx->h_ends[c];
            if (end < done || (cands_out && do_coarse && end > cap_out)) break;  // capacity errors are reported below
            CU(fetch(done, end, ctx->d2h));
            done = end;
        }
    }
    int h_counters[4];
    CU(cudaMemcpyAsync(h_counters, b.counters, sizeof(h_counters), cudaMemcpyDeviceToHost, cs));
    CU(cudaStreamSynchronize(cs));
    if (early) CU(cudaStreamSynchronize(ctx->d2h));  // nothing may still be writing caller memory if we fail below
    CU(cudaGetLastError());
    const int total = h_counters[0];
    if (h_counters[1]) return fail(ctx, UWSPR_B200_E_CAPACITY, "more candidates than max_candidates of the context");
    if (total_out) *total_out = total;
    if (do_coarse) {
        if (cands_out && total > cap_out) return fail(ctx, UWSPR_B200_E_CAPACITY, "more candidates than the caller's cap");
    } else if (cands_in && total != total_in) {
        return fail(ctx, UWSPR_B200_E_PARAM, "sum of npk differs from total");
    }
    if (npk_out) CU(cudaMemcpyAsync(npk_out, b.npk, sizeof(int) * nwin, cudaMemcpyDeviceToHost, cs));
    if (cands_out && !do_coarse && total)  // the caller's own list, echoed
        CU(cudaMemcpyAsync(cands_out, b.cands, sizeof(uwspr_b200_candidate_t) * (size_t)total, cudaMemcpyDeviceToHost, cs));
    CU(fetch(done, total, cs));
    CU(cudaEventRecord(ctx->ev_end, cs));
    CU(cudaStreamSynchronize(cs));
    for (int c = 0; c < nchunks; c++) {
        float t;
        for (int q = 0; q < 3; q++) {
            CU(cudaEventElapsedTime(&t, ctx->ev[4 * c + q], ctx->ev[4 * c + q + 1]));
            ctx->ms[q] += t;
        }
    }
    CU(cudaEventElapsedTime(&ctx->ms[3], ctx->ev_begin, ctx->ev_end));
    if (ctx->knobs.trace) {
        float k = 0.f, c0 = 0.f, c1 = 0.f;
        cudaEventElapsedTime(&k, ctx->ev_begin, ctx->ev_kend);
        if (host) {
            cudaEventElapsedTime(&c0, ctx->ev_begin, ctx->ev_cp0);
            cudaEventElapsedTime(&c1, ctx->ev_begin, ctx->ev_cp1);
        }
        fprintf(stderr, "uwspr_b200 trace: chunk kernels start..end (ms):");
        for (int c = 0; c < nchunks; c++) {
            float a = 0.f, z = 0.f;
            cudaEventElapsedTime(&a, ctx->ev_begin, ctx->ev[4 * c]);
            cudaEventElapsedTime(&z, ctx->ev_begin, ctx->ev[4 * c + 3]);
            fprintf(stderr, " [%d w%d] %.2f..%.2f", c, chunks[c].nw, a, z);
        }
        fprintf(stderr, "\n");
        fprintf(stderr, "uwspr_b200 trace: nwin %d chunks %d | first copy starts %.3f ms, last copy ends %.3f ms, "
                        "kernels end %.3f ms, results on host %.3f ms\n", nwin, nchunks, c0, c1, k, ctx->ms[3]);
    }
    ctx->have_coarse = true;
    // the fine path writes b.refined[g], b.jig[g * jig_count + t] and b.soft[(g * jig_count + t) * 162] at the
    // call-wide candidate index g (the work list's running total), for host-fed and resident input alike
    ctx->have_fine = do_fine;
    ctx->last_jig_count = jig_count;
    ctx->last_nwin = nwin;
    ctx->last_total = total;
    ctx->last_samples = samples;
    ctx->last_stride = win_stride;
    return UWSPR_B200_OK;
}

// Every failure leaves through here: nothing may still be copying into the caller's buffers or running on
// the context's streams once an error status has been returned, and a candidate list left by a call that
// failed half way must not be used by a following fine(cands == NULL).
int run(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int nwin, bool do_coarse,
        bool do_fine, const int32_t *npk_in, const uwspr_b200_candidate_t *cands_in, int total_in, int jig_first,
        int jig_count, int32_t *npk_out, uwspr_b200_candidate_t *cands_out, int cap_out, int32_t *total_out,
        uwspr_b200_refined_t *refined_out, uwspr_b200_jiggle_t *jig_out, uint8_t *soft_out, int wins_per_chan = 0,
        int64_t chan_stride = 0)
{
    // the public entry points pass one stream: every window of the call belongs to channel 0
    if (wins_per_chan <= 0) wins_per_chan = std::max(nwin, 1);
    const int rc = run_impl(ctx, samples, space, win_stride, wins_per_chan, chan_stride, nwin, do_coarse, do_fine, npk_in, cands_in, total_in, jig_first,
                            jig_count, npk_out, cands_out, cap_out, total_out, refined_out, jig_out, soft_out);
    if (rc != UWSPR_B200_OK && ctx) {
        cudaStream_t all[5] = { ctx->compute, ctx->compute2, ctx->compute3, ctx->copy, ctx->d2h };
        for (cudaStream_t q : all)
            if (q) cudaStreamSynchronize(q);
        cudaGetLastError();
        ctx->have_coarse = false;
        ctx->have_fine = false;
        ctx->last_nwin = 0;
    }
    return rc;
}

}  // namespace

extern "C" {

const char *uwspr_b200_status_string(int status)
{
    switch (status) {
    case UWSPR_B200_OK: return "ok";
    case UWSPR_B200_E_PARAM: return "parameter outside the supported domain";
    case UWSPR_B200_E_CUDA: return "CUDA error";
    case UWSPR_B200_E_CAPACITY: return "candidate capacity exceeded";
    case UWSPR_B200_E_NOMEM: return "out of memory";
    case UWSPR_B200_E_STATE: return "call sequence error";
    default: return "unknown status";
    }
}

const char *uwspr_b200_last_error(const uwspr_b200_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : "";
}

static thread_local std::string g_create_error;   // per thread: contexts may be created concurrently
UWSPR_B200_API const char *uwspr_b200_create_error(void) { return g_create_error.c_str(); }

int uwspr_b200_create(const uwspr_b200_params_t *params, uwspr_b200_ctx **ctx_out)
{
    if (!params || !ctx_out) return UWSPR_B200_E_PARAM;
    *ctx_out = nullptr;
    uwspr_b200_ctx *ctx = new uwspr_b200_ctx();
    ctx->prm = *params;
    auto bail = [&](int st) {
        g_create_error = ctx->err;
        uwspr_b200_destroy(ctx);
        return st;
    };
    const uwspr_b200_params_t &p = ctx->prm;
    // domain of the reference's own constants
    if (p.spb != 256) return bail(fail(ctx, UWSPR_B200_E_PARAM, "spb must be 256 (the fine stage of the reference hard-codes 256 samples per symbol)"));
    if (p.fl != UW_NP) return bail(fail(ctx, UWSPR_B200_E_PARAM, "fl must be 45000 (npoints is a literal in the reference)"));
    if (p.fs <= 0 || p.maxfreqs < 1 || p.maxdrift < 0 || p.halfbandwidth < 1)
        return bail(fail(ctx, UWSPR_B200_E_PARAM, "fs, maxfreqs, halfbandwidth must be positive and maxdrift non-negative"));
    if (p.halfbandwidth > (int)((float)p.fs / 2.0))  // FDR_impl.cc:82-90 (the reference exits)
        return bail(fail(ctx, UWSPR_B200_E_PARAM, "half pass bandwidth must be lower than the max frequency range"));
    std::vector<uint32_t> off4;
    std::vector<short> hyp_unique;
    int rc = build_tables(ctx, off4, hyp_unique);
    if (rc) return bail(rc);

    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return bail(fail(ctx, UWSPR_B200_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(ce)));
    if (p.device < 0 || p.device >= ndev) return bail(fail(ctx, UWSPR_B200_E_PARAM, "device ordinal out of range"));
    ctx->device = p.device;
#define CUC(call)                                                                                          \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return bail(fail(ctx, UWSPR_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_))); \
    } while (0)
    CUC(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = prop.multiProcessorCount;
    UwDims &d = ctx->d;
    ctx->max_windows = p.max_windows > 0 ? p.max_windows : 1;
    ctx->chunk_windows = std::min(ctx->max_windows, 16384);
    ctx->knobs = read_knobs();
    const long long def_cap = (long long)ctx->max_windows * d.maxcand;
    ctx->max_candidates = p.max_candidates > 0 ? p.max_candidates : (int)std::min<long long>(def_cap, 1 << 22);
    Buffers &b = ctx->b;
    const size_t cw = (size_t)ctx->chunk_windows, cap = (size_t)ctx->max_candidates;
    CUC(cudaMalloc(&b.amp, cw * d.n_rows * d.nbp * sizeof(float)));
    CUC(cudaMalloc(&b.psavg, cw * d.nbp * sizeof(float)));
    CUC(cudaMalloc(&b.peaks, cw * d.maxcand * sizeof(UwPeak)));
    CUC(cudaMalloc(&b.items, cap * sizeof(UwItem)));
    CUC(cudaMalloc(&b.cands, cap * sizeof(uwspr_b200_candidate_t)));
    CUC(cudaMalloc(&b.refined, cap * sizeof(uwspr_b200_refined_t)));
    CUC(cudaMalloc(&b.jig, cap * UWSPR_B200_NJIG * sizeof(uwspr_b200_jiggle_t)));
    CUC(cudaMalloc(&b.soft, cap * UWSPR_B200_NJIG * UW_NSYM));
    CUC(cudaMalloc(&b.counters, kCounterInts * sizeof(int)));
    CUC(cudaMemset(b.counters, 0, kCounterInts * sizeof(int)));
    // 16 384 candidates per pass on every stream: with 4 096 on the second and third, a 4 096-window host-fed chunk
    // needed two passes (host-fed 100 000-window stream: 4 096 / 8 192 / 16 384 -> 247 / 283 / 294 k windows/s)
    for (int q = 0; q < 3; q++) CUC(uw_fine_work_alloc(&b.fine[q], std::min(ctx->max_candidates, 16384)));
    // tables
    std::vector<float> window(UW_FFT_N);
    for (int i = 0; i < d.size; i++) window[i] = (float)sin((M_PI / (d.size - 1)) * i);  // FDR_impl.cc:103-105
    std::vector<float2> tw(UW_FFT_N);
    for (int t = 0; t < UW_FFT_N; t++) {
        const double a = -2.0 * M_PI * t / UW_FFT_N;
        tw[t] = make_float2((float)cos(a), (float)sin(a));
    }
    CUC(cudaMalloc(&b.window, UW_FFT_N * sizeof(float)));
    CUC(cudaMalloc(&b.twiddle, UW_FFT_N * sizeof(float2)));
    CUC(cudaMalloc(&b.off4, off4.size() * sizeof(uint32_t)));
    CUC(cudaMalloc(&b.hyp_unique, hyp_unique.size() * sizeof(short)));
    CUC(cudaMemcpy(b.window, window.data(), UW_FFT_N * sizeof(float), cudaMemcpyHostToDevice));
    CUC(cudaMemcpy(b.twiddle, tw.data(), UW_FFT_N * sizeof(float2), cudaMemcpyHostToDevice));
    CUC(cudaMemcpy(b.off4, off4.data(), off4.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CUC(cudaMemcpy(b.hyp_unique, hyp_unique.data(), hyp_unique.size() * sizeof(short), cudaMemcpyHostToDevice));
    CUC(cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->copy, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->compute2, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->d2h, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->compute3, cudaStreamNonBlocking));
    CUC(cudaEventCreateWithFlags(&ctx->ev_join3, cudaEventDisableTiming));
    CUC(cudaHostAlloc(&ctx->h_ends, sizeof(int) * (kMaxChunks + 4), cudaHostAllocDefault));
    CUC(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    for (int q = 0; q < 3; q++) {
        CUC(cudaEventCreateWithFlags(&ctx->ev_h2d[q], cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&ctx->ev_free[q], cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&ctx->ev_wl[q], cudaEventDisableTiming));
    }
    CUC(cudaEventCreate(&ctx->ev_begin));
    CUC(cudaEventCreate(&ctx->ev_cp0));
    CUC(cudaEventCreate(&ctx->ev_cp1));
    CUC(cudaEventCreate(&ctx->ev_kend));
    CUC(cudaEventCreate(&ctx->ev_end));
    const Knobs &kn = ctx->knobs;
    UwFineLaunch &fl = ctx->fine_launch;
    if (uw_coarse_setup(d) || uw_fine_setup(ctx->sm_count, !kn.no_lag_share, !kn.no_fine_reuse, &fl) || uw_fano_setup())
        return bail(fail(ctx, UWSPR_B200_E_CUDA, "cannot reserve shared memory for the kernels (not an sm_100a device?)"));
    ctx->grid_coarse = ctx->sm_count * uw_coarse_blocks_per_sm(d);
    ctx->fano_grid = ctx->sm_count * uw_fano_blocks_per_sm();
    if (kn.trace)
        fprintf(stderr, "uwspr_b200 trace: fine path: %d + %d + %d resident CTAs per SM (points, lags, lag share%s), slices of %d candidates\n",
                fl.grid_points / ctx->sm_count, fl.grid_lags / ctx->sm_count, fl.grid_share / ctx->sm_count,
                fl.lag_share ? "" : " off", b.fine[0].slice);
    CUC(cudaDeviceSynchronize());
#undef CUC
    *ctx_out = ctx;
    return UWSPR_B200_OK;
}

void uwspr_b200_destroy(uwspr_b200_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->pending.valid()) ctx->pending.wait();
    cudaSetDevice(ctx->device);
    Buffers &b = ctx->b;
    void *ptrs[] = { b.x_stage[0], b.x_stage[1], b.x_stage[2], b.amp, b.ps_dbg, b.psavg, b.peaks, b.npk, b.base, b.items,
                     b.cands, b.refined, b.jig, b.soft, b.counters, b.window, b.twiddle, b.off4, b.hyp_unique,
                     b.dec_first_ok, b.dec_tasks, b.dec_task_cycles, b.dec_task_msg, b.dec_counters, b.dec_out, b.mettab, b.rows };
    for (void *q : ptrs)
        if (q) cudaFree(q);
    for (UwFineWork &w : b.fine) uw_fine_work_free(&w);
    for (cudaEvent_t e : ctx->ev) cudaEventDestroy(e);
    for (int q = 0; q < 3; q++) {
        if (ctx->ev_h2d[q]) cudaEventDestroy(ctx->ev_h2d[q]);
        if (ctx->ev_free[q]) cudaEventDestroy(ctx->ev_free[q]);
        if (ctx->ev_wl[q]) cudaEventDestroy(ctx->ev_wl[q]);
    }
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_cp0) cudaEventDestroy(ctx->ev_cp0);
    if (ctx->ev_cp1) cudaEventDestroy(ctx->ev_cp1);
    if (ctx->ev_kend) cudaEventDestroy(ctx->ev_kend);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->compute && ctx->own_compute) cudaStreamDestroy(ctx->compute);
    if (ctx->copy) cudaStreamDestroy(ctx->copy);
    if (ctx->compute2) cudaStreamDestroy(ctx->compute2);
    if (ctx->d2h) cudaStreamDestroy(ctx->d2h);
    if (ctx->compute3) cudaStreamDestroy(ctx->compute3);
    if (ctx->ev_join3) cudaEventDestroy(ctx->ev_join3);
    if (ctx->h_ends) cudaFreeHost(ctx->h_ends);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    delete ctx;
}

int uwspr_b200_info(const uwspr_b200_ctx *ctx, uwspr_b200_info_t *info)
{
    if (!ctx || !info) return UWSPR_B200_E_PARAM;
    const UwDims &d = ctx->d;
    info->size = d.size;
    info->m = d.m;
    info->hpbm = d.hpbm;
    info->n_rows = d.n_rows;
    info->finpb = d.finpb;
    info->noiseidx = d.noiseidx;
    info->df = d.df;
    info->min_snr = d.min_snr;
    info->bin_lo = d.bin_lo;
    info->n_bins = d.n_bins;
    info->n_lin = d.n_lin;
    info->n_unique = d.n_unique;
    info->max_cand_per_window = d.maxcand;
    info->max_windows = ctx->max_windows;
    info->max_candidates = ctx->max_candidates;
    info->sm_count = ctx->sm_count;
    return UWSPR_B200_OK;
}

static int busy(uwspr_b200_ctx *ctx)
{
    return (ctx && ctx->pending.valid()) ? fail(ctx, UWSPR_B200_E_STATE, "a submitted call has not been waited for (uwspr_b200_wait)") : 0;
}

int uwspr_b200_coarse(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int nwin,
                      int32_t *npk, uwspr_b200_candidate_t *cands, int cap, int32_t *total)
{
    if (busy(ctx)) return UWSPR_B200_E_STATE;
    return run(ctx, samples, space, win_stride, nwin, true, false, nullptr, nullptr, 0, 0, 0, npk, cands, cap, total,
               nullptr, nullptr, nullptr);
}

int uwspr_b200_fine(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int nwin,
                    const int32_t *npk, const uwspr_b200_candidate_t *cands, int total, int jig_first,
                    int jig_count, uwspr_b200_refined_t *refined, uwspr_b200_jiggle_t *jig, uint8_t *soft)
{
    if (busy(ctx)) return UWSPR_B200_E_STATE;
    return run(ctx, samples, space, win_stride, nwin, false, true, npk, cands, total, jig_first, jig_count, nullptr,
               nullptr, 0, nullptr, refined, jig, soft);
}

int uwspr_b200_coarse_fine(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int nwin,
                           int jig_first, int jig_count, int32_t *npk, uwspr_b200_candidate_t *cands, int cap,
                           int32_t *total, uwspr_b200_refined_t *refined, uwspr_b200_jiggle_t *jig, uint8_t *soft)
{
    if (busy(ctx)) return UWSPR_B200_E_STATE;
    return run(ctx, samples, space, win_stride, nwin, true, true, nullptr, nullptr, 0, jig_first, jig_count, npk, cands,
               cap, total, refined, jig, soft);
}

}  // extern "C"

int uw_coarse_fine_channels(uwspr_b200_ctx *ctx, const float *samples, int64_t win_stride, int wins_per_chan,
                            int64_t chan_stride, int nchan, int jig_first, int jig_count, int32_t *npk,
                            uwspr_b200_candidate_t *cands, int cap, int32_t *total)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (busy(ctx)) return UWSPR_B200_E_STATE;
    if (wins_per_chan < 1 || nchan < 1 || (long long)wins_per_chan * nchan > INT_MAX ||
        (nchan > 1 && chan_stride < (wins_per_chan - 1) * win_stride + ctx->d.fl))
        return fail(ctx, UWSPR_B200_E_PARAM, "bad channel geometry");
    return run(ctx, samples, UWSPR_B200_DEVICE, win_stride, wins_per_chan * nchan, true, true, nullptr, nullptr, 0, jig_first,
               jig_count, npk, cands, cap, total, nullptr, nullptr, nullptr, wins_per_chan, chan_stride);
}

extern "C" {

int uwspr_b200_coarse_fine_submit(uwspr_b200_ctx *ctx, const float *samples, int space, int64_t win_stride, int nwin,
                                  int jig_first, int jig_count, int32_t *npk, uwspr_b200_candidate_t *cands, int cap,
                                  int32_t *total, uwspr_b200_refined_t *refined, uwspr_b200_jiggle_t *jig, uint8_t *soft)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (ctx->pending.valid()) return fail(ctx, UWSPR_B200_E_STATE, "one submission at a time per context: wait for the previous one");
    // run() drives copies and kernels with stream waits and a few event synchronisations of its own; on its own
    // thread none of them blocks the caller (a GNU Radio message handler returns at once and picks the results up later)
    std::packaged_task<int()> task([=]() {
        return run(ctx, samples, space, win_stride, nwin, true, true, nullptr, nullptr, 0, jig_first, jig_count, npk, cands, cap,
                   total, refined, jig, soft);
    });
    std::future<int> fut = task.get_future();
    std::thread(std::move(task)).detach();
    ctx->pending = std::move(fut);   // the worker thread never touches `pending`; the synchronous entry points check it
    return UWSPR_B200_OK;
}

int uwspr_b200_poll(uwspr_b200_ctx *ctx)
{
    if (!ctx || !ctx->pending.valid()) return -1;
    return ctx->pending.wait_for(std::chrono::seconds(0)) == std::future_status::ready ? 1 : 0;
}

int uwspr_b200_wait(uwspr_b200_ctx *ctx)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (!ctx->pending.valid()) return fail(ctx, UWSPR_B200_E_STATE, "nothing was submitted");
    return ctx->pending.get();
}

}  // extern "C"

namespace {

int ensure_mettab(uwspr_b200_ctx *ctx)
{
    Buffers &b = ctx->b;
    if (b.mettab) return UWSPR_B200_OK;
    CU(cudaMalloc(&b.mettab, sizeof(WSPR_METTAB)));
    // on the context's stream: the kernels run there, and that stream does not wait for the legacy default stream
    CU(cudaMemcpyAsync(b.mettab, WSPR_METTAB, sizeof(WSPR_METTAB), cudaMemcpyHostToDevice, ctx->compute));
    CU(cudaStreamSynchronize(ctx->compute));
    return UWSPR_B200_OK;
}

int ensure_decoder(uwspr_b200_ctx *ctx)
{
    Buffers &b = ctx->b;
    const int rc = ensure_mettab(ctx);
    if (rc || b.dec_out) return rc;
    const size_t cap = (size_t)ctx->max_candidates, ntask = cap * UWSPR_B200_NJIG;
    CU(cudaMalloc(&b.dec_first_ok, cap * sizeof(int)));
    CU(cudaMalloc(&b.dec_tasks, ntask * sizeof(int)));
    CU(cudaMalloc(&b.dec_task_cycles, ntask * sizeof(uint32_t)));
    CU(cudaMalloc(&b.dec_task_msg, ntask * sizeof(unsigned long long)));
    CU(cudaMalloc(&b.dec_counters, 2 * sizeof(int)));
    CU(cudaMalloc(&b.dec_out, cap * (1 + 7 + sizeof(int32_t) + sizeof(uint32_t))));
    return UWSPR_B200_OK;
}

// (maxcycles * nbits + 1) * delta must fit in int32: the device decoder keeps its threshold in 32 bits (fano.cu)
bool fano_domain(uint32_t nbits, int delta, uint32_t maxcycles)
{
    if (nbits < 32 || nbits > 81 || delta <= 0 || maxcycles < 1) return false;
    const unsigned long long steps = (unsigned long long)maxcycles * nbits + 1;
    return steps * (unsigned long long)delta <= (unsigned long long)INT32_MAX;
}

int decode_impl(uwspr_b200_ctx *ctx, const uwspr_b200_refined_t *refined, const uwspr_b200_jiggle_t *jig,
                const uint8_t *soft, int space, int ncand, int jig_count, uint8_t *decoded, int8_t *messages7,
                int32_t *idt_used, uint32_t *fano_cycles, int *ndecoded)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_decoder(ctx);
    if (rc) return rc;
    Buffers &b = ctx->b;
    cudaStream_t cs = ctx->compute;
    if (refined) {
        // the caller's inputs replace the fine results of the last call on the device
        ctx->have_fine = false;
        const cudaMemcpyKind k = space == UWSPR_B200_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
        const size_t n = (size_t)ncand;
        CU(cudaMemcpyAsync(b.refined, refined, n * sizeof(uwspr_b200_refined_t), k, cs));
        CU(cudaMemcpyAsync(b.jig, jig, n * jig_count * sizeof(uwspr_b200_jiggle_t), k, cs));
        CU(cudaMemcpyAsync(b.soft, soft, n * jig_count * UW_NSYM, k, cs));
    }
    const size_t cap = (size_t)ctx->max_candidates;
    uint8_t *d_dec = b.dec_out;
    int8_t *d_msg = reinterpret_cast<int8_t *>(b.dec_out + cap);
    int32_t *d_idt = reinterpret_cast<int32_t *>(b.dec_out + 8 * cap);
    uint32_t *d_cyc = reinterpret_cast<uint32_t *>(b.dec_out + 12 * cap);
    uw_launch_fano_candidates(b.refined, b.jig, b.soft, ncand, jig_count, b.mettab, b.dec_first_ok, b.dec_tasks,
                              b.dec_counters, b.dec_task_cycles, b.dec_task_msg, ctx->fano_grid, d_dec, d_msg, d_idt, d_cyc, cs);
    ctx->launches += jig_count > 0 ? 3 : 2;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(decoded, d_dec, (size_t)ncand, cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(messages7, d_msg, (size_t)ncand * 7, cudaMemcpyDeviceToHost, cs));
    if (idt_used) CU(cudaMemcpyAsync(idt_used, d_idt, (size_t)ncand * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
    if (fano_cycles) CU(cudaMemcpyAsync(fano_cycles, d_cyc, (size_t)ncand * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
    CU(cudaStreamSynchronize(cs));
    int n = 0;
    for (int g = 0; g < ncand; g++) n += decoded[g];
    *ndecoded = n;
    return UWSPR_B200_OK;
}

int fano_rows_impl(uwspr_b200_ctx *ctx, const uint8_t *symbols, int space, int n, uint32_t nbits, int delta,
                   uint32_t maxcycles, int32_t *status, uint32_t *metric, uint32_t *cycles, uint32_t *maxnp, uint8_t *data11)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_mettab(ctx);
    if (rc) return rc;
    Buffers &b = ctx->b;
    // symbols, then the four counters and data11, each array 16-byte aligned
    const size_t m = (size_t)n, sym_bytes = (m * UW_NSYM + 15) & ~(size_t)15, cnt_bytes = (m * sizeof(uint32_t) + 15) & ~(size_t)15;
    const size_t need = sym_bytes + 4 * cnt_bytes + m * 11;
    if (need > b.rows_cap) {
        if (b.rows) cudaFree(b.rows);
        b.rows = nullptr;
        b.rows_cap = 0;
        CU(cudaMalloc(&b.rows, need));
        b.rows_cap = need;
    }
    cudaStream_t cs = ctx->compute;
    uint8_t *d_sym = b.rows;
    int32_t *d_status = reinterpret_cast<int32_t *>(b.rows + sym_bytes);
    uint32_t *d_metric = reinterpret_cast<uint32_t *>(b.rows + sym_bytes + cnt_bytes);
    uint32_t *d_cycles = reinterpret_cast<uint32_t *>(b.rows + sym_bytes + 2 * cnt_bytes);
    uint32_t *d_maxnp = reinterpret_cast<uint32_t *>(b.rows + sym_bytes + 3 * cnt_bytes);
    uint8_t *d_data = b.rows + sym_bytes + 4 * cnt_bytes;
    const uint8_t *src = symbols;
    if (space == UWSPR_B200_HOST) {
        CU(cudaMemcpyAsync(d_sym, symbols, m * UW_NSYM, cudaMemcpyHostToDevice, cs));
        src = d_sym;
    }
    uw_launch_fano_rows(src, n, (int)nbits, delta, maxcycles, b.mettab, d_status, d_metric, d_cycles, d_maxnp, d_data, cs);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(status, d_status, m * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(metric, d_metric, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(cycles, d_cycles, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(maxnp, d_maxnp, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, cs));
    CU(cudaMemcpyAsync(data11, d_data, m * 11, cudaMemcpyDeviceToHost, cs));
    CU(cudaStreamSynchronize(cs));
    return UWSPR_B200_OK;
}

// as run(): nothing may still run on the context's stream once an error status has been returned
int settle(uwspr_b200_ctx *ctx, int rc)
{
    if (rc != UWSPR_B200_OK) {
        cudaStreamSynchronize(ctx->compute);
        cudaGetLastError();
    }
    return rc;
}

}  // namespace

extern "C" {

int uwspr_b200_decode_device(uwspr_b200_ctx *ctx, const uwspr_b200_refined_t *refined, const uwspr_b200_jiggle_t *jig,
                             const uint8_t *soft, int space, int64_t ncand, int jig_count, uint8_t *decoded,
                             int8_t *messages7, int32_t *idt_used, uint32_t *fano_cycles)
{
    if (!ctx) return -UWSPR_B200_E_PARAM;
    if (busy(ctx)) return -UWSPR_B200_E_STATE;
    if (ncand < 0 || jig_count < 0 || jig_count > UWSPR_B200_NJIG)
        return -fail(ctx, UWSPR_B200_E_PARAM, "ncand < 0 or jig_count outside [0, 17]");
    if (!refined && !jig && !soft) {
        if (!ctx->have_fine) return -fail(ctx, UWSPR_B200_E_STATE, "no fine results on the device: call uwspr_b200_fine / coarse_fine first");
        if (ncand != ctx->last_total || jig_count != ctx->last_jig_count)
            return -fail(ctx, UWSPR_B200_E_PARAM, "ncand / jig_count differ from the last fine call's candidate total / jiggle count");
    } else {
        if (!refined || !jig || !soft) return -fail(ctx, UWSPR_B200_E_PARAM, "refined, jig and soft: all given or all NULL");
        if (space != UWSPR_B200_HOST && space != UWSPR_B200_DEVICE) return -fail(ctx, UWSPR_B200_E_PARAM, "space must be HOST or DEVICE");
        if (ncand > ctx->max_candidates) return -fail(ctx, UWSPR_B200_E_CAPACITY, "more candidates than max_candidates");
    }
    if (ncand == 0) return 0;
    if (!decoded || !messages7) return -fail(ctx, UWSPR_B200_E_PARAM, "decoded and messages7 are required");
    int n = 0;
    const int rc = settle(ctx, decode_impl(ctx, refined, jig, soft, space, (int)ncand, jig_count, decoded, messages7, idt_used,
                                           fano_cycles, &n));
    return rc ? -rc : n;
}

int uwspr_b200_fano_batch(uwspr_b200_ctx *ctx, const uint8_t *symbols, int space, int64_t n, uint32_t nbits, int delta,
                          uint32_t maxcycles, int32_t *status, uint32_t *metric, uint32_t *cycles, uint32_t *maxnp,
                          uint8_t *data11)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (!fano_domain(nbits, delta, maxcycles))
        return fail(ctx, UWSPR_B200_E_PARAM, "need 32 <= nbits <= 81, delta > 0, maxcycles >= 1 and (maxcycles*nbits + 1)*delta < 2^31");
    if (n < 0 || n > INT_MAX - 64) return fail(ctx, UWSPR_B200_E_PARAM, "row count out of range");
    if (space != UWSPR_B200_HOST && space != UWSPR_B200_DEVICE) return fail(ctx, UWSPR_B200_E_PARAM, "space must be HOST or DEVICE");
    if (busy(ctx)) return UWSPR_B200_E_STATE;
    if (n == 0) return UWSPR_B200_OK;
    if (!symbols || !status || !metric || !cycles || !maxnp || !data11) return fail(ctx, UWSPR_B200_E_PARAM, "NULL buffer");
    return settle(ctx, fano_rows_impl(ctx, symbols, space, (int)n, nbits, delta, maxcycles, status, metric, cycles, maxnp, data11));
}

int uwspr_b200_host_alloc(void **ptr, size_t bytes)
{
    if (!ptr) return UWSPR_B200_E_PARAM;
    return cudaHostAlloc(ptr, bytes, cudaHostAllocDefault) == cudaSuccess ? UWSPR_B200_OK : UWSPR_B200_E_NOMEM;
}

void uwspr_b200_host_free(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
}

UWSPR_B200_API int uwspr_b200_set_debug(uwspr_b200_ctx *ctx, int keep_power)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    CU(cudaSetDevice(ctx->device));
    if (keep_power && !ctx->b.ps_dbg)
        CU(cudaMalloc(&ctx->b.ps_dbg, (size_t)ctx->chunk_windows * ctx->d.n_rows * ctx->d.nbp * sizeof(float)));
    ctx->debug_ps = keep_power != 0;
    return UWSPR_B200_OK;
}

/* use the caller's CUDA stream (a cudaStream_t passed as void*) for all kernels, so that
 * events recorded by the caller on that stream bracket the work; NULL restores the
 * context's own stream */
UWSPR_B200_API int uwspr_b200_set_stream(uwspr_b200_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    static_assert(sizeof(void *) == sizeof(cudaStream_t), "stream handle size");
    if (cuda_stream) {
        if (ctx->own_compute && ctx->compute) cudaStreamDestroy(ctx->compute);
        ctx->compute = (cudaStream_t)cuda_stream;
        ctx->own_compute = false;
    } else if (!ctx->own_compute) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking));
        ctx->own_compute = true;
    }
    return UWSPR_B200_OK;
}

int uwspr_b200_debug_spectrogram(uwspr_b200_ctx *ctx, int win, float *ps, float *psavg)
{
    if (!ctx) return UWSPR_B200_E_PARAM;
    if (!ctx->debug_ps || !ctx->b.ps_dbg) return fail(ctx, UWSPR_B200_E_STATE, "enable uwspr_b200_set_debug first");
    // the chunk buffers keep the last chunk (device input) or the last chunks of every buffer set (host input)
    const int cw = ctx->last_cw > 0 ? ctx->last_cw : 1;
    const std::vector<UwChunk> &chunks = ctx->last_chunks;
    const UwChunk *ch = nullptr;
    for (const UwChunk &q : chunks)
        if (win >= q.w0 && win < q.w0 + q.nw) ch = &q;
    if (win < 0 || win >= ctx->last_nwin || !ch || ch->group < chunks.back().group - (ctx->last_sets - 1))
        return fail(ctx, UWSPR_B200_E_PARAM, "window is not in the chunks still held on the device");
    const size_t slot = (size_t)ch->set * cw + (size_t)ch->slot + (size_t)(win - ch->w0);
    CU(cudaSetDevice(ctx->device));
    const UwDims &d = ctx->d;
    std::vector<float> tmp((size_t)d.n_rows * d.nbp);
    if (ps) {
        CU(cudaMemcpy(tmp.data(), ctx->b.ps_dbg + slot * d.n_rows * d.nbp, tmp.size() * sizeof(float),
                      cudaMemcpyDeviceToHost));
        for (int r = 0; r < d.n_rows; r++) memcpy(ps + (size_t)r * d.n_bins, &tmp[(size_t)r * d.nbp], sizeof(float) * d.n_bins);
    }
    if (psavg) CU(cudaMemcpy(psavg, ctx->b.psavg + slot * d.nbp, sizeof(float) * d.n_bins, cudaMemcpyDeviceToHost));
    return UWSPR_B200_OK;
}

int uwspr_b200_last_timing(const uwspr_b200_ctx *ctx, float ms[4])
{
    if (!ctx || !ms) return UWSPR_B200_E_PARAM;
    for (int q = 0; q < 4; q++) ms[q] = ctx->ms[q];
    return UWSPR_B200_OK;
}

int64_t uwspr_b200_launch_count(const uwspr_b200_ctx *ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
