// Kernel 1: half-symbol-step spectrogram + normalizer + peak pick for a batch of windows.
//
// Replaces, per window, lib/FDR_impl.cc:222-319 of the reference:
//   :222-254  348 half-sine-windowed 512-point forward DFTs at a 128-sample hop, |X|^2,
//             fft-shift
//   :257-263  column sums psavg[j] (sequential over rows, fp32)
//   :265-291  +-3-bin smoothing, 30th-percentile noise floor, SNR normalisation and clamp
//   :293-306  strict local maxima -> candidate frequencies
//   :309-319  stable descending sort on snr
//
// One CTA (256 threads) per window.  Four 64-thread groups each run one radix-8x8x8
// Stockham FFT per iteration (87 iterations cover the 348 rows); the two inter-pass
// exchanges go through shared memory, the window and twiddles live in registers / shared
// memory.  The four rows of an iteration overlap (hop 128, length 512) and read 896 consecutive
// samples, of which the next iteration keeps 384: the window's samples are staged through a
// shared-memory ring of three 512-sample blocks, one TMA bulk copy (cp.async.bulk, 4 KB) per
// iteration issued two blocks ahead and tracked by an mbarrier, so every sample crosses
// L2 -> shared memory once and no thread holds prefetched samples in registers.  Only the bins the rest of the path can touch are kept ([bin_lo, bin_lo+n_bins),
// 42 of 512 at halfbandwidth 10): their amplitudes sqrt(ps) are written once to HBM for
// the coarse-search kernel (powersum() takes the sqrt of every ps it reads,
// FDR_impl.cc:199-205; IEEE sqrtf is deterministic, so hoisting it is exact), and their
// powers are summed per column in row order by one owner thread per bin.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kGroups = 4;
constexpr int kBlk = kGroups * UW_HOP;   // samples an iteration advances by (512) = one ring block
constexpr int kRingBlocks = 3;

// ---- TMA bulk copy + mbarrier (sm_90+ PTX; SASS: UBLKCP / SYNCS) ----
__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion is counted on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@!p bra WAIT_%=;\n}" ::"r"(smem_addr(bar)),
                 "r"(parity)
                 : "memory");
}

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
// multiply by -i
__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }

// 8-point forward DFT, natural order in and out.  The complex additions are packed (FADD2: the same two fp32
// additions as the scalar pair, one issue slot); multiplications by -i and by exp(-i pi/4) work on the halves.
__device__ __forceinline__ uw_f2 pk2(float2 a) { return uw_pk(a.x, a.y); }
__device__ __forceinline__ float2 up2(uw_f2 a) { return make_float2(uw_lo(a), uw_hi(a)); }
__device__ __forceinline__ void fft8(float2 *v)
{
    const float h = 0.70710678118654752440f;
    const uw_f2 v0 = pk2(v[0]), v1 = pk2(v[1]), v2 = pk2(v[2]), v3 = pk2(v[3]), v4 = pk2(v[4]), v5 = pk2(v[5]), v6 = pk2(v[6]),
                v7 = pk2(v[7]);
    const uw_f2 a0 = uw_add2(v0, v4), a4 = uw_sub2(v0, v4);
    const uw_f2 a1 = uw_add2(v1, v5);
    const float2 t5 = up2(uw_sub2(v1, v5));
    const uw_f2 a2 = uw_add2(v2, v6);
    const float2 t6 = up2(uw_sub2(v2, v6));
    const uw_f2 a3 = uw_add2(v3, v7);
    const float2 t7 = up2(uw_sub2(v3, v7));
    const uw_f2 a5 = uw_pk((t5.x + t5.y) * h, (t5.y - t5.x) * h);   // * exp(-i pi/4)
    const uw_f2 a6 = uw_pk(t6.y, -t6.x);                             // * exp(-i pi/2)
    const uw_f2 a7 = uw_pk((t7.y - t7.x) * h, -(t7.x + t7.y) * h);  // * exp(-3i pi/4)
    const uw_f2 b0 = uw_add2(a0, a2), b2 = uw_sub2(a0, a2), b1 = uw_add2(a1, a3);
    const float2 d13 = up2(uw_sub2(a1, a3));
    const uw_f2 b3 = uw_pk(d13.y, -d13.x);                           // -i (a1 - a3)
    const uw_f2 b4 = uw_add2(a4, a6), b6 = uw_sub2(a4, a6), b5 = uw_add2(a5, a7);
    const float2 d57 = up2(uw_sub2(a5, a7));
    const uw_f2 b7 = uw_pk(d57.y, -d57.x);                           // -i (a5 - a7)
    v[0] = up2(uw_add2(b0, b1));
    v[4] = up2(uw_sub2(b0, b1));
    v[2] = up2(uw_add2(b2, b3));
    v[6] = up2(uw_sub2(b2, b3));
    v[1] = up2(uw_add2(b4, b5));
    v[5] = up2(uw_sub2(b4, b5));
    v[3] = up2(uw_add2(b6, b7));
    v[7] = up2(uw_sub2(b6, b7));
}

// Exchange layout: entry i of a 512-point exchange lives in slot i ^ sw(i), sw = i[6:4] on bits 0..2 and i[6] on
// bit 3.  A 64-bit shared access is served half a warp at a time from sixteen 8-byte slots; with this swizzle the
// sixteen lanes of every half-warp hit sixteen different slots in all three access patterns of the Stockham passes
// (stores to 8j + r, loads from j + 64r, stores to 64(j/8) + j%8 + 8r).  The padded layout this replaces (one spare
// slot per 8) served the stores but made every load a two-wavefront access: 18 % of the kernel's shared wavefronts.

struct __align__(16) SpecSmem {
    float2 xring[kRingBlocks][kBlk];               // the window's samples, block b in slot b % 3
    float2 buf[kGroups][UW_FFT_N];   // inter-pass exchange, one FFT per group, swizzled (see above)
    float2 tw1[8][8];                // pass-1 twiddles exp(-2 pi i 8 r k / 512), [r][k]
    float2 tw2[8][64];               // pass-2 twiddles exp(-2 pi i r j / 512), [r][j]
    float psrow[kGroups][UW_FFT_N];  // powers of the kept bins of the four rows of this iteration
    float psavg[UW_FFT_N];           // column sums of the kept bins
    float smspec[UW_FFT_N];          // smoothed / normalised spectrum, finpb entries
    float noise;
    int npk;
    UwPeak peaks[256];
    UwPeak sorted[256];
    uint64_t bar[kRingBlocks];       // one mbarrier per ring slot
};

// 4 CTAs/SM (64 registers) measured 4.6 % faster than 3 (80 registers) and 20 % faster than 2;
// 64-thread named barriers for the group-local exchanges measured 2 % slower than __syncthreads
// FULL: the row count is a multiple of the four groups (348 = 4 x 87 for the reference's frame length), no row tests
template <bool FULL>
__global__ void __launch_bounds__(kThreads, 4)
k_spectrogram(UwDims d, const float2 *__restrict__ x, UwGeom geom, int nwin,
              const float *__restrict__ window, const float2 *__restrict__ twiddle,
              float *__restrict__ amp, float *__restrict__ ps_dbg, float *__restrict__ psavg_out,
              UwPeak *__restrict__ peaks_out, int *__restrict__ npk_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SpecSmem &sm = *reinterpret_cast<SpecSmem *>(smem_raw);
    const int tid = threadIdx.x;
    const int g = tid >> 6, j = tid & 63;
    const int win = blockIdx.x;
    if (win >= nwin) return;
    const float2 *xw = x + uw_window_offset(geom, win);

    // twiddles laid out so that the lanes of a warp read consecutive words (no bank conflicts)
    for (int t = tid; t < 64; t += kThreads) sm.tw1[t >> 3][t & 7] = twiddle[(8 * (t >> 3) * (t & 7)) & (UW_FFT_N - 1)];
    for (int t = tid; t < 512; t += kThreads) sm.tw2[t >> 6][t & 63] = twiddle[((t >> 6) * (t & 63)) & (UW_FFT_N - 1)];
    float wj[8];
#pragma unroll
    for (int r = 0; r < 8; r++) wj[r] = window[j + 64 * r];

    // this thread owns the column sums of kept bins tid and tid+256
    float acc0 = 0.0f, acc1 = 0.0f;
    const int nb = d.n_bins;
    // which of this thread's eight pass-2 outputs X[j + 64 r] fall in the kept bins
    unsigned keep = 0;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int c = ((j + 64 * r + UW_FFT_N / 2) & (UW_FFT_N - 1)) - d.bin_lo;
        if (c >= 0 && c < nb) keep |= 1u << r;
    }
    __syncthreads();

    const int n_iter = (d.n_rows + kGroups - 1) / kGroups;
    // Sample staging.  Iteration `it` reads samples [512 it, 512 it + 896): ring blocks it and it + 1; block it + 2
    // is fetched while it runs.  Windows that start on a 16-byte boundary use one bulk copy per block (thread 0
    // arms the slot's mbarrier with the byte count and issues it); others (odd sample strides such as the 9 s
    // sliding window) copy with plain loads, ordered by the loop's own barriers.
    const int nblk = (d.fl + kBlk - 1) / kBlk;
    const bool bulk = (reinterpret_cast<unsigned long long>(xw) & 15ull) == 0ull;
    auto fetch_block = [&](int b, int slot) {
        if (b >= nblk) return;
        const int cnt = min(kBlk, d.fl - b * kBlk);          // the last block is short (45000 = 87 * 512 + 456)
        float2 *dst = sm.xring[slot];
        if (bulk) {
            if (tid == 0) {
                mbar_expect_tx(&sm.bar[slot], (unsigned)cnt * 8u);
                bulk_g2s(dst, xw + (long long)b * kBlk, (unsigned)cnt * 8u, &sm.bar[slot]);
            }
        } else {
            for (int t = tid; t < cnt; t += kThreads) dst[t] = __ldg(xw + (long long)b * kBlk + t);
        }
    };
    if (tid == 0) {
#pragma unroll
        for (int q = 0; q < kRingBlocks; q++) mbar_init(&sm.bar[q], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    fetch_block(0, 0);
    fetch_block(1, 1);
    if (bulk) mbar_wait(&sm.bar[0], 0);
    __syncthreads();
    // Everything the loop indexes with is fixed per thread: the exchange positions of the three passes, the twiddle
    // columns, and which of the eight samples of a row come from the second of the iteration's two ring blocks
    // (offset 128 g + j + 64 r >= 512, i.e. r >= 8 - 2 g: the same for a whole warp).
    // Swizzled slots, r = 0..7 (derivation in the layout comment; sw depends on bits 4..6 of the entry only):
    //   pass-0 stores, entry 8j + r:            ex0 + (r ^ k7),  k7 = (j/2) % 8
    //   loads, entry j + 64r:                    (r odd ? ex1o : ex1e) + 64r
    //   pass-1 stores, entry 64(j/8) + j%8 + 8r: ex2 + ((j%4) ^ (r/2)) + 16(r/2) + (r odd ? ex2s : 0)
    const int jb = (j >> 3) & 1;
    const int k7 = (j >> 1) & 7;
    float2 *const ex0 = &sm.buf[g][16 * (j >> 1) + ((8 * (j & 1)) ^ (jb << 3))];
    const float2 *const ex1e = &sm.buf[g][(j & 48) + ((j & 15) ^ (j >> 4))];
    const float2 *const ex1o = &sm.buf[g][(j & 48) + ((j & 15) ^ ((j >> 4) | 12))];
    float2 *const ex2 = &sm.buf[g][64 * (j >> 3) + 4 * (((j >> 2) & 1) ^ jb) + 8 * jb];
    const int ex2s = jb ? -8 : 8;
    const int j3 = j & 3;
    const float2 *const tw1c = &sm.tw1[0][j & 7];
    const float2 *const tw2c = &sm.tw2[0][j];
    const int r_hi = 8 - 2 * g;
    const int base = UW_HOP * g + j;
    int s0 = 0;                              // ring slot of block `it`
    unsigned waited = 1u;                    // bit s: parity of the next wait on slot s (slot 0 was waited for once)
    float *amp_row = amp + ((long long)win * d.n_rows + g) * d.nbp;
    float *dbg_row = ps_dbg ? ps_dbg + ((long long)win * d.n_rows + g) * d.nbp : nullptr;
    const long long row_step = (long long)kGroups * d.nbp;
    for (int it = 0; it < n_iter; it++) {
        const int row = it * kGroups + g;
        const bool live = FULL || row < d.n_rows;
        const int s1 = s0 == kRingBlocks - 1 ? 0 : s0 + 1, s2 = s0 == 0 ? kRingBlocks - 1 : s0 - 1;
        float2 v[8];
        // block it + 1 has landed (use k of a slot completes phase k of its mbarrier)
        if (bulk && it + 1 < nblk) {
            mbar_wait(&sm.bar[s1], (waited >> s1) & 1u);
            waited ^= 1u << s1;
        }
        if (live) {
            const float2 *lo = &sm.xring[s0][base], *hi = &sm.xring[s1][base] - kBlk;
#pragma unroll
            for (int r = 0; r < 8; r++) {
                const float2 xv = (r >= r_hi ? hi : lo)[64 * r];
                // FDR_impl.cc:230-231: the fp32 sample times the fp32 window, rounded once
                v[r] = make_float2(__fmul_rn(xv.x, wj[r]), __fmul_rn(xv.y, wj[r]));
            }
            // pass 0 (Ns = 1): no twiddles; out[8j + r] = X[r]
            fft8(v);
#pragma unroll
            for (int r = 0; r < 8; r++) ex0[r ^ k7] = v[r];
        }
        __syncthreads();
        // every thread has read its samples of this iteration: the slot of block it - 1 is free for block it + 2
        fetch_block(it + 2, s2);
        if (live) {
            // pass 1 (Ns = 8)
#pragma unroll
            for (int r = 0; r < 8; r++) {
                float2 sv = ((r & 1) ? ex1o : ex1e)[64 * r];
                v[r] = (r == 0) ? sv : cmul(sv, tw1c[8 * r]);
            }
            fft8(v);
        }
        __syncthreads();
        if (live) {
#pragma unroll
            for (int r = 0; r < 8; r++) ex2[(j3 ^ (r >> 1)) + 16 * (r >> 1) + ((r & 1) ? ex2s : 0)] = v[r];
        }
        __syncthreads();
        if (live && keep) {
            // pass 2 (Ns = 64): thread j ends with X[j + 64 r].  Narrow pass bands keep one output
            // per thread at most (X[j] below DC+, X[j+448] above): those are summed directly
#pragma unroll
            for (int r = 0; r < 8; r++) {
                float2 sv = ((r & 1) ? ex1o : ex1e)[64 * r];
                v[r] = (r == 0) ? sv : cmul(sv, tw2c[64 * r]);
            }
            if (keep == 0x01u) {
                v[0] = cadd(cadd(cadd(v[0], v[4]), cadd(v[2], v[6])), cadd(cadd(v[1], v[5]), cadd(v[3], v[7])));
            } else if (keep == 0x80u) {
                // X[7] = d0 + d1 e^{i pi/4} + i d2 + d3 e^{3 i pi/4},  dn = v[n] - v[n+4]
                const float h = 0.70710678118654752440f;
                const float2 d0 = csub(v[0], v[4]), d1 = csub(v[1], v[5]), d2 = csub(v[2], v[6]), d3 = csub(v[3], v[7]);
                const float2 e1 = make_float2((d1.x - d1.y) * h, (d1.x + d1.y) * h);
                const float2 e2 = make_float2(-d2.y, d2.x);
                const float2 e3 = make_float2(-(d3.x + d3.y) * h, (d3.x - d3.y) * h);
                v[7] = cadd(cadd(d0, e2), cadd(e1, e3));
            } else {
                fft8(v);
            }
#pragma unroll
            for (int r = 0; r < 8; r++) {
                // narrow bands keep exactly one output per thread (r = 0 or r = 7): skip the other tests
                if ((keep == 0x01u && r != 0) || (keep == 0x80u && r != 7)) continue;
                const int kbin = j + 64 * r;                 // FFT bin (0 = DC)
                const int sh = (kbin + UW_FFT_N / 2) & (UW_FFT_N - 1);  // index after the shift of :247-248
                const int c = sh - d.bin_lo;
                if (c >= 0 && c < nb) {
                    // :252 ps = re*re + im*im, three roundings
                    float p = __fadd_rn(__fmul_rn(v[r].x, v[r].x), __fmul_rn(v[r].y, v[r].y));
                    sm.psrow[g][c] = p;
                    amp_row[c] = __fsqrt_rn(p);
                    if (dbg_row) dbg_row[c] = p;
                }
            }
        }
        amp_row += row_step;
        if (dbg_row) dbg_row += row_step;
        s0 = s1;
        __syncthreads();
        // :257-263 column sums in row order
        {
            const int rows_here = FULL ? kGroups : min(kGroups, d.n_rows - it * kGroups);
            if (tid < nb) {
#pragma unroll
                for (int q = 0; q < kGroups; q++)
                    if (q < rows_here) acc0 = __fadd_rn(acc0, sm.psrow[q][tid]);
            }
            if (tid + kThreads < nb) {
#pragma unroll
                for (int q = 0; q < kGroups; q++)
                    if (q < rows_here) acc1 = __fadd_rn(acc1, sm.psrow[q][tid + kThreads]);
            }
        }
        // psrow is rewritten only after the next iteration's three barriers
    }
    if (tid < nb) sm.psavg[tid] = acc0;
    if (tid + kThreads < nb) sm.psavg[tid + kThreads] = acc1;
    __syncthreads();
    if (psavg_out) {
        for (int c = tid; c < nb; c += kThreads) psavg_out[(long long)win * d.nbp + c] = sm.psavg[c];
    }

    // :265-275 smoothing over +-3 bins, accumulated in the order j = -3..3 from 0.0f
    const int band0 = d.m - d.hpbm - d.bin_lo;  // kept-bin index of shifted bin m-hpbm
    for (int i = tid; i < d.finpb; i += kThreads) {
        float a = 0.0f;
#pragma unroll
        for (int q = -3; q <= 3; q++) a = __fadd_rn(a, sm.psavg[band0 + i + q]);
        sm.smspec[i] = a;
    }
    __syncthreads();
    // :277-285 the noiseidx-th smallest value (qsort + pick), found by rank counting;
    // ties are broken by index so exactly one element has each rank
    for (int i = tid; i < d.finpb; i += kThreads) {
        const float vi = sm.smspec[i];
        int rank = 0;
        for (int q = 0; q < d.finpb; q++) {
            const float vq = sm.smspec[q];
            rank += (vq < vi) || (vq == vi && q < i);
        }
        if (rank == d.noiseidx) sm.noise = vi;
    }
    __syncthreads();
    const float noise = sm.noise;
    __syncthreads();
    // :287-291
    for (int i = tid; i < d.finpb; i += kThreads) {
        float q = __fdiv_rn(sm.smspec[i], noise);
        float s = __fsub_rn(q, 1.0f);  // (double)q - 1.0 stored to float == fp32 subtraction
        if (s < d.min_snr) s = d.floor_val;
        sm.psrow[0][i] = s;  // reuse as the normalised spectrum
    }
    __syncthreads();
    // :293-306 strict local maxima, first maxfreqs in bin order.  One thread walks the
    // (short) pass band so that the order and the cap are exactly the reference's.
    if (tid == 0) {
        int n = 0;
        const float *s = sm.psrow[0];
        for (int i = 1; i < d.finpb - 1; i++) {
            if (s[i] > s[i - 1] && s[i] > s[i + 1] && n < d.maxcand) {
                sm.peaks[n].freq = __fmul_rn((float)(i - d.hpbm), d.df);
                // 10*log10f(x): evaluated in double and rounded, then the fp32 product
                sm.peaks[n].snr = __fmul_rn(10.0f, (float)log10((double)s[i]));
                n++;
            }
        }
        sm.npk = n;
    }
    __syncthreads();
    const int npk = sm.npk;
    // :311-319 stable descending sort: rank = #greater + #equal before
    if (tid < npk) {
        const float si = sm.peaks[tid].snr;
        int rank = 0;
        for (int q = 0; q < npk; q++) {
            const float sq = sm.peaks[q].snr;
            rank += (sq > si) || (sq == si && q < tid);
        }
        sm.sorted[rank] = sm.peaks[tid];
    }
    __syncthreads();
    if (tid < npk) peaks_out[(long long)win * d.maxcand + tid] = sm.sorted[tid];
    if (tid == 0) npk_out[win] = npk;
}

// Exclusive scan of npk over the windows of one chunk + expansion into the compact work
// list.  counters: [0] running total over the chunks of this call (in/out), [1] overflow
// flag; set: the chunk's own {coarse ticket, fine ticket, end of its items} (chunks in
// flight on different streams use different sets).  Item indices are
// global to the call (so results land compactly, window-major); item.win is relative to
// the chunk.
__global__ void __launch_bounds__(1024)
k_worklist(const int *__restrict__ npk, int nwin, int cap, int *__restrict__ base,
           UwItem *__restrict__ items, int *__restrict__ counters, int *__restrict__ set)
{
    __shared__ int part[1024];
    const int tid = threadIdx.x;
    const int run0 = counters[0];
    const int per = (nwin + 1023) / 1024;
    const int lo = min(nwin, tid * per), hi = min(nwin, lo + per);
    int s = 0;
    for (int w = lo; w < hi; w++) s += max(npk[w], 0);
    part[tid] = s;
    __syncthreads();
    // Hillis-Steele inclusive scan over the 1024 partial sums
    for (int off = 1; off < 1024; off <<= 1) {
        int v = (tid >= off) ? part[tid - off] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    int run = run0 + part[tid] - s;
    for (int w = lo; w < hi; w++) {
        base[w] = run;
        const int n = max(npk[w], 0);   // the host rejects negative counts; never index below the list
        for (int q = 0; q < n; q++)
            if (run + q < cap) {
                items[run + q].win = w;
                items[run + q].slot = q;
            }
        run += n;
    }
    if (tid == 1023) {
        const int end = run0 + part[1023];
        counters[0] = end;
        if (end > cap) counters[1] = 1;
        set[0] = run0;  // coarse ticket
        set[1] = run0;  // fine ticket
        set[2] = min(end, cap);  // end of this chunk's items
    }
}

}  // namespace

void uw_launch_spectrogram(const UwDims &d, const float2 *x, const UwGeom &geom, int nwin,
                           const float *window, const float2 *twiddle, float *amp, float *ps_dbg,
                           float *psavg, UwPeak *peaks, int *npk, cudaStream_t s)
{
    static bool attr_set = false;   // above the 48 KB default: opt in once (the attribute belongs to the function)
    if (!attr_set) {
        cudaFuncSetAttribute(k_spectrogram<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SpecSmem));
        cudaFuncSetAttribute(k_spectrogram<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SpecSmem));
        attr_set = true;
    }
    if (d.n_rows % kGroups == 0)
        k_spectrogram<true><<<nwin, kThreads, sizeof(SpecSmem), s>>>(d, x, geom, nwin, window, twiddle, amp, ps_dbg, psavg,
                                                                     peaks, npk);
    else
        k_spectrogram<false><<<nwin, kThreads, sizeof(SpecSmem), s>>>(d, x, geom, nwin, window, twiddle, amp, ps_dbg, psavg,
                                                                      peaks, npk);
}

void uw_launch_worklist(const int *npk, int nwin, int cap, int *base, UwItem *items, int *counters,
                        int *set, cudaStream_t s)
{
    k_worklist<<<1, 1024, 0, s>>>(npk, nwin, cap, base, items, counters, set);
}
