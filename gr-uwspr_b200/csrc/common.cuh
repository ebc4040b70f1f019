// Shared declarations of the uwspr_b200 CUDA path (sm_100a).
//
// Arithmetic contract: the reference decides candidates by strict comparisons of fp32
// sums, and its CPU build cannot contract a*b+c into an FMA (x86-64 baseline).  All
// translation units are therefore compiled with -fmad=false and every expression that
// mirrors a reference line is written with the round-to-nearest intrinsics
// (__fadd_rn, __fmul_rn, __fdiv_rn, __fsqrt_rn) in the reference's evaluation order.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "uwspr_b200.h"

#define UW_NSYM 162
#define UW_FFT_N 512
#define UW_HOP 128
#define UW_NK0 26          // half-symbol start offsets searched, FDR_impl.cc:346
#define UW_NIFR 5          // if0-2 .. if0+2, FDR_impl.cc:344
#define UW_NTRAJ 125       // slm.cc:76-116
#define UW_SPS 256         // samples per symbol in the fine stage (literal in the reference)
#define UW_NP 45000        // npoints, sync_and_demodulate_impl.cc:92
#define UW_MAX_TILE_W 40   // widest amplitude tile (bins) one coarse CTA stages
#define UW_MAX_UNIQUE 192  // most distinct bin-offset sequences supported
#define UW_NQUAD 41        // ceil(162/4) packed offset words per sequence

// Scalar description of one context, passed by value to the kernels.
struct UwDims {
    int fl, n_rows, size, m, hpbm, finpb, noiseidx, maxfreqs, maxcand, maxdrift, cf;
    float df, min_snr, floor_val, threshold;
    int bin_lo, n_bins, nbp;        // kept bins [bin_lo, bin_lo+n_bins), row pitch nbp floats
    int n_lin, n_hyp, n_unique;     // 2*maxdrift+1, n_lin+125, distinct offset sequences
    int off_min, off_max, tile_w;   // bin offsets span [off_min, off_max]; tile_w = 11 + off_max - off_min
    int nonlinear_intended_t;
    uint32_t sync_words[6];         // WSPR sync vector, bit i at word i/32 bit i%32 (reference lib/pr3.h)
};

// one entry of the compact work list: which window, which candidate slot of that window
struct UwItem {
    int win, slot;
};

// per-window staging record written by the spectrogram kernel (before the coarse search)
struct UwPeak {
    float freq, snr;
};

// Where the windows of one launch live.  Window w of the launch is window W = w0 + w of the call;
// the call's windows are channel-major, per_chan per channel: window W = c*per_chan + k starts at
//     x + c*chan_stride + k*win_stride,  x = the call's first sample.
// A single stream is one channel (per_chan >= the call's window count, chan_stride unused).
struct UwGeom {
    long long win_stride, chan_stride;
    int per_chan, w0;
};

// offset, in samples from the call's first sample, of window w of the launch; non-decreasing in w when
// chan_stride >= (per_chan - 1)*win_stride
__host__ __device__ __forceinline__ long long uw_window_offset(const UwGeom &g, int w)
{
    const int W = g.w0 + w;
    const int c = W / g.per_chan;
    return (long long)c * g.chan_stride + (long long)(W - c * g.per_chan) * g.win_stride;
}

__device__ __forceinline__ int uw_sync_bit(const uint32_t *words, int i)
{
    return (int)((words[i >> 5] >> (i & 31)) & 1u);
}

// ---- packed fp32 pairs (sm_100a: add/sub/fma.rn.f32x2 -> FADD2 / FFMA2) ------------------
// One issue slot carries two independent IEEE round-to-nearest operations, each bit-identical
// to its scalar form.  The kernels that mirror reference sums are bound by issue slots and
// the fp32 pipe (no FMA contraction allowed), so they pair two accumulation chains that
// share an operand (two tones against one sample, two bins against one shift).
// ptxas contracts mul.rn.f32x2 followed by add.rn.f32x2 into one FFMA2 even under
// --fmad=false, which would round once instead of twice.  The product is therefore issued
// as fma(a, b, -0.0) with the -0.0 pair in a kernel parameter (opaque to ptxas):
// a*b + (-0) is a*b rounded once, sign of zero included, and an FFMA2 cannot be merged
// with the addition that consumes it.
typedef unsigned long long uw_f2;
#define UW_NEGZERO2 0x8000000080000000ull

__device__ __forceinline__ uw_f2 uw_pk(float lo, float hi)
{
    uw_f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float uw_lo(uw_f2 v)
{
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
    return a;
}
__device__ __forceinline__ float uw_hi(uw_f2 v)
{
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
    return b;
}
__device__ __forceinline__ uw_f2 uw_add2(uw_f2 a, uw_f2 b)
{
    uw_f2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uw_f2 uw_sub2(uw_f2 a, uw_f2 b)
{
    uw_f2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// both products rounded once each; nz must be UW_NEGZERO2 read from a kernel parameter
__device__ __forceinline__ uw_f2 uw_mul2(uw_f2 a, uw_f2 b, uw_f2 nz)
{
    uw_f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(nz));
    return r;
}
// a*b + c with one rounding per lane (callers use it where the product is exact)
__device__ __forceinline__ uw_f2 uw_fma2(uw_f2 a, uw_f2 b, uw_f2 c)
{
    uw_f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// scalar times pair (the scalar is broadcast by the instruction's operand form)
__device__ __forceinline__ uw_f2 uw_mul2s(float a, uw_f2 b, uw_f2 nz) { return uw_mul2(uw_pk(a, a), b, nz); }

// launches (defined in the .cu files)
void uw_launch_spectrogram(const UwDims &d, const float2 *x, const UwGeom &geom, int nwin,
                           const float *window, const float2 *twiddle, float *amp, float *ps_dbg,
                           float *psavg, UwPeak *peaks, int *npk, cudaStream_t s);
void uw_launch_worklist(const int *npk, int nwin, int cap, int *base, UwItem *items, int *counters,
                        int *set, cudaStream_t s);
void uw_launch_coarse(const UwDims &d, const float *amp, const UwPeak *peaks, const UwItem *items,
                      const int *total, int cap, const uint32_t *off4, const short *hyp_unique,
                      uwspr_b200_candidate_t *cands, int *ticket, int grid, cudaStream_t s);
// The fine path's workspace for `slice` candidates (fine.cu): chain state, tone magnitudes, constant-frequency tone
// tables and the work counters of the heavy launches.  One per compute stream: sequences on different streams run
// concurrently.  Alloc makes one allocation and zeroes the counters; free releases it (a zeroed workspace is empty).
struct UwFineWork {
    void *state;                       // chain state per candidate (private to fine.cu); start of the allocation
    float4 *pbuf, *pE, *pbest, *tables;
    int *tickets;
    int slice;                         // candidates one pass of the stage sequence handles
};
cudaError_t uw_fine_work_alloc(UwFineWork *w, int slice);
void uw_fine_work_free(UwFineWork *w);
// How the fine path launches, fixed when a context is created (uw_fine_setup).
struct UwFineLaunch {
    int grid_points, grid_lags, grid_share;   // resident CTAs of R1, R2 and R3 on the whole device
    bool lag_share;   // the lag searches of stages A and D through R3; off: through R1 (reference path for tests)
    bool reuse;       // stage E takes jiggle 0 from the chain; off: evaluates it again (reference path for tests)
};
// the stage sequence of the fine path over work-list entries *begin + slice0 + [0, w.slice); returns the launches issued
int uw_launch_fine(const UwDims &d, const float2 *x, const UwGeom &geom, const UwItem *items, const int *begin,
                   const int *end, int cap, const uwspr_b200_candidate_t *cands, int jig_first, int jig_count,
                   uwspr_b200_refined_t *refined, uwspr_b200_jiggle_t *jig, uint8_t *soft, int slice0,
                   const UwFineWork &w, const UwFineLaunch &l, cudaStream_t s);
// uwspr_b200_coarse_fine over nchan channels of device-resident samples, wins_per_chan windows each (window
// c*wins_per_chan + k at samples + 2*(c*chan_stride + k*win_stride) floats), all jiggles' results left on the device
// for uwspr_b200_decode_device; npk / cands are host outputs in that channel-major window order (capi.cu)
int uw_coarse_fine_channels(uwspr_b200_ctx *ctx, const float *samples, int64_t win_stride, int wins_per_chan,
                            int64_t chan_stride, int nchan, int jig_first, int jig_count, int32_t *npk,
                            uwspr_b200_candidate_t *cands, int cap, int32_t *total);
// kernel launches a front-end stream has issued (frontend.cu)
int64_t uw_frontend_stream_launches(const uwspr_b200_frontend_stream *s);
size_t uw_coarse_smem_bytes(const UwDims &d);
int uw_coarse_setup(const UwDims &d);
// reserves the fine kernels' shared memory and fills *l for a device of sm_count SMs; nonzero on failure
int uw_fine_setup(int sm_count, bool lag_share, bool reuse, UwFineLaunch *l);
int uw_coarse_blocks_per_sm(const UwDims &d);
// the Fano decoder (fano.cu).  Candidate form: task list, decoder tasks and per-candidate reduction over
// refined[ncand], jig/soft[ncand][jig_count]; workspaces first_ok[ncand], tasks/task_cycles/task_msg
// [ncand*jig_count], counters[2]; grid = resident blocks of the decoder kernel.
void uw_launch_fano_candidates(const uwspr_b200_refined_t *refined, const uwspr_b200_jiggle_t *jig, const uint8_t *soft,
                               int ncand, int jig_count, const short *mettab, int *first_ok, int *tasks, int *counters,
                               uint32_t *task_cycles, unsigned long long *task_msg, int grid, uint8_t *decoded,
                               int8_t *msg7, int32_t *idt_used, uint32_t *fano_cycles, cudaStream_t s);
// raw form: n rows of 162 de-interleaved symbols -> uwspr_b200_fano's outputs per row
void uw_launch_fano_rows(const uint8_t *symbols, int n, int nbits, int delta, uint32_t maxcycles, const short *mettab,
                         int32_t *status, uint32_t *metric, uint32_t *cycles, uint32_t *maxnp, uint8_t *data11, cudaStream_t s);
int uw_fano_setup();
int uw_fano_blocks_per_sm();
