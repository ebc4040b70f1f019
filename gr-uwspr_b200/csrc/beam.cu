// Narrowband delay-and-sum beamformer at complex baseband (k_beamform): B beams from C channels of 375-sps streams,
//
//     y_b[n] = sum_{c=0}^{C-1} w[b][c] * x_c[n - d[b][c]],   x_c[m] = 0 for m < 0,
//
// w complex, d an integer sample delay in [0, 8192].  After the front-end's mix-down by fc, a passband delay tau is an
// envelope delay plus the phase e^{-i 2 pi fc tau}: integer delays and complex weights steer any geometry to within
// half a sample of envelope error (1.3 ms at 375 sps, against a 683 ms symbol).
//
// Fixed arithmetic.  The accumulator of output (b, n) starts at (0, 0) and adds the channels in ascending c, each as
//     re = fmaf(wr, xr, re); re = fmaf(-wi, xi, re); im = fmaf(wr, xi, im); im = fmaf(wi, xr, im);
// The operands are w[b][c] and x_c[n - d[b][c]] (0 when n - d < 0) and nothing else, so output (b, n) depends only on
// (b, n) and the inputs: not on the tile or beam group it falls in, the launch it belongs to, how many outputs a launch
// makes, or where x_c[n - d] was read from (the current piece of a stream or the history kept from earlier pieces).
// That is the argument of k_frontend's stream form (DESIGN 7.1): a stream pushed in any split produces the one-shot's
// outputs bit for bit.  Tensor cores would reorder the sum; the kernel is bound by memory and latency, not by the fp32
// pipe, so it keeps the scalar fmaf chain.
//
// Layout.  One CTA of 256 threads per (tile of kTile = 128 outputs, group of kGroup = 32 beams).  Warp v owns beams
// 4v .. 4v+3 of the group and lane l outputs n0 + l + 32 r, r = 0..3: 16 complex accumulators per thread.  Channels go
// through shared memory one after another, double-buffered with 8-byte cp.async: for channel c the CTA stages the
// group's 32 weights and delays and the segment x_c[h + n0 - dhi, h + n0 + kTile - dlo), where [dlo, dhi] is the
// range of the group's delays on that channel (precomputed on the host).  Segments start at any sample, so TMA's
// 16-byte alignment does not hold; cp.async's source size of 0 zero-fills the samples before the start of the stream
// and past the end of the launch's input in the same instruction.  The lanes of a warp read 32 consecutive samples
// (two wavefronts per 8-byte load) and one broadcast weight.  Shared memory per CTA is 2 x (kTile + max span) samples
// plus the tables, sized per launch: a few KB for an array's fan of beams, 130 KB when a group's delays on one channel
// span all of [0, 8192].  Weights never have to fit shared memory as a whole: a CTA holds one channel's at a time.
#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"

namespace {

constexpr int kTile = 128;      // outputs per CTA
constexpr int kGroup = 32;      // beams per CTA
constexpr int kThreads = 256;   // 8 warps x 4 beams
constexpr int kPerLane = kTile / 32;
constexpr int kBeamsPerWarp = kGroup / (kThreads / 32);

__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
// 8 bytes global -> shared; ok == false writes zeros and reads nothing
__device__ __forceinline__ void cp8(void *dst, const void *src, bool ok)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_addr(dst)), "l"(src), "r"(ok ? 8 : 0) : "memory");
}
__device__ __forceinline__ void cp4(void *dst, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One stage: the group's weights and delays on one channel, then the channel's segment.
struct StageHead {
    float2 w[kGroup];
    int d[kGroup];
};

// in: channel c at in + c*in_stride; output j of the launch reads in-buffer index h + j - d (zero below 0 and at or
// above h + n_out).  w, d: [group][nchan][kGroup] (padding beams have w = 0, d = dlo); span: [group][nchan] (dlo, dhi).
__global__ void __launch_bounds__(kThreads)
k_beamform(const float2 *__restrict__ in, long long in_stride, long long h, int nchan, const float2 *__restrict__ w,
           const int *__restrict__ d, const int2 *__restrict__ span, int maxspan, int nbeam, float2 *__restrict__ out,
           long long out_stride, long long n_out)
{
    extern __shared__ __align__(16) unsigned char bf_smem[];
    const int seg = kTile + maxspan;
    const size_t stage_bytes = sizeof(StageHead) + (size_t)seg * sizeof(float2);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n0 = (long long)blockIdx.x * kTile;
    const int grp = blockIdx.y;
    const long long qend = h + n_out;   // first in-buffer index past the launch's input

    auto stage = [&](int c, int buf) {
        unsigned char *base = bf_smem + buf * stage_bytes;
        StageHead *hd = reinterpret_cast<StageHead *>(base);
        float2 *xs = reinterpret_cast<float2 *>(base + sizeof(StageHead));
        const size_t t = (size_t)grp * nchan + c;
        if (tid < kGroup) cp8(&hd->w[tid], w + t * kGroup + tid, true);
        else if (tid < 2 * kGroup) cp4(&hd->d[tid - kGroup], d + t * kGroup + tid - kGroup);
        const int2 s = span[t];
        const long long q0 = h + n0 - s.y;
        const int cnt = kTile + s.y - s.x;
        const float2 *row = in + (long long)c * in_stride;
        for (int i = tid; i < cnt; i += kThreads) {
            const long long q = q0 + i;
            const bool ok = q >= 0 && q < qend;
            cp8(xs + i, ok ? row + q : row, ok);
        }
    };

    float2 acc[kBeamsPerWarp][kPerLane];
#pragma unroll
    for (int k = 0; k < kBeamsPerWarp; k++)
#pragma unroll
        for (int r = 0; r < kPerLane; r++) acc[k][r] = make_float2(0.0f, 0.0f);
    const int b_first = grp * kGroup + warp * kBeamsPerWarp;   // this warp's first beam
    const int nb_warp = min(kBeamsPerWarp, nbeam - b_first);   // <= 0: padding warp, it only stages

    stage(0, 0);
    cp_commit();
    for (int c = 0; c < nchan; c++) {
        const int buf = c & 1;
        if (c + 1 < nchan) stage(c + 1, buf ^ 1);
        cp_commit();
        cp_wait<1>();
        __syncthreads();
        const unsigned char *base = bf_smem + buf * stage_bytes;
        const StageHead *hd = reinterpret_cast<const StageHead *>(base);
        const float2 *xs = reinterpret_cast<const float2 *>(base + sizeof(StageHead));
        const int dhi = span[(size_t)grp * nchan + c].y;
#pragma unroll
        for (int k = 0; k < kBeamsPerWarp; k++) {
            if (k < nb_warp) {
                const float2 wv = hd->w[warp * kBeamsPerWarp + k];
                const float nwi = -wv.y;
                // output n0 + j reads segment slot j + dhi - d
                const float2 *xb = xs + (dhi - hd->d[warp * kBeamsPerWarp + k]) + lane;
#pragma unroll
                for (int r = 0; r < kPerLane; r++) {
                    const float2 x = xb[32 * r];
                    acc[k][r].x = fmaf(wv.x, x.x, acc[k][r].x);
                    acc[k][r].x = fmaf(nwi, x.y, acc[k][r].x);
                    acc[k][r].y = fmaf(wv.x, x.y, acc[k][r].y);
                    acc[k][r].y = fmaf(wv.y, x.x, acc[k][r].y);
                }
            }
        }
        __syncthreads();   // the buffer is staged again two channels on
    }
#pragma unroll
    for (int k = 0; k < kBeamsPerWarp; k++) {
        if (k >= nb_warp) continue;
        float2 *o = out + (long long)(b_first + k) * out_stride;
#pragma unroll
        for (int r = 0; r < kPerLane; r++) {
            const long long n = n0 + lane + 32 * r;
            if (n < n_out) o[n] = acc[k][r];
        }
    }
}

}  // namespace

int uw_beams_check(int nchan, const float *weights, const int32_t *delays, int nbeam)
{
    if (!weights || !delays || nchan < 1 || nchan > 1024 || nbeam < 1 || nbeam > 1024) return UWSPR_B200_E_PARAM;
    const size_t n = (size_t)nbeam * nchan;
    for (size_t i = 0; i < n; i++) {
        if (!std::isfinite(weights[2 * i]) || !std::isfinite(weights[2 * i + 1])) return UWSPR_B200_E_PARAM;
        if (delays[i] < 0 || delays[i] > UW_BEAM_MAX_DELAY) return UWSPR_B200_E_PARAM;
    }
    return UWSPR_B200_OK;
}

cudaError_t uw_beams_upload(UwBeams *b, int nchan, const float *weights, const int32_t *delays, int nbeam)
{
    const int ngroup = (nbeam + kGroup - 1) / kGroup;
    const size_t nt = (size_t)ngroup * nchan;
    std::vector<float2> w(nt * kGroup, make_float2(0.0f, 0.0f));
    std::vector<int> d(nt * kGroup, 0);
    std::vector<int2> span(nt);
    int maxspan = 0, dmax = 0;
    for (int g = 0; g < ngroup; g++)
        for (int c = 0; c < nchan; c++) {
            const size_t t = (size_t)g * nchan + c;
            int lo = INT32_MAX, hi = 0;
            for (int k = 0; k < kGroup && g * kGroup + k < nbeam; k++) {
                const size_t i = (size_t)(g * kGroup + k) * nchan + c;
                w[t * kGroup + k] = make_float2(weights[2 * i], weights[2 * i + 1]);
                d[t * kGroup + k] = delays[i];
                lo = std::min(lo, (int)delays[i]);
                hi = std::max(hi, (int)delays[i]);
            }
            for (int k = nbeam - g * kGroup; k < kGroup; k++) d[t * kGroup + k] = lo;   // padding beams: never read
            span[t] = make_int2(lo, hi);
            maxspan = std::max(maxspan, hi - lo);
            dmax = std::max(dmax, hi);
        }
    *b = UwBeams();
    b->nbeam = nbeam;
    b->nchan = nchan;
    b->ngroup = ngroup;
    b->maxspan = maxspan;
    b->dmax = dmax;
    cudaError_t e = cudaMalloc(&b->w, w.size() * sizeof(float2));
    if (e == cudaSuccess) e = cudaMalloc(&b->d, d.size() * sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc(&b->span, span.size() * sizeof(int2));
    if (e == cudaSuccess) e = cudaMemcpy(b->w, w.data(), w.size() * sizeof(float2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(b->d, d.data(), d.size() * sizeof(int), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(b->span, span.data(), span.size() * sizeof(int2), cudaMemcpyHostToDevice);
    b->smem = 2 * (sizeof(StageHead) + (size_t)(kTile + maxspan) * sizeof(float2));
    // opt in to the largest any delay matrix needs (133 888 bytes), so that beam sets of any size share the kernel
    const size_t most = 2 * (sizeof(StageHead) + (size_t)(kTile + UW_BEAM_MAX_DELAY) * sizeof(float2));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_beamform, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most);
    if (e != cudaSuccess) uw_beams_free(b);
    return e;
}

void uw_beams_free(UwBeams *b)
{
    if (b->w) cudaFree(b->w);
    if (b->d) cudaFree(b->d);
    if (b->span) cudaFree(b->span);
    *b = UwBeams();
}

void uw_launch_beamform(const UwBeams &b, const float2 *in, long long in_stride, long long h, float2 *out,
                        long long out_stride, long long n_out, cudaStream_t s)
{
    const dim3 grid((unsigned)((n_out + kTile - 1) / kTile), (unsigned)b.ngroup);
    k_beamform<<<grid, kThreads, b.smem, s>>>(in, in_stride, h, b.nchan, b.w, b.d, b.span, b.maxspan, b.nbeam, out,
                                              out_stride, n_out);
}

#define BF_CU(call)                                                                                  \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            if (d_in_own) cudaFree(d_in_own);                                                        \
            if (d_out_own) cudaFree(d_out_own);                                                      \
            uw_beams_free(&bm);                                                                      \
            return UWSPR_B200_E_CUDA;                                                                \
        }                                                                                            \
    } while (0)

extern "C" int uwspr_b200_beamform(int device, const float *in, int space_in, int64_t in_stride, int nchan, int64_t n,
                                   const float *weights, const int32_t *delays, int nbeam, float *out, int space_out,
                                   int64_t out_stride)
{
    if (!in || !out || n < 0 || in_stride < n || out_stride < n || (space_in != UWSPR_B200_HOST && space_in != UWSPR_B200_DEVICE) ||
        (space_out != UWSPR_B200_HOST && space_out != UWSPR_B200_DEVICE) || uw_beams_check(nchan, weights, delays, nbeam))
        return UWSPR_B200_E_PARAM;
    if (n == 0) return UWSPR_B200_OK;
    void *d_in_own = nullptr, *d_out_own = nullptr;
    UwBeams bm;
    BF_CU(cudaSetDevice(device));
    const float2 *d_in = reinterpret_cast<const float2 *>(in);
    if (space_in == UWSPR_B200_HOST) {
        const size_t bytes = ((size_t)(nchan - 1) * (size_t)in_stride + (size_t)n) * sizeof(float2);
        BF_CU(cudaMalloc(&d_in_own, bytes));
        BF_CU(cudaMemcpy(d_in_own, in, bytes, cudaMemcpyHostToDevice));
        d_in = reinterpret_cast<const float2 *>(d_in_own);
    }
    float2 *d_out = reinterpret_cast<float2 *>(out);
    if (space_out == UWSPR_B200_HOST) {
        BF_CU(cudaMalloc(&d_out_own, ((size_t)(nbeam - 1) * (size_t)out_stride + (size_t)n) * sizeof(float2)));
        d_out = reinterpret_cast<float2 *>(d_out_own);
    }
    BF_CU(uw_beams_upload(&bm, nchan, weights, delays, nbeam));
    uw_launch_beamform(bm, d_in, (long long)in_stride, 0, d_out, (long long)out_stride, (long long)n, 0);
    BF_CU(cudaGetLastError());
    if (space_out == UWSPR_B200_HOST)
        // beam by beam: the caller's memory between two beams (out_stride > n) is not touched
        BF_CU(cudaMemcpy2D(out, (size_t)out_stride * sizeof(float2), d_out_own, (size_t)out_stride * sizeof(float2),
                           (size_t)n * sizeof(float2), (size_t)nbeam, cudaMemcpyDeviceToHost));
    else
        BF_CU(cudaDeviceSynchronize());
    uw_beams_free(&bm);
    if (d_in_own) cudaFree(d_in_own);
    if (d_out_own) cudaFree(d_out_own);
    return UWSPR_B200_OK;
}
