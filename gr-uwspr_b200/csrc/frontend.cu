// Front-end ahead of the hot path (SURVEY 8(f) row 4): real audio at fs_in (12 kHz in the
// reference flowgraphs) -> mix down by fc -> FIR low-pass -> keep every `decim`-th sample ->
// complex64 at 375 sps, the stream uwspr.sliding_window_stream_to_pdu consumes.
//
// In the reference this is done by stock GNU Radio blocks, not by gr-uwspr code
// (examples/WaveFilePlusNoiseDecode.grc:834-958 two freq_xlating_fft_filter_ccc, :1753-1810
// rational_resampler decim 32).  One translating decimating FIR with caller-supplied taps
// replaces the cascade:
//
//     y[m] = sum_k taps[k] * x[n - k] * exp(-2 pi i fc (n - k) / fs_in),  n = m * decim + delay
//
// with x[n] = 0 outside [0, n_in) (the zero history of a GNU Radio FIR).  It pays off when many
// channels of audio are already on the device (the 64-hydrophone array of BASELINE.json
// configs[4]): the 375-sps output feeds uwspr_b200_coarse_fine as a device pointer.
// taps may be complex (uwspr_b200_frontend_ctaps): the flowgraph's cascade - real band-pass around fc,
// translate by fc + low-pass, rational resampler 1/32 - collapses into one complex composite filter
// (h_bp[k] e^{-i w k}) * h_lp * h_rs applied to the mixed-down input (uwspr_b200/binding.py flowgraph_taps).
// GNU Radio itself is not available here: oracle/gr_frontend.py restates its blocks one by one in
// float64 from their published algorithms (gr-filter 3.7: firdes, freq_xlating_fft_filter, rational_resampler)
// and the GPU test compares this kernel with that chain; tests/test_gpu_parity.py also checks the formula above
// against a float64 numpy evaluation.
#include <algorithm>
#include <string>

#include "common.cuh"

namespace {

constexpr int kFeOut = 64;      // outputs per CTA
constexpr int kFeThreads = 256; // 8 warps x 8 outputs

// sample r of channel chan of a buffer in the input format (the conversion of blocks_wavfile_source for int16)
__device__ __forceinline__ float fe_load(const void *p, int fmt, long long chan_stride, int chan, long long r)
{
    const long long i = (long long)chan * chan_stride + r;
    return fmt ? (float)reinterpret_cast<const short *>(p)[i] * (1.0f / 32768.0f) : reinterpret_cast<const float *>(p)[i];
}

// Outputs m_first + [0, n_out) of every channel.  Input sample n (absolute index from the start of the stream) is
// audio[n - base] for base <= n < base + n_in, hist[n - base + nhist] for base - nhist <= n < base, else 0.
// The one-shot front-end is base = 0, nhist = 0, m_first = 0.  Everything an output computes depends on n alone
// (the sample, the oscillator phase from the absolute index, the position in the tap sum), so a stream pushed in
// pieces produces the one-shot's outputs bit for bit.
template <bool CTAPS>
__global__ void __launch_bounds__(kFeThreads)
k_frontend(const void *__restrict__ audio, int fmt, long long chan_stride, long long n_in, long long base,
           const void *__restrict__ hist, long long hist_stride, int nhist,
           const float *__restrict__ taps, int ntaps, int decim, int delay, double cyc_per_sample,
           float2 *__restrict__ out, long long out_stride, long long m_first, long long n_out)
{
    extern __shared__ __align__(16) unsigned char fe_smem[];
    float2 *z = reinterpret_cast<float2 *>(fe_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long m0 = m_first + (long long)blockIdx.x * kFeOut;
    const int chan = blockIdx.y;
    const int span = (kFeOut - 1) * decim + ntaps;
    const long long nb = m0 * decim + delay - (ntaps - 1);   // input index of z[0]
    for (int t = tid; t < span; t += kFeThreads) {
        const long long n = nb + t, r = n - base;
        float v = 0.0f;
        if (r >= 0 && r < n_in) v = fe_load(audio, fmt, chan_stride, chan, r);
        else if (r < 0 && r >= -nhist) v = fe_load(hist, fmt, hist_stride, chan, r + nhist);
        // local oscillator exp(-2 pi i fc n / fs): the phase in turns, reduced in double
        double turns = (double)n * cyc_per_sample;
        turns -= floor(turns);
        double sn, cs;
        sincospi(2.0 * turns, &sn, &cs);
        z[t] = make_float2(v * (float)cs, -v * (float)sn);
    }
    __syncthreads();
    float2 acc[8];
#pragma unroll
    for (int o = 0; o < 8; o++) acc[o] = make_float2(0.0f, 0.0f);
    const float2 *zw = z + (warp * 8) * decim + (ntaps - 1);
    for (int k = lane; k < ntaps; k += 32) {
        const float h = CTAPS ? __ldg(taps + 2 * k) : __ldg(taps + k);
        const float hi = CTAPS ? __ldg(taps + 2 * k + 1) : 0.0f;
#pragma unroll
        for (int o = 0; o < 8; o++) {
            const float2 s = zw[o * decim - k];
            acc[o].x = fmaf(h, s.x, acc[o].x);
            acc[o].y = fmaf(h, s.y, acc[o].y);
            if (CTAPS) {
                acc[o].x = fmaf(-hi, s.y, acc[o].x);
                acc[o].y = fmaf(hi, s.x, acc[o].y);
            }
        }
    }
#pragma unroll
    for (int o = 0; o < 8; o++) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            acc[o].x += __shfl_xor_sync(0xffffffffu, acc[o].x, d);
            acc[o].y += __shfl_xor_sync(0xffffffffu, acc[o].y, d);
        }
        const long long m = m0 - m_first + warp * 8 + o;
        if (lane == 0 && m < n_out) out[(long long)chan * out_stride + m] = acc[o];
    }
}

void launch_frontend(bool ctaps, int nchan, size_t smem, cudaStream_t st, const void *audio, int fmt, long long chan_stride,
                     long long n_in, long long base, const void *hist, long long hist_stride, int nhist, const float *taps,
                     int ntaps, int decim, int delay, double cyc, float2 *out, long long out_stride, long long m_first,
                     long long n_out)
{
    const dim3 grid((unsigned)((n_out + kFeOut - 1) / kFeOut), (unsigned)nchan);
    if (ctaps)
        k_frontend<true><<<grid, kFeThreads, smem, st>>>(audio, fmt, chan_stride, n_in, base, hist, hist_stride, nhist, taps,
                                                         ntaps, decim, delay, cyc, out, out_stride, m_first, n_out);
    else
        k_frontend<false><<<grid, kFeThreads, smem, st>>>(audio, fmt, chan_stride, n_in, base, hist, hist_stride, nhist, taps,
                                                          ntaps, decim, delay, cyc, out, out_stride, m_first, n_out);
}

thread_local std::string g_fe_error;

int fe_fail(int st, const std::string &msg)
{
    g_fe_error = msg;
    return st;
}

// *smem: shared memory one CTA stages; E_PARAM when it does not fit the device
int smem_fits(int device, int ntaps, int decim, size_t *smem)
{
    *smem = ((size_t)(kFeOut - 1) * decim + ntaps) * sizeof(float2);
    int optin = 0;
    cudaError_t e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess && *smem <= (size_t)optin) {
        e = cudaFuncSetAttribute(k_frontend<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_frontend<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    }
    if (e != cudaSuccess) return fe_fail(UWSPR_B200_E_CUDA, std::string("front-end set-up: ") + cudaGetErrorString(e));
    if (*smem > (size_t)optin) return fe_fail(UWSPR_B200_E_PARAM, "ntaps + 63*decim samples do not fit shared memory");
    return UWSPR_B200_OK;
}

bool fe_args_ok(int nchan, int fmt, int ntaps, int decim, int delay, double fs_in)
{
    return nchan >= 1 && nchan <= 65535 && ntaps >= 1 && ntaps <= 16384 && decim >= 1 && decim <= 4096 && delay >= 0 &&
           fs_in > 0.0 && (fmt == 0 || fmt == 1);
}

}  // namespace

#define FE_CU(call)                                                                                \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            if (d_audio_own) cudaFree(d_audio_own);                                                \
            if (d_out_own) cudaFree(d_out_own);                                                    \
            if (d_taps) cudaFree(d_taps);                                                          \
            return fe_fail(UWSPR_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
        }                                                                                          \
    } while (0)

extern "C" const char *uwspr_b200_frontend_error(void) { return g_fe_error.c_str(); }

static int frontend_impl(bool ctaps, int device, const void *audio, int fmt, int space_in, int64_t chan_stride, int nchan,
                         int64_t n_in, const float *taps, int ntaps, int decim, int delay, double fc,
                         double fs_in, float *out, int space_out, int64_t out_stride, int64_t *n_out_p)
{
    if (!audio || !taps || !out || nchan < 1 || n_in < 1 || ntaps < 1 || ntaps > 16384 || decim < 1 || decim > 4096 ||
        delay < 0 || !(fs_in > 0.0) || (fmt != 0 && fmt != 1) || chan_stride < n_in)
        return fe_fail(UWSPR_B200_E_PARAM, "bad front-end arguments");
    if (nchan > 65535) return fe_fail(UWSPR_B200_E_PARAM, "more than 65535 channels in one call (grid.y limit)");
    const int64_t n_out = n_in / decim;
    if (n_out_p) *n_out_p = n_out;
    if (n_out == 0) return UWSPR_B200_OK;
    if (out_stride < n_out) return fe_fail(UWSPR_B200_E_PARAM, "out_stride shorter than the output");
    void *d_audio_own = nullptr, *d_out_own = nullptr;
    float *d_taps = nullptr;
    FE_CU(cudaSetDevice(device));
    const size_t esz = fmt ? sizeof(short) : sizeof(float);
    const void *d_audio = audio;
    if (space_in == UWSPR_B200_HOST) {
        const size_t bytes = ((size_t)(nchan - 1) * (size_t)chan_stride + (size_t)n_in) * esz;
        FE_CU(cudaMalloc(&d_audio_own, bytes));
        FE_CU(cudaMemcpy(d_audio_own, audio, bytes, cudaMemcpyHostToDevice));
        d_audio = d_audio_own;
    }
    float2 *d_out = reinterpret_cast<float2 *>(out);
    const size_t out_bytes = ((size_t)(nchan - 1) * (size_t)out_stride + (size_t)n_out) * sizeof(float2);
    if (space_out == UWSPR_B200_HOST) {
        FE_CU(cudaMalloc(&d_out_own, out_bytes));
        d_out = reinterpret_cast<float2 *>(d_out_own);
    }
    const size_t tap_bytes = sizeof(float) * (size_t)ntaps * (ctaps ? 2 : 1);
    FE_CU(cudaMalloc(&d_taps, tap_bytes));
    FE_CU(cudaMemcpy(d_taps, taps, tap_bytes, cudaMemcpyHostToDevice));
    size_t smem = 0;
    const int fit = smem_fits(device, ntaps, decim, &smem);
    if (fit != UWSPR_B200_OK) {
        cudaFree(d_taps);
        if (d_audio_own) cudaFree(d_audio_own);
        if (d_out_own) cudaFree(d_out_own);
        return fit;
    }
    launch_frontend(ctaps, nchan, smem, 0, d_audio, fmt, (long long)chan_stride, (long long)n_in, 0, nullptr, 0, 0, d_taps, ntaps,
                    decim, delay, fc / fs_in, d_out, (long long)out_stride, 0, (long long)n_out);
    FE_CU(cudaGetLastError());
    if (space_out == UWSPR_B200_HOST)
        // channel by channel: the caller's memory between two channels (out_stride > n_out) is not touched
        FE_CU(cudaMemcpy2D(out, (size_t)out_stride * sizeof(float2), d_out_own, (size_t)out_stride * sizeof(float2),
                           (size_t)n_out * sizeof(float2), (size_t)nchan, cudaMemcpyDeviceToHost));
    else
        FE_CU(cudaDeviceSynchronize());
    cudaFree(d_taps);
    if (d_audio_own) cudaFree(d_audio_own);
    if (d_out_own) cudaFree(d_out_own);
    return UWSPR_B200_OK;
}

extern "C" int uwspr_b200_frontend(int device, const void *audio, int fmt, int space_in, int64_t chan_stride, int nchan,
                                   int64_t n_in, const float *taps, int ntaps, int decim, int delay, double fc,
                                   double fs_in, float *out, int space_out, int64_t out_stride, int64_t *n_out_p)
{
    return frontend_impl(false, device, audio, fmt, space_in, chan_stride, nchan, n_in, taps, ntaps, decim, delay, fc, fs_in, out,
                         space_out, out_stride, n_out_p);
}

extern "C" int uwspr_b200_frontend_ctaps(int device, const void *audio, int fmt, int space_in, int64_t chan_stride, int nchan,
                                         int64_t n_in, const float *taps_iq, int ntaps, int decim, int delay, double fc,
                                         double fs_in, float *out, int space_out, int64_t out_stride, int64_t *n_out_p)
{
    return frontend_impl(true, device, audio, fmt, space_in, chan_stride, nchan, n_in, taps_iq, ntaps, decim, delay, fc, fs_in, out,
                         space_out, out_stride, n_out_p);
}

// ---- the same kernel as a stream ------------------------------------------------------------------------------------
// State per channel: the last ntaps - 1 + decim input samples (in the input format) and the count of samples pushed.
// Output m reads x[n - k], n = m*decim + delay, 0 <= k < ntaps: once every sample up to n has been pushed it is
// computed from the current piece and the history, and nothing older than ntaps - 1 samples before the first
// sample of a push is needed again.
namespace {
constexpr int64_t kFePiece = 1 << 18;   // input samples per channel per launch: bounds the staging buffers
}

struct uwspr_b200_frontend_stream {
    int device = 0, nchan = 0, fmt = 0, ntaps = 0, decim = 0, delay = 0;
    bool ctaps = false, broken = false;
    double cyc = 0.0;
    size_t esz = 0, smem = 0;
    int64_t hist_cap = 0, nhist = 0;   // history capacity and valid samples per channel
    int64_t n_total = 0, m_next = 0;   // input samples pushed, outputs produced (per channel)
    int64_t out_pitch = 0, launches = 0;
    float *taps = nullptr;
    void *in = nullptr;                // host-fed piece [nchan][kFePiece]
    float2 *out = nullptr;             // outputs of a piece bound for the host [nchan][out_pitch]
    void *hist[2] = { nullptr, nullptr };
    int cur = 0;
    cudaStream_t st = nullptr;

    int64_t outputs_below(int64_t n) const { return n > delay ? (n - delay + decim - 1) / decim : 0; }
};

extern "C" void uwspr_b200_frontend_stream_destroy(uwspr_b200_frontend_stream *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->st) cudaStreamSynchronize(s->st);
    void *ptrs[] = { s->taps, s->in, s->out, s->hist[0], s->hist[1] };
    for (void *q : ptrs)
        if (q) cudaFree(q);
    if (s->st) cudaStreamDestroy(s->st);
    delete s;
}

extern "C" int uwspr_b200_frontend_stream_create(int device, int nchan, int fmt, const float *taps, int ntaps, int complex_taps,
                                                 int decim, int delay, double fc, double fs_in, uwspr_b200_frontend_stream **out)
{
    if (!out) return fe_fail(UWSPR_B200_E_PARAM, "NULL output pointer");
    *out = nullptr;
    if (!taps || !fe_args_ok(nchan, fmt, ntaps, decim, delay, fs_in)) return fe_fail(UWSPR_B200_E_PARAM, "bad front-end arguments");
    uwspr_b200_frontend_stream *s = new uwspr_b200_frontend_stream();
    s->device = device;
    s->nchan = nchan;
    s->fmt = fmt;
    s->ntaps = ntaps;
    s->decim = decim;
    s->delay = delay;
    s->ctaps = complex_taps != 0;
    s->cyc = fc / fs_in;
    s->esz = fmt ? sizeof(short) : sizeof(float);
    s->hist_cap = (int64_t)ntaps - 1 + decim;
    s->out_pitch = kFePiece / decim + 1;
    auto bail = [&](int st) {
        uwspr_b200_frontend_stream_destroy(s);
        return st;
    };
#define FS_CU(call)                                                                                             \
    do {                                                                                                        \
        cudaError_t e_ = (call);                                                                                \
        if (e_ != cudaSuccess) return bail(fe_fail(UWSPR_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_))); \
    } while (0)
    FS_CU(cudaSetDevice(device));
    const int fit = smem_fits(device, ntaps, decim, &s->smem);
    if (fit != UWSPR_B200_OK) return bail(fit);
    const size_t tap_bytes = sizeof(float) * (size_t)ntaps * (s->ctaps ? 2 : 1);
    FS_CU(cudaMalloc(&s->taps, tap_bytes));
    FS_CU(cudaMemcpy(s->taps, taps, tap_bytes, cudaMemcpyHostToDevice));
    FS_CU(cudaMalloc(&s->in, (size_t)nchan * kFePiece * s->esz));
    FS_CU(cudaMalloc(&s->out, (size_t)nchan * s->out_pitch * sizeof(float2)));
    for (int q = 0; q < 2; q++) FS_CU(cudaMalloc(&s->hist[q], (size_t)nchan * s->hist_cap * s->esz));
    FS_CU(cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking));
#undef FS_CU
    *out = s;
    return UWSPR_B200_OK;
}

extern "C" int64_t uwspr_b200_frontend_stream_outputs(const uwspr_b200_frontend_stream *s) { return s ? s->m_next : 0; }

int64_t uw_frontend_stream_launches(const uwspr_b200_frontend_stream *s) { return s ? s->launches : 0; }

static int stream_push(uwspr_b200_frontend_stream *s, const char *audio, bool host_in, int64_t chan_stride, int64_t n_in,
                       float2 *out, bool host_out, int64_t out_stride)
{
#define SP_CU(call)                                                                                          \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess) return fe_fail(UWSPR_B200_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)
    SP_CU(cudaSetDevice(s->device));
    const size_t esz = s->esz, C = (size_t)s->nchan;
    int64_t written = 0;
    for (int64_t off = 0; off < n_in; off += kFePiece) {
        const int64_t n = std::min(kFePiece, n_in - off);
        const char *src = audio + (size_t)off * esz;
        int64_t sstride = chan_stride;
        if (host_in) {
            SP_CU(cudaMemcpy2DAsync(s->in, kFePiece * esz, src, (size_t)chan_stride * esz, (size_t)n * esz, C,
                                    cudaMemcpyHostToDevice, s->st));
            src = static_cast<const char *>(s->in);
            sstride = kFePiece;
        }
        const int64_t m_end = s->outputs_below(s->n_total + n), cnt = m_end - s->m_next;
        if (cnt > 0) {
            float2 *dst = host_out ? s->out : out + written;
            launch_frontend(s->ctaps, s->nchan, s->smem, s->st, src, s->fmt, sstride, n, s->n_total, s->hist[s->cur], s->hist_cap,
                            (int)s->nhist, s->taps, s->ntaps, s->decim, s->delay, s->cyc, dst, host_out ? s->out_pitch : out_stride,
                            s->m_next, cnt);
            s->launches++;
            SP_CU(cudaGetLastError());
            if (host_out)
                SP_CU(cudaMemcpy2DAsync(out + written, (size_t)out_stride * sizeof(float2), s->out, (size_t)s->out_pitch * sizeof(float2),
                                        (size_t)cnt * sizeof(float2), C, cudaMemcpyDeviceToHost, s->st));
            written += cnt;
            s->m_next = m_end;
        }
        // the new history is the last `keep` samples of (old history, this piece), written to the other buffer
        const int64_t keep = std::min(s->hist_cap, s->nhist + n), from_old = std::max<int64_t>(0, keep - n);
        char *h_new = static_cast<char *>(s->hist[s->cur ^ 1]);
        const char *h_old = static_cast<const char *>(s->hist[s->cur]);
        const size_t hp = (size_t)s->hist_cap * esz;
        if (from_old > 0)
            SP_CU(cudaMemcpy2DAsync(h_new, hp, h_old + (size_t)(s->nhist - from_old) * esz, hp, (size_t)from_old * esz, C,
                                    cudaMemcpyDeviceToDevice, s->st));
        SP_CU(cudaMemcpy2DAsync(h_new + (size_t)from_old * esz, hp, src + (size_t)(n - (keep - from_old)) * esz, (size_t)sstride * esz,
                                (size_t)(keep - from_old) * esz, C, cudaMemcpyDeviceToDevice, s->st));
        s->cur ^= 1;
        s->nhist = keep;
        s->n_total += n;
    }
    SP_CU(cudaStreamSynchronize(s->st));
#undef SP_CU
    return UWSPR_B200_OK;
}

extern "C" int uwspr_b200_frontend_stream_push(uwspr_b200_frontend_stream *s, const void *audio, int space_in, int64_t chan_stride,
                                               int64_t n_in, float *out, int space_out, int64_t out_stride, int64_t out_cap,
                                               int64_t *n_out)
{
    if (n_out) *n_out = 0;
    if (!s || n_in < 0 || (n_in > 0 && !audio) || (space_in != UWSPR_B200_HOST && space_in != UWSPR_B200_DEVICE) ||
        (space_out != UWSPR_B200_HOST && space_out != UWSPR_B200_DEVICE) || chan_stride < n_in || out_cap < 0 ||
        out_stride < out_cap)   // the strides are also the pitches of the 2-D copies, one channel included
        return fe_fail(UWSPR_B200_E_PARAM, "bad front-end stream arguments");
    if (s->broken) return fe_fail(UWSPR_B200_E_STATE, "an earlier push failed: the stream's state is lost");
    const int64_t cnt = s->outputs_below(s->n_total + n_in) - s->m_next;
    if (cnt > 0 && !out) return fe_fail(UWSPR_B200_E_PARAM, "NULL output buffer");
    if (cnt > out_cap) return fe_fail(UWSPR_B200_E_CAPACITY, "the push produces more outputs than out_cap");
    if (n_in == 0) return UWSPR_B200_OK;
    const int rc = stream_push(s, static_cast<const char *>(audio), space_in == UWSPR_B200_HOST, chan_stride, n_in,
                               reinterpret_cast<float2 *>(out), space_out == UWSPR_B200_HOST, out_stride);
    if (rc != UWSPR_B200_OK) {
        s->broken = true;
        cudaStreamSynchronize(s->st);
        cudaGetLastError();
        return rc;
    }
    if (n_out) *n_out = cnt;
    return UWSPR_B200_OK;
}
