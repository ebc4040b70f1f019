// The receive chain of nchan channels (gr::uwspr::array_receiver, host/blocks.h) and its C entry points,
// uwspr_b200_array_receiver_* and the one-channel uwspr_b200_receiver_*.
//
// Device ring: one complex64 buffer, channel c at c*pitch samples, pitch >= (K-1)*stride + fl + kRingPiece for
// K = batch windows.  Channel c's 375-sps stream from the start of window d_next_window occupies [0, d_fill) of
// its row; the front-end (or the copy of complex input) appends straight into the row.  A batch is one
// coarse_fine submission over the channel-major windows c*K + k at c*pitch + k*stride (uw_coarse_fine_channels),
// then the decoder on the results left on the device.  The unread tail of every row then moves to the front of
// the second buffer, which becomes the ring: source and destination would overlap within one buffer whenever
// the tail is longer than K*stride (41 625 samples at shift 9 s and K = 1).
#include <string.h>

#include <algorithm>
#include <climits>

#include "common.cuh"
#include "blocks.h"

namespace {

// 375-sps samples one append may add per channel beyond a full batch: the ring always has that much room
// when a push piece starts, since every complete batch has been run by then
constexpr int64_t kRingPiece = 16384;

int check_args(const uwspr_b200_params_t *p, const uwspr_b200_input_t *in, int nchan, int shift_seconds, int batch_windows)
{
    if (!p || !in || nchan < 1 || batch_windows < 1 || p->fs <= 0) return UWSPR_B200_E_PARAM;
    const long long stride = (long long)shift_seconds * p->fs;
    if (stride <= 0 || stride > p->fl) return UWSPR_B200_E_PARAM;
    if (in->kind < 0 || in->kind > 2) return UWSPR_B200_E_PARAM;
    if (in->kind > 0) {
        if (!in->taps || in->ntaps < 1 || in->ntaps > 16384 || in->decim < 1 || in->decim > 4096 || in->delay < 0 ||
            !(in->fs_in > 0.0) || in->fs_in / in->decim != (double)p->fs)
            return UWSPR_B200_E_PARAM;
    }
    if ((long long)nchan * batch_windows > INT_MAX / 2) return UWSPR_B200_E_PARAM;
    return UWSPR_B200_OK;
}

void cuda_check(cudaError_t e, const char *what)
{
    if (e != cudaSuccess) throw gr::uwspr::context_error(UWSPR_B200_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

}  // namespace

namespace gr {
namespace uwspr {

array_receiver::array_receiver(const uwspr_b200_params_t &params, const uwspr_b200_input_t &input, int nchan, int shift_seconds,
                               int batch_windows)
{
    int st = check_args(&params, &input, nchan, shift_seconds, batch_windows);
    if (st) throw context_error(st, "bad receiver arguments");
    d_device = params.device;
    d_kind = input.kind;
    d_nchan = nchan;
    d_fl = params.fl;
    d_stride = shift_seconds * params.fs;
    d_batch = batch_windows;
    uwspr_b200_params_t p = params;
    p.max_windows = nchan * batch_windows;
    try {
        st = uwspr_b200_create(&p, &d_ctx);
        if (st) throw context_error(st, uwspr_b200_create_error());
        uwspr_b200_info_t info;
        uwspr_b200_info(d_ctx, &info);
        d_cap = info.max_candidates;
        if (d_kind > 0) {
            d_decim = input.decim;
            st = uwspr_b200_frontend_stream_create(params.device, nchan, d_kind - 1, input.taps, input.ntaps, input.complex_taps,
                                                   input.decim, input.delay, input.fc, input.fs_in, &d_fe);
            if (st) throw context_error(st, uwspr_b200_frontend_error());
        }
        // rows start on 64-sample boundaries: every channel's windows keep the alignment a single stream's have
        d_pitch = ((int64_t)(batch_windows - 1) * d_stride + d_fl + kRingPiece + 63) / 64 * 64;
        cuda_check(cudaSetDevice(params.device), "cudaSetDevice");
        for (int q = 0; q < 2; q++) cuda_check(cudaMalloc(&d_ring[q], (size_t)nchan * d_pitch * sizeof(float2)), "cudaMalloc");
        cudaStream_t s;
        cuda_check(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "cudaStreamCreate");
        d_stream = s;
    } catch (...) {
        release();
        throw;
    }
    d_npk.resize((size_t)nchan * batch_windows);
    d_cands.resize(d_cap);
    d_decoded.resize(d_cap);
    d_blobs.resize((size_t)d_cap * 7);
}

array_receiver::~array_receiver() { release(); }

void array_receiver::release()
{
    if (d_stream) {
        cudaStreamSynchronize(static_cast<cudaStream_t>(d_stream));
        cudaStreamDestroy(static_cast<cudaStream_t>(d_stream));
        d_stream = nullptr;
    }
    for (void *&q : d_ring) {
        if (q) cudaFree(q);
        q = nullptr;
    }
    uwspr_b200_frontend_stream_destroy(d_fe);
    d_fe = nullptr;
    uwspr_b200_destroy(d_ctx);
    d_ctx = nullptr;
}

int64_t array_receiver::launch_count() const { return uwspr_b200_launch_count(d_ctx) + uw_frontend_stream_launches(d_fe); }

void array_receiver::push(const void *data, int space, int64_t chan_stride, int64_t n)
{
    cudaStream_t st = static_cast<cudaStream_t>(d_stream);
    cuda_check(cudaSetDevice(d_device), "cudaSetDevice");
    const size_t esz = d_kind == 0 ? sizeof(float2) : d_kind == 1 ? sizeof(float) : sizeof(short);
    for (int64_t off = 0; off < n;) {
        // the ring has room for kRingPiece samples at least (process() ran every complete batch)
        float2 *row0 = static_cast<float2 *>(d_ring[d_cur]) + d_fill;
        const int64_t room = d_pitch - d_fill;
        const char *src = static_cast<const char *>(data) + (size_t)off * esz;
        int64_t take, got;
        if (d_kind == 0) {
            take = got = std::min(room, n - off);
            cuda_check(cudaMemcpy2DAsync(row0, (size_t)d_pitch * sizeof(float2), src, (size_t)chan_stride * esz,
                                         (size_t)take * sizeof(float2), (size_t)d_nchan,
                                         space == UWSPR_B200_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st),
                       "cudaMemcpy2DAsync");
            cuda_check(cudaStreamSynchronize(st), "cudaStreamSynchronize");
        } else {
            // take samples produce at most ceil(take / decim) <= room outputs
            take = std::min(n - off, room * d_decim);
            const int rc = uwspr_b200_frontend_stream_push(d_fe, src, space, chan_stride, take, reinterpret_cast<float *>(row0),
                                                           UWSPR_B200_DEVICE, d_pitch, room, &got);
            if (rc) throw context_error(rc, uwspr_b200_frontend_error());
        }
        off += take;
        d_fill += got;
        process(false);
    }
}

void array_receiver::flush() { process(true); }

void array_receiver::process(bool all)
{
    for (;;) {
        const int64_t have = d_fill >= d_fl ? 1 + (d_fill - d_fl) / d_stride : 0;
        if (have == 0 || (have < d_batch && !all)) break;
        run_batch((int)std::min<int64_t>(have, d_batch));
    }
}

void array_receiver::run_batch(int nb)
{
    const float *ring = static_cast<const float *>(d_ring[d_cur]);
    int32_t total = 0;
    int st = uw_coarse_fine_channels(d_ctx, ring, d_stride, nb, d_pitch, d_nchan, 0, UWSPR_B200_NJIG, d_npk.data(),
                                     d_cands.data(), d_cap, &total);
    if (st) throw context_error(st, uwspr_b200_last_error(d_ctx));
    const int got = uwspr_b200_decode_device(d_ctx, nullptr, nullptr, nullptr, UWSPR_B200_DEVICE, total, UWSPR_B200_NJIG,
                                             d_decoded.data(), d_blobs.data(), nullptr, nullptr);
    if (got < 0) throw context_error(-got, uwspr_b200_last_error(d_ctx));
    // results are channel-major (window c*nb + k); messages are published window by window, channel by channel
    std::vector<int> base((size_t)d_nchan * nb + 1, 0);
    for (int i = 0; i < d_nchan * nb; i++) base[i + 1] = base[i] + d_npk[i];
    for (int k = 0; k < nb; k++)
        for (int c = 0; c < d_nchan; c++)
            for (int g = base[c * nb + k]; g < base[c * nb + k + 1]; g++) {
                if (!d_decoded[g]) continue;
                message_pdu m;
                memcpy(m.blob, &d_blobs[(size_t)g * 7], 7);
                m.candidate = d_cands[g];
                m.window = d_next_window + k;
                m.channel = c;
                d_msgs.push_back(m);
            }
    // window k = s_c[k*stride, k*stride + fl): what no later window reads is dropped, the rest moves to the front
    const int64_t done = (int64_t)nb * d_stride, tail = d_fill - done;
    cudaStream_t s = static_cast<cudaStream_t>(d_stream);
    if (tail > 0) {
        cuda_check(cudaMemcpy2DAsync(d_ring[d_cur ^ 1], (size_t)d_pitch * sizeof(float2), ring + 2 * done,
                                     (size_t)d_pitch * sizeof(float2), (size_t)tail * sizeof(float2), (size_t)d_nchan,
                                     cudaMemcpyDeviceToDevice, s),
                   "cudaMemcpy2DAsync");
        cuda_check(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    }
    d_cur ^= 1;
    d_fill = tail;
    d_next_window += nb;
}

bool array_receiver::pop(message_pdu &out)
{
    if (d_msgs.empty()) return false;
    out = d_msgs.front();
    d_msgs.pop_front();
    return true;
}

}  // namespace uwspr
}  // namespace gr

// ------------------------------------------------------------------ C entry points
namespace {

struct rx_handle {
    gr::uwspr::array_receiver rx;
    bool broken = false;   // a push failed half way: the ring and the front-end state are lost
    template <class... A> rx_handle(A &&...a) : rx(std::forward<A>(a)...) {}
};

template <class F> int guarded(F &&f)
{
    try {
        f();
    } catch (const gr::uwspr::context_error &e) {
        return e.status;
    } catch (const std::bad_alloc &) {
        return UWSPR_B200_E_NOMEM;
    } catch (const std::exception &) {
        return UWSPR_B200_E_PARAM;
    }
    return UWSPR_B200_OK;
}

int create(const uwspr_b200_params_t *params, const uwspr_b200_input_t *input, int nchan, int shift_seconds, int batch_windows,
           rx_handle **out)
{
    if (!out) return UWSPR_B200_E_PARAM;
    *out = nullptr;
    const int st = check_args(params, input, nchan, shift_seconds, batch_windows);
    if (st) return st;
    return guarded([&] { *out = new rx_handle(*params, *input, nchan, shift_seconds, batch_windows); });
}

int push(rx_handle *h, const void *data, int space, int64_t chan_stride, int64_t n, int flush)
{
    if (!h || n < 0 || (n > 0 && !data) || (space != UWSPR_B200_HOST && space != UWSPR_B200_DEVICE)) return UWSPR_B200_E_PARAM;
    if (h->broken) return UWSPR_B200_E_STATE;
    const int st = guarded([&] {
        if (n > 0) h->rx.push(data, space, chan_stride, n);
        if (flush) h->rx.flush();
    });
    if (st) h->broken = true;
    return st;
}

}  // namespace

extern "C" {

int uwspr_b200_array_receiver_create(const uwspr_b200_params_t *params, const uwspr_b200_input_t *input, int nchan,
                                     int shift_seconds, int batch_windows, uwspr_b200_array_receiver **out)
{
    return create(params, input, nchan, shift_seconds, batch_windows, reinterpret_cast<rx_handle **>(out));
}

void uwspr_b200_array_receiver_destroy(uwspr_b200_array_receiver *rx) { delete reinterpret_cast<rx_handle *>(rx); }

int uwspr_b200_array_receiver_push(uwspr_b200_array_receiver *rx, const void *data, int space, int64_t chan_stride,
                                   int64_t n_per_chan, int flush)
{
    rx_handle *h = reinterpret_cast<rx_handle *>(rx);
    if (chan_stride < n_per_chan) return UWSPR_B200_E_PARAM;   // also the pitch of the copies, one channel included
    return push(h, data, space, chan_stride, n_per_chan, flush);
}

int uwspr_b200_array_receiver_pop(uwspr_b200_array_receiver *rx, int32_t *channel, int64_t *window, uwspr_b200_candidate_t *cand,
                                  int8_t *message7)
{
    if (!rx) return 0;
    gr::uwspr::message_pdu m;
    if (!reinterpret_cast<rx_handle *>(rx)->rx.pop(m)) return 0;
    if (channel) *channel = m.channel;
    if (window) *window = m.window;
    if (cand) *cand = m.candidate;
    if (message7) memcpy(message7, m.blob, 7);
    return 1;
}

int64_t uwspr_b200_array_receiver_windows(const uwspr_b200_array_receiver *rx)
{
    return rx ? reinterpret_cast<const rx_handle *>(rx)->rx.windows_done() : 0;
}

int64_t uwspr_b200_array_receiver_launch_count(const uwspr_b200_array_receiver *rx)
{
    return rx ? reinterpret_cast<const rx_handle *>(rx)->rx.launch_count() : 0;
}

// one channel of 375-sps complex samples
int uwspr_b200_receiver_create(const uwspr_b200_params_t *params, int shift_seconds, int batch_windows, uwspr_b200_receiver **out)
{
    uwspr_b200_input_t in;
    memset(&in, 0, sizeof(in));
    return create(params, &in, 1, shift_seconds, std::max(1, batch_windows), reinterpret_cast<rx_handle **>(out));
}

void uwspr_b200_receiver_destroy(uwspr_b200_receiver *rx) { delete reinterpret_cast<rx_handle *>(rx); }

int uwspr_b200_receiver_push(uwspr_b200_receiver *rx, const float *iq, int64_t n_complex, int flush)
{
    return push(reinterpret_cast<rx_handle *>(rx), iq, UWSPR_B200_HOST, n_complex, n_complex, flush);
}

int uwspr_b200_receiver_pop(uwspr_b200_receiver *rx, int8_t *message7, int64_t *window, uwspr_b200_candidate_t *cand)
{
    return uwspr_b200_array_receiver_pop(reinterpret_cast<uwspr_b200_array_receiver *>(rx), nullptr, window, cand, message7);
}

int64_t uwspr_b200_receiver_windows(const uwspr_b200_receiver *rx)
{
    return uwspr_b200_array_receiver_windows(reinterpret_cast<const uwspr_b200_array_receiver *>(rx));
}

}  // extern "C"
