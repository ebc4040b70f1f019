// Host-side mirror of the three gr-uwspr blocks that bracket the hot path, on top of the C ABI.
//
// GNU Radio 3.7 is not available in the build image, so these classes keep the reference's
// factory signatures and handler semantics but exchange plain-data PDUs instead of PMTs
// (the four schemas are listed in SURVEY.md 8(b)); INTEGRATION.md shows the PMT glue.
//
//   gr::uwspr::FDR::make(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold)
//        include/uwspr/FDR.h:49-50, handler lib/FDR_impl.cc:214-456
//   gr::uwspr::sync_and_demodulate::make(fs, fl, spb, maxdrift, maxfreqs, cf)
//        include/uwspr/sync_and_demodulate.h:49, handler lib/sync_and_demodulate_impl.cc:315-534
//   gr::uwspr::sliding_window_stream_to_pdu::make(fs, fl, shift, C)
//        include/uwspr/sliding_window_stream_to_pdu.h:52, work() lib/sliding_window_stream_to_pdu_impl.cc:98-138
//
// `array_receiver` is the batched form north_star asks for: C channels of audio (or 375-sps samples) go
// through a front-end stream into a ring on the device, and the sliding window hands every channel's
// overlapping windows to the device in one submission per batch, decoded where they are.  It owns device
// memory, so it is defined with the kernels' host code (csrc/receiver.cu); uwspr_b200_receiver_* is the same
// class with one channel.
#ifndef UWSPR_B200_HOST_BLOCKS_H
#define UWSPR_B200_HOST_BLOCKS_H

#include <complex>
#include <cstdint>
#include <cstdio>
#include <ctime>
#include <deque>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "uwspr_b200.h"

namespace gr {
namespace uwspr {

typedef std::complex<float> gr_complex;

// PDU (1): sliding window -> FDR : fl complex samples
typedef std::shared_ptr<const std::vector<gr_complex>> samples_ptr;
// PDU (2): FDR -> sync_and_demodulate : the same sample vector + npk candidates
struct candidates_pdu {
    samples_ptr samples;
    std::vector<uwspr_b200_candidate_t> candidates;
};
// PDU (3): sync_and_demodulate -> WSPR_unpacker : first 7 bytes of the decoded data
struct message_pdu {
    int8_t blob[7];
    uwspr_b200_candidate_t candidate;  // not in the reference's PDU; kept for logging
    int64_t window;                    // index of the window it came from (receiver only)
    int32_t channel = 0;               // channel it came from (receiver only)
};

// text the reference appends to messagelog.txt for one decoded frame, without the two
// wall-clock lines ("Handoff time", "Elapsed time") that precede it (sync_and_demodulate_impl.cc:508-525)
std::string format_message_log(int framecount, const uwspr_b200_candidate_t &cand, const int8_t blob[7]);

class context_error : public std::runtime_error
{
public:
    context_error(int status, const std::string &what) : std::runtime_error(what), status(status) {}
    int status;
};

class FDR
{
public:
    typedef std::shared_ptr<FDR> sptr;
    static sptr make(int fs, int fl, int spb, int maxdrift, int maxfreqs, int halfbandwidth, int cf, int threshold);
    ~FDR();
    void set_msg_out(std::function<void(const candidates_pdu &)> h) { d_out = h; }
    // message handler of port "in"
    void transform(samples_ptr window);

private:
    FDR() {}
    uwspr_b200_ctx *d_ctx = nullptr;
    int d_fl = 0, d_maxfreqs = 0;
    std::function<void(const candidates_pdu &)> d_out;
};

class sync_and_demodulate
{
public:
    typedef std::shared_ptr<sync_and_demodulate> sptr;
    static sptr make(int fs, int fl, int spb, int maxdrift, int maxfreqs, int cf);
    ~sync_and_demodulate();
    void set_msg_out(std::function<void(const message_pdu &)> h) { d_out = h; }
    // message handler of port "in": one message_pdu per decoded candidate, in candidate order
    void demodulate(const candidates_pdu &pdu);
    int framecount() const { return d_framecount; }
    // the reference appends every decode to ./messagelog.txt (sync_and_demodulate_impl.cc:98-108,
    // :507-526); off by default here, same text when enabled
    void set_message_log(const std::string &path);

private:
    sync_and_demodulate() {}
    uwspr_b200_ctx *d_ctx = nullptr;
    int d_fl = 0, d_framecount = 0;
    FILE *d_log = nullptr;
    time_t d_start = 0;
    std::function<void(const message_pdu &)> d_out;
};

class sliding_window_stream_to_pdu
{
public:
    typedef std::shared_ptr<sliding_window_stream_to_pdu> sptr;
    static sptr make(int fs, int fl, int shift, int C);
    void set_msg_out(std::function<void(samples_ptr)> h) { d_out = h; }
    // same contract as the reference's work(): consumes noutput_items, emits at most one window
    int work(int noutput_items, const gr_complex *in);

private:
    sliding_window_stream_to_pdu() {}
    int d_fs = 0, d_fl = 0, d_shift = 0;
    size_t d_capacity = 0;
    std::deque<gr_complex> d_buffer;
    long d_count = 0;
    std::function<void(samples_ptr)> d_out;
};

// Receive chain of nchan channels in lockstep: front-end stream -> ring of 375-sps streams on the device ->
// one coarse+fine submission per `batch` windows of every channel -> decoder on the device.
class array_receiver
{
public:
    // throws context_error (E_PARAM for the checks of uwspr_b200_array_receiver_create)
    array_receiver(const uwspr_b200_params_t &params, const uwspr_b200_input_t &input, int nchan, int shift_seconds,
                   int batch_windows);
    ~array_receiver();
    // n samples of every channel, channel c at data + c*chan_stride samples; runs a submission whenever `batch`
    // complete windows are buffered on every channel
    void push(const void *data, int space, int64_t chan_stride, int64_t n);
    // processes every complete window still buffered
    void flush();
    bool pop(message_pdu &out);
    int64_t windows_done() const { return d_next_window; }
    int64_t launch_count() const;

private:
    void release();
    void process(bool all);
    void run_batch(int per_chan);
    uwspr_b200_ctx *d_ctx = nullptr;
    uwspr_b200_frontend_stream *d_fe = nullptr;
    void *d_stream = nullptr;                // cudaStream_t of the ring copies
    void *d_ring[2] = { nullptr, nullptr };  // complex64 [nchan][d_pitch]: the ring and the buffer its tail moves to
    int d_cur = 0;
    int d_device, d_kind, d_nchan, d_fl, d_stride, d_batch, d_cap, d_decim = 1;
    int64_t d_pitch = 0, d_fill = 0;         // samples per channel of the ring, and those held (from window d_next_window)
    int64_t d_next_window = 0;
    std::deque<message_pdu> d_msgs;
    std::vector<int32_t> d_npk;
    std::vector<uwspr_b200_candidate_t> d_cands;
    std::vector<uint8_t> d_decoded;
    std::vector<int8_t> d_blobs;
};

}  // namespace uwspr
}  // namespace gr

#endif
