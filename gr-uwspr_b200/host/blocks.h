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
// `receiver` is the batched form north_star asks for: the sliding window hands many
// overlapping windows (and, with one receiver per channel, many channels) to the device in
// one submission -- the ring's contiguous span plus a stride, so every sample crosses PCIe
// once -- and runs the host-side decoder on what comes back.
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

// Batched receive chain of one stream (one channel): sliding window -> coarse+fine on the
// device for up to `batch` windows per submission -> host decoder.
class receiver
{
public:
    receiver(const uwspr_b200_params_t &fdr_params, int shift_seconds, int batch_windows);
    ~receiver();
    // appends stream samples; runs a submission whenever `batch` complete windows are buffered
    void push(const gr_complex *in, size_t n);
    // processes every complete window still buffered
    void flush();
    bool pop(message_pdu &out);
    int64_t windows_done() const { return d_next_window; }

private:
    void run_batch(int nwin);
    uwspr_b200_ctx *d_ctx = nullptr;
    int d_fl, d_stride, d_batch, d_cap;
    std::vector<gr_complex> d_stream;  // samples from the start of window d_next_window
    int64_t d_next_window = 0;
    std::deque<message_pdu> d_msgs;
    std::vector<int32_t> d_npk;
    std::vector<uwspr_b200_candidate_t> d_cands;
};

}  // namespace uwspr
}  // namespace gr

#endif
