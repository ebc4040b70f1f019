// Host-side mirror of the gr-uwspr blocks around the hot path (see blocks.h).
#include "blocks.h"

#include <string.h>

#include <algorithm>

namespace gr {
namespace uwspr {

namespace {

uwspr_b200_ctx *make_ctx(const uwspr_b200_params_t &p)
{
    uwspr_b200_ctx *ctx = nullptr;
    const int st = uwspr_b200_create(&p, &ctx);
    if (st != UWSPR_B200_OK) throw context_error(st, uwspr_b200_create_error());
    return ctx;
}

void check(uwspr_b200_ctx *ctx, int st)
{
    if (st != UWSPR_B200_OK) throw context_error(st, uwspr_b200_last_error(ctx));
}

}  // namespace

std::string format_message_log(int framecount, const uwspr_b200_candidate_t &c, const int8_t blob[7])
{
    char buf[512];
    int n = snprintf(buf, sizeof(buf), "Frame: %d\nBaseband freq is %2.2f Hz\n(6 Hz) SNR is %2.2f dB\n", framecount, c.freq, c.snr);
    if (c.m_type == 0)
        n += snprintf(buf + n, sizeof(buf) - n, "Linear drift is %2.2f Hz\n", c.m_linear.drift);
    else  // the reference does not end this line
        n += snprintf(buf + n, sizeof(buf) - n, "Nonlinear drift  V=:(%2.2f,%2.2f) p=(%d,%d)", c.m_nonlinear.V1,
                      c.m_nonlinear.V2, c.m_nonlinear.p1, c.m_nonlinear.p2);
    n += snprintf(buf + n, sizeof(buf) - n, "Data: ");
    for (int i = 0; i < 7; i++) n += snprintf(buf + n, sizeof(buf) - n, "%02x", (unsigned)(unsigned char)blob[i]);
    snprintf(buf + n, sizeof(buf) - n, "\n\n");
    return std::string(buf);
}

// ------------------------------------------------------------------------------ FDR
FDR::sptr FDR::make(int fs, int fl, int spb, int maxdrift, int maxfreqs, int halfbandwidth, int cf, int threshold)
{
    sptr b(new FDR());
    uwspr_b200_params_t p = { fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, 0, 1, maxfreqs, 0 };
    b->d_ctx = make_ctx(p);  // the reference exit()s on a bad half pass bandwidth (FDR_impl.cc:85-90); this throws
    b->d_fl = fl;
    b->d_maxfreqs = maxfreqs;
    return b;
}

FDR::~FDR() { uwspr_b200_destroy(d_ctx); }

void FDR::transform(samples_ptr window)
{
    if (!window || (int)window->size() != d_fl) throw std::invalid_argument("FDR: window must hold fl samples");
    candidates_pdu out;
    out.samples = window;  // the reference forwards the same vector object (FDR_impl.cc:450)
    out.candidates.resize(d_maxfreqs);
    int32_t npk = 0, total = 0;
    check(d_ctx, uwspr_b200_coarse(d_ctx, reinterpret_cast<const float *>(window->data()), UWSPR_B200_HOST, d_fl, 1, &npk,
                                   out.candidates.data(), d_maxfreqs, &total));
    out.candidates.resize(npk);
    if (d_out) d_out(out);
}

// -------------------------------------------------------------- sync_and_demodulate
sync_and_demodulate::sptr sync_and_demodulate::make(int fs, int fl, int spb, int maxdrift, int maxfreqs, int cf)
{
    sptr b(new sync_and_demodulate());
    // halfbandwidth / threshold do not enter the fine stage; any valid values do
    uwspr_b200_params_t p = { fs, fl, spb, maxdrift, maxfreqs, 10, cf, 10, 0, 1, maxfreqs, 0 };
    b->d_ctx = make_ctx(p);
    b->d_fl = fl;
    return b;
}

sync_and_demodulate::~sync_and_demodulate()
{
    if (d_log) fclose(d_log);
    uwspr_b200_destroy(d_ctx);
}

void sync_and_demodulate::set_message_log(const std::string &path)
{
    if (d_log) fclose(d_log);
    d_log = fopen(path.c_str(), "a");  // :98
    if (!d_log) throw std::runtime_error("cannot open message log " + path);  // the reference dereferences NULL here
    time(&d_start);
    fprintf(d_log, "Start time: %s\n", asctime(localtime(&d_start)));  // :105-107
    fflush(d_log);
}

void sync_and_demodulate::demodulate(const candidates_pdu &pdu)
{
    const int npk = (int)pdu.candidates.size();
    if (npk == 0) return;
    std::vector<uwspr_b200_refined_t> refined(npk);
    std::vector<uwspr_b200_jiggle_t> jig((size_t)npk * UWSPR_B200_NJIG);
    std::vector<uint8_t> soft((size_t)npk * UWSPR_B200_NJIG * UWSPR_B200_NSYM);
    int32_t npk32 = npk;
    check(d_ctx, uwspr_b200_fine(d_ctx, reinterpret_cast<const float *>(pdu.samples->data()), UWSPR_B200_HOST, d_fl, 1,
                                 &npk32, pdu.candidates.data(), npk, 0, UWSPR_B200_NJIG, refined.data(), jig.data(),
                                 soft.data()));
    for (int j = 0; j < npk; j++) {  // sync_and_demodulate_impl.cc:389
        message_pdu m;
        int32_t idt;
        uint32_t cycles;
        if (uwspr_b200_decode_candidate(&refined[j], &jig[(size_t)j * UWSPR_B200_NJIG],
                                        &soft[(size_t)j * UWSPR_B200_NJIG * UWSPR_B200_NSYM], UWSPR_B200_NJIG, m.blob, &idt,
                                        &cycles)) {
            d_framecount++;  // :492
            if (d_log) {     // :507-526
                time_t now;
                time(&now);
                const long dt = (long)difftime(now, d_start);
                fprintf(d_log, "Handoff time : %sElapsed time: %02d:%02d:%02d\n", asctime(localtime(&now)),
                        (int)((dt / 3600) % 24), (int)((dt / 60) % 60), (int)(dt % 60));
                fputs(format_message_log(d_framecount, pdu.candidates[j], m.blob).c_str(), d_log);
                fflush(d_log);
            }
            m.candidate = pdu.candidates[j];
            m.window = -1;
            if (d_out) d_out(m);  // :528-530
        }
    }
}

// ------------------------------------------------------ sliding_window_stream_to_pdu
sliding_window_stream_to_pdu::sptr sliding_window_stream_to_pdu::make(int fs, int fl, int shift, int C)
{
    sptr b(new sliding_window_stream_to_pdu());
    b->d_fs = fs;
    b->d_fl = fl;
    b->d_shift = shift;
    b->d_capacity = (size_t)C * fl;  // sliding_window_stream_to_pdu_impl.cc:65
    return b;
}

int sliding_window_stream_to_pdu::work(int noutput_items, const gr_complex *in)
{
    for (int i = 0; i < noutput_items; i++) {  // :108-110 (a full circular buffer drops its oldest element)
        if (d_buffer.size() == d_capacity && d_capacity) d_buffer.pop_front();
        d_buffer.push_back(in[i]);
    }
    d_count += noutput_items;
    if (d_count >= d_fl) {  // :113
        std::shared_ptr<std::vector<gr_complex>> w(new std::vector<gr_complex>(d_fl));
        const int adv = d_shift * d_fs;
        for (int i = 0; i < adv; i++) {  // :118-126 pop shift*fs samples into the PDU
            (*w)[i] = d_buffer.front();
            d_buffer.pop_front();
        }
        for (int i = 0; i < d_fl - adv; i++) (*w)[adv + i] = d_buffer[i];  // :128-131 peek the rest
        d_count -= adv;                                                     // :135
        if (d_out) d_out(w);
    }
    return noutput_items;
}

}  // namespace uwspr
}  // namespace gr

extern "C" {

int uwspr_b200_format_message_log(int framecount, const uwspr_b200_candidate_t *cand, const int8_t *message7, char *text,
                                  size_t text_cap)
{
    if (!cand || !message7 || !text) return UWSPR_B200_E_PARAM;
    const std::string s = gr::uwspr::format_message_log(framecount, *cand, message7);
    if (s.size() + 1 > text_cap) return UWSPR_B200_E_CAPACITY;
    memcpy(text, s.c_str(), s.size() + 1);
    return UWSPR_B200_OK;
}

}  // extern "C"
