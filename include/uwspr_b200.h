/* uwspr_b200 -- C ABI of the B200-native receive hot path of gr-uwspr.
 *
 * One shared library, libuwspr_b200.so, replaces the arithmetic of two GNU Radio
 * blocks of the reference (all citations are file:line under the reference tree):
 *
 *   uwspr.FDR                 FDR_impl::transform                 lib/FDR_impl.cc:214-456
 *   uwspr.sync_and_demodulate sync_and_demodulate_impl::demodulate lib/sync_and_demodulate_impl.cc:315-482
 *                             (up to, not including, deinterleave + Fano::fano at :476-478)
 *
 * The entry points take plain pointers and sizes; there are no C++, torch or GNU
 * Radio types in any signature.  Every function returns an int status
 * (UWSPR_B200_OK == 0); nothing in the library calls exit() or throws across the
 * boundary (the reference exits on bad parameters, lib/FDR_impl.cc:85-90).
 * A context is bound to one CUDA device and may be used by one thread at a time
 * (uwspr_b200_coarse_fine_submit / uwspr_b200_wait give a non-blocking form);
 * distinct contexts are independent (the reference's blocks are never re-entered
 * either: GNU Radio 3.7 runs one handler invocation at a time per block).
 *
 * There is no CPU fallback: if no CUDA device is usable, uwspr_b200_create fails
 * with UWSPR_B200_E_CUDA.
 */
#ifndef UWSPR_B200_H
#define UWSPR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UWSPR_B200_API __attribute__((visibility("default")))

enum {
    UWSPR_B200_OK = 0,
    UWSPR_B200_E_PARAM = 1,    /* parameters outside the domain (see uwspr_b200_create) */
    UWSPR_B200_E_CUDA = 2,     /* CUDA runtime error; text in uwspr_b200_last_error */
    UWSPR_B200_E_CAPACITY = 3, /* more candidates than the caller's / context's capacity */
    UWSPR_B200_E_NOMEM = 4,
    UWSPR_B200_E_STATE = 5     /* call sequence error (e.g. fetch before any submission) */
};

enum { UWSPR_B200_HOST = 0, UWSPR_B200_DEVICE = 1 }; /* memory space of a sample pointer */

#define UWSPR_B200_NSYM 162     /* channel symbols per frame                       */
#define UWSPR_B200_NJIG 17      /* jiggled shifts of the final peak-up, idt = 0..16 (sync_and_demodulate_impl.cc:460) */

/* candidate_t of the reference, byte for byte: lib/candidate_t.h:27-50
 * (48 bytes, alignment 8; offsets freq 0, snr 4, drift 8, sync 12, shift 16,
 * m_type 20, union 24: V1 24, V2 32, p1 40, p2 44). */
typedef struct {
    float freq;      /* baseband frequency, Hz                                      */
    float snr;       /* 10*log10 of the normalised smoothed spectrum at the peak    */
    float drift;     /* unused by the reference (never written); always 0 here      */
    float sync;      /* coarse sync metric                                          */
    int32_t shift;   /* start of frame in samples (128 * half-symbol index)         */
    int32_t m_type;  /* 0 = linear drift model, 1 = nonlinear (straight-line) model */
    union {
        struct { float drift; } m_linear;
        struct { double V1, V2; int32_t p1, p2; } m_nonlinear;
    };
} uwspr_b200_candidate_t;

/* Result of the refinement chain of demodulate() for one candidate: the values of
 * f1, shift1, drift1, sync1 when the peak-up loop starts (:457) and worth_a_try (:453). */
typedef struct {
    float f1;
    int32_t shift1;
    float drift1;
    float sync1;
    int32_t worth_a_try; /* sync1 > minsync1 (0.10) after the coarse-grid stages */
    int32_t reserved;
} uwspr_b200_refined_t;

/* One mode-2 evaluation of the peak-up loop (:461-475): jiggle index idt uses
 * shift1 + 8*(+-ceil(idt/2)).  gate = sync > minsync2 (0.12) && rms > minrms (40.625):
 * the condition under which the reference hands the symbols to the Fano decoder. */
typedef struct {
    float sync;
    float rms;
    int32_t shift;
    int32_t gate;
} uwspr_b200_jiggle_t;

/* Constructor arguments of the two blocks.  fs..threshold are the eight ints of
 * uwspr.FDR(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold)
 * (include/uwspr/FDR.h:49-50; grc/uwspr_FDR.xml:7); sync_and_demodulate takes the
 * first five and cf (include/uwspr/sync_and_demodulate.h:49). */
typedef struct {
    int32_t fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold;
    int32_t device;             /* CUDA device ordinal                                         */
    int32_t max_windows;        /* largest nwin of one call; 0 = 1                             */
    int32_t max_candidates;     /* capacity of the compact candidate list of one call;
                                   0 = max_windows * min(maxfreqs, (finpb-1)/2)               */
    int32_t nonlinear_intended_t; /* 0 (default): the nonlinear fine branch uses t == 0, as the
                                   compiled reference behaves (uninitialised `t`,
                                   sync_and_demodulate_impl.cc:177-180); 1: t = i*111/162     */
} uwspr_b200_params_t;

typedef struct uwspr_b200_ctx uwspr_b200_ctx;

/* Domain: spb == 256, fl == 45000 (the reference's fine stage hard-codes 256 samples per
 * symbol and npoints = 45000, sync_and_demodulate_impl.cc:92,146,191,204), halfbandwidth
 * <= fs/2 (FDR_impl.cc:85-90) and small enough that every bin the reference touches exists
 * (it reads out of bounds beyond ~180 Hz at fs = 375), maxfreqs >= 1. */
UWSPR_B200_API int uwspr_b200_create(const uwspr_b200_params_t *params, uwspr_b200_ctx **ctx_out);
UWSPR_B200_API void uwspr_b200_destroy(uwspr_b200_ctx *ctx);
UWSPR_B200_API const char *uwspr_b200_last_error(const uwspr_b200_ctx *ctx);
UWSPR_B200_API const char *uwspr_b200_status_string(int status);
/* text of the failure of the last uwspr_b200_create that returned non-zero on the calling thread */
UWSPR_B200_API const char *uwspr_b200_create_error(void);

/* Derived constants of the FDR constructor (FDR_impl.cc:81-137), for callers and tests. */
typedef struct {
    int32_t size, m, hpbm, n_rows, finpb, noiseidx;
    float df, min_snr;
    int32_t bin_lo, n_bins;      /* kept spectrogram bins [bin_lo, bin_lo + n_bins) (shifted index, DC = m) */
    int32_t n_lin, n_unique;     /* linear hypotheses, distinct bin-offset sequences among the 2*maxdrift+1+125 */
    int32_t max_cand_per_window; /* min(maxfreqs, (finpb-1)/2) */
    int32_t max_windows, max_candidates;
    int32_t sm_count;
} uwspr_b200_info_t;
UWSPR_B200_API int uwspr_b200_info(const uwspr_b200_ctx *ctx, uwspr_b200_info_t *info);

/* ---- FDR_impl::transform for nwin windows --------------------------------------------
 * samples: interleaved complex64 (I, Q), window w = samples[w*win_stride, w*win_stride + fl)
 * (win_stride in complex samples: fl for independent windows, shift*fs for the sliding
 * window of lib/sliding_window_stream_to_pdu_impl.cc:113-135).  space says where `samples`
 * lives.  Outputs (host pointers, any may be NULL):
 *   npk[nwin]         candidates per window (FDR_impl.cc:293-306,414)
 *   cands[cap]        compact, window-major; within a window in the reference's order
 *                     (descending snr, stable; FDR_impl.cc:311-319) with the coarse
 *                     estimates of :339-409 filled in
 *   *total            sum of npk
 * The candidate list also stays on the device for a following uwspr_b200_fine(..., cands == NULL). */
UWSPR_B200_API int uwspr_b200_coarse(uwspr_b200_ctx *ctx, const float *samples, int space,
                                     int64_t win_stride, int nwin, int32_t *npk,
                                     uwspr_b200_candidate_t *cands, int cap, int32_t *total);

/* ---- sync_and_demodulate_impl::demodulate up to the decoder ----------------------------
 * Same sample arguments.  npk/cands: the candidate lists (host pointers, compact layout as
 * returned by uwspr_b200_coarse); pass cands == NULL to use the list left on the device by
 * the preceding uwspr_b200_coarse call on the same windows.
 * For every candidate: the refinement chain :404-456, then mode-2 evaluations for jiggle
 * indices idt in [jig_first, jig_first + jig_count) (:460-475).
 * Outputs (host pointers, any may be NULL), g = compact candidate index:
 *   refined[g]
 *   jig[g*jig_count + t]
 *   soft[(g*jig_count + t)*162 + i]   soft symbols as sync_and_demodulate() returns them
 *                                     (before deinterleave); all 0 when !worth_a_try
 */
UWSPR_B200_API int uwspr_b200_fine(uwspr_b200_ctx *ctx, const float *samples, int space,
                                   int64_t win_stride, int nwin, const int32_t *npk,
                                   const uwspr_b200_candidate_t *cands, int total, int jig_first,
                                   int jig_count, uwspr_b200_refined_t *refined,
                                   uwspr_b200_jiggle_t *jig, uint8_t *soft);

/* ---- both stages in one submission (candidates never leave the device in between) ------ */
UWSPR_B200_API int uwspr_b200_coarse_fine(uwspr_b200_ctx *ctx, const float *samples, int space,
                                          int64_t win_stride, int nwin, int jig_first,
                                          int jig_count, int32_t *npk,
                                          uwspr_b200_candidate_t *cands, int cap, int32_t *total,
                                          uwspr_b200_refined_t *refined, uwspr_b200_jiggle_t *jig,
                                          uint8_t *soft);

/* ---- non-blocking form of uwspr_b200_coarse_fine ----------------------------------------
 * _submit starts the same work on a thread owned by the context and returns at once (a GNU Radio
 * message handler does not stall for the batch); the caller keeps every buffer alive and untouched
 * until uwspr_b200_wait() returns the call's status.  uwspr_b200_poll(): 1 = finished, 0 = still
 * running, -1 = nothing submitted.  One submission per context at a time; the synchronous entry points
 * return UWSPR_B200_E_STATE while one is outstanding.  Kernels run on the stream given to
 * uwspr_b200_set_stream(), as for the synchronous calls. */
UWSPR_B200_API int uwspr_b200_coarse_fine_submit(uwspr_b200_ctx *ctx, const float *samples, int space,
                                                 int64_t win_stride, int nwin, int jig_first,
                                                 int jig_count, int32_t *npk,
                                                 uwspr_b200_candidate_t *cands, int cap, int32_t *total,
                                                 uwspr_b200_refined_t *refined,
                                                 uwspr_b200_jiggle_t *jig, uint8_t *soft);
UWSPR_B200_API int uwspr_b200_poll(uwspr_b200_ctx *ctx);
UWSPR_B200_API int uwspr_b200_wait(uwspr_b200_ctx *ctx);

/* ---- host side of the path that stays on the CPU (north_star: "Fano decoding and
 * WSPR_unpacker stay host-side") -------------------------------------------------------- */
/* lib/sync_and_demodulate_impl.cc:265-282, in place on 162 bytes */
UWSPR_B200_API void uwspr_b200_deinterleave(uint8_t *sym162);
/* lib/Fano.cc:110-252 with the metric table of :36-45; symbols are deinterleaved soft symbols.
 * Returns 0 on success, -1 on time-out (data11 then holds the decoder's partial path). */
UWSPR_B200_API int uwspr_b200_fano(uint32_t *metric, uint32_t *cycles, uint32_t *maxnp,
                                   uint8_t *data11, const uint8_t *symbols162, uint32_t nbits,
                                   int delta, uint32_t maxcycles);
/* The peak-up/decode loop :457-490 over precomputed jiggles of one candidate: walks
 * idt = 0.., runs the decoder where gate is set, stops at the first success.
 * Returns 1 and fills message7 (the published blob, :484-490,528-530) if decoded, else 0. */
UWSPR_B200_API int uwspr_b200_decode_candidate(const uwspr_b200_refined_t *refined,
                                               const uwspr_b200_jiggle_t *jig, const uint8_t *soft,
                                               int jig_count, int8_t *message7, int32_t *idt_used,
                                               uint32_t *fano_cycles);
/* The same loop over `ncand` candidates as uwspr_b200_fine() returns them (refined[ncand],
 * jig[ncand][jig_count], soft[ncand][jig_count][162]), spread over `nthreads` host threads
 * (<= 0: one per online core).  Candidates are independent in the reference too (one
 * demodulate() loop iteration each, :405), so the outputs do not depend on the thread count:
 * decoded[g] = 0/1, messages[g*7..], idt_used[g], fano_cycles[g] (the last two may be NULL).
 * Returns the number of decoded candidates, or a negative status. */
UWSPR_B200_API int uwspr_b200_decode_batch(const uwspr_b200_refined_t *refined,
                                           const uwspr_b200_jiggle_t *jig, const uint8_t *soft,
                                           int64_t ncand, int jig_count, int nthreads,
                                           uint8_t *decoded, int8_t *messages7, int32_t *idt_used,
                                           uint32_t *fano_cycles);

/* ---- the same decoder on the device (sm_100a; bit-identical to the two host entry points above) ------
 * uwspr_b200_decode_device: uwspr_b200_decode_batch's loop with every gated (candidate, jiggle) decoded by
 * its own device thread; same outputs (host pointers; idt_used and fano_cycles may be NULL) and the same
 * return value: the number of decoded candidates, or a negative status.
 * refined == jig == soft == NULL: decodes the results the last uwspr_b200_fine / uwspr_b200_coarse_fine call
 * on this context left on the device (so a coarse_fine(..., soft = NULL) never copies soft symbols to the
 * host); ncand and jig_count must equal that call's candidate total and jiggle count (else E_PARAM), and
 * E_STATE if no such results exist.  Otherwise the three inputs are read from `space` (HOST or DEVICE);
 * they are copied into the context's device result buffers, which replaces the results of the last call,
 * and more than max_candidates is E_CAPACITY.  E_STATE while a submission is outstanding.  Runs on the
 * stream of uwspr_b200_set_stream. */
UWSPR_B200_API int uwspr_b200_decode_device(uwspr_b200_ctx *ctx, const uwspr_b200_refined_t *refined,
                                            const uwspr_b200_jiggle_t *jig, const uint8_t *soft, int space,
                                            int64_t ncand, int jig_count, uint8_t *decoded, int8_t *messages7,
                                            int32_t *idt_used, uint32_t *fano_cycles);
/* uwspr_b200_fano on n independent rows of 162 de-interleaved symbols (symbols[n*162] in `space`), one
 * device thread each; every output (host pointers, n entries; data11: n x 11 bytes, zero past nbits/8)
 * equals uwspr_b200_fano's for that row, the partial path of a time-out included.  Domain:
 * 32 <= nbits <= 81, delta > 0, maxcycles >= 1 and (maxcycles*nbits + 1)*delta < 2^31; outside it, or with
 * a NULL ctx, E_PARAM before any CUDA call.  Returns a status. */
UWSPR_B200_API int uwspr_b200_fano_batch(uwspr_b200_ctx *ctx, const uint8_t *symbols, int space, int64_t n,
                                         uint32_t nbits, int delta, uint32_t maxcycles, int32_t *status,
                                         uint32_t *metric, uint32_t *cycles, uint32_t *maxnp, uint8_t *data11);

/* ---- WSPR_unpacker's text: lib/helpers.cc:494-590 (unpk_) -------------------------------
 * message7 -> "CALL GRID dBm" (type 1), "PFX/CALL dBm" (type 2) or "<CALL> GRID6 dBm" (type 3).
 * hashtab: caller-owned callsign hash table of uwspr_b200_hashtab_bytes() zero-initialised
 * bytes (the reference keeps one per unpacker block and persists it in hashtable.txt).
 * Returns the reference's `noprint` flag (0 = print), or -1 on bad arguments. */
UWSPR_B200_API size_t uwspr_b200_hashtab_bytes(void);
UWSPR_B200_API int uwspr_b200_unpack(const int8_t *message7, char *hashtab, char *text, size_t text_cap);

/* Transmit direction, for synthetic inputs and tests (the reference ships only the receiver):
 * "CALL", "GRID" (4 characters), dBm -> the 7-byte type-1 message uwspr_b200_unpack() reads back
 * (inverse of lib/helpers.cc:321-434), and message -> the 162 four-level channel symbols
 * (encoder lib/Fano.cc:81-100, interleaver inverse of sync_and_demodulate_impl.cc:265-282,
 * symbol = 2*data + pr3[i]). */
UWSPR_B200_API int uwspr_b200_pack_type1(const char *call, const char *grid4, int dbm, int8_t *message7);
UWSPR_B200_API void uwspr_b200_channel_symbols(const int8_t *message7, uint8_t *symbols162);

/* ---- upstream of the path ---------------------------------------------------------------
 * uwspr.c2file_source's reader (lib/c2file_source_impl.cc:75-96): 45000 complex samples at
 * 375 sps as I - jQ (the reference flips the quadrature sign at :91) into iq[2*45000];
 * name15 (15 bytes), type and freq_mhz may be NULL.  E_PARAM if the file cannot be read or is short. */
UWSPR_B200_API int uwspr_b200_read_c2(const char *path, float *iq, char *name15, int32_t *type, double *freq_mhz);

/* Front-end on the device (stock GNU Radio blocks in the reference's flowgraphs,
 * examples/WaveFilePlusNoiseDecode.grc:834-958,1753-1810): real audio -> mix down by fc ->
 * FIR -> keep every decim-th sample:
 *     y[m] = sum_k taps[k] * x[n-k] * exp(-2 pi i fc (n-k) / fs_in),  n = m*decim + delay,
 * x = 0 outside [0, n_in).  audio: nchan channels of n_in samples, chan_stride apart, fmt 0 =
 * float32, 1 = int16 (scaled by 1/32768 like blocks_wavfile_source); out: complex64, channel c at
 * out + 2*c*out_stride floats, *n_out = n_in / decim samples each.  space_in / space_out say
 * where the buffers live; a device output feeds uwspr_b200_coarse_fine directly. */
UWSPR_B200_API int uwspr_b200_frontend(int device, const void *audio, int fmt, int space_in,
                                       int64_t chan_stride, int nchan, int64_t n_in,
                                       const float *taps, int ntaps, int decim, int delay, double fc,
                                       double fs_in, float *out, int space_out, int64_t out_stride,
                                       int64_t *n_out);
/* The same with complex taps (taps_iq: ntaps pairs re, im).  The cascade of the reference's flowgraph
 * (examples/WaveFilePlusNoiseDecode.grc: freq_xlating_fft_filter_ccc with a real band-pass at centre 0 (:834-893),
 * freq_xlating_fft_filter_ccc at centre 1500 Hz with a low-pass (:894-958), rational_resampler_xxx 1/32 (:1753-1810))
 * is one such filter with delay 0: composite = (h_bp[k] e^{-i w k}) * h_lp * h_rs, w = 2 pi fc / fs_in. */
UWSPR_B200_API int uwspr_b200_frontend_ctaps(int device, const void *audio, int fmt, int space_in,
                                             int64_t chan_stride, int nchan, int64_t n_in,
                                             const float *taps_iq, int ntaps, int decim, int delay, double fc,
                                             double fs_in, float *out, int space_out, int64_t out_stride,
                                             int64_t *n_out);
/* text of the last front-end failure (one-shot or stream) on the calling thread */
UWSPR_B200_API const char *uwspr_b200_frontend_error(void);

/* The front-end as a stream that keeps its state between pushes (audio read in pieces, a GNU Radio work() call
 * at a time).  After N input samples per channel in total, in any split, the stream has produced exactly the
 * outputs m with m*decim + delay < N, and each equals, bit for bit, output m of uwspr_b200_frontend (real taps) or
 * uwspr_b200_frontend_ctaps (complex_taps != 0: taps holds ntaps pairs re, im) run once over any input that holds
 * those samples.  State per channel: the last ntaps - 1 + decim samples in the input format and the sample count.
 * create allocates every buffer; a push allocates nothing, runs on a stream owned by the object, works through
 * its input in pieces of bounded size and returns when its outputs are written.
 * create: E_PARAM for the arguments uwspr_b200_frontend rejects, and when ntaps + 63*decim samples do not fit
 * shared memory (a device query).  push: audio holds n_in samples of each of the nchan channels, chan_stride
 * apart, in `space_in`; the new outputs go to out (complex64, channel c at out + 2*c*out_stride floats) in
 * `space_out`, *n_out of them per channel; more than out_cap is E_CAPACITY and consumes nothing.  After any other
 * failure of a push the stream's state is lost: later pushes return E_STATE.  chan_stride < n_in or
 * out_stride < out_cap is E_PARAM, for one channel too. */
typedef struct uwspr_b200_frontend_stream uwspr_b200_frontend_stream;
UWSPR_B200_API int uwspr_b200_frontend_stream_create(int device, int nchan, int fmt, const float *taps, int ntaps,
                                                     int complex_taps, int decim, int delay, double fc, double fs_in,
                                                     uwspr_b200_frontend_stream **out);
UWSPR_B200_API int uwspr_b200_frontend_stream_push(uwspr_b200_frontend_stream *s, const void *audio, int space_in,
                                                   int64_t chan_stride, int64_t n_in, float *out, int space_out,
                                                   int64_t out_stride, int64_t out_cap, int64_t *n_out);
/* outputs produced so far, per channel */
UWSPR_B200_API int64_t uwspr_b200_frontend_stream_outputs(const uwspr_b200_frontend_stream *s);
UWSPR_B200_API void uwspr_b200_frontend_stream_destroy(uwspr_b200_frontend_stream *s);

/* The text the reference appends to messagelog.txt for one decoded frame
 * (lib/sync_and_demodulate_impl.cc:508-525), without the two wall-clock lines before it. */
UWSPR_B200_API int uwspr_b200_format_message_log(int framecount, const uwspr_b200_candidate_t *cand,
                                                 const int8_t *message7, char *text, size_t text_cap);

/* ---- batched receive chain of one stream (one hydrophone channel) -----------------------
 * The sliding window of lib/sliding_window_stream_to_pdu_impl.cc:98-138 (window k =
 * stream[k*shift*fs, k*shift*fs + fl)) feeding the device `batch_windows` windows per
 * submission, then the decoder on the device (uwspr_b200_decode_device on the results left there; no soft
 * symbol crosses PCIe).  Messages come out in (window, candidate) order, one per decoded candidate, no
 * de-duplication -- as the reference publishes them.  It is the array receiver below with one channel of kind 0. */
typedef struct uwspr_b200_receiver uwspr_b200_receiver;
UWSPR_B200_API int uwspr_b200_receiver_create(const uwspr_b200_params_t *params, int shift_seconds,
                                              int batch_windows, uwspr_b200_receiver **out);
UWSPR_B200_API void uwspr_b200_receiver_destroy(uwspr_b200_receiver *rx);
/* appends n_complex stream samples (interleaved I,Q); flush != 0 also processes every complete
 * window still buffered */
UWSPR_B200_API int uwspr_b200_receiver_push(uwspr_b200_receiver *rx, const float *iq, int64_t n_complex, int flush);
/* returns 1 and fills the outputs (any may be NULL) while decoded messages are queued */
UWSPR_B200_API int uwspr_b200_receiver_pop(uwspr_b200_receiver *rx, int8_t *message7, int64_t *window,
                                           uwspr_b200_candidate_t *cand);
UWSPR_B200_API int64_t uwspr_b200_receiver_windows(const uwspr_b200_receiver *rx);

/* ---- receive chain of nchan channels in lockstep, from audio or 375-sps samples to messages ---------------
 * Channel c's stream s_c is its input (kind 0) or the output of a uwspr_b200_frontend_stream over its audio
 * (kinds 1 and 2).  Window k of channel c is s_c[k*shift*fs, k*shift*fs + fl).  The streams live in a ring on the
 * device; once batch_windows windows are complete on every channel, one coarse_fine submission covers all
 * nchan * batch_windows windows (17 jiggles, nothing copied back but the candidate list), then
 * uwspr_b200_decode_device decodes them where they are.  Messages come out in (window, channel, candidate) order,
 * one per decoded candidate, without de-duplication, and do not depend on batch_windows or on how the input is
 * split into pushes.  params->max_windows is ignored (nchan * batch_windows); params->max_candidates as for
 * uwspr_b200_create. */
typedef struct {
    int32_t kind;            /* 0: complex64 at params->fs (no front-end), 1: float32 audio, 2: int16 audio */
    const float *taps;       /* kinds 1, 2: ntaps real taps, or ntaps (re, im) pairs when complex_taps != 0 */
    int32_t ntaps, complex_taps, decim, delay;
    double fc, fs_in;        /* fs_in / decim must equal params->fs */
} uwspr_b200_input_t;
typedef struct uwspr_b200_array_receiver uwspr_b200_array_receiver;
/* E_PARAM before any CUDA call: NULL pointers, nchan < 1, batch_windows < 1, shift*fs outside (0, fl], a bad kind,
 * and for kinds 1 and 2 ntaps outside 1..16384, decim outside 1..4096, delay < 0 or fs_in / decim != fs.
 * E_PARAM after a device query: ntaps + 63*decim samples do not fit shared memory.  Otherwise as uwspr_b200_create. */
UWSPR_B200_API int uwspr_b200_array_receiver_create(const uwspr_b200_params_t *params, const uwspr_b200_input_t *input,
                                                    int nchan, int shift_seconds, int batch_windows,
                                                    uwspr_b200_array_receiver **out);
/* n_per_chan samples of every channel (complex64 for kind 0, else the audio format), channel c at
 * data + c*chan_stride samples (chan_stride >= n_per_chan, else E_PARAM), in `space`; flush != 0 then processes
 * every complete window still buffered.
 * A failing batch returns its status (E_CAPACITY when its candidates exceed max_candidates); the receiver's state
 * is then lost and later pushes return E_STATE. */
UWSPR_B200_API int uwspr_b200_array_receiver_push(uwspr_b200_array_receiver *rx, const void *data, int space,
                                                  int64_t chan_stride, int64_t n_per_chan, int flush);
/* returns 1 and fills the outputs (any may be NULL) while decoded messages are queued, else 0 */
UWSPR_B200_API int uwspr_b200_array_receiver_pop(uwspr_b200_array_receiver *rx, int32_t *channel, int64_t *window,
                                                 uwspr_b200_candidate_t *cand, int8_t *message7);
/* windows processed per channel */
UWSPR_B200_API int64_t uwspr_b200_array_receiver_windows(const uwspr_b200_array_receiver *rx);
/* kernel launches issued so far (front-end, search and decoder) */
UWSPR_B200_API int64_t uwspr_b200_array_receiver_launch_count(const uwspr_b200_array_receiver *rx);
UWSPR_B200_API void uwspr_b200_array_receiver_destroy(uwspr_b200_array_receiver *rx);

/* ---- utilities ------------------------------------------------------------------------- */
/* pinned host memory for sample / result buffers (cudaHostAlloc / cudaFreeHost) */
UWSPR_B200_API int uwspr_b200_host_alloc(void **ptr, size_t bytes);
UWSPR_B200_API void uwspr_b200_host_free(void *ptr);

/* Run all kernels on the caller's CUDA stream (a cudaStream_t passed as void*), so that
 * events the caller records on that stream bracket the work; NULL restores the context's
 * own stream.  Calls remain synchronous with respect to the host. */
UWSPR_B200_API int uwspr_b200_set_stream(uwspr_b200_ctx *ctx, void *cuda_stream);

/* keep_power != 0: later coarse calls also keep |X|^2 of the kept bins for
 * uwspr_b200_debug_spectrogram (costs one extra device buffer and its writes) */
UWSPR_B200_API int uwspr_b200_set_debug(uwspr_b200_ctx *ctx, int keep_power);

/* test hook: power spectrogram rows of window `win` of the last coarse call, restricted to
 * the kept bins: ps[n_rows][n_bins] (FDR_impl.cc:246-253), and psavg[n_bins] (:257-263) */
UWSPR_B200_API int uwspr_b200_debug_spectrogram(uwspr_b200_ctx *ctx, int win, float *ps, float *psavg);

/* device time, in ms, of the stages of the last call (CUDA events on the context's stream):
 * [0] spectrogram+normalizer+peaks, [1] coarse search, [2] fine sync + soft symbols, [3] whole call
 * including copies */
UWSPR_B200_API int uwspr_b200_last_timing(const uwspr_b200_ctx *ctx, float ms[4]);
/* number of kernel launches issued by this context so far */
UWSPR_B200_API int64_t uwspr_b200_launch_count(const uwspr_b200_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* UWSPR_B200_H */
