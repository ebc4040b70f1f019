"""uwspr_b200 -- Python face of libuwspr_b200.so (ctypes over the C ABI in include/uwspr_b200.h).

Mirrors the two reference blocks on the hot path:

    FDR(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold)   (include/uwspr/FDR.h:49-50)
    sync_and_demodulate(fs, fl, spb, maxdrift, maxfreqs, cf)             (include/uwspr/sync_and_demodulate.h:49)

There is no CPU fallback: importing works anywhere, but constructing a context needs the
in-tree CUDA library and a CUDA device, and fails loudly otherwise.
"""
from .binding import (  # noqa: F401
    CAND_DTYPE, JIG_DTYPE, REFINED_DTYPE, NJIG, NSYM, Context, FDR, UwsprError, lib_path, load_library,
    sync_and_demodulate, deinterleave, fano, fano_batch, decode_candidates, EXPORTED_SYMBOLS, Receiver, ArrayReceiver, FrontendStream,
    WSPR_unpacker,
    pack_type1, channel_symbols, format_message_log, read_c2, frontend, lowpass_taps, flowgraph_taps, firdes_low_pass, firdes_band_pass, resampler_taps,
)
