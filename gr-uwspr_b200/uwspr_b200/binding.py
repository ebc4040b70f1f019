import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
NSYM = 162
NJIG = 17
HOST, DEVICE = 0, 1

# every symbol include/uwspr_b200.h declares
EXPORTED_SYMBOLS = [
    "uwspr_b200_create", "uwspr_b200_destroy", "uwspr_b200_last_error", "uwspr_b200_status_string",
    "uwspr_b200_create_error", "uwspr_b200_info", "uwspr_b200_coarse", "uwspr_b200_fine", "uwspr_b200_coarse_fine",
    "uwspr_b200_deinterleave", "uwspr_b200_fano", "uwspr_b200_decode_candidate", "uwspr_b200_decode_batch",
    "uwspr_b200_host_alloc",
    "uwspr_b200_host_free", "uwspr_b200_set_stream", "uwspr_b200_set_debug", "uwspr_b200_debug_spectrogram",
    "uwspr_b200_last_timing", "uwspr_b200_launch_count",
    "uwspr_b200_receiver_create", "uwspr_b200_receiver_destroy", "uwspr_b200_receiver_push", "uwspr_b200_receiver_pop",
    "uwspr_b200_receiver_windows", "uwspr_b200_hashtab_bytes", "uwspr_b200_unpack", "uwspr_b200_format_message_log",
    "uwspr_b200_pack_type1", "uwspr_b200_channel_symbols", "uwspr_b200_read_c2", "uwspr_b200_frontend", "uwspr_b200_frontend_ctaps",
    "uwspr_b200_frontend_error", "uwspr_b200_coarse_fine_submit", "uwspr_b200_poll", "uwspr_b200_wait",
    "uwspr_b200_decode_device", "uwspr_b200_fano_batch",
    "uwspr_b200_frontend_stream_create", "uwspr_b200_frontend_stream_push", "uwspr_b200_frontend_stream_outputs",
    "uwspr_b200_frontend_stream_destroy", "uwspr_b200_array_receiver_create", "uwspr_b200_array_receiver_push",
    "uwspr_b200_array_receiver_pop", "uwspr_b200_array_receiver_windows", "uwspr_b200_array_receiver_launch_count",
    "uwspr_b200_array_receiver_destroy", "uwspr_b200_beamform", "uwspr_b200_array_receiver_create_beams",
]

CAND_DTYPE = np.dtype(
    {
        # candidate_t of the reference (lib/candidate_t.h:27-50)
        "names": ["freq", "snr", "drift", "sync", "shift", "m_type", "lin_drift", "V1", "V2", "p1", "p2"],
        "formats": ["<f4", "<f4", "<f4", "<f4", "<i4", "<i4", "<f4", "<f8", "<f8", "<i4", "<i4"],
        "offsets": [0, 4, 8, 12, 16, 20, 24, 24, 32, 40, 44],
        "itemsize": 48,
    }
)
REFINED_DTYPE = np.dtype([("f1", "<f4"), ("shift1", "<i4"), ("drift1", "<f4"), ("sync1", "<f4"), ("worth_a_try", "<i4"), ("reserved", "<i4")])
JIG_DTYPE = np.dtype([("sync", "<f4"), ("rms", "<f4"), ("shift", "<i4"), ("gate", "<i4")])


class Params(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "fs", "fl", "spb", "maxdrift", "maxfreqs", "halfbandwidth", "cf", "threshold",
        "device", "max_windows", "max_candidates", "nonlinear_intended_t")]


class Input(C.Structure):
    _fields_ = [("kind", C.c_int32), ("taps", C.c_void_p), ("ntaps", C.c_int32), ("complex_taps", C.c_int32),
                ("decim", C.c_int32), ("delay", C.c_int32), ("fc", C.c_double), ("fs_in", C.c_double)]


class Beams(C.Structure):
    _fields_ = [("nbeam", C.c_int32), ("weights", C.c_void_p), ("delays", C.c_void_p)]


class Info(C.Structure):
    _fields_ = [
        ("size", C.c_int32), ("m", C.c_int32), ("hpbm", C.c_int32), ("n_rows", C.c_int32), ("finpb", C.c_int32),
        ("noiseidx", C.c_int32), ("df", C.c_float), ("min_snr", C.c_float), ("bin_lo", C.c_int32), ("n_bins", C.c_int32),
        ("n_lin", C.c_int32), ("n_unique", C.c_int32), ("max_cand_per_window", C.c_int32), ("max_windows", C.c_int32),
        ("max_candidates", C.c_int32), ("sm_count", C.c_int32),
    ]


class UwsprError(RuntimeError):
    def __init__(self, status, text):
        super().__init__("uwspr_b200 status %d: %s" % (status, text))
        self.status = status


def lib_path():
    # UWSPR_B200_LIB selects another build of the same library (to compare another build with this one)
    return os.environ.get("UWSPR_B200_LIB") or os.path.join(os.path.dirname(_HERE), "libuwspr_b200.so")


_lib = None


def load_library():
    """loads the in-tree CUDA library; raises if it has not been built (no fallback)"""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise UwsprError(-1, "libuwspr_b200.so is not built (run __graft_entry__.build() or make -C gr-uwspr_b200); "
                             "there is no CPU fallback for the CUDA path")
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.uwspr_b200_create.restype = C.c_int
    L.uwspr_b200_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.uwspr_b200_destroy.argtypes = [vp]
    L.uwspr_b200_last_error.restype = C.c_char_p
    L.uwspr_b200_last_error.argtypes = [vp]
    L.uwspr_b200_status_string.restype = C.c_char_p
    L.uwspr_b200_status_string.argtypes = [C.c_int]
    L.uwspr_b200_create_error.restype = C.c_char_p
    L.uwspr_b200_info.restype = C.c_int
    L.uwspr_b200_info.argtypes = [vp, C.POINTER(Info)]
    L.uwspr_b200_coarse.restype = C.c_int
    L.uwspr_b200_coarse.argtypes = [vp, vp, C.c_int, i64, C.c_int, vp, vp, C.c_int, vp]
    L.uwspr_b200_fine.restype = C.c_int
    L.uwspr_b200_fine.argtypes = [vp, vp, C.c_int, i64, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.uwspr_b200_coarse_fine.restype = C.c_int
    L.uwspr_b200_coarse_fine.argtypes = [vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp, vp, vp]
    L.uwspr_b200_coarse_fine_submit.restype = C.c_int
    L.uwspr_b200_coarse_fine_submit.argtypes = L.uwspr_b200_coarse_fine.argtypes
    L.uwspr_b200_poll.restype = C.c_int
    L.uwspr_b200_poll.argtypes = [vp]
    L.uwspr_b200_wait.restype = C.c_int
    L.uwspr_b200_wait.argtypes = [vp]
    L.uwspr_b200_deinterleave.argtypes = [vp]
    L.uwspr_b200_fano.restype = C.c_int
    L.uwspr_b200_fano.argtypes = [vp, vp, vp, vp, vp, C.c_uint32, C.c_int, C.c_uint32]
    L.uwspr_b200_decode_candidate.restype = C.c_int
    L.uwspr_b200_decode_candidate.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp]
    L.uwspr_b200_decode_batch.restype = C.c_int
    L.uwspr_b200_decode_batch.argtypes = [vp, vp, vp, C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp]
    L.uwspr_b200_decode_device.restype = C.c_int
    L.uwspr_b200_decode_device.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp]
    L.uwspr_b200_fano_batch.restype = C.c_int
    L.uwspr_b200_fano_batch.argtypes = [vp, vp, C.c_int, C.c_int64, C.c_uint32, C.c_int, C.c_uint32, vp, vp, vp, vp, vp]
    L.uwspr_b200_pack_type1.restype = C.c_int
    L.uwspr_b200_pack_type1.argtypes = [C.c_char_p, C.c_char_p, C.c_int, vp]
    L.uwspr_b200_channel_symbols.restype = None
    L.uwspr_b200_channel_symbols.argtypes = [vp, vp]
    L.uwspr_b200_read_c2.restype = C.c_int
    L.uwspr_b200_read_c2.argtypes = [C.c_char_p, vp, vp, vp, vp]
    L.uwspr_b200_frontend.restype = C.c_int
    L.uwspr_b200_frontend.argtypes = [C.c_int, vp, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int64, vp, C.c_int, C.c_int,
                                      C.c_int, C.c_double, C.c_double, vp, C.c_int, C.c_int64, vp]
    L.uwspr_b200_frontend_ctaps.restype = C.c_int
    L.uwspr_b200_frontend_ctaps.argtypes = L.uwspr_b200_frontend.argtypes
    L.uwspr_b200_frontend_error.restype = C.c_char_p
    L.uwspr_b200_host_alloc.restype = C.c_int
    L.uwspr_b200_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    L.uwspr_b200_host_free.argtypes = [vp]
    L.uwspr_b200_set_stream.restype = C.c_int
    L.uwspr_b200_set_stream.argtypes = [vp, vp]
    L.uwspr_b200_set_debug.restype = C.c_int
    L.uwspr_b200_set_debug.argtypes = [vp, C.c_int]
    L.uwspr_b200_debug_spectrogram.restype = C.c_int
    L.uwspr_b200_debug_spectrogram.argtypes = [vp, C.c_int, vp, vp]
    L.uwspr_b200_last_timing.restype = C.c_int
    L.uwspr_b200_last_timing.argtypes = [vp, vp]
    L.uwspr_b200_launch_count.restype = i64
    L.uwspr_b200_launch_count.argtypes = [vp]
    L.uwspr_b200_receiver_create.restype = C.c_int
    L.uwspr_b200_receiver_create.argtypes = [C.POINTER(Params), C.c_int, C.c_int, C.POINTER(vp)]
    L.uwspr_b200_receiver_destroy.argtypes = [vp]
    L.uwspr_b200_receiver_push.restype = C.c_int
    L.uwspr_b200_receiver_push.argtypes = [vp, vp, i64, C.c_int]
    L.uwspr_b200_receiver_pop.restype = C.c_int
    L.uwspr_b200_receiver_pop.argtypes = [vp, vp, vp, vp]
    L.uwspr_b200_receiver_windows.restype = i64
    L.uwspr_b200_receiver_windows.argtypes = [vp]
    L.uwspr_b200_frontend_stream_create.restype = C.c_int
    L.uwspr_b200_frontend_stream_create.argtypes = [C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                                    C.c_double, C.POINTER(vp)]
    L.uwspr_b200_frontend_stream_push.restype = C.c_int
    L.uwspr_b200_frontend_stream_push.argtypes = [vp, vp, C.c_int, i64, i64, vp, C.c_int, i64, i64, C.POINTER(i64)]
    L.uwspr_b200_frontend_stream_outputs.restype = i64
    L.uwspr_b200_frontend_stream_outputs.argtypes = [vp]
    L.uwspr_b200_frontend_stream_destroy.argtypes = [vp]
    L.uwspr_b200_array_receiver_create.restype = C.c_int
    L.uwspr_b200_array_receiver_create.argtypes = [C.POINTER(Params), C.POINTER(Input), C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.uwspr_b200_array_receiver_push.restype = C.c_int
    L.uwspr_b200_array_receiver_push.argtypes = [vp, vp, C.c_int, i64, i64, C.c_int]
    L.uwspr_b200_array_receiver_pop.restype = C.c_int
    L.uwspr_b200_array_receiver_pop.argtypes = [vp, vp, vp, vp, vp]
    L.uwspr_b200_array_receiver_windows.restype = i64
    L.uwspr_b200_array_receiver_windows.argtypes = [vp]
    L.uwspr_b200_array_receiver_launch_count.restype = i64
    L.uwspr_b200_array_receiver_launch_count.argtypes = [vp]
    L.uwspr_b200_array_receiver_destroy.argtypes = [vp]
    L.uwspr_b200_array_receiver_create_beams.restype = C.c_int
    L.uwspr_b200_array_receiver_create_beams.argtypes = [C.POINTER(Params), C.POINTER(Input), C.c_int, C.POINTER(Beams), C.c_int,
                                                         C.c_int, C.POINTER(vp)]
    L.uwspr_b200_beamform.restype = C.c_int
    L.uwspr_b200_beamform.argtypes = [C.c_int, vp, C.c_int, i64, C.c_int, i64, vp, vp, C.c_int, vp, C.c_int, i64]
    L.uwspr_b200_hashtab_bytes.restype = C.c_size_t
    L.uwspr_b200_unpack.restype = C.c_int
    L.uwspr_b200_unpack.argtypes = [vp, vp, vp, C.c_size_t]
    _lib = L
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _buffer_arg(a, dtype):
    """(pointer, space, keep-alive, byte size) of a numpy array (host) or a contiguous CUDA tensor (device)"""
    if hasattr(a, "data_ptr") and getattr(a, "is_cuda", False):
        if not a.is_contiguous():
            raise ValueError("CUDA tensors must be contiguous")
        return C.c_void_p(a.data_ptr()), DEVICE, a, a.numel() * a.element_size()
    h = np.ascontiguousarray(a, dtype=dtype)
    return _p(h), HOST, h, h.nbytes


def _samples_arg(samples):
    """accepts a numpy complex64 array (host) or (device_pointer:int, n_complex:int) for device memory"""
    if isinstance(samples, tuple):
        return C.c_void_p(int(samples[0])), DEVICE, None
    a = np.ascontiguousarray(samples, dtype=np.complex64)
    return _p(a), HOST, a


class Context:
    """one uwspr_b200_ctx: both blocks' arithmetic for batches of windows on one GPU"""

    def __init__(self, fs=375, fl=45000, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10,
                 device=0, max_windows=1, max_candidates=0, nonlinear_intended_t=0):
        self.L = load_library()
        self.prm = Params(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, device, max_windows,
                          max_candidates, nonlinear_intended_t)
        h = C.c_void_p()
        st = self.L.uwspr_b200_create(C.byref(self.prm), C.byref(h))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_create_error().decode() or self.L.uwspr_b200_status_string(st).decode())
        self.h = h
        self.fl = fl
        self._pinned = []
        self._fine = None          # (candidate total, jiggle count) of the fine results on the device
        self._coarse_total = 0     # candidates of the list on the device
        inf = Info()
        self._check(self.L.uwspr_b200_info(self.h, C.byref(inf)))
        self.info = inf

    def _check(self, st):
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_last_error(self.h).decode() or self.L.uwspr_b200_status_string(st).decode())

    def close(self):
        if getattr(self, "h", None):
            for ptr in getattr(self, "_pinned", []):
                self.L.uwspr_b200_host_free(ptr)
            self._pinned = []
            self.L.uwspr_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        self._check(self.L.uwspr_b200_set_stream(self.h, C.c_void_p(cuda_stream_ptr) if cuda_stream_ptr else None))

    def set_debug(self, on=True):
        self._check(self.L.uwspr_b200_set_debug(self.h, int(on)))

    def _nwin(self, samples, nwin, stride):
        if nwin is not None:
            return nwin
        a = np.asarray(samples)
        if a.ndim == 2:
            return a.shape[0]
        return 1 + (a.size - self.fl) // stride

    # ---- FDR_impl::transform for a batch --------------------------------------------------
    def coarse(self, samples, nwin=None, stride=None, fetch=True):
        stride = self.fl if stride is None else stride
        ptr, space, keep = _samples_arg(samples)
        nwin = self._nwin(samples, nwin, stride) if not isinstance(samples, tuple) else nwin
        cap = self.info.max_candidates
        npk = np.zeros(nwin, np.int32) if fetch else None
        cands = np.zeros(cap, CAND_DTYPE) if fetch else None
        total = C.c_int32(0)
        self._check(self.L.uwspr_b200_coarse(self.h, ptr, space, stride, nwin, _p(npk), _p(cands), cap, C.byref(total)))
        self._fine = None
        self._coarse_total = total.value
        if not fetch:
            return total.value
        return npk, cands[: total.value].copy()

    # ---- demodulate() up to the decoder ---------------------------------------------------
    def fine(self, samples, npk=None, cands=None, nwin=None, stride=None, jig_first=0, jig_count=NJIG, fetch=True):
        stride = self.fl if stride is None else stride
        ptr, space, keep = _samples_arg(samples)
        nwin = self._nwin(samples, nwin, stride) if not isinstance(samples, tuple) else nwin
        if cands is not None:
            cands = np.ascontiguousarray(cands, dtype=CAND_DTYPE)
            npk = np.ascontiguousarray(npk, dtype=np.int32)
            total = len(cands)
        else:
            total = 0
        n_out = total if cands is not None else self.info.max_candidates
        refined = np.zeros(n_out, REFINED_DTYPE) if fetch else None
        jig = np.zeros((n_out, jig_count), JIG_DTYPE) if fetch else None
        soft = np.zeros((n_out, jig_count, NSYM), np.uint8) if fetch else None
        self._check(self.L.uwspr_b200_fine(self.h, ptr, space, stride, nwin, _p(npk), _p(cands), total, jig_first,
                                           jig_count, _p(refined), _p(jig), _p(soft)))
        self._fine = (total if cands is not None else self._coarse_total, jig_count)
        return refined, jig, soft

    def result_buffers(self, nwin, jig_count=NJIG, pinned=True):
        """caller-owned result buffers for coarse_fine(out=...), page-locked so the device->host
        copies run at link speed (cudaHostAlloc through uwspr_b200_host_alloc)"""
        cap = self.info.max_candidates
        spec = [("npk", (nwin,), np.dtype(np.int32)), ("cands", (cap,), CAND_DTYPE), ("refined", (cap,), REFINED_DTYPE),
                ("jig", (cap, jig_count), JIG_DTYPE), ("soft", (cap, jig_count, NSYM), np.dtype(np.uint8))]
        out = {}
        for name, shape, dt in spec:
            n = int(np.prod(shape)) * dt.itemsize
            if pinned:
                ptr = C.c_void_p()
                st = self.L.uwspr_b200_host_alloc(C.byref(ptr), max(n, 1))
                if st != 0:
                    raise UwsprError(st, "cannot allocate pinned host memory")
                raw = (C.c_ubyte * max(n, 1)).from_address(ptr.value)
                self._pinned.append(ptr)
                out[name] = np.frombuffer(raw, dtype=dt, count=int(np.prod(shape))).reshape(shape)
            else:
                out[name] = np.zeros(shape, dt)
        return out

    def coarse_fine(self, samples, nwin=None, stride=None, jig_first=0, jig_count=NJIG, fetch=True, out=None):
        stride = self.fl if stride is None else stride
        ptr, space, keep = _samples_arg(samples)
        nwin = self._nwin(samples, nwin, stride) if not isinstance(samples, tuple) else nwin
        cap = self.info.max_candidates
        total = C.c_int32(0)
        if not fetch:
            self._check(self.L.uwspr_b200_coarse_fine(self.h, ptr, space, stride, nwin, jig_first, jig_count, None, None,
                                                      0, C.byref(total), None, None, None))
            self._fine = (total.value, jig_count)
            self._coarse_total = total.value
            return total.value
        if out is not None:
            # views into the caller's buffers, no copies
            self._check(self.L.uwspr_b200_coarse_fine(self.h, ptr, space, stride, nwin, jig_first, jig_count,
                                                      _p(out["npk"]), _p(out["cands"]), cap, C.byref(total),
                                                      _p(out["refined"]), _p(out["jig"]), _p(out["soft"])))
            t = total.value
            self._fine = (t, jig_count)
            self._coarse_total = t
            return out["npk"][:nwin], out["cands"][:t], out["refined"][:t], out["jig"][:t], out["soft"][:t]
        npk = np.zeros(nwin, np.int32)
        cands = np.zeros(cap, CAND_DTYPE)
        refined = np.zeros(cap, REFINED_DTYPE)
        jig = np.zeros((cap, jig_count), JIG_DTYPE)
        soft = np.zeros((cap, jig_count, NSYM), np.uint8)
        self._check(self.L.uwspr_b200_coarse_fine(self.h, ptr, space, stride, nwin, jig_first, jig_count, _p(npk),
                                                  _p(cands), cap, C.byref(total), _p(refined), _p(jig), _p(soft)))
        t = total.value
        self._fine = (t, jig_count)
        self._coarse_total = t
        return npk, cands[:t].copy(), refined[:t].copy(), jig[:t].copy(), soft[:t].copy()

    def submit(self, samples, out, nwin=None, stride=None, jig_first=0, jig_count=NJIG):
        """non-blocking coarse_fine into the caller's result buffers (result_buffers()); returns at once.
        wait() returns the same tuple coarse_fine(out=...) returns; poll() says whether it is ready."""
        stride = self.fl if stride is None else stride
        ptr, space, keep = _samples_arg(samples)
        nwin = self._nwin(samples, nwin, stride) if not isinstance(samples, tuple) else nwin
        total = C.c_int32(0)
        self._pending = (keep, out, nwin, total, jig_count)
        self._check(self.L.uwspr_b200_coarse_fine_submit(self.h, ptr, space, stride, nwin, jig_first, jig_count, _p(out["npk"]),
                                                         _p(out["cands"]), self.info.max_candidates, C.byref(total),
                                                         _p(out["refined"]), _p(out["jig"]), _p(out["soft"])))

    def poll(self):
        return int(self.L.uwspr_b200_poll(self.h))

    def wait(self):
        keep, out, nwin, total, jig_count = self._pending
        self._check(self.L.uwspr_b200_wait(self.h))
        self._pending = None
        t = total.value
        self._fine = (t, jig_count)
        self._coarse_total = t
        return out["npk"][:nwin], out["cands"][:t], out["refined"][:t], out["jig"][:t], out["soft"][:t]

    # ---- the decoder on the device ---------------------------------------------------------
    def decode(self, refined=None, jig=None, soft=None, jig_count=NJIG, cycles=False):
        """uwspr_b200_decode_device: the list decode_candidates() returns -- (candidate index, 7-byte message, idt
        used) per decoded candidate, in candidate order -- and with cycles=True also the decoder cycles of every
        candidate (a uint32 array), as (list, cycles).  Without inputs it decodes the results the last fine /
        coarse_fine call left on the device (jig_count must be that call's); otherwise refined [n], jig [n, jig_count]
        and soft [n, jig_count, 162] are numpy arrays (host) or contiguous CUDA tensors holding the same bytes."""
        if refined is None and jig is None and soft is None:
            ncand = self._fine[0] if self._fine else 0
            args, space = (None, None, None), HOST
        else:
            r, space, kr, nbytes = _buffer_arg(refined, REFINED_DTYPE)
            j, sj, kj, _ = _buffer_arg(jig, JIG_DTYPE)
            s, ss, ks, _ = _buffer_arg(soft, np.uint8)
            if not space == sj == ss:
                raise ValueError("refined, jig and soft must all be on the host or all on the device")
            ncand = nbytes // REFINED_DTYPE.itemsize
            args = (r, j, s)
        n = max(ncand, 1)
        decoded = np.zeros(n, np.uint8)
        msgs = np.zeros((n, 7), np.int8)
        idt = np.zeros(n, np.int32)
        cyc = np.zeros(n, np.uint32)
        got = self.L.uwspr_b200_decode_device(self.h, *args, space, ncand, jig_count, _p(decoded), _p(msgs), _p(idt), _p(cyc))
        if got < 0:
            self._check(-got)
        out = [(int(g), msgs[g].view(np.uint8).copy(), int(idt[g])) for g in np.flatnonzero(decoded[:ncand])]
        return (out, cyc[:ncand].copy()) if cycles else out

    def debug_spectrogram(self, win=0):
        ps = np.zeros((self.info.n_rows, self.info.n_bins), np.float32)
        psavg = np.zeros(self.info.n_bins, np.float32)
        self._check(self.L.uwspr_b200_debug_spectrogram(self.h, win, _p(ps), _p(psavg)))
        return ps, psavg

    def last_timing(self):
        ms = (C.c_float * 4)()
        self._check(self.L.uwspr_b200_last_timing(self.h, ms))
        return [float(v) for v in ms]

    def launch_count(self):
        return int(self.L.uwspr_b200_launch_count(self.h))


def deinterleave(sym):
    s = np.array(sym, dtype=np.uint8, copy=True)
    load_library().uwspr_b200_deinterleave(_p(s))
    return s


def fano(symbols, delta=60, maxcycles=10000, nbits=81):
    s = np.ascontiguousarray(symbols, dtype=np.uint8)
    data = np.zeros(11, np.uint8)
    metric, cycles, maxnp = C.c_uint32(), C.c_uint32(), C.c_uint32()
    r = load_library().uwspr_b200_fano(C.byref(metric), C.byref(cycles), C.byref(maxnp), _p(data), _p(s), nbits, delta, maxcycles)
    return r, data, metric.value, cycles.value, maxnp.value


def fano_batch(ctx, symbols, delta=60, maxcycles=10000, nbits=81):
    """uwspr_b200_fano_batch: fano() on every row of symbols [n, 162] (de-interleaved; numpy or a CUDA tensor) on
    ctx's device.  Returns arrays mirroring fano()'s tuple: status [n] (0 / -1), data [n, 11], metric, cycles,
    maxnp [n]."""
    ptr, space, keep, nbytes = _buffer_arg(symbols, np.uint8)
    n = nbytes // NSYM
    status = np.zeros(n, np.int32)
    data = np.zeros((n, 11), np.uint8)
    metric, cycles, maxnp = (np.zeros(n, np.uint32) for _ in range(3))
    ctx._check(ctx.L.uwspr_b200_fano_batch(ctx.h, ptr, space, n, nbits, delta, maxcycles, _p(status), _p(metric),
                                           _p(cycles), _p(maxnp), _p(data)))
    return status, data, metric, cycles, maxnp


def decode_candidates(refined, jig, soft, nthreads=0):
    """the peak-up/decode loop (sync_and_demodulate_impl.cc:457-490) over fetched results, spread over
    `nthreads` host threads (0: all cores); returns a list of (candidate index, 7-byte message, idt used)
    in candidate order"""
    L = load_library()
    jig = np.ascontiguousarray(jig)
    soft = np.ascontiguousarray(soft)
    refined = np.ascontiguousarray(refined)
    n = len(refined)
    if n == 0:
        return []
    decoded = np.zeros(n, np.uint8)
    msgs = np.zeros((n, 7), np.int8)
    idt = np.zeros(n, np.int32)
    got = L.uwspr_b200_decode_batch(_p(refined), _p(jig), _p(soft), n, jig.shape[1], int(nthreads), _p(decoded),
                                    _p(msgs), _p(idt), None)
    if got < 0:
        raise UwsprError(-got, L.uwspr_b200_status_string(-got).decode())
    return [(int(g), msgs[g].view(np.uint8).copy(), int(idt[g])) for g in np.flatnonzero(decoded)]


class FDR:
    """uwspr.FDR: same constructor arguments as the reference block (include/uwspr/FDR.h:49-50).
    transform(window) -> candidate array, as FDR_impl::transform publishes it."""

    def __init__(self, fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, device=0, max_windows=1, ctx=None):
        self.ctx = ctx or Context(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, device=device,
                                  max_windows=max_windows)

    def transform(self, window):
        npk, cands = self.ctx.coarse(np.asarray(window).reshape(1, -1))
        return cands


class sync_and_demodulate:
    """uwspr.sync_and_demodulate (include/uwspr/sync_and_demodulate.h:49).
    demodulate(window, candidates) -> list of 7-byte messages, one per decoded candidate, in
    candidate order (sync_and_demodulate_impl.cc:389-531)."""

    def __init__(self, fs, fl, spb, maxdrift, maxfreqs, cf, device=0, ctx=None):
        self.ctx = ctx or Context(fs, fl, spb, maxdrift, maxfreqs, 10, cf, 10, device=device, max_windows=1,
                                  max_candidates=max(1, maxfreqs))

    def demodulate(self, window, candidates):
        cands = np.ascontiguousarray(candidates, dtype=CAND_DTYPE)
        if len(cands) == 0:
            return []
        npk = np.array([len(cands)], np.int32)
        refined, jig, soft = self.ctx.fine(np.asarray(window).reshape(1, -1), npk, cands)
        return [m for _, m, _ in decode_candidates(refined, jig, soft)]


class Receiver:
    """batched receive chain of one stream: sliding window (shift seconds) -> device -> host decoder"""

    def __init__(self, fs=375, fl=45000, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10,
                 shift=9, batch_windows=16, device=0):
        self.L = load_library()
        prm = Params(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, device, batch_windows, 0, 0)
        h = C.c_void_p()
        st = self.L.uwspr_b200_receiver_create(C.byref(prm), shift, batch_windows, C.byref(h))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_create_error().decode() or self.L.uwspr_b200_status_string(st).decode())
        self.h = h

    def push(self, samples, flush=False):
        a = np.ascontiguousarray(samples, dtype=np.complex64)
        st = self.L.uwspr_b200_receiver_push(self.h, _p(a), a.size, int(flush))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_status_string(st).decode())
        out = []
        msg = np.zeros(7, np.int8)
        win = C.c_int64()
        cand = np.zeros(1, CAND_DTYPE)
        while self.L.uwspr_b200_receiver_pop(self.h, _p(msg), C.byref(win), _p(cand)):
            out.append((win.value, msg.view(np.uint8).copy(), cand[0].copy()))
        return out

    def windows_done(self):
        return int(self.L.uwspr_b200_receiver_windows(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.uwspr_b200_receiver_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def read_c2(path):
    """uwspr.c2file_source's reader: (complex64[45000] = I - jQ, name, type, dial frequency in MHz)"""
    iq = np.zeros(45000, np.complex64)
    name = C.create_string_buffer(15)
    typ, freq = C.c_int32(), C.c_double()
    st = load_library().uwspr_b200_read_c2(os.fsencode(path), _p(iq), name, C.byref(typ), C.byref(freq))
    if st != 0:
        raise UwsprError(st, "cannot read 45000 samples from %r" % (path,))
    return iq, name.value.decode("latin1"), typ.value, freq.value


def lowpass_taps(ntaps=513, cutoff=150.0, fs_in=12000.0):
    """Hamming-windowed sinc low-pass with unit DC gain (what gnuradio.filter.firdes.low_pass designs)"""
    k = np.arange(ntaps) - (ntaps - 1) / 2
    h = np.sinc(2 * cutoff / fs_in * k) * np.hamming(ntaps)
    return (h / h.sum()).astype(np.float32)


def _window(name, ntaps, beta):
    """gr::filter::firdes::window (firdes.cc, GNU Radio 3.7): Hamming 0.54 - 0.46 cos(2 pi n / (N-1)); Kaiser
    I0(beta sqrt(1 - (2n/(N-1) - 1)^2)) / I0(beta)"""
    n = np.arange(ntaps, dtype=np.float64)
    if name == "hamming":
        return 0.54 - 0.46 * np.cos(2 * np.pi * n / (ntaps - 1))
    t = 2 * n / (ntaps - 1) - 1
    return np.i0(beta * np.sqrt(np.maximum(0.0, 1 - t * t))) / np.i0(beta)


def _ntaps(fs, width, window, beta):
    """firdes::compute_ntaps: attenuation of the window (Hamming 53 dB, Kaiser beta/0.1102 + 8.7) * fs / (22 width),
    made odd"""
    att = 53.0 if window == "hamming" else beta / 0.1102 + 8.7
    n = int(att * fs / (22.0 * width))
    return n | 1


def firdes_low_pass(gain, fs, cutoff, width, window="hamming", beta=6.76):
    """gnuradio.filter.firdes.low_pass: windowed sinc, unit gain at DC times `gain`"""
    nt = _ntaps(fs, width, window, beta)
    m = (nt - 1) // 2
    n = np.arange(-m, m + 1, dtype=np.float64)
    w0 = 2 * np.pi * cutoff / fs
    h = np.where(n == 0, w0 / np.pi, np.sin(n * w0) / np.where(n == 0, 1.0, n * np.pi)) * _window(window, nt, beta)
    return h * (gain / h.sum())


def firdes_band_pass(gain, fs, low, high, width, window="hamming", beta=6.76):
    """gnuradio.filter.firdes.band_pass: difference of two windowed sincs, unit gain at the band centre"""
    nt = _ntaps(fs, width, window, beta)
    m = (nt - 1) // 2
    n = np.arange(-m, m + 1, dtype=np.float64)
    w0, w1 = 2 * np.pi * low / fs, 2 * np.pi * high / fs
    h = np.where(n == 0, (w1 - w0) / np.pi, (np.sin(n * w1) - np.sin(n * w0)) / np.where(n == 0, 1.0, n * np.pi))
    h = h * _window(window, nt, beta)
    return h * (gain / (h * np.cos(n * (w0 + w1) * 0.5)).sum())


def resampler_taps(interp, decim, fractional_bw=0.4):
    """gnuradio.filter.rational_resampler.design_filter: Kaiser (beta 7) low-pass at the narrower of the two rates"""
    rate = float(interp) / float(decim)
    if rate >= 1.0:
        width = 0.5 - fractional_bw
        mid = 0.5 - width / 2
    else:
        width = rate * (0.5 - fractional_bw)
        mid = rate * 0.5 - width / 2
    return firdes_low_pass(interp, interp, mid, width, "kaiser", 7.0)


def flowgraph_taps(fs_in=12000.0, fc=1500.0, half_bandwidth=10.0, width=10.0, decim=32):
    """Composite complex taps of the reference flowgraph's front-end (examples/WaveFilePlusNoiseDecode.grc): band-pass
    fc -+ half_bandwidth at centre 0 (:322-383, :834-893), translation by fc with a low-pass at fc + half_bandwidth
    (:384-420, :894-958), rational resampler 1/decim with its default taps (:1753-1810).  With x'[n] = x[n] e^{-iwn}
    the cascade is y[m] = sum_j g[j] x'[m decim - j], g = (h_bp[k] e^{-iwk}) * h_lp * h_rs: pass g to frontend() with
    delay 0."""
    h1 = firdes_band_pass(1.0, fs_in, fc - half_bandwidth, fc + half_bandwidth, width)
    h2 = firdes_low_pass(1.0, fs_in, fc + half_bandwidth, width)
    h3 = resampler_taps(1, decim)
    w = 2 * np.pi * fc / fs_in
    g = np.convolve(np.convolve(h1 * np.exp(-1j * w * np.arange(len(h1))), h2), h3)
    return g.astype(np.complex64)


def frontend(audio, taps=None, decim=32, fc=1500.0, fs_in=12000.0, delay=None, device=0, out_device_ptr=None,
             out_stride=None):
    """real audio [nchan, n] or [n] (float32, or int16 PCM) at fs_in -> complex64 at fs_in/decim on the GPU
    (uwspr_b200_frontend, or uwspr_b200_frontend_ctaps when the taps are complex).  `audio` may be a numpy array or a
    (device pointer, dtype, shape) tuple; the result is a numpy array, or stays on the device when out_device_ptr is
    given.  delay defaults to the filter's group delay."""
    L = load_library()
    taps, ctaps, delay = _frontend_taps(taps, fs_in, delay)
    if isinstance(audio, tuple):
        ptr, dtype, shape = audio
        space_in = 1
    else:
        a = np.ascontiguousarray(audio)
        if a.dtype != np.int16:
            a = np.ascontiguousarray(a, dtype=np.float32)
        ptr, dtype, shape, space_in = _p(a), a.dtype, a.shape, 0
    fmt = 1 if np.dtype(dtype) == np.int16 else 0
    nchan, n_in = (1, shape[0]) if len(shape) == 1 else shape
    n_out = n_in // decim if decim > 0 else 0   # the library reports the bad argument
    stride = n_out if out_stride is None else int(out_stride)
    got = C.c_int64()
    if out_device_ptr is None:
        out = np.zeros((nchan, stride), np.complex64)
        optr, space_out = _p(out), 0
    else:
        out, optr, space_out = None, C.c_void_p(int(out_device_ptr)), 1
    entry = L.uwspr_b200_frontend_ctaps if ctaps else L.uwspr_b200_frontend
    st = entry(device, ptr, fmt, space_in, n_in, nchan, n_in, _p(taps), len(taps), decim, delay, fc, fs_in,
               optr, space_out, stride, C.byref(got))
    if st != 0:
        raise UwsprError(st, L.uwspr_b200_frontend_error().decode())
    if out is None:
        return got.value
    out = out[:, :got.value]
    return out[0] if len(shape) == 1 else out


def _frontend_taps(taps, fs_in, delay):
    """(taps as float32 array, complex?, delay): complex taps go as (re, im) pairs; delay defaults to the group delay"""
    ctaps = taps is not None and np.iscomplexobj(taps)
    if ctaps:
        taps = np.ascontiguousarray(taps, dtype=np.complex64)
    else:
        taps = lowpass_taps(fs_in=fs_in) if taps is None else np.ascontiguousarray(taps, dtype=np.float32)
    delay = (len(taps) - 1) // 2 if delay is None else int(delay)
    return taps, ctaps, delay


def _channels_arg(data, dtype):
    """(pointer, space, keep-alive, nchan, n per channel, channel stride) of [nchan, n] / [n] samples: a numpy array
    (converted to dtype) or a (device pointer, dtype, shape) tuple of contiguous device memory"""
    if isinstance(data, tuple):
        ptr, dt, shape = data
        if np.dtype(dt) != np.dtype(dtype):
            raise ValueError("device samples are %s, expected %s" % (np.dtype(dt), np.dtype(dtype)))
        nchan, n = (1, shape[0]) if len(shape) == 1 else shape
        return C.c_void_p(int(ptr.value if isinstance(ptr, C.c_void_p) else ptr)), DEVICE, None, nchan, n, n
    a = np.ascontiguousarray(data, dtype=dtype)
    nchan, n = (1, a.shape[0]) if a.ndim == 1 else a.shape
    return _p(a), HOST, a, nchan, n, n


class FrontendStream:
    """frontend() as a stream (uwspr_b200_frontend_stream): push(audio [nchan, n]) returns the outputs the new samples
    complete, complex64 [nchan, m]; after N samples in any split they equal frontend() over all N bit for bit.
    fmt is np.float32 or np.int16 (PCM scaled by 1/32768); complex taps select the _ctaps form."""

    def __init__(self, nchan, taps=None, decim=32, fc=1500.0, fs_in=12000.0, delay=None, fmt=np.float32, device=0):
        self.L = load_library()
        self.taps, ctaps, self.delay = _frontend_taps(taps, fs_in, delay)
        self.nchan, self.decim, self.fmt = nchan, decim, np.dtype(fmt)
        self.pushed = 0   # samples per channel so far
        h = C.c_void_p()
        st = self.L.uwspr_b200_frontend_stream_create(device, nchan, 1 if self.fmt == np.int16 else 0, _p(self.taps), len(self.taps),
                                                      int(ctaps), decim, self.delay, fc, fs_in, C.byref(h))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_frontend_error().decode())
        self.h = h

    def pending(self, n):
        """outputs a push of n more samples per channel produces"""
        N = self.pushed + n
        return max(0, (N - self.delay + self.decim - 1) // self.decim) - self.outputs()

    def push(self, audio, out_device_ptr=None, out_stride=None):
        """audio: numpy [nchan, n] / [n] or a (device pointer, dtype, shape) tuple.  Returns complex64 [nchan, m], or
        m when out_device_ptr is given (the outputs are then written there, channel c at out_stride samples)"""
        ptr, space, keep, nchan, n, stride = _channels_arg(audio, self.fmt)
        if nchan != self.nchan:
            raise ValueError("expected %d channels" % self.nchan)
        cap = self.pending(n)
        got = C.c_int64()
        if out_device_ptr is None:
            out = np.zeros((nchan, max(cap, 1)), np.complex64)
            optr, ospace, ostride = _p(out), HOST, max(cap, 1)
        else:
            out, optr, ospace = None, C.c_void_p(int(out_device_ptr)), DEVICE
            ostride = cap if out_stride is None else int(out_stride)
        st = self.L.uwspr_b200_frontend_stream_push(self.h, ptr, space, stride, n, optr, ospace, ostride, cap, C.byref(got))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_frontend_error().decode())
        self.pushed += n
        return got.value if out is None else out[:, :got.value]

    def outputs(self):
        return int(self.L.uwspr_b200_frontend_stream_outputs(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.uwspr_b200_frontend_stream_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_INPUT_KINDS = {"complex64": (0, np.complex64), "float32": (1, np.float32), "int16": (2, np.int16)}


def _beam_tables(weights, delays, nchan=None):
    """(weights as [nbeam, nchan] complex64, delays as [nbeam, nchan] int32); the shapes must agree"""
    w = np.ascontiguousarray(weights, dtype=np.complex64)
    d = np.ascontiguousarray(delays, dtype=np.int32)
    if w.ndim != 2 or d.shape != w.shape or (nchan is not None and w.shape[1] != nchan):
        raise ValueError("weights and delays must both be [nbeam, nchan]%s" % ("" if nchan is None else " with nchan %d" % nchan))
    return w, d


def beamform(x, weights, delays, device=0, out_device_ptr=None, out_stride=None):
    """delay-and-sum beams on the GPU (uwspr_b200_beamform): y_b[n] = sum_c weights[b, c] x_c[n - delays[b, c]], x_c = 0
    before its first sample.  x: numpy [nchan, n] complex64, or a (device pointer, dtype, shape) tuple as frontend()
    accepts; weights [nbeam, nchan] complex, delays [nbeam, nchan] integers in [0, 8192].  Returns complex64
    [nbeam, n], or n when out_device_ptr is given (beam b is then written at out_device_ptr + 8*b*out_stride bytes)."""
    L = load_library()
    ptr, space, keep, nchan, n, stride = _channels_arg(x, np.complex64)
    w, d = _beam_tables(weights, delays, nchan)
    nbeam = w.shape[0]
    if out_device_ptr is None:
        out = np.zeros((nbeam, n), np.complex64)
        optr, ospace, ostride = _p(out), HOST, n
    else:
        out, optr, ospace = None, C.c_void_p(int(out_device_ptr)), DEVICE
        ostride = n if out_stride is None else int(out_stride)
    st = L.uwspr_b200_beamform(device, ptr, space, stride, nchan, n, _p(w), _p(d), nbeam, optr, ospace, ostride)
    if st != 0:
        raise UwsprError(st, L.uwspr_b200_status_string(st).decode())
    return n if out is None else out


def plane_wave_steering(positions_m, directions, sound_speed=1500.0, fc=1500.0, fs=375.0):
    """(weights [nbeam, nchan] complex64, delays [nbeam, nchan] int32) of delay-and-sum beams steered at plane waves.
    positions_m: [nchan, 2 or 3] hydrophone positions in metres; directions: [nbeam, same dimension] unit vectors
    pointing from the array towards each source.  A plane wave from u reaches hydrophone c at tau_c = -(p_c . u) / c_s
    (relative to the origin).  Beam b delays channel c by d_c = round((tau_max - tau_c) fs) samples at baseband, so
    that every channel lines up with the last arrival, and its weight removes the carrier phase of the whole
    alignment delay tau_max - tau_c, integer part and residual fraction: after the mix-down by fc a passband delay tau
    is the phase e^{-i 2 pi fc tau} (the envelope error left by rounding is under half a sample).  Weights are
    normalised to sum |w_c|^2 = 1, so a beam's noise level in independent noise equals one hydrophone's."""
    p = np.asarray(positions_m, dtype=np.float64)
    u = np.asarray(directions, dtype=np.float64)
    if u.ndim == 1:
        u = u[None, :]
    if p.ndim != 2 or u.ndim != 2 or p.shape[1] != u.shape[1] or p.shape[1] not in (2, 3):
        raise ValueError("positions [nchan, 2 or 3] and directions [nbeam, same dimension]")
    tau = -(u @ p.T) / sound_speed                       # [nbeam, nchan] arrival times, s
    align = tau.max(axis=1, keepdims=True) - tau         # delay that lines channel c up with the last arrival
    delays = np.rint(align * fs).astype(np.int32)
    weights = np.exp(-2j * np.pi * fc * align) / np.sqrt(p.shape[0])
    return weights.astype(np.complex64), delays


class ArrayReceiver:
    """receive chain of nchan channels in lockstep (uwspr_b200_array_receiver): 375-sps complex64 input, or float32 /
    int16 audio at fs_in through the front-end stream (taps, decim, fc, delay as for frontend()); sliding windows of
    `shift` seconds, batch_windows windows of every channel per submission, decoded on the device.
    push(data [nchan, n], flush) returns [(channel, window, message7, candidate)] in (window, channel, candidate) order.
    beams=(weights [nbeam, nchan] complex64, delays [nbeam, nchan] int32) decodes nbeam delay-and-sum beams of the
    channels instead (uwspr_b200_array_receiver_create_beams; plane_wave_steering makes them): `channel` is then the
    beam index, and the order is (window, beam, candidate)."""

    def __init__(self, nchan, fs=375, fl=45000, spb=256, maxdrift=0, maxfreqs=200, halfbandwidth=10, cf=1500, threshold=10,
                 shift=9, batch_windows=16, input="complex64", taps=None, decim=32, fc=1500.0, fs_in=12000.0, delay=None,
                 device=0, max_candidates=0, beams=None):
        self.L = load_library()
        kind, self.dtype = _INPUT_KINDS[input]
        prm = Params(fs, fl, spb, maxdrift, maxfreqs, halfbandwidth, cf, threshold, device, 0, max_candidates, 0)
        if kind == 0:
            inp = Input(0, None, 0, 0, 0, 0, 0.0, 0.0)
        else:
            self.taps, ctaps, delay = _frontend_taps(taps, fs_in, delay)
            inp = Input(kind, _p(self.taps), len(self.taps), int(ctaps), decim, delay, fc, fs_in)
        self.nchan = nchan
        h = C.c_void_p()
        if beams is None:
            st = self.L.uwspr_b200_array_receiver_create(C.byref(prm), C.byref(inp), nchan, shift, batch_windows, C.byref(h))
        else:
            w, d = _beam_tables(*beams, nchan=nchan)
            bm = Beams(w.shape[0], _p(w), _p(d))
            st = self.L.uwspr_b200_array_receiver_create_beams(C.byref(prm), C.byref(inp), nchan, C.byref(bm), shift,
                                                                batch_windows, C.byref(h))
        if st != 0:
            text = self.L.uwspr_b200_create_error().decode() if st == 2 else ""
            raise UwsprError(st, text or self.L.uwspr_b200_status_string(st).decode())
        self.h = h

    def push(self, data, flush=False):
        ptr, space, keep, nchan, n, stride = _channels_arg(data, self.dtype)
        if nchan != self.nchan:
            raise ValueError("expected %d channels" % self.nchan)
        st = self.L.uwspr_b200_array_receiver_push(self.h, ptr, space, stride, n, int(flush))
        if st != 0:
            raise UwsprError(st, self.L.uwspr_b200_status_string(st).decode())
        out = []
        chan, win = C.c_int32(), C.c_int64()
        msg = np.zeros(7, np.int8)
        cand = np.zeros(1, CAND_DTYPE)
        while self.L.uwspr_b200_array_receiver_pop(self.h, C.byref(chan), C.byref(win), _p(cand), _p(msg)):
            out.append((chan.value, win.value, msg.view(np.uint8).copy(), cand[0].copy()))
        return out

    def windows_done(self):
        return int(self.L.uwspr_b200_array_receiver_windows(self.h))

    def launch_count(self):
        return int(self.L.uwspr_b200_array_receiver_launch_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.L.uwspr_b200_array_receiver_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pack_type1(call, grid, dbm):
    """"CALL", "GRID", dBm -> the 7-byte type-1 message (what WSPR_unpacker turns back into text)"""
    msg = np.zeros(7, np.int8)
    st = load_library().uwspr_b200_pack_type1(call.encode(), grid.encode(), int(dbm), _p(msg))
    if st != 0:
        raise UwsprError(st, "not a type-1 message: %r %r %r" % (call, grid, dbm))
    return msg.view(np.uint8)


def channel_symbols(message7):
    """7-byte message -> the 162 four-level channel symbols (0..3) a WSPR transmitter keys"""
    msg = np.ascontiguousarray(message7).view(np.uint8)
    assert msg.size == 7
    out = np.zeros(162, np.uint8)
    load_library().uwspr_b200_channel_symbols(_p(msg), _p(out))
    return out


def format_message_log(framecount, cand, message7):
    """the text the reference appends to messagelog.txt for a decoded frame (without its two clock lines)"""
    L = load_library()
    L.uwspr_b200_format_message_log.restype = C.c_int
    L.uwspr_b200_format_message_log.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    c = np.zeros(1, CAND_DTYPE)
    c[0] = cand
    m = np.ascontiguousarray(message7, dtype=np.uint8)
    text = np.zeros(512, np.uint8)
    st = L.uwspr_b200_format_message_log(framecount, _p(c), _p(m), _p(text), text.size)
    if st != 0:
        raise UwsprError(st, L.uwspr_b200_status_string(st).decode())
    return bytes(text).split(b"\0")[0].decode("latin1")


class WSPR_unpacker:
    """uwspr.WSPR_unpacker's text (lib/helpers.cc:494-590): unpack(message7) -> (noprint, "CALL GRID dBm")"""

    def __init__(self):
        self.L = load_library()
        self.hashtab = np.zeros(self.L.uwspr_b200_hashtab_bytes(), np.uint8)

    def unpack(self, message7):
        m = np.ascontiguousarray(message7, dtype=np.uint8)
        text = np.zeros(64, np.uint8)
        noprint = self.L.uwspr_b200_unpack(_p(m), _p(self.hashtab), _p(text), text.size)
        return noprint, bytes(text).split(b"\0")[0].decode("latin1")
