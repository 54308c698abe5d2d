"""ctypes binding of libb2video.so (include/b2video.h).

This is the only place the Python host side touches native code.  There is no CPU
fallback: if the CUDA library is missing or fails to load, `lib()` raises — the
product path must fail loudly (and never routes through oracle/).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B2V_LIB") or os.path.join(_HERE, "libb2video.so")      # B2V_LIB: A/B runs against another build (tools/)

B2V_OK, B2V_EINVAL, B2V_ECUDA, B2V_ENOMEM, B2V_ESTATE, B2V_ETIMEOUT = 0, -1, -2, -3, -4, -5
B2V_RC_CBR, B2V_RC_CQP = 0, 1
B2V_HDR_NONE, B2V_HDR_PIXELFLUX = 0, 1
B2V_FLAG_SPS_EVERY_IDR, B2V_FLAG_NO_ENCODE, B2V_FLAG_TIMING, B2V_FLAG_DEVICE_TIMER, B2V_FLAG_TIMING_CSC, B2V_FLAG_JPEG = 1, 2, 4, 8, 16, 32


class B2VSettings(C.Structure):
    _fields_ = [
        ("src_w", C.c_int32), ("src_h", C.c_int32), ("dst_w", C.c_int32), ("dst_h", C.c_int32),
        ("fps", C.c_double), ("device", C.c_int32), ("rc_mode", C.c_int32),
        ("bitrate_kbps", C.c_int32), ("crf", C.c_int32), ("gop", C.c_int32),
        ("slice_rows", C.c_int32), ("header_mode", C.c_int32), ("ring_slots", C.c_int32),
        ("flags", C.c_int32), ("paintover_trigger_frames", C.c_int32), ("paintover_crf", C.c_int32), ("stripe_rows", C.c_int32), ("idr_slice_mbs", C.c_int32), ("paintover_burst_frames", C.c_int32),
    ]


class B2VFrame(C.Structure):
    _fields_ = [
        ("data", C.POINTER(C.c_ubyte)), ("size", C.c_int32), ("frame_id", C.c_int32),
        ("is_key", C.c_int32), ("qp", C.c_int32), ("pts90k", C.c_int64), ("capture_ns", C.c_int64),
        ("y_start", C.c_int32), ("height", C.c_int32),
    ]


class B2VStats(C.Structure):
    _fields_ = [
        ("frames_submitted", C.c_int64), ("frames_delivered", C.c_int64), ("key_frames", C.c_int64),
        ("bytes_out", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("ms_csc", C.c_double), ("ms_intra", C.c_double), ("ms_inter", C.c_double),
        ("ms_cavlc", C.c_double), ("ms_slice", C.c_double), ("ms_pack", C.c_double),
        ("ms_total_gpu", C.c_double),
        ("n_csc", C.c_int64), ("n_intra", C.c_int64), ("n_inter", C.c_int64),
        ("n_cavlc", C.c_int64), ("n_slice", C.c_int64), ("n_pack", C.c_int64),
        ("ms_csc_device", C.c_double), ("n_csc_device", C.c_int64),
        ("ns_wait_event", C.c_int64), ("ns_wait_event_max", C.c_int64), ("n_event_sleeps", C.c_int64),
        ("ns_wait_job", C.c_int64), ("ns_callback", C.c_int64), ("ns_wait_out_slot", C.c_int64),
        ("ns_wait_ring", C.c_int64), ("ns_submit", C.c_int64),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


FRAME_CB = C.CFUNCTYPE(None, C.POINTER(B2VFrame), C.c_void_p)

# every symbol include/b2video.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("b2v_abi_version", C.c_int, []),
    ("b2v_device_count", C.c_int, []),
    ("b2v_create", C.c_int, [C.POINTER(B2VSettings), FRAME_CB, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("b2v_destroy", None, [C.c_void_p]),
    ("b2v_ring_acquire", C.c_void_p, [C.c_void_p, C.POINTER(C.c_int32)]),
    ("b2v_ring_submit", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64]),
    ("b2v_ring_release", C.c_int, [C.c_void_p, C.c_int32]),
    ("b2v_resident_upload", C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
    ("b2v_submit_resident", C.c_int, [C.c_void_p, C.c_int32, C.c_int64]),
    ("b2v_flush", C.c_int, [C.c_void_p]),
    ("b2v_set_framerate", C.c_int, [C.c_void_p, C.c_double]),
    ("b2v_set_bitrate_kbps", C.c_int, [C.c_void_p, C.c_int32]),
    ("b2v_set_qp", C.c_int, [C.c_void_p, C.c_int32]),
    ("b2v_set_gop", C.c_int, [C.c_void_p, C.c_int32]),
    ("b2v_set_resolution", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    ("b2v_request_idr", C.c_int, [C.c_void_p]),
    ("b2v_get_stats", C.c_int, [C.c_void_p, C.POINTER(B2VStats)]),
    ("b2v_reset_stats", C.c_int, [C.c_void_p]),
    ("b2v_coded_size", C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("b2v_csc_nv12", C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    ("b2v_get_recon", C.c_int, [C.c_void_p, C.c_void_p]),
    ("b2v_bench_csc", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    ("b2v_bench_csc_burst", C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    ("b2v_timer_start", C.c_int, [C.c_void_p]),
    ("b2v_timer_stop", C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    ("b2v_last_error", C.c_char_p, []),
    ("b2v_rtp_h264_packetize", C.c_int, [C.c_char_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                         C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32)]),
]

_lib = None
_lock = threading.Lock()


class B2VError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libb2video error {code}: {msg}")
        self.code = code


def lib():
    """Load libb2video.so (built in-tree by `__graft_entry__.build()`); raises if absent."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(
                    f"{LIB_PATH} is missing — build it with "
                    "`python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU fallback for the video hot path)")
            l = C.CDLL(LIB_PATH)
            for name, res, args in SYMBOLS:
                fn = getattr(l, name)          # AttributeError here = header/library mismatch
                fn.restype = res
                fn.argtypes = args
            if l.b2v_abi_version() != 3:
                raise ImportError("libb2video ABI version mismatch")
            _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise B2VError(rc, (lib().b2v_last_error() or b"").decode("utf-8", "replace"))
    return rc
