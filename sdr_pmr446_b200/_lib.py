"""ctypes binding of libpmr446_b200.so (the C ABI declared in include/pmr446_b200.h).

The shared library is built in-tree by `make -C sdr_pmr446_b200/csrc` (see __graft_entry__.build).
There is no Python or CPU fallback: if the library is missing, loading fails loudly.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpmr446_b200.so")
_LIB = None

OK, EINVAL, ENODEV, ECUDA, ERANGE, ENOMEM = 0, -1, -2, -3, -4, -5
FMT_CF32, FMT_CU8, FMT_CS16, FMT_CS8 = 0, 1, 2, 3


class Config(C.Structure):
    """pmr446_config (include/pmr446_b200.h)."""
    _fields_ = [("n_streams", C.c_int), ("device", C.c_int), ("fs_in", C.c_uint), ("in_fmt", C.c_int),
                ("num_channels", C.c_uint), ("channel_width", C.c_uint), ("pfb_m", C.c_uint), ("pfb_as", C.c_float),
                ("resamp_as", C.c_float), ("dc_alpha", C.c_float), ("kf", C.c_float), ("audio_gain", C.c_float),
                ("lowpass", C.c_int), ("waterfall", C.c_uint), ("max_chunk", C.c_uint),
                ("hp_taps", C.c_void_p), ("hp_len", C.c_uint), ("lp_taps", C.c_void_p), ("lp_len", C.c_uint),
                ("deemph_b0", C.c_float), ("deemph_b1", C.c_float), ("deemph_a1", C.c_float), ("deemph_fir", C.c_int),
                ("dsd_rate", C.c_uint)]


class Outputs(C.Structure):
    """pmr446_outputs (include/pmr446_b200.h)."""
    _fields_ = [("res", C.c_void_p), ("res_ld", C.c_longlong), ("chan", C.c_void_p), ("demod", C.c_void_p),
                ("lpcomp", C.c_void_p), ("audio", C.c_void_p), ("pcm", C.c_void_p), ("ld", C.c_longlong),
                ("ascii", C.c_void_p), ("peak", C.c_void_p), ("psd", C.c_void_p), ("rssi", C.c_void_p), ("chan_edge", C.c_void_p),
                ("dsd_audio", C.c_void_p), ("dsd_pcm", C.c_void_p), ("dsd_ld", C.c_longlong)]


class RxConfig(C.Structure):
    """pmr446_rx_config (include/pmr446_b200.h)."""
    _fields_ = [("chain", Config), ("squelch_level", C.c_float), ("channel_mask", C.c_ulonglong), ("lock_mode", C.c_int),
                ("ctcss_block", C.c_uint), ("ctcss_dc_alpha", C.c_float)]


class RxStatus(C.Structure):
    """pmr446_rx_status (include/pmr446_b200.h)."""
    _fields_ = [("state", C.c_int), ("active_chan", C.c_int), ("rssi", C.c_float), ("n_audio", C.c_uint),
                ("tone_detected", C.c_int), ("ctcss_index", C.c_int), ("ctcss_freq", C.c_float), ("max_power", C.c_float),
                ("events", C.c_int)]


class RxOutputs(C.Structure):
    """pmr446_rx_outputs (include/pmr446_b200.h)."""
    _fields_ = [("rssi", C.c_void_p), ("status", C.c_void_p), ("audio", C.c_void_p), ("pcm", C.c_void_p),
                ("ctcss_in", C.c_void_p), ("ctcss_power", C.c_void_p), ("ld", C.c_longlong), ("ascii", C.c_void_p),
                ("peak", C.c_void_p)]


class DsdConfig(C.Structure):
    """dsd446_config (include/pmr446_b200.h)."""
    _fields_ = [("n_streams", C.c_int), ("device", C.c_int), ("fs_in", C.c_uint), ("in_fmt", C.c_int),
                ("fs_sig", C.c_uint), ("fs_audio", C.c_uint), ("max_chunk", C.c_uint),
                ("dc_alpha", C.c_float), ("resamp_as", C.c_float), ("kf", C.c_float)]


class DsdOutputs(C.Structure):
    _fields_ = [("res", C.c_void_p), ("fm", C.c_void_p), ("res_ld", C.c_longlong), ("audio", C.c_void_p),
                ("pcm", C.c_void_p), ("out_ld", C.c_longlong)]


EXPORTS = [
    "pmr446_default_config", "pmr446_batch_create", "pmr446_batch_destroy", "pmr446_batch_max_res",
    "pmr446_batch_max_ns", "pmr446_batch_execute", "pmr446_batch_execute_device", "pmr446_batch_last_launches",
    "pmr446_batch_gather_channel", "pmr446_batch_max_dsd", "pmr446_batch_last_dsd",
    "pmr446_batch_reset", "pmr446_last_error", "pmr446_host_alloc", "pmr446_host_free", "pmr446_measure_fp32_peak", "pmr446_batch_timing",
    "pmr446_batch_get_timings",
    "pmr446_rx_default_config", "pmr446_receiver_create", "pmr446_receiver_destroy", "pmr446_receiver_max_ns",
    "pmr446_receiver_execute", "pmr446_receiver_execute_device", "pmr446_receiver_last_launches", "pmr446_receiver_reset",
    "dsd446_default_config", "dsd446_batch_create", "dsd446_batch_destroy", "dsd446_batch_max_res",
    "dsd446_batch_max_out", "dsd446_batch_last_launches", "dsd446_batch_execute", "dsd446_batch_execute_device", "dsd446_batch_reset",
    "pmr446_design_msresamp", "pmr446_design_pfbch", "pmr446_design_asgram_window", "pmr446_design_nco_dtheta",
    "pmr446_count_resampled", "pmr446_describe_frontend", "pmr446_bytes_per_sample",
]


def build(force=False):
    src = os.path.join(_HERE, "csrc")
    deps = [os.path.join(src, f) for f in os.listdir(src)] + [os.path.join(_HERE, "..", "include", f) for f in
                                                              ("pmr446_b200.h", "pmr446_taps.h")]
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(d) > os.path.getmtime(LIB_PATH) for d in deps):
        subprocess.check_call(["make", "-C", src, "-s"])
    return LIB_PATH


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.pmr446_default_config.argtypes = [C.POINTER(Config)]
        L.pmr446_default_config.restype = None
        L.pmr446_batch_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.pmr446_batch_destroy.argtypes = [C.c_void_p]
        L.pmr446_batch_max_res.argtypes = [C.c_void_p]
        L.pmr446_batch_max_res.restype = C.c_longlong
        L.pmr446_batch_max_ns.argtypes = [C.c_void_p]
        L.pmr446_batch_max_ns.restype = C.c_longlong
        L.pmr446_batch_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(Outputs),
                                           C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.pmr446_batch_execute_device.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(Outputs),
                                                  C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.c_void_p]
        L.pmr446_batch_last_launches.argtypes = [C.c_void_p]
        L.pmr446_batch_max_dsd.argtypes = [C.c_void_p]
        L.pmr446_batch_max_dsd.restype = C.c_longlong
        L.pmr446_batch_last_dsd.argtypes = [C.c_void_p]
        L.pmr446_batch_last_dsd.restype = C.c_longlong
        L.pmr446_batch_gather_channel.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]
        L.pmr446_batch_reset.argtypes = [C.c_void_p]
        L.pmr446_last_error.restype = C.c_char_p
        L.pmr446_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_ulonglong]
        L.pmr446_host_free.argtypes = [C.c_void_p]
        L.pmr446_measure_fp32_peak.argtypes = [C.POINTER(C.c_double), C.c_void_p]
        L.pmr446_batch_timing.argtypes = [C.c_void_p, C.c_int]
        L.pmr446_batch_get_timings.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]
        L.pmr446_rx_default_config.argtypes = [C.POINTER(RxConfig)]
        L.pmr446_rx_default_config.restype = None
        L.pmr446_receiver_create.argtypes = [C.POINTER(RxConfig), C.POINTER(C.c_void_p)]
        L.pmr446_receiver_destroy.argtypes = [C.c_void_p]
        L.pmr446_receiver_max_ns.argtypes = [C.c_void_p]
        L.pmr446_receiver_max_ns.restype = C.c_longlong
        L.pmr446_receiver_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(RxOutputs), C.POINTER(C.c_uint)]
        L.pmr446_receiver_execute_device.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(RxOutputs),
                                                     C.POINTER(C.c_uint), C.c_void_p]
        L.pmr446_receiver_last_launches.argtypes = [C.c_void_p]
        L.pmr446_receiver_reset.argtypes = [C.c_void_p]
        L.dsd446_default_config.argtypes = [C.POINTER(DsdConfig)]
        L.dsd446_default_config.restype = None
        L.dsd446_batch_create.argtypes = [C.POINTER(DsdConfig), C.POINTER(C.c_void_p)]
        L.dsd446_batch_destroy.argtypes = [C.c_void_p]
        L.dsd446_batch_max_res.argtypes = [C.c_void_p]
        L.dsd446_batch_max_res.restype = C.c_longlong
        L.dsd446_batch_max_out.argtypes = [C.c_void_p]
        L.dsd446_batch_max_out.restype = C.c_longlong
        L.dsd446_batch_last_launches.argtypes = [C.c_void_p]
        L.dsd446_batch_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(DsdOutputs),
                                           C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.dsd446_batch_execute_device.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint, C.POINTER(DsdOutputs),
                                                  C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.c_void_p]
        L.dsd446_batch_reset.argtypes = [C.c_void_p]
        L.pmr446_design_msresamp.argtypes = [C.c_float, C.c_float, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_uint),
                                             C.POINTER(C.c_uint), C.c_void_p, C.c_void_p]
        L.pmr446_design_pfbch.argtypes = [C.c_uint, C.c_uint, C.c_float, C.c_void_p]
        L.pmr446_design_asgram_window.argtypes = [C.c_uint, C.c_void_p]
        L.pmr446_design_nco_dtheta.argtypes = [C.c_float]
        L.pmr446_design_nco_dtheta.restype = C.c_uint
        L.pmr446_count_resampled.argtypes = [C.c_float, C.c_float, C.c_longlong]
        L.pmr446_count_resampled.restype = C.c_longlong
        L.pmr446_describe_frontend.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_char_p, C.c_int]
        L.pmr446_bytes_per_sample.argtypes = [C.c_int]
        _LIB = L
    return _LIB


def bytes_per_sample(in_fmt):
    """Bytes per IQ sample of an in_fmt, as the library reads it (cu8 and cs8 2, cs16 4, anything else cf32, 8)."""
    return lib().pmr446_bytes_per_sample(int(in_fmt))


class Pmr446Error(RuntimeError):
    def __init__(self, code, where):
        msg = lib().pmr446_last_error()
        super().__init__("%s failed with code %d: %s" % (where, code, msg.decode() if msg else ""))
        self.code = code


def check(code, where):
    if code != OK:
        raise Pmr446Error(code, where)
