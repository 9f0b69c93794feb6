"""ctypes front-end of the CPU oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.  PARITY UNPINNED.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  It restates the reference chains of /root/reference/src/sdr_pmr446.c:788-913
and /root/reference/src/dsd_in.c:159-180 (see oracle/chains.c, oracle/liquid_subset.c).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FMT_CF32, FMT_CU8 = 0, 1


class PmrCfg(C.Structure):
    _fields_ = [("fs_in", C.c_uint), ("in_fmt", C.c_int), ("num_channels", C.c_uint), ("channel_width", C.c_uint),
                ("pfb_m", C.c_uint), ("pfb_as", C.c_float), ("resamp_as", C.c_float), ("dc_alpha", C.c_float),
                ("kf", C.c_float), ("audio_gain", C.c_float), ("lowpass", C.c_int), ("waterfall", C.c_uint),
                ("chunk", C.c_uint), ("active_only", C.c_int), ("channelize_only", C.c_int), ("deemph_fir", C.c_int)]


class PmrOut(C.Structure):
    _fields_ = [("dcblocked", C.c_void_p), ("res", C.c_void_p), ("chan", C.c_void_p), ("demod", C.c_void_p),
                ("lpcomp", C.c_void_p), ("audio", C.c_void_p), ("pcm", C.c_void_p), ("ld", C.c_uint),
                ("ascii", C.c_void_p), ("peak", C.c_void_p), ("psd", C.c_void_p)]


class DsdCfg(C.Structure):
    _fields_ = [("fs_in", C.c_uint), ("in_fmt", C.c_int), ("fs_sig", C.c_uint), ("fs_audio", C.c_uint),
                ("chunk", C.c_uint), ("dc_alpha", C.c_float), ("resamp_as", C.c_float), ("kf", C.c_float)]


class RxCfg(C.Structure):
    _fields_ = [("chain", PmrCfg), ("squelch_level", C.c_float), ("channel_mask", C.c_ulonglong), ("lock_mode", C.c_int),
                ("ctcss_block", C.c_uint), ("ctcss_dc_alpha", C.c_float)]


class RxStatus(C.Structure):
    _fields_ = [("state", C.c_int), ("active_chan", C.c_int), ("rssi", C.c_float), ("n_audio", C.c_uint),
                ("tone_detected", C.c_int), ("ctcss_index", C.c_int), ("ctcss_freq", C.c_float), ("max_power", C.c_float),
                ("events", C.c_int)]


class RxOut(C.Structure):
    _fields_ = [("rssi", C.c_void_p), ("audio", C.c_void_p), ("pcm", C.c_void_p), ("ctcss_in", C.c_void_p),
                ("ctcss_power", C.c_void_p), ("chan", C.c_void_p), ("ld", C.c_uint)]


class Knobs(C.Structure):
    _fields_ = [("resamp_npfb", C.c_int), ("resamp_fc_mode", C.c_int), ("kaiser_r_mode", C.c_int),
                ("asgram_avg", C.c_int), ("asgram_keep_buf", C.c_int)]


def build(force=False):
    so = os.path.join(_HERE, "liboracle_pmr446.so")
    srcs = [os.path.join(_HERE, f) for f in ("liquid_subset.c", "chains.c", "receiver.c", "liquid_subset.h", "chains.h", "receiver.h", "resamp_tmpl.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.oracle_pmr_create.restype = C.c_void_p
        L.oracle_pmr_create.argtypes = [C.POINTER(PmrCfg)]
        L.oracle_pmr_destroy.argtypes = [C.c_void_p]
        L.oracle_pmr_default_cfg.argtypes = [C.POINTER(PmrCfg)]
        L.oracle_pmr_res_size.argtypes = [C.c_void_p]
        L.oracle_pmr_chan_size.argtypes = [C.c_void_p]
        L.oracle_pmr_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.POINTER(PmrOut), C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.oracle_rx_default_cfg.argtypes = [C.POINTER(RxCfg)]
        L.oracle_rx_create.restype = C.c_void_p
        L.oracle_rx_create.argtypes = [C.POINTER(RxCfg)]
        L.oracle_rx_destroy.argtypes = [C.c_void_p]
        L.oracle_rx_chan_size.argtypes = [C.c_void_p]
        L.oracle_rx_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.POINTER(RxOut), C.POINTER(RxStatus), C.POINTER(C.c_uint)]
        L.oracle_dsd_create.restype = C.c_void_p
        L.oracle_dsd_create.argtypes = [C.POINTER(DsdCfg)]
        L.oracle_dsd_destroy.argtypes = [C.c_void_p]
        L.oracle_dsd_default_cfg.argtypes = [C.POINTER(DsdCfg)]
        L.oracle_dsd_res_size.argtypes = [C.c_void_p]
        L.oracle_dsd_out_size.argtypes = [C.c_void_p]
        L.oracle_dsd_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.oracle_liquid_get_knobs.restype = C.POINTER(Knobs)
        L.liquid_firdes_kaiser.argtypes = [C.c_uint, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.liquid_kaiser.restype = C.c_float
        L.liquid_kaiser.argtypes = [C.c_uint, C.c_uint, C.c_float]
        L.kaiser_beta_As.restype = C.c_float
        L.kaiser_beta_As.argtypes = [C.c_float]
        L.msresamp_crcf_create.restype = C.c_void_p
        L.msresamp_crcf_create.argtypes = [C.c_float, C.c_float]
        L.msresamp_crcf_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p, C.POINTER(C.c_uint)]
        L.msresamp_crcf_destroy.argtypes = [C.c_void_p]
        L.oracle_msresamp_crcf_plan.argtypes = [C.c_void_p, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_float),
                                                C.POINTER(C.c_uint), C.POINTER(C.c_uint)]
        L.msresamp_rrrf_create.restype = C.c_void_p
        L.msresamp_rrrf_create.argtypes = [C.c_float, C.c_float]
        L.msresamp_rrrf_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p, C.POINTER(C.c_uint)]
        L.msresamp_rrrf_destroy.argtypes = [C.c_void_p]
        L.nco_crcf_create.restype = C.c_void_p
        L.nco_crcf_create.argtypes = [C.c_int]
        L.nco_crcf_set_frequency.argtypes = [C.c_void_p, C.c_float]
        L.oracle_nco_crcf_get_dtheta_u32.restype = C.c_uint
        L.oracle_nco_crcf_get_dtheta_u32.argtypes = [C.c_void_p]
        L.nco_crcf_destroy.argtypes = [C.c_void_p]
        L.firpfbch_crcf_create_kaiser.restype = C.c_void_p
        L.firpfbch_crcf_create_kaiser.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_float]
        L.firpfbch_crcf_analyzer_execute.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.firpfbch_crcf_destroy.argtypes = [C.c_void_p]
        L.iirfilt_crcf_create_dc_blocker.restype = C.c_void_p
        L.iirfilt_crcf_create_dc_blocker.argtypes = [C.c_float]
        L.iirfilt_crcf_execute_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p]
        L.iirfilt_crcf_destroy.argtypes = [C.c_void_p]
        L.iirfilt_rrrf_create.restype = C.c_void_p
        L.iirfilt_rrrf_create.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint]
        L.iirfilt_rrrf_execute_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p]
        L.iirfilt_rrrf_destroy.argtypes = [C.c_void_p]
        L.freqdem_create.restype = C.c_void_p
        L.freqdem_create.argtypes = [C.c_float]
        L.freqdem_demodulate_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p]
        L.freqdem_destroy.argtypes = [C.c_void_p]
        L.firfilt_rrrf_create.restype = C.c_void_p
        L.firfilt_rrrf_create.argtypes = [C.c_void_p, C.c_uint]
        L.firfilt_rrrf_execute_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p]
        L.firfilt_rrrf_destroy.argtypes = [C.c_void_p]
        L.asgramcf_create.restype = C.c_void_p
        L.asgramcf_create.argtypes = [C.c_uint]
        L.asgramcf_set_scale.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.asgramcf_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
        L.asgramcf_execute.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.asgramcf_destroy.argtypes = [C.c_void_p]
        L.oracle_fft_forward.argtypes = [C.c_uint, C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pmr_default_cfg(**kw):
    cfg = PmrCfg()
    lib().oracle_pmr_default_cfg(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


def dsd_default_cfg(**kw):
    cfg = DsdCfg()
    lib().oracle_dsd_default_cfg(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


class PmrOracle:
    """One stream of the PMR446 chain, all channels demodulated (reference loop body :795-913)."""

    def __init__(self, cfg=None, **kw):
        self.cfg = cfg if cfg is not None else pmr_default_cfg(**kw)
        self.h = lib().oracle_pmr_create(C.byref(self.cfg))
        if not self.h:
            raise RuntimeError("oracle_pmr_create failed")
        self.M = self.cfg.num_channels
        self.res_size = lib().oracle_pmr_res_size(self.h)
        self.chan_size = lib().oracle_pmr_chan_size(self.h)

    def close(self):
        if self.h:
            lib().oracle_pmr_destroy(self.h)
            self.h = None

    __del__ = close

    def execute(self, iq, want=("res", "chan", "demod", "lpcomp", "audio", "pcm")):
        """Process one chunk (<= cfg.chunk samples).  Returns dict of per-chunk arrays."""
        iq = np.ascontiguousarray(iq)
        n = iq.shape[0] // 2 if self.cfg.in_fmt == FMT_CU8 else iq.shape[0]
        M, ld = self.M, self.chan_size
        bufs = {}
        out = PmrOut()
        out.ld = ld
        if "dcblocked" in want:
            bufs["dcblocked"] = np.zeros(n, np.complex64)
        if "res" in want:
            bufs["res"] = np.zeros(self.res_size, np.complex64)
        if "chan" in want:
            bufs["chan"] = np.zeros((M, ld), np.complex64)
        for k in ("demod", "lpcomp", "audio"):
            if k in want:
                bufs[k] = np.zeros((M, ld), np.float32)
        if "pcm" in want:
            bufs["pcm"] = np.zeros((M, ld), np.int16)
        W = self.cfg.waterfall
        if W:
            bufs["ascii"] = np.zeros(W, np.uint8)
            bufs["peak"] = np.zeros(2, np.float32)
            bufs["psd"] = np.zeros(4 * W, np.float32)
        for k, v in bufs.items():
            setattr(out, k, v.ctypes.data)
        ny, ns = C.c_uint(0), C.c_uint(0)
        rc = lib().oracle_pmr_execute(self.h, _p(iq), n, C.byref(out), C.byref(ny), C.byref(ns))
        if rc:
            raise RuntimeError("oracle_pmr_execute rc=%d" % rc)
        r = {"ny": ny.value, "ns": ns.value}
        for k, v in bufs.items():
            if k == "res":
                r[k] = v[:ny.value]
            elif k in ("chan", "demod", "lpcomp", "audio", "pcm"):
                r[k] = v[:, :ns.value]
            else:
                r[k] = v
        return r

    def run(self, iq, chunk=None, want=("res", "chan", "demod", "lpcomp", "audio", "pcm")):
        """Process a whole capture in chunks; concatenates outputs along time."""
        chunk = chunk or self.cfg.chunk
        step = 2 * chunk if self.cfg.in_fmt == FMT_CU8 else chunk
        parts = []
        for o in range(0, iq.shape[0], step):
            parts.append(self.execute(iq[o:o + step], want))
        r = {"ny": sum(p["ny"] for p in parts), "ns": sum(p["ns"] for p in parts)}
        for k in parts[0]:
            if k in ("ny", "ns"):
                continue
            if k in ("ascii", "peak", "psd"):
                r[k] = np.stack([p[k] for p in parts])
            else:
                r[k] = np.concatenate([p[k] for p in parts], axis=-1)
        return r


class RxOracle:
    """One stream of the reference receiver: RSSI, squelch/selector state machine, the selected channel's
    demodulation chain and the CTCSS detector (src/sdr_pmr446.c:828-908; oracle/receiver.c)."""

    STATUS_FIELDS = ("state", "active_chan", "rssi", "n_audio", "tone_detected", "ctcss_index", "ctcss_freq", "max_power", "events")

    def __init__(self, squelch_level=18.0, channel_mask=2 ** 64 - 1, lock_mode=0, ctcss_block=2441, ctcss_dc_alpha=0.0005, **chain_kw):
        self.cfg = RxCfg()
        lib().oracle_rx_default_cfg(C.byref(self.cfg))
        for k, v in chain_kw.items():
            if not hasattr(self.cfg.chain, k):
                raise AttributeError(k)
            setattr(self.cfg.chain, k, v)
        self.cfg.squelch_level = squelch_level
        self.cfg.channel_mask = channel_mask
        self.cfg.lock_mode = lock_mode
        self.cfg.ctcss_block = ctcss_block
        self.cfg.ctcss_dc_alpha = ctcss_dc_alpha
        self.h = lib().oracle_rx_create(C.byref(self.cfg))
        if not self.h:
            raise RuntimeError("oracle_rx_create failed")
        self.M = self.cfg.chain.num_channels
        self.chan_size = lib().oracle_rx_chan_size(self.h)

    def close(self):
        if self.h:
            lib().oracle_rx_destroy(self.h)
            self.h = None

    __del__ = close

    def execute(self, iq):
        """One chunk -> dict(status fields, rssi_ch [M], chan [M, ns], audio, pcm, ctcss_in [n_audio], ctcss_power [38], ns)."""
        iq = np.ascontiguousarray(iq)
        n = iq.shape[0] // 2 if self.cfg.chain.in_fmt == FMT_CU8 else iq.shape[0]
        ld = self.chan_size
        bufs = {"rssi": np.zeros(self.M, np.float32), "audio": np.zeros(ld, np.float32), "pcm": np.zeros(ld, np.int16),
                "ctcss_in": np.zeros(ld, np.float32), "ctcss_power": np.zeros(38, np.float32), "chan": np.zeros((self.M, ld), np.complex64)}
        out = RxOut()
        out.ld = ld
        for k, v in bufs.items():
            setattr(out, k, v.ctypes.data)
        st, ns = RxStatus(), C.c_uint(0)
        rc = lib().oracle_rx_execute(self.h, _p(iq), n, C.byref(out), C.byref(st), C.byref(ns))
        if rc:
            raise RuntimeError("oracle_rx_execute rc=%d" % rc)
        r = {k: getattr(st, k) for k in self.STATUS_FIELDS}
        r["ns"] = ns.value
        r["rssi_ch"] = bufs["rssi"]
        r["ctcss_power"] = bufs["ctcss_power"]
        r["chan"] = bufs["chan"][:, :ns.value]
        for k in ("audio", "pcm", "ctcss_in"):
            r[k] = bufs[k][:st.n_audio]
        return r

    def run(self, iq, chunk=None):
        """Whole capture in chunks -> list of per-chunk dicts."""
        chunk = chunk or self.cfg.chain.chunk
        step = 2 * chunk if self.cfg.chain.in_fmt == FMT_CU8 else chunk
        return [self.execute(iq[o:o + step]) for o in range(0, iq.shape[0], step)]


class DsdOracle:
    """One stream of the dsd_in chain (reference loop body src/dsd_in.c:167-175)."""

    def __init__(self, cfg=None, **kw):
        self.cfg = cfg if cfg is not None else dsd_default_cfg(**kw)
        self.h = lib().oracle_dsd_create(C.byref(self.cfg))
        self.res_size = lib().oracle_dsd_res_size(self.h)
        self.out_size = lib().oracle_dsd_out_size(self.h)

    def close(self):
        if self.h:
            lib().oracle_dsd_destroy(self.h)
            self.h = None

    __del__ = close

    def execute(self, iq):
        iq = np.ascontiguousarray(iq)
        n = iq.shape[0] // 2 if self.cfg.in_fmt == FMT_CU8 else iq.shape[0]
        res = np.zeros(self.res_size, np.complex64)
        fm = np.zeros(self.res_size, np.float32)
        audio = np.zeros(self.out_size, np.float32)
        pcm = np.zeros(self.out_size, np.int16)
        ny, nz = C.c_uint(0), C.c_uint(0)
        rc = lib().oracle_dsd_execute(self.h, _p(iq), n, _p(res), _p(fm), _p(audio), _p(pcm), C.byref(ny), C.byref(nz))
        if rc:
            raise RuntimeError("oracle_dsd_execute rc=%d" % rc)
        return {"ny": ny.value, "nz": nz.value, "res": res[:ny.value], "fm": fm[:ny.value], "audio": audio[:nz.value],
                "pcm": pcm[:nz.value]}

    def run(self, iq, chunk=None):
        chunk = chunk or self.cfg.chunk
        step = 2 * chunk if self.cfg.in_fmt == FMT_CU8 else chunk
        parts = [self.execute(iq[o:o + step]) for o in range(0, iq.shape[0], step)]
        r = {"ny": sum(p["ny"] for p in parts), "nz": sum(p["nz"] for p in parts)}
        for k in ("res", "fm", "audio", "pcm"):
            r[k] = np.concatenate([p[k] for p in parts])
        return r
