"""Host-side mirror of the reference's processing chains over the C ABI.

`PmrBatch` is `proc_chain_t` + the loop body of /root/reference/src/sdr_pmr446.c:788-913 for
n_streams streams; `DsdBatch` the same for /root/reference/src/dsd_in.c:159-180.  They only
marshal buffers: every sample is computed by the CUDA kernels in libpmr446_b200.so.

Two call styles, as in include/pmr446_b200.h:
  execute(iq)            host numpy buffers in and out (H2D/D2H inside the call)
  execute_device(iq, ..) torch CUDA tensors in and out, enqueued on the current torch stream
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import FMT_CF32, FMT_CS8, FMT_CS16, FMT_CU8, Config, Outputs, bytes_per_sample, check, lib  # noqa: F401 (formats re-exported)

PMR_OUTPUTS = ("res", "chan", "demod", "lpcomp", "audio", "pcm")
DSD_OUTPUTS = ("dsd_audio", "dsd_pcm")   # per-channel DSD feed, PmrBatch(dsd_rate=48000)


def _samples(iq, bps):
    """IQ samples per row of a host array in the handle's format (any dtype: the row is read as bytes)."""
    return iq.shape[1] * iq.itemsize // bps


def _columns(chunk, iq, bps):
    """Array columns that hold `chunk` IQ samples."""
    return chunk * bps // iq.itemsize


def default_config(**kw):
    cfg = Config()
    lib().pmr446_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError("pmr446_config has no field %r" % k)
        setattr(cfg, k, v)
    return cfg


class PmrBatch:
    def __init__(self, cfg=None, **kw):
        self.cfg = cfg if cfg is not None else default_config(**kw)
        self._keep = []
        h = C.c_void_p()
        check(lib().pmr446_batch_create(C.byref(self.cfg), C.byref(h)), "pmr446_batch_create")
        self.h = h
        self.S = self.cfg.n_streams
        self.M = self.cfg.num_channels
        self.max_res = lib().pmr446_batch_max_res(self.h)
        self.max_ns = lib().pmr446_batch_max_ns(self.h)
        self.max_dsd = lib().pmr446_batch_max_dsd(self.h)
        self.bytes_per_sample = bytes_per_sample(self.cfg.in_fmt)

    def close(self):
        if getattr(self, "h", None) and lib is not None:
            try:
                lib().pmr446_batch_destroy(self.h)
            except TypeError:  # interpreter shutdown
                pass
            self.h = None

    __del__ = close

    def reset(self):
        check(lib().pmr446_batch_reset(self.h), "pmr446_batch_reset")

    @property
    def last_launches(self):
        return lib().pmr446_batch_last_launches(self.h)

    @property
    def last_dsd(self):
        """dsd_audio / dsd_pcm samples per row the last execute call wrote."""
        return lib().pmr446_batch_last_dsd(self.h)

    TIMING_TAGS = ("start", "dc_carry", "cascade0", "cascade1", "cascade2", "hist_save", "channelize", "audio", "waterfall",
                   "gather", "dsd")

    def timing(self, enable=True):
        check(lib().pmr446_batch_timing(self.h, int(enable)), "pmr446_batch_timing")

    def get_timings(self):
        """dict tag -> (total_ms, intervals) since timing(True)."""
        n = len(self.TIMING_TAGS)
        ms = (C.c_double * n)()
        cnt = (C.c_longlong * n)()
        check(lib().pmr446_batch_get_timings(self.h, ms, cnt, n), "pmr446_batch_get_timings")
        return {t: (ms[i], cnt[i]) for i, t in enumerate(self.TIMING_TAGS) if cnt[i]}

    # ---- host buffers ------------------------------------------------------------------------
    def execute(self, iq, want=PMR_OUTPUTS):
        """iq: [S, n*2] uint8 (cu8), int16 (cs16) or int8 (cs8), or [S, n] complex64 (cf32).  Returns dict of numpy arrays."""
        iq = np.ascontiguousarray(iq)
        if iq.ndim == 1:
            iq = iq[None, :]
        assert iq.shape[0] == self.S
        n = _samples(iq, self.bytes_per_sample)
        S, M, ld, rld = self.S, self.M, self.max_ns, self.max_res
        bufs = {}
        out = Outputs()
        out.ld, out.res_ld = ld, rld
        if "res" in want:
            bufs["res"] = np.zeros((S, rld), np.complex64)
        if "chan" in want:
            bufs["chan"] = np.zeros((S, M, ld), np.complex64)
        for k in ("demod", "lpcomp", "audio"):
            if k in want:
                bufs[k] = np.zeros((S, M, ld), np.float32)
        if "pcm" in want:
            bufs["pcm"] = np.zeros((S, M, ld), np.int16)
        W = self.cfg.waterfall
        if W and "ascii" in want:
            bufs["ascii"] = np.zeros((S, W), np.uint8)
            bufs["peak"] = np.zeros((S, 2), np.float32)
            bufs["psd"] = np.zeros((S, 4 * W), np.float32)
        if "rssi" in want:
            bufs["rssi"] = np.zeros((S, M), np.float32)
        if "chan_edge" in want:
            bufs["chan_edge"] = np.zeros((S, M, 2), np.complex64)
        out.dsd_ld = self.max_dsd
        if "dsd_audio" in want:
            bufs["dsd_audio"] = np.zeros((S, M, self.max_dsd), np.float32)
        if "dsd_pcm" in want:
            bufs["dsd_pcm"] = np.zeros((S, M, self.max_dsd), np.int16)
        for k, v in bufs.items():
            setattr(out, k, v.ctypes.data)
        ny, ns = C.c_uint(0), C.c_uint(0)
        check(lib().pmr446_batch_execute(self.h, iq.ctypes.data, iq.strides[0], n, C.byref(out), C.byref(ny), C.byref(ns)),
              "pmr446_batch_execute")
        r = {"ny": ny.value, "ns": ns.value}
        for k, v in bufs.items():
            if k == "res":
                r[k] = v[:, :ny.value]
            elif k in DSD_OUTPUTS:
                r[k] = v[:, :, :self.last_dsd]
            elif k in ("chan", "demod", "lpcomp", "audio", "pcm"):
                r[k] = v[:, :, :ns.value]
            else:
                r[k] = v
        return r

    def run(self, iq, chunk=None, want=PMR_OUTPUTS):
        """Whole capture in chunks of `chunk` samples; outputs concatenated along time."""
        chunk = chunk or self.cfg.max_chunk
        if iq.ndim == 1:
            iq = iq[None, :]
        step = _columns(chunk, iq, self.bytes_per_sample)
        parts = [self.execute(iq[:, o:o + step], want) for o in range(0, iq.shape[1], step)]
        r = {"ny": sum(p["ny"] for p in parts), "ns": sum(p["ns"] for p in parts)}
        for k in parts[0]:
            if k in ("ny", "ns"):
                continue
            if k in ("ascii", "peak", "psd", "rssi", "chan_edge"):
                r[k] = np.stack([p[k] for p in parts], axis=1)
            else:
                r[k] = np.concatenate([p[k] for p in parts], axis=-1)
        return r

    # ---- device buffers (torch tensors are only used as device memory + stream handles) ---------
    def execute_device(self, iq, n, outputs, stream_ptr=None):
        """iq: torch CUDA tensor [S, row] (uint8 or complex64/float32 view); outputs: dict name ->
        torch CUDA tensor laid out as in include/pmr446_b200.h plus 'ld'/'res_ld'/'dsd_ld'.  Asynchronous; the DSD feed's
        count per row is last_dsd once the call returns."""
        import torch
        out = Outputs()
        out.ld = int(outputs.get("ld", self.max_ns))
        out.res_ld = int(outputs.get("res_ld", self.max_res))
        out.dsd_ld = int(outputs.get("dsd_ld", self.max_dsd))
        for k in ("res", "chan", "demod", "lpcomp", "audio", "pcm", "ascii", "peak", "psd", "rssi", "chan_edge") + DSD_OUTPUTS:
            t = outputs.get(k)
            if t is not None:
                setattr(out, k, t.data_ptr())
        if stream_ptr is None:
            stream_ptr = torch.cuda.current_stream().cuda_stream
        ny, ns = C.c_uint(0), C.c_uint(0)
        stride = iq.stride(0) * iq.element_size()
        check(lib().pmr446_batch_execute_device(self.h, iq.data_ptr(), stride, n, C.byref(out), C.byref(ny), C.byref(ns),
                                                C.c_void_p(stream_ptr)), "pmr446_batch_execute_device")
        return ny.value, ns.value


class PmrReceiver:
    """n_streams reference receivers: RSSI, squelch / selector, selected-channel audio, CTCSS detector
    (/root/reference/src/sdr_pmr446.c:828-908).  Keyword arguments not named below configure the DSP chain."""

    STATUS_FIELDS = ("state", "active_chan", "rssi", "n_audio", "tone_detected", "ctcss_index", "ctcss_freq", "max_power", "events")

    def __init__(self, squelch_level=18.0, channel_mask=2 ** 64 - 1, lock_mode=0, ctcss_block=2441, ctcss_dc_alpha=0.0005, **chain_kw):
        self.cfg = _lib.RxConfig()
        lib().pmr446_rx_default_config(C.byref(self.cfg))
        for k, v in chain_kw.items():
            if not hasattr(self.cfg.chain, k):
                raise AttributeError("pmr446_config has no field %r" % k)
            setattr(self.cfg.chain, k, v)
        self.cfg.squelch_level = squelch_level
        self.cfg.channel_mask = channel_mask
        self.cfg.lock_mode = lock_mode
        self.cfg.ctcss_block = ctcss_block
        self.cfg.ctcss_dc_alpha = ctcss_dc_alpha
        h = C.c_void_p()
        check(lib().pmr446_receiver_create(C.byref(self.cfg), C.byref(h)), "pmr446_receiver_create")
        self.h = h
        self.S = self.cfg.chain.n_streams
        self.M = self.cfg.chain.num_channels
        self.max_ns = lib().pmr446_receiver_max_ns(self.h)
        self.bytes_per_sample = bytes_per_sample(self.cfg.chain.in_fmt)

    def close(self):
        if getattr(self, "h", None) and lib is not None:
            try:
                lib().pmr446_receiver_destroy(self.h)
            except TypeError:  # interpreter shutdown
                pass
            self.h = None

    __del__ = close

    def reset(self):
        check(lib().pmr446_receiver_reset(self.h), "pmr446_receiver_reset")

    @property
    def last_launches(self):
        return lib().pmr446_receiver_last_launches(self.h)

    def execute(self, iq):
        """One chunk of every stream (host buffers).  Returns dict: status fields as [S] arrays, rssi_ch [S, M],
        audio / pcm / ctcss_in [S, ns] (valid for stream s up to n_audio[s]), ctcss_power [S, 38], ns."""
        iq = np.ascontiguousarray(iq)
        if iq.ndim == 1:
            iq = iq[None, :]
        assert iq.shape[0] == self.S
        n = _samples(iq, self.bytes_per_sample)
        S, M, ld = self.S, self.M, self.max_ns
        status = (_lib.RxStatus * S)()
        bufs = {"rssi": np.zeros((S, M), np.float32), "audio": np.zeros((S, ld), np.float32), "pcm": np.zeros((S, ld), np.int16),
                "ctcss_in": np.zeros((S, ld), np.float32), "ctcss_power": np.zeros((S, 38), np.float32)}
        out = _lib.RxOutputs()
        out.ld = ld
        out.status = C.addressof(status)
        for k, v in bufs.items():
            setattr(out, k, v.ctypes.data)
        ns = C.c_uint(0)
        check(lib().pmr446_receiver_execute(self.h, iq.ctypes.data, iq.strides[0], n, C.byref(out), C.byref(ns)),
              "pmr446_receiver_execute")
        r = {k: np.array([getattr(status[s], k) for s in range(S)]) for k in self.STATUS_FIELDS}
        r["ns"] = ns.value
        r["rssi_ch"] = bufs["rssi"]
        r["ctcss_power"] = bufs["ctcss_power"]
        for k in ("audio", "pcm", "ctcss_in"):
            r[k] = bufs[k][:, :ns.value]
        return r

    def execute_device(self, iq, n, outputs, stream_ptr=None):
        """iq: torch CUDA tensor [S, row]; outputs: dict name -> torch CUDA tensor laid out as pmr446_rx_outputs
        ('rssi', 'status' (uint8 [S, sizeof(pmr446_rx_status)]), 'audio', 'pcm', 'ctcss_in', 'ctcss_power', 'ascii', 'peak') plus
        'ld'.  Asynchronous; returns ns."""
        import torch
        out = _lib.RxOutputs()
        out.ld = int(outputs.get("ld", self.max_ns))
        for k in ("rssi", "status", "audio", "pcm", "ctcss_in", "ctcss_power", "ascii", "peak"):
            t = outputs.get(k)
            if t is not None:
                setattr(out, k, t.data_ptr())
        if stream_ptr is None:
            stream_ptr = torch.cuda.current_stream().cuda_stream
        ns = C.c_uint(0)
        stride = iq.stride(0) * iq.element_size()
        check(lib().pmr446_receiver_execute_device(self.h, iq.data_ptr(), stride, n, C.byref(out), C.byref(ns), C.c_void_p(stream_ptr)),
              "pmr446_receiver_execute_device")
        return ns.value

    def run(self, iq, chunk=None):
        """Whole capture in chunks -> list of per-chunk dicts."""
        chunk = chunk or self.cfg.chain.max_chunk
        if iq.ndim == 1:
            iq = iq[None, :]
        step = _columns(chunk, iq, self.bytes_per_sample)
        return [self.execute(iq[:, o:o + step]) for o in range(0, iq.shape[1], step)]


def dsd_default_config(**kw):
    cfg = _lib.DsdConfig()
    lib().dsd446_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError("dsd446_config has no field %r" % k)
        setattr(cfg, k, v)
    return cfg


class DsdBatch:
    """n_streams copies of the dsd_in chain (/root/reference/src/dsd_in.c:167-175)."""

    def __init__(self, cfg=None, **kw):
        self.cfg = cfg if cfg is not None else dsd_default_config(**kw)
        h = C.c_void_p()
        check(lib().dsd446_batch_create(C.byref(self.cfg), C.byref(h)), "dsd446_batch_create")
        self.h = h
        self.S = self.cfg.n_streams
        self.max_res = lib().dsd446_batch_max_res(self.h)
        self.max_out = lib().dsd446_batch_max_out(self.h)
        self.bytes_per_sample = bytes_per_sample(self.cfg.in_fmt)

    def close(self):
        if getattr(self, "h", None) and lib is not None:
            try:
                lib().dsd446_batch_destroy(self.h)
            except TypeError:  # interpreter shutdown
                pass
            self.h = None

    __del__ = close

    def reset(self):
        check(lib().dsd446_batch_reset(self.h), "dsd446_batch_reset")

    @property
    def last_launches(self):
        return lib().dsd446_batch_last_launches(self.h)

    def execute(self, iq):
        iq = np.ascontiguousarray(iq)
        if iq.ndim == 1:
            iq = iq[None, :]
        assert iq.shape[0] == self.S
        n = _samples(iq, self.bytes_per_sample)
        S = self.S
        res = np.zeros((S, self.max_res), np.complex64)
        fm = np.zeros((S, self.max_res), np.float32)
        audio = np.zeros((S, self.max_out), np.float32)
        pcm = np.zeros((S, self.max_out), np.int16)
        out = _lib.DsdOutputs(res.ctypes.data, fm.ctypes.data, self.max_res, audio.ctypes.data, pcm.ctypes.data, self.max_out)
        ny, nz = C.c_uint(0), C.c_uint(0)
        check(lib().dsd446_batch_execute(self.h, iq.ctypes.data, iq.strides[0], n, C.byref(out), C.byref(ny), C.byref(nz)),
              "dsd446_batch_execute")
        return {"ny": ny.value, "nz": nz.value, "res": res[:, :ny.value], "fm": fm[:, :ny.value],
                "audio": audio[:, :nz.value], "pcm": pcm[:, :nz.value]}

    def run(self, iq, chunk=None):
        chunk = chunk or self.cfg.max_chunk
        if iq.ndim == 1:
            iq = iq[None, :]
        step = _columns(chunk, iq, self.bytes_per_sample)
        parts = [self.execute(iq[:, o:o + step]) for o in range(0, iq.shape[1], step)]
        r = {"ny": sum(p["ny"] for p in parts), "nz": sum(p["nz"] for p in parts)}
        for k in ("res", "fm", "audio", "pcm"):
            r[k] = np.concatenate([p[k] for p in parts], axis=-1)
        return r

    def execute_device(self, iq, n, res=None, fm=None, audio=None, pcm=None, stream_ptr=None):
        import torch
        out = _lib.DsdOutputs()
        out.res_ld = self.max_res
        out.out_ld = self.max_out
        for k, t in (("res", res), ("fm", fm), ("audio", audio), ("pcm", pcm)):
            if t is not None:
                setattr(out, k, t.data_ptr())
        if stream_ptr is None:
            stream_ptr = torch.cuda.current_stream().cuda_stream
        ny, nz = C.c_uint(0), C.c_uint(0)
        stride = iq.stride(0) * iq.element_size()
        check(lib().dsd446_batch_execute_device(self.h, iq.data_ptr(), stride, n, C.byref(out), C.byref(ny), C.byref(nz),
                                                C.c_void_p(stream_ptr)), "dsd446_batch_execute_device")
        return ny.value, nz.value


def measure_fp32_peak():
    v = C.c_double(0.0)
    check(lib().pmr446_measure_fp32_peak(C.byref(v), None), "pmr446_measure_fp32_peak")
    return v.value
