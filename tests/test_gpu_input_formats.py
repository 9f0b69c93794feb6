"""CS16 and CS8 input on the GPU.  Both conversions (x / 32768, x / 128) are exact in float32, so a handle fed integers
must return bitwise what the same handle type returns when fed the converted cf32 samples: every output array and every
count of every call, for the batch, receiver and dsd_in chains.

Call shapes: 3 streams (2 at 20 Msps) read from rows wider than the chunk (iq_stride > row), uneven chunks including
0, 1 and 7 samples, host-buffer and device-buffer calls alternating on one handle, device rows that start one sample past
a 32-byte boundary (only the guarded per-sample loader can read them), full-scale samples including -32768 and -128, and
a reset in the middle of the run.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BITS = {"cs16": 15, "cs8": 7}
RESET = "reset"


def _fmt(name):
    from sdr_pmr446_b200 import _lib
    return {"cs16": _lib.FMT_CS16, "cs8": _lib.FMT_CS8, "cf32": _lib.FMT_CF32}[name]


def _captures(name, fs, S, n, M=16, seed=446):
    """[S, 2n] interleaved integers of format `name` and the [S, n] complex64 samples they stand for."""
    from sdr_pmr446_b200 import synth
    make = synth.make_cs16 if name == "cs16" else synth.make_cs8
    q = np.stack([make(synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=synth.rotated_carriers(s, M)), n, seed + s)
                  for s in range(S)])
    full = 1 << BITS[name]
    q[:, 4000:4100:2] = -full           # a full-scale burst: the most negative value and the largest positive one
    q[:, 4001:4100:2] = full - 1
    q[:, 9001::7919] = -full
    x = (q.astype(np.float32) * np.float32(2.0 ** -BITS[name])).view(np.complex64)
    return q, x


class _Src:
    """A capture's rows inside wider rows (iq_stride > row), `lead` bytes after the row start, on the host and the device."""

    def __init__(self, a, lead):
        import torch
        raw = np.ascontiguousarray(a).view(np.uint8)
        S, nb = raw.shape
        stride = (lead + nb + 96 + 31) // 32 * 32
        full = np.zeros((S, stride), np.uint8)
        full[:, lead:lead + nb] = raw
        self.host = full[:, lead:lead + nb]
        self.dev = torch.from_numpy(full).cuda()[:, lead:lead + nb]
        assert self.host.strides[0] == stride > nb and self.dev.stride(0) == stride

    def host_ptr(self, off, bps):
        return self.host.ctypes.data + off * bps, self.host.strides[0]

    def dev_view(self, off, n, bps):
        return self.dev[:, off * bps:(off + n) * bps]


def _arrays(shapes, device):
    import torch
    return {k: (torch.from_numpy(np.zeros(s, t)).cuda() if device else np.zeros(s, t)) for k, (s, t) in shapes.items()}


def _to_host(arrs):
    import torch
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in arrs.items()}


def _call_pmr(b, src, off, n, device):
    from sdr_pmr446_b200._lib import Outputs, check, lib
    S, M, ld, rld, W = b.S, b.M, b.max_ns, b.max_res, b.cfg.waterfall
    shapes = {"res": ((S, rld), np.complex64), "chan": ((S, M, ld), np.complex64), "demod": ((S, M, ld), np.float32),
              "lpcomp": ((S, M, ld), np.float32), "audio": ((S, M, ld), np.float32), "pcm": ((S, M, ld), np.int16)}
    if W:
        shapes.update(ascii=((S, W), np.uint8), peak=((S, 2), np.float32), psd=((S, 4 * W), np.float32))
    arrs = _arrays(shapes, device)
    if device:
        ny, ns = b.execute_device(src.dev_view(off, n, b.bytes_per_sample), n, dict(arrs, ld=ld, res_ld=rld))
    else:
        out = Outputs()
        out.ld, out.res_ld = ld, rld
        for k, v in arrs.items():
            setattr(out, k, v.ctypes.data)
        cy, cs = C.c_uint(), C.c_uint()
        ptr, stride = src.host_ptr(off, b.bytes_per_sample)
        check(lib().pmr446_batch_execute(b.h, ptr, stride, n, C.byref(out), C.byref(cy), C.byref(cs)), "pmr446_batch_execute")
        ny, ns = cy.value, cs.value
    return dict(_to_host(arrs), ny=ny, ns=ns)


def _call_rx(r, src, off, n, device):
    from sdr_pmr446_b200 import _lib
    S, M, ld, W = r.S, r.M, r.max_ns, r.cfg.chain.waterfall
    shapes = {"rssi": ((S, M), np.float32), "status": ((S, C.sizeof(_lib.RxStatus)), np.uint8), "audio": ((S, ld), np.float32),
              "pcm": ((S, ld), np.int16), "ctcss_in": ((S, ld), np.float32), "ctcss_power": ((S, 38), np.float32)}
    if W:
        shapes.update(ascii=((S, W), np.uint8), peak=((S, 2), np.float32))
    arrs = _arrays(shapes, device)
    if device:
        ns = r.execute_device(src.dev_view(off, n, r.bytes_per_sample), n, dict(arrs, ld=ld))
    else:
        out = _lib.RxOutputs()
        out.ld = ld
        for k, v in arrs.items():
            setattr(out, k, v.ctypes.data)
        cs = C.c_uint()
        ptr, stride = src.host_ptr(off, r.bytes_per_sample)
        _lib.check(_lib.lib().pmr446_receiver_execute(r.h, ptr, stride, n, C.byref(out), C.byref(cs)), "pmr446_receiver_execute")
        ns = cs.value
    return dict(_to_host(arrs), ns=ns)


def _call_dsd(d, src, off, n, device):
    from sdr_pmr446_b200 import _lib
    S = d.S
    shapes = {"res": ((S, d.max_res), np.complex64), "fm": ((S, d.max_res), np.float32), "audio": ((S, d.max_out), np.float32),
              "pcm": ((S, d.max_out), np.int16)}
    arrs = _arrays(shapes, device)
    if device:
        ny, nz = d.execute_device(src.dev_view(off, n, d.bytes_per_sample), n, **arrs)
    else:
        out = _lib.DsdOutputs(arrs["res"].ctypes.data, arrs["fm"].ctypes.data, d.max_res, arrs["audio"].ctypes.data,
                              arrs["pcm"].ctypes.data, d.max_out)
        cy, cz = C.c_uint(), C.c_uint()
        ptr, stride = src.host_ptr(off, d.bytes_per_sample)
        _lib.check(_lib.lib().dsd446_batch_execute(d.h, ptr, stride, n, C.byref(out), C.byref(cy), C.byref(cz)), "dsd446_batch_execute")
        ny, nz = cy.value, cz.value
    return dict(_to_host(arrs), ny=ny, nz=nz)


def _compare(name, make, call, q, x, sizes, lead):
    """Feeds q to make(name's format) and x to make(cf32) call by call (`sizes` samples per stream, RESET = reset both
    handles), host and device calls alternating, and requires every result of every call to be bitwise equal."""
    hi, hf = make(_fmt(name)), make(_fmt("cf32"))
    assert (hi.bytes_per_sample, hf.bytes_per_sample) == ({"cs16": 4, "cs8": 2}[name], 8)
    si, sf = _Src(q, lead * hi.bytes_per_sample), _Src(x, lead * hf.bytes_per_sample)
    off, produced = 0, 0
    for k, n in enumerate(sizes):
        if n == RESET:
            hi.reset()
            hf.reset()
            continue
        device = k % 2 == 1
        ri, rf = call(hi, si, off, n, device), call(hf, sf, off, n, device)
        assert ri.keys() == rf.keys()
        for key in rf:
            if isinstance(rf[key], np.ndarray):
                assert ri[key].shape == rf[key].shape and ri[key].tobytes() == rf[key].tobytes(), (k, n, device, key)
            else:
                assert ri[key] == rf[key], (k, n, device, key)
                produced += rf[key]
        off += n
    assert off <= x.shape[1] and produced > 0
    hi.close()
    hf.close()


# 0, 1 and 7-sample calls, chunk edges off the 16-sample grid, a reset in the middle
def _sizes(chunk):
    return [chunk, 0, 1, 7, chunk - 8, chunk // 3 + 5, RESET, chunk, 13, chunk // 2, chunk]


@pytest.mark.parametrize("name", ["cs16", "cs8"])
@pytest.mark.parametrize("fs,lead", [(1024000, 0), (2400000, 1), (3200000, 0)])
def test_batch_to_200k_with_waterfall(name, fs, lead):
    """1.024 Msps ([5,10] | resampler), 2.4 Msps ([3,5] | tile[10]: the cf32 plan, not the fused cu8 kernel) and 3.2 Msps
    ([3,5] | [10] + resampler) -> 200 kHz: res, chan, demod, lpcomp, audio, pcm and a W = 120 waterfall."""
    from sdr_pmr446_b200 import chain
    chunk = fs // 25
    sizes = _sizes(chunk)
    q, x = _captures(name, fs, 3, sum(s for s in sizes if s != RESET) + 64)
    make = lambda f: chain.PmrBatch(n_streams=3, fs_in=fs, in_fmt=f, audio_gain=1.0, max_chunk=chunk, waterfall=120)  # noqa: E731
    _compare(name, make, _call_pmr, q, x, sizes, lead)


@pytest.mark.parametrize("name", ["cs16", "cs8"])
def test_batch_generic_channelizer_and_time_sliced_copy(name):
    """M = 20 (the generic channelizer, 250 kHz from 1.024 Msps) and a host call of 600 000 samples, which is cut in time
    into sub-chunks whose copies overlap the kernels."""
    from sdr_pmr446_b200 import chain
    sizes = [7, 600000, 1, 0, 50000, RESET, 40001]
    q, x = _captures(name, 1024000, 3, sum(s for s in sizes if s != RESET) + 64, M=20)
    make = lambda f: chain.PmrBatch(n_streams=3, fs_in=1024000, in_fmt=f, num_channels=20, audio_gain=1.0, max_chunk=600000)  # noqa: E731
    _compare(name, make, _call_pmr, q, x, sizes, 1)


@pytest.mark.parametrize("name", ["cs16", "cs8"])
def test_batch_rate_one_1600_channels(name):
    """Rate 1.0 (20 Msps into 1600 channels): the resampler alone behind the DC_SCAN pre-pass (dc_local_kernel)."""
    from sdr_pmr446_b200 import chain
    sizes = _sizes(32000)
    q, x = _captures(name, 20000000, 2, sum(s for s in sizes if s != RESET) + 64, M=1600)
    make = lambda f: chain.PmrBatch(n_streams=2, fs_in=20000000, in_fmt=f, num_channels=1600, audio_gain=1.0, max_chunk=32000)  # noqa: E731
    _compare(name, make, _call_pmr, q, x, sizes, 0)


@pytest.mark.parametrize("name", ["cs16", "cs8"])
def test_receiver_2400k(name):
    """The receiver: RSSI, every status field and event, selected audio / pcm, the CTCSS branch and powers, waterfall row."""
    from sdr_pmr446_b200 import chain
    chunk = 120000
    sizes = _sizes(chunk) + [chunk] * 4
    q, x = _captures(name, 2400000, 3, sum(s for s in sizes if s != RESET) + 64)
    make = lambda f: chain.PmrReceiver(n_streams=3, fs_in=2400000, in_fmt=f, max_chunk=chunk, audio_gain=1.0, waterfall=64)  # noqa: E731
    _compare(name, make, _call_rx, q, x, sizes, 0)


@pytest.mark.parametrize("name", ["cs16", "cs8"])
@pytest.mark.parametrize("fs", [1024000, 2400000])
def test_dsd_in(name, fs):
    """dsd_in at 1.024 and 2.4 Msps (the cf32 cascades, not the six-stage cu8 kernel): res, fm, audio, pcm, ny, nz."""
    from sdr_pmr446_b200 import chain
    chunk = 100000
    sizes = _sizes(chunk)
    q, x = _captures(name, fs, 3, sum(s for s in sizes if s != RESET) + 64)
    make = lambda f: chain.DsdBatch(n_streams=3, fs_in=fs, in_fmt=f, max_chunk=chunk)  # noqa: E731
    _compare(name, make, _call_dsd, q, x, sizes, 1)


@pytest.mark.parametrize("name,flag", [("cs16", "-16"), ("cs8", "-s8")])
def test_rx_file_harness_integer_capture(tmp_path, name, flag):
    """pmr446_rx_file on an integer capture writes the WAV and the log lines of the cf32 run on the converted capture."""
    import rx_scenarios as sc
    from sdr_pmr446_b200 import synth
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "host"), "-s"])
    make = synth.make_cs16 if name == "cs16" else synth.make_cs8
    q = make(synth.CaptureSpec(fs=float(sc.FS), carriers=sc.keyed_two_calls()), int(2.0 * sc.FS), 446)
    (tmp_path / "cap.int").write_bytes(q.tobytes())
    (q.astype(np.float32) * np.float32(2.0 ** -BITS[name])).tofile(tmp_path / "cap.cf32")
    runs = {}
    for kind, args in (("int", [flag]), ("cf32", [])):
        wav = tmp_path / ("%s.wav" % kind)
        p = subprocess.run([os.path.join(ROOT, "host", "pmr446_rx_file")] + args + ["-g", "1.0", "-o", str(wav), str(tmp_path / ("cap." + kind))],
                           check=True, capture_output=True, text=True)
        runs[kind] = (wav.read_bytes(), p.stderr)
    assert "Tuned to channel 2" in runs["cf32"][1] and "Acquired CTCSS code" in runs["cf32"][1]
    assert runs["int"][1] == runs["cf32"][1]
    assert len(runs["int"][0]) > 44 + 2 * 20000 and runs["int"][0] == runs["cf32"][0]
