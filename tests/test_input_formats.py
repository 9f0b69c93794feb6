"""CS16 and CS8 input formats without a GPU: the ABI constants and symbols, the front-end plans they get, the byte width
every layer uses, and the synthetic quantisers at full scale."""
import ctypes as C
import os
import re

import numpy as np

from sdr_pmr446_b200 import _lib, chain, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_format_constants_and_symbol_are_exported():
    hdr = open(os.path.join(ROOT, "include", "pmr446_b200.h")).read()
    consts = dict((k, int(v)) for k, v in re.findall(r"#define PMR446_FMT_(\w+) (\d+)", hdr))
    assert consts == {"CF32": 0, "CU8": 1, "CS16": 2, "CS8": 3}
    assert (_lib.FMT_CF32, _lib.FMT_CU8, _lib.FMT_CS16, _lib.FMT_CS8) == (0, 1, 2, 3)
    assert (chain.FMT_CS16, chain.FMT_CS8) == (2, 3)
    assert "pmr446_bytes_per_sample" in _lib.EXPORTS
    assert hasattr(_lib.lib(), "pmr446_bytes_per_sample")


def test_bytes_per_sample_python_equals_library():
    L = _lib.lib()
    expect = {_lib.FMT_CU8: 2, _lib.FMT_CS8: 2, _lib.FMT_CS16: 4, _lib.FMT_CF32: 8, 4: 8, 7: 8, -1: 8, 1 << 20: 8}
    for fmt, bps in expect.items():
        assert L.pmr446_bytes_per_sample(fmt) == bps, fmt
        assert _lib.bytes_per_sample(fmt) == bps, fmt


def test_integer_formats_get_the_cf32_plans():
    """The same 300-rate sweep test_abi.py runs: CS16 and CS8 describe exactly the cf32 plan (the fused and front6 cu8
    kernels are never chosen for them), and every one of those plans has its kernels instantiated for the new loaders."""
    L = _lib.lib()
    buf = C.create_string_buffer(256)

    def plan(rate, fmt):
        rc = L.pmr446_describe_frontend(np.float32(rate), 60.0, fmt, 1, buf, 256)
        assert rc == 0, (rate, fmt, L.pmr446_last_error())
        return buf.value.decode()

    named = [(200000, 2400000), (200000, 1024000), (200000, 3200000), (12500, 2400000), (12500, 1024000), (1, 1)]
    rng = np.random.default_rng(7)
    rates = [float(np.exp(lr)) for lr in rng.uniform(np.log(1e-4), 0.0, 300)] + [a / b for a, b in named]
    for r in rates:
        ref = plan(r, _lib.FMT_CF32)
        assert plan(r, _lib.FMT_CS16) == ref, r
        assert plan(r, _lib.FMT_CS8) == ref, r
        assert "fused" not in ref and "front6" not in ref
    assert plan(200000 / 2400000, _lib.FMT_CS16) == "cascade[3,5] | tile[10]+arb"


def test_quantisers_round_trip_at_full_scale():
    for to, bits, dt in ((synth.to_cs16, 16, np.int16), (synth.to_cs8, 8, np.int8)):
        full = 1 << (bits - 1)
        q = np.array([-full, full - 1, 0, 1, -1, full // 2, -full // 2, full - 2, -full + 1, -full], dt)   # interleaved I, Q
        # the float32 value the library computes, x / 2^(bits-1), is exact: integer -> cf32 -> integer is the identity
        f = q.astype(np.float32) / np.float32(full)
        assert np.array_equal(f.astype(np.float64) * full, q.astype(np.float64))
        back = to(f[0::2].astype(np.complex128) + 1j * f[1::2])
        assert back.dtype == dt and np.array_equal(back, q)
        # beyond full scale: saturated, not wrapped
        sat = to(np.array([2.0 - 2.0j, -2.0 + 2.0j, 1.0 - 1.0j]))
        assert list(sat) == [full - 1, -full, -full, full - 1, full - 1, -full]


def test_make_integer_captures_quantise_the_cf32_capture():
    spec = synth.CaptureSpec(fs=1024000.0)
    x = synth.make_cf64(spec, 5000, 9)
    assert np.array_equal(synth.make_cs16(spec, 5000, 9), synth.to_cs16(x))
    assert np.array_equal(synth.make_cs8(spec, 5000, 9), synth.to_cs8(x))
    q = synth.make_cs16(spec, 5000, 9).astype(np.float64) / 32768
    assert np.max(np.abs(q[0::2] - x.real)) <= 0.5 / 32768 + 1e-12
