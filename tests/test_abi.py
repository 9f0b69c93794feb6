"""C-ABI checks that need no GPU: the library loads, exports every symbol include/pmr446_b200.h declares,
refuses to run without a device (no CPU fallback), and its host-side filter design / sample-count
bookkeeping equals the oracle's (i.e. liquid-dsp's formulas, SURVEY.md Appendix A.2-A.8, A.13)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import oracle as orc
from sdr_pmr446_b200 import _lib, chain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    txt = open(os.path.join(ROOT, "include", "pmr446_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b((?:pmr446|dsd446)_\w+)\s*\(", txt)))


def test_every_declared_symbol_is_exported():
    L = _lib.lib()
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), n
    assert set(_lib.EXPORTS) <= set(names)


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.Pmr446Error) as e:
        chain.PmrBatch()
    assert e.value.code == _lib.ENODEV
    with pytest.raises(_lib.Pmr446Error) as e:
        chain.DsdBatch()
    assert e.value.code == _lib.ENODEV


def test_bad_arguments_are_rejected():
    L = _lib.lib()
    assert L.pmr446_batch_create(None, None) == _lib.EINVAL
    cfg = chain.default_config(num_channels=1)   # outside [2, 4096]: refused before a device is selected
    h = C.c_void_p()
    assert L.pmr446_batch_create(C.byref(cfg), C.byref(h)) == _lib.EINVAL and not h.value
    assert b"num_channels" in L.pmr446_last_error()
    assert L.pmr446_batch_execute(None, None, 0, 0, None, None, None) == _lib.EINVAL
    assert b"null" in L.pmr446_last_error()


def test_default_config_is_the_reference_setup():
    c = chain.default_config()
    assert (c.fs_in, c.num_channels, c.channel_width, c.pfb_m, c.max_chunk) == (1024000, 16, 12500, 13, 100000)
    assert (c.pfb_as, c.resamp_as, c.kf, c.audio_gain) == (80.0, 60.0, 0.5, 4.0)
    assert abs(c.dc_alpha - 0.0005) < 1e-9 and abs(c.deemph_a1 - 0.014602874461272194) < 1e-8
    d = chain.dsd_default_config()
    assert (d.fs_in, d.fs_sig, d.fs_audio, d.max_chunk) == (1024000, 12500, 48000, 200000)


@pytest.mark.parametrize("rate", [200000 / 1024000, 200000 / 2400000, 12500 / 2400000, 12500 / 1024000, 1.0, 48000 / 12500])
def test_msresamp_design_equals_oracle(rate):
    L, O = _lib.lib(), orc.lib()
    st, m, step, npfb = C.c_uint(), (C.c_uint * 16)(), C.c_uint(), C.c_uint()
    hb = np.zeros((16, 20), np.float32)
    pfb = np.zeros((256, 14), np.float32)
    assert L.pmr446_design_msresamp(rate, 60.0, C.byref(st), m, C.byref(step), C.byref(npfb), hb.ctypes.data, pfb.ctypes.data) == 0
    if rate <= 1.0:
        q = O.msresamp_crcf_create(rate, 60.0)
        ost, om, ra, ostep, onpfb = C.c_uint(), (C.c_uint * 16)(), C.c_float(), C.c_uint(), C.c_uint()
        O.oracle_msresamp_crcf_plan(q, C.byref(ost), om, C.byref(ra), C.byref(ostep), C.byref(onpfb))
        assert (st.value, list(m)[:st.value], step.value, npfb.value) == (ost.value, list(om)[:ost.value], ostep.value, onpfb.value)
        # behavioural check of the taps: impulse response of the oracle object vs a convolution built from the product's taps
        n = 1 << (st.value + 7)
        x = np.zeros(n, np.complex64)
        x[0] = 1.0
        y = np.zeros(n, np.complex64)
        ny = C.c_uint()
        O.msresamp_crcf_execute(q, x.ctypes.data, n, y.ctypes.data, C.byref(ny))
        O.msresamp_crcf_destroy(q)
        assert L.pmr446_count_resampled(rate, 60.0, n) == ny.value
        # total DC gain of the product design: each half-band stage has gain 2 (x zeta = 1), each bank row ~1
        for g in range(st.value):
            assert abs(1.0 + hb[g, :2 * m[g]].sum() - 2.0) < 2e-3
        assert np.max(np.abs(pfb.sum(axis=1) - 1.0)) < 2e-3
    else:
        assert st.value == 1 and m[0] == 10 and step.value == 8738134


def test_pfbch_and_window_design_equal_oracle():
    L, O = _lib.lib(), orc.lib()
    taps = np.zeros((16, 26), np.float32)
    assert L.pmr446_design_pfbch(16, 13, 80.0, taps.ctypes.data) == 0
    h = np.zeros(417, np.float32)
    O.liquid_firdes_kaiser(417, 0.5 / 16, 80.0, 0.0, h.ctypes.data)
    ref = h[:416].reshape(26, 16).T          # ref[i, n] = h[i + 16 n]
    assert np.array_equal(taps, ref)
    assert abs(taps.sum() - 16.0005) < 1e-3   # Appendix B
    w = np.zeros(120, np.float32)
    assert L.pmr446_design_asgram_window(120, w.ctypes.data) == 0
    hann = 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(120) / 119)
    g = np.sqrt(2) / (np.sqrt(np.mean(hann ** 2)) * np.sqrt(480))
    assert np.max(np.abs(w - g * hann)) < 1e-6
    assert L.pmr446_design_nco_dtheta(np.float32(-0.5 * 15 / 16 * 2 * np.pi)) == 0x88000000


@pytest.mark.parametrize("rate", [200000 / 1024000, 200000 / 2400000])
def test_resampled_count_matches_oracle_for_any_length(rate):
    L, O = _lib.lib(), orc.lib()
    rng = np.random.default_rng(5)
    q = O.msresamp_crcf_create(rate, 60.0)
    total_in = total_out = 0
    for n in [0, 1, 7, 16, 1000, 4097] + list(rng.integers(1, 5000, 20)):
        n = int(n)
        x = np.zeros(max(n, 1), np.complex64)
        y = np.zeros(max(n, 1) + 8, np.complex64)
        ny = C.c_uint()
        O.msresamp_crcf_execute(q, x.ctypes.data, n, y.ctypes.data, C.byref(ny))
        total_in += n
        total_out += ny.value
        assert L.pmr446_count_resampled(rate, 60.0, total_in) == total_out
    O.msresamp_crcf_destroy(q)


def test_receiver_argument_checks_need_no_device():
    """pmr446_receiver_create validates its own arguments before touching the GPU (reference: exits when the channel
    mask is empty, src/sdr_pmr446.c:725; MAX_CHANNELS 64, :18)."""
    L = _lib.lib()
    cfg = _lib.RxConfig()
    L.pmr446_rx_default_config(C.byref(cfg))
    assert cfg.squelch_level == 18.0 and cfg.ctcss_block == 2441 and cfg.lock_mode == 0 and cfg.chain.num_channels == 16
    h = C.c_void_p()
    cfg.channel_mask = 0xFFFF0000            # no enabled channel among the 16
    assert L.pmr446_receiver_create(C.byref(cfg), C.byref(h)) == _lib.EINVAL and not h.value
    assert b"channel_mask" in L.pmr446_last_error()
    L.pmr446_rx_default_config(C.byref(cfg))
    cfg.chain.num_channels = 80
    assert L.pmr446_receiver_create(C.byref(cfg), C.byref(h)) == _lib.EINVAL
    L.pmr446_rx_default_config(C.byref(cfg))
    cfg.chain.deemph_fir = 1
    assert L.pmr446_receiver_create(C.byref(cfg), C.byref(h)) == _lib.EINVAL
    assert L.pmr446_receiver_create(None, C.byref(h)) == _lib.EINVAL
    assert L.pmr446_receiver_max_ns(None) == 0 and L.pmr446_receiver_destroy(None) == _lib.OK


def test_every_decimating_rate_has_a_frontend_plan():
    """msresamp_crcf_create(rate, 60) accepts any rate (src/sdr_pmr446.c:425-426): every decimating rate must be cut into
    instantiated kernels (VERDICT r01 item 8), and the BASELINE plans must keep their intended shape."""
    import ctypes as C

    import numpy as np
    from sdr_pmr446_b200 import _lib
    L = _lib.lib()
    buf = C.create_string_buffer(256)

    def plan(fs_in, fs_out, fmt):
        rc = L.pmr446_describe_frontend(np.float32(fs_out) / np.float32(fs_in), 60.0, fmt, 1, buf, 256)
        assert rc == 0, (fs_in, fs_out, fmt, L.pmr446_last_error())
        return buf.value.decode()

    assert plan(2400000, 200000, 1) == "fused[3,5,10]+arb"                       # configs[2]: one launch
    assert plan(2400000, 200000, 0) == "cascade[3,5] | tile[10]+arb"
    assert plan(1024000, 200000, 1) == "cascade[5,10] | cascade[]+arb"           # configs[0]
    assert plan(2400000, 12500, 1) == "front6[3,3,3,3,3,5] | tile[10]+arb"             # configs[1]: six half-bands in one launch
    assert plan(1024000, 12500, 1) == "front6[3,3,3,3,5,10] | cascade[]+arb"           # dsd_in at the reference's own rate
    assert plan(20000000, 20000000, 0) == "cascade[]+arb"                        # configs[3]: rate 1.0
    assert plan(3200000, 200000, 1) == "cascade[3,5] | cascade[10]+arb"
    rng = np.random.default_rng(7)
    rates = list(rng.uniform(np.log(1e-4), 0.0, 300))
    for lr in rates:
        r = float(np.exp(lr))
        for fmt in (0, 1):
            rc = L.pmr446_describe_frontend(np.float32(r), 60.0, fmt, 1, buf, 256)
            assert rc == 0, (r, fmt, L.pmr446_last_error())
    assert L.pmr446_describe_frontend(np.float32(1.5), 60.0, 0, 1, buf, 256) != 0      # interpolation is msresamp_rrrf's job (dsd_in)


def test_makefile_lists_every_kernel_header():
    """A header missing from HDRS means an edit to it does not rebuild the library that travels to the GPU box."""
    import glob
    import os
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sdr_pmr446_b200", "csrc")
    mk = open(os.path.join(root, "Makefile")).read().replace("\\\n", " ")
    hdrs = set(re.search(r"^HDRS\s*=\s*(.*)$", mk, re.M).group(1).split())
    have = {os.path.basename(p) for p in glob.glob(os.path.join(root, "*.cuh")) + glob.glob(os.path.join(root, "*.hpp"))}
    assert have <= hdrs, sorted(have - hdrs)


def test_library_reads_no_environment_variables():
    """The library's behaviour is a function of its configuration struct alone, not of the environment of the process that loads it."""
    import glob
    import os
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sdr_pmr446_b200", "csrc")
    srcs = [p for ext in ("*.cu", "*.cuh", "*.hpp") for p in glob.glob(os.path.join(root, ext))]
    assert srcs
    hits = [os.path.basename(p) for p in srcs if re.search(r"\bgetenv\b", open(p).read())]
    assert not hits, hits
