"""Shared helpers for the parity tests."""
import numpy as np

# north_star tolerances (BASELINE.json): float stage outputs within 1e-4 relative RMS of the
# reference chain, final s16 audio within +-1 LSB.
REL_RMS_TOL = 1e-4
PCM_TOL_LSB = 1


def rel_rms(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    den = np.sqrt(np.mean(np.abs(b.astype(np.complex128 if np.iscomplexobj(b) else np.float64)) ** 2))
    num = np.sqrt(np.mean(np.abs(a.astype(np.complex128 if np.iscomplexobj(a) else np.float64) - b) ** 2))
    return float(num / den) if den > 0 else float(num)


def active_channels(spec_carriers):
    """0-based channel indices that carry a signal (discriminator parity is only meaningful there, SURVEY.md 7)."""
    return sorted({c.channel - 1 for c in spec_carriers})


# ---- the filter design the library runs with (host-only entry points, no GPU needed) ----------------------------------
def design_pfbch(M, m=13, as_db=80.0):
    """firpfbch_crcf_create_kaiser(ANALYZER, M, m, as) branch taps [M][2m], taps[i][n] = h[i + n M]."""
    import ctypes as C

    from sdr_pmr446_b200._lib import check, lib
    t = np.zeros((M, 2 * m), np.float32)
    check(lib().pmr446_design_pfbch(M, m, C.c_float(as_db), t.ctypes.data), "pmr446_design_pfbch")
    return t


def nco_offset(M):
    """The channelizer's mix-down frequency -0.5 (M - 1) / M 2 pi as pmr446_batch_create and the oracle form it in float32."""
    import math
    o = np.float32(np.float32(np.float32(-0.5) * np.float32(M - 1)) / np.float32(M)) * np.float32(2)
    return float(np.float32(float(o) * math.pi))


def design_dtheta(M):
    """32-bit NCO increment of the channelizer's mix-down."""
    from sdr_pmr446_b200._lib import lib
    return int(lib().pmr446_design_nco_dtheta(nco_offset(M)))


def design_msresamp(rate, as_db=60.0):
    """msresamp_crcf_create(rate, as) / msresamp_rrrf_create as the library plans it: dict of stages, m, step, npfb,
    hb [16][20] and pfb [npfb][14] (the form tests/stage_ref.py takes)."""
    import ctypes as C

    from sdr_pmr446_b200._lib import check, lib
    st, m, step, npfb = C.c_uint(), (C.c_uint * 16)(), C.c_uint(), C.c_uint()
    hb, pfb = np.zeros((16, 20), np.float32), np.zeros((256, 14), np.float32)
    check(lib().pmr446_design_msresamp(np.float32(rate), as_db, C.byref(st), m, C.byref(step), C.byref(npfb), hb.ctypes.data,
                                       pfb.ctypes.data), "pmr446_design_msresamp")
    return dict(stages=st.value, m=list(m)[:st.value], step=step.value, npfb=npfb.value, hb=hb, pfb=pfb[:npfb.value])


def describe_frontend(rate, fmt, with_dc=1, as_db=60.0):
    """pmr446_describe_frontend: the plan string of the front end ("fused[3,5,10]+arb", "cascade[3,5] | tile[10]+arb", ...)."""
    import ctypes as C

    from sdr_pmr446_b200._lib import check, lib
    buf = C.create_string_buffer(256)
    check(lib().pmr446_describe_frontend(np.float32(rate), as_db, fmt, with_dc, buf, 256), "pmr446_describe_frontend")
    return buf.value.decode()


def design_asgram_window(W):
    from sdr_pmr446_b200._lib import check, lib
    w = np.zeros(W, np.float32)
    check(lib().pmr446_design_asgram_window(W, w.ctypes.data), "pmr446_design_asgram_window")
    return w
