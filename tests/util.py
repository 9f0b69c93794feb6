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


def design_asgram_window(W):
    from sdr_pmr446_b200._lib import check, lib
    w = np.zeros(W, np.float32)
    check(lib().pmr446_design_asgram_window(W, w.ctypes.data), "pmr446_design_asgram_window")
    return w
