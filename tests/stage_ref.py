"""Float64 references of single stages of the PMR446 chain (plain NumPy, complex128 / float64).

Each function takes the previous stage's output as given (for a GPU test: the GPU's own float32 output of that
stage) and computes one stage exactly, so a comparison measures only the rounding of the stage under test and not the
error accumulated upstream.  The conventions are the ones oracle/liquid_subset.c and oracle/chains.c restate from
liquid-dsp:

  channelize  nco_crcf_mix_down with theta_j = j dtheta mod 2^32 (sample j from stream start), then the firpfbch
              analyzer: sample M f + k of frame f enters branch M - 1 - k, X[k] = sum_n taps[M-1-k][n] x[M (f-n) + k]
              with taps[i][n] = h[i + n M] (pmr446_design_pfbch), y = forward M-point DFT of X; freqdem against the
              previous frame (frame -1 = 0).
  audio       firfilt (HP) from zero state, wdelayf((hp_len - 1) / 2) minus HP = lpcomp, gain, one-pole
              iirfilt b = {b0, b1}, a = {1, a1} from zero state, optional LP firfilt, s16 = trunc(clip(32767 a)).
  asgram      one call = one row: the window buffer starts at zero, a transform of the last W samples every
              floor(W / 2) samples of the call, 4 W-point zero-padded DFT, power averaged over the call's
              transforms, FFT-shifted, 10 log10(max(p, 1e-12)); row characters from the maximum of 4 bins against
              the levels -40 + 2 j dB (asgramcf_set_scale(-40, 2)).
"""
import numpy as np
from scipy import signal

LEVEL_CHARS = b" .,-+*&NM#"
ASGRAM_REF, ASGRAM_DIV = -40.0, 2.0


def nco_phase(n, dtheta, j0=0):
    """theta_j / 2^32 for samples j0 .. j0 + n - 1, from exact integer phases."""
    j = np.arange(j0, j0 + n, dtype=np.uint64)
    th = (j * np.uint64(dtheta)) & np.uint64(0xFFFFFFFF)
    return th.astype(np.float64) / 4294967296.0


def discriminator(chan, kf):
    """freqdem over the frames of every channel: arg(conj(y[f-1]) y[f]) / (2 pi kf), y[-1] = 0.

    The products are formed component-wise as liquid does, so frame 0's arg(conj(0) y) keeps the sign of zero the
    reference itself produces (+-pi or 0)."""
    y = np.asarray(chan, np.complex128)
    prev = np.concatenate([np.zeros(y.shape[:-1] + (1,), np.complex128), y[..., :-1]], axis=-1)
    re = prev.real * y.real + prev.imag * y.imag
    im = prev.real * y.imag - prev.imag * y.real
    return np.arctan2(im, re) / (2.0 * np.pi * float(kf))


def channelize(res, M, taps, dtheta, kf):
    """res: un-mixed resampler output [n] from stream start; taps [M][2m].  Returns chan [M][F], demod [M][F], F = n // M."""
    x = np.asarray(res, np.complex128)
    F = x.shape[0] // M
    x = x[:F * M] * np.exp(-2j * np.pi * nco_phase(F * M, dtheta))
    fr = x.reshape(F, M)                                   # fr[f, k] = x[M f + k]
    t = np.asarray(taps, np.float64).reshape(M, -1)[::-1]  # t[k, n] = taps[M - 1 - k][n]
    X = np.zeros((F, M), np.complex128)
    for n in range(t.shape[1]):
        X[n:] += t[:, n] * fr[:F - n]
    chan = np.fft.fft(X, axis=1).T
    return chan, discriminator(chan, kf)


def to_pcm(audio):
    return np.trunc(np.clip(np.asarray(audio, np.float64) * 32767.0, -32768.0, 32767.0)).astype(np.int16)


def audio(demod_row, hp, lp, gain, b0, b1, a1):
    """One discriminator row (or [rows][n]) from stream start -> (lpcomp, audio, pcm).  lp = None: no low-pass."""
    x = np.asarray(demod_row, np.float64)
    hp = np.asarray(hp, np.float64)
    hpo = signal.lfilter(hp, [1.0], x, axis=-1)
    d = (hp.shape[0] - 1) // 2
    delayed = np.zeros_like(x)
    delayed[..., d:] = x[..., :x.shape[-1] - d]
    lpcomp = delayed - hpo
    y = signal.lfilter([float(b0), float(b1)], [1.0, float(a1)], float(gain) * hpo, axis=-1)
    if lp is not None:
        y = signal.lfilter(np.asarray(lp, np.float64), [1.0], y, axis=-1)
    return lpcomp, y, to_pcm(y)


def asgram_row(res, W, window):
    """One asgramcf_write + asgramcf_execute over one call's samples -> (psd [4W], peak [2], ascii [W] bytes, transforms)."""
    x = np.asarray(res, np.complex128)
    w = np.asarray(window, np.float64)
    nfft, hop = 4 * W, W // 2
    nt = x.shape[0] // hop
    if nt == 0:
        return None, np.zeros(2), np.full(W, ord(" "), np.uint8), 0
    xp = np.concatenate([np.zeros(W, np.complex128), x])
    ends = W + hop * np.arange(1, nt + 1)                  # a transform after every hop-th sample of the call
    frames = xp[ends[:, None] - W + np.arange(W)[None, :]] * w
    acc = np.sum(np.abs(np.fft.fft(frames, n=nfft, axis=1)) ** 2, axis=0)
    acc = np.fft.fftshift(acc)
    psd = 10.0 * np.log10(np.where(acc > 1e-12, acc, 1e-12) / nt)   # as liquid: a NaN power (W = 2: 0 x inf window) reads 1e-12
    i = int(np.argmax(psd))
    peak = np.array([psd[i], i / nfft - 0.5])
    val = psd.reshape(W, 4).max(axis=1)
    ascii = asgram_chars(val)
    return psd, peak, ascii, nt


def asgram_chars(val):
    """Level characters of the per-column maxima (dB)."""
    lev = np.sum(val[:, None] > ASGRAM_REF + ASGRAM_DIV * np.arange(10)[None, :], axis=1)   # levels are increasing
    chars = np.frombuffer(LEVEL_CHARS, np.uint8)
    return np.where(lev == 0, chars[0], chars[np.maximum(lev - 1, 0)])


# ---- comparisons of a float32 stage output with its float64 reference; each returns the worst measured error ------------
def wrapped(a):
    return (a + np.pi) % (2 * np.pi) - np.pi


def check_chan(chan, ref, tol_ch, tol_stage):
    """Per channel: error RMS <= tol_ch of that channel's RMS + tol_stage of the whole stage's RMS."""
    ref = np.asarray(ref, np.complex128)
    stage = np.sqrt(np.mean(np.abs(ref) ** 2))
    worst = 0.0
    for c in range(ref.shape[0]):
        e = np.sqrt(np.mean(np.abs(chan[c] - ref[c]) ** 2))
        r = np.sqrt(np.mean(np.abs(ref[c]) ** 2))
        assert e <= tol_ch * r + tol_stage * stage, (c, e / r, e / stage)
        worst = max(worst, e / (tol_ch * r + tol_stage * stage))
    return worst


def check_demod(demod, chan_used, chan_ref, kf, tol_rad):
    """demod (float32, units of the discriminator) against the float64 discriminator of the channel samples it was computed
    from, and against the reference's demod on samples where the angle is well conditioned."""
    k = 2 * np.pi * kf
    own = discriminator(chan_used, kf)
    d = np.abs(wrapped((demod.astype(np.float64) - own) * k))
    y = np.abs(np.asarray(chan_used, np.complex128))
    ok = np.ones_like(y, bool)
    ok[:, 0] = False                                        # arg(conj(0) y): sign-of-zero dependent
    ok[:, 1:] &= (y[:, 1:] > 0) & (y[:, :-1] > 0)
    assert np.max(d[ok]) < tol_rad, float(np.max(d[ok]))
    # against the reference's channel samples: error cone of the channel error over the magnitudes
    e = np.abs(np.asarray(chan_used, np.complex128) - chan_ref)
    ya = np.abs(chan_ref)
    cone = np.full_like(ya, np.inf)
    cone[:, 1:] = e[:, 1:] / ya[:, 1:] + e[:, :-1] / ya[:, :-1]
    ref_d = discriminator(chan_ref, kf)
    good = cone < 1e-3
    assert np.mean(good) > 0.5
    dd = np.abs(wrapped((demod.astype(np.float64) - ref_d) * k))
    assert np.all(dd[good] <= 2 * cone[good] + tol_rad), float(np.max(dd[good] - 2 * cone[good]))
    return float(np.max(d[ok]))


def check_pcm(pcm, audio64, max_abs_err):
    """s16 equal to trunc(clip(32767 a)) of the float64 audio, except +-1 where a * 32767 lies within the audio error of an
    integer (truncation can go either way there)."""
    v = np.asarray(audio64, np.float64) * 32767.0
    want = to_pcm(audio64).astype(np.int32)
    d = np.abs(pcm.astype(np.int32) - want)
    assert d.max() <= 1, int(d.max())
    near = np.abs(v - np.round(v)) <= max(0.05, 2.0 * max_abs_err * 32767.0)
    assert np.all(d[~near] == 0), int(np.sum(d[~near] != 0))
    return int(np.sum(d != 0))


def check_asgram(psd, peak, ascii, psd64, peak64, tol_db):
    """psd within tol_db on bins within 60 dB of the row peak; peak value within tol_db, its bin unless the top two bins are
    closer than tol_db; characters equal except where a column maximum lies within tol_db of a level edge."""
    top = np.max(psd64)
    sel = psd64 > top - 60.0
    err = float(np.max(np.abs(psd[sel] - psd64[sel])))
    assert err < tol_db, err
    assert abs(peak[0] - peak64[0]) < tol_db
    second = np.sort(psd64)[-2]
    if top - second > tol_db:
        assert abs(peak[1] - peak64[1]) < 1e-6, (peak, peak64)
    val = psd64.reshape(-1, 4).max(axis=1)
    edges = ASGRAM_REF + ASGRAM_DIV * np.arange(10)
    near = np.min(np.abs(val[:, None] - edges[None, :]), axis=1) < tol_db
    assert np.all((ascii == asgram_chars(val)) | near)
    return err
