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
  convert     raw IQ -> the float32 value the chain works on: cu8 (u8 - 127.4f) * (1 / 128) in float32 (the subtraction
              is exact), cs16 x 2^-15, cs8 x 2^-7, cf32 as is.
  dc_block    iirfilt_crcf_create_dc_blocker(alpha): y[n] = v[n] - v[n-1], v[n] = x[n] + c v[n-1] from zero state, with
              the effective feedback c = fl32(1 - alpha) (liquid stores a1 = -1 + alpha in float32; DESIGN 4).
  msresamp    msresamp_crcf / msresamp_rrrf with the plan of pmr446_design_msresamp (stages, m, step, npfb, hb[16][20]
              newest-first, pfb[npfb][14] newest-first), all state zero at stream start.
              decimation: half-band stages from the highest index down, each output o = sum_j hb[g][j] x[2 (o - j)] +
              x[2 (o - m) + 1] (resamp2_decim: even samples into the filter branch, odd ones into the delay branch),
              then the scale 2^-stages, then the arbitrary resampler.
              arbitrary resampler: output j = sum_k pfb[row_j][k] u[pos_j - k], pos_j = (j step) >> 24, row_j = ((j step)
              mod 2^24) >> (24 - log2 npfb), in exact integers; after n inputs there are ceil(n 2^24 / step) outputs.
              interpolation (rate > 1): the arbitrary resampler first, then the half-band stages from index 0 up, each
              input n giving y[2 n] = x[n - m] (delay branch) and y[2 n + 1] = sum_j hb[g][j] x[n - j] (filter branch;
              resamp2_interp, msresamp2_interp), no scale.
  receiver    (oracle/receiver.c) rssi = 20 log10(mean |y|) per channel and call; the squelch / selector step and the
              38-tone Goertzel bank restated bit-exactly in float32 (NumPy rounds every operation and never fuses, the
              oracle builds with -ffp-contract=off and the kernels use explicitly rounded operations); the selected
              stream = the active channel's frames of every tuned call, sample 0 of a call discriminated against the last
              frame of the previous tuned call's then-active channel (0 at start and after a detune); the CTCSS branch's
              iirfilt_rrrf DC blocker v0 = x - a1 v1, y = v0 - v1 with a1 = fl32(-1 + alpha).
"""
import numpy as np
from scipy import signal

LEVEL_CHARS = b" .,-+*&NM#"
ASGRAM_REF, ASGRAM_DIV = -40.0, 2.0
FMT_CF32, FMT_CU8, FMT_CS16, FMT_CS8 = 0, 1, 2, 3


def convert(iq, fmt):
    """Raw capture (interleaved I, Q for the integer formats, complex64 for cf32) -> complex128 of the float32 values."""
    if fmt == FMT_CF32:
        return np.asarray(iq, np.complex64).astype(np.complex128)
    iq = np.asarray(iq)
    if fmt == FMT_CU8:
        v = (iq.astype(np.float32) - np.float32(127.4)) * np.float32(1.0 / 128.0)
    elif fmt == FMT_CS16:
        v = iq.astype(np.float64) * 2.0 ** -15
    elif fmt == FMT_CS8:
        v = iq.astype(np.float64) * 2.0 ** -7
    else:
        raise ValueError("unknown input format %r" % (fmt,))
    v = v.astype(np.float64)
    return v[0::2] + 1j * v[1::2]


def dc_block(x, alpha):
    c = float(np.float32(1.0) - np.float32(alpha))
    return signal.lfilter([1.0, -1.0], [1.0, -c], np.asarray(x, np.complex128))


def _arb(x, plan):
    """The arbitrary resampler over x from stream start (zero history)."""
    step, pfb = int(plan["step"]), np.asarray(plan["pfb"], np.float64)
    bits = int(plan["npfb"]).bit_length() - 1
    taps = pfb.shape[1]
    n = x.shape[0]
    J = (n * (1 << 24) + step - 1) // step
    ph = np.arange(J, dtype=np.uint64) * np.uint64(step)
    pos = (ph >> np.uint64(24)).astype(np.int64)
    row = ((ph & np.uint64((1 << 24) - 1)) >> np.uint64(24 - bits)).astype(np.int64)
    xp = np.concatenate([np.zeros(taps - 1, x.dtype), x])
    out = np.zeros(J, x.dtype)
    for k in range(taps):
        out += pfb[row, k] * xp[pos - k + taps - 1]
    return out


def msresamp_decim(x, plan):
    """msresamp_crcf (rate <= 1) over x from stream start."""
    x = np.asarray(x, np.complex128)
    stages = int(plan["stages"])
    for g in range(stages - 1, -1, -1):
        m = int(plan["m"][g])
        h = np.asarray(plan["hb"][g][:2 * m], np.float64)
        n = x.shape[0] // 2
        ev, od = x[0:2 * n:2], x[1:2 * n:2]
        y = signal.lfilter(h, [1.0], ev)
        y[m:] += od[:max(n - m, 0)]
        x = y
    return _arb(x * 2.0 ** -stages, plan)


def msresamp_interp_real(x, plan):
    """msresamp_rrrf (rate > 1) over x from stream start."""
    y = _arb(np.asarray(x, np.float64), plan)
    for g in range(int(plan["stages"])):
        m = int(plan["m"][g])
        h = np.asarray(plan["hb"][g][:2 * m], np.float64)
        out = np.zeros(2 * y.shape[0])
        out[2 * m::2] = y[:max(y.shape[0] - m, 0)]
        out[1::2] = signal.lfilter(h, [1.0], y)
        y = out
    return y


def front_end(iq, fmt, plan, alpha, with_dc=True):
    """Raw capture -> the front end's output `res` (conversion, DC blocker, msresamp_crcf)."""
    x = convert(iq, fmt)
    return msresamp_decim(dc_block(x, alpha) if with_dc else x, plan)


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


def check_res(out, ref, tol_rms, tol_max):
    """A resampler output (complex or real) against its float64 reference: error RMS <= tol_rms of the reference RMS over
    the whole output, and EVERY sample's |error| <= tol_max of that RMS (an RMS over N samples lets k sparse errors of
    tol_rms sqrt(N / k) through: segment starts, tile and chunk edges are where such errors come from).  Returns both
    measured ratios (error RMS, worst sample) over the reference RMS."""
    out, ref = np.asarray(out), np.asarray(ref)
    assert out.shape == ref.shape, (out.shape, ref.shape)
    stage = np.sqrt(np.mean(np.abs(ref) ** 2))
    e = np.abs(out.astype(np.complex128 if np.iscomplexobj(out) else np.float64) - ref)
    rms, worst = float(np.sqrt(np.mean(e ** 2)) / stage), float(np.max(e, initial=0.0) / stage)
    assert rms <= tol_rms, ("rms", rms)
    assert worst <= tol_max, ("sample", int(np.argmax(e)), worst)
    return rms, worst


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


# ---- receiver (oracle/receiver.c, pmr446_receiver_*) ---------------------------------------------------------------------
CTCSS_FREQS = np.array([67.0, 71.9, 74.4, 77.0, 79.7, 82.5, 85.4, 88.5, 91.5, 94.8, 97.4, 100.0, 103.5, 107.2, 110.9, 114.8,
                        118.8, 123.0, 127.3, 131.8, 136.5, 141.3, 146.2, 151.4, 156.7, 162.2, 167.9, 173.8, 179.9, 186.2,
                        192.8, 203.5, 210.7, 218.1, 225.7, 233.6, 241.8, 250.3], np.float32)   # include/pmr446_taps.h
EV_TUNED, EV_CHANGED, EV_DETUNED, EV_CTCSS_ACQUIRED, EV_CTCSS_CHANGED, EV_CTCSS_LOST = 1, 2, 4, 8, 16, 32
_F = np.float32


def rssi(chan):
    """20 log10(mean |y|) of every channel of one call (float64); a call with no frame gives NaN (0 / 0)."""
    y = np.asarray(chan, np.complex128)
    if y.shape[-1] == 0:
        return np.full(y.shape[:-1], np.nan)
    return 20.0 * np.log10(np.mean(np.abs(y), axis=-1))


def ctcss_coef(channel_width=12500):
    """2 cos(2 pi f / fs_audio) per tone in float32, as pmr446_receiver_create and the oracle form it: the argument is
    rounded to float32 and cosf of it (correctly rounded here) doubled."""
    arg = ((2.0 * np.pi * CTCSS_FREQS.astype(np.float64)) / float(channel_width)).astype(np.float32)
    return (_F(2.0) * np.cos(arg.astype(np.float64)).astype(np.float32)).astype(np.float32)


def tone_bank_state():
    """ctcss_detector_reset: the tone bank's state (u0, u1 and the last block's powers, all float32)."""
    z = np.zeros(len(CTCSS_FREQS), np.float32)
    return {"u0": z.copy(), "u1": z.copy(), "power": z.copy(), "max_power": _F(0.0), "index": 0, "samp": 0, "tone": 0}


def rx_state():
    """A receiver's state at creation and after reset (proc_scanning, no channel, ctcss_freq -1)."""
    return {"state": 0, "active": -1, "rssi": _F(0.0), "ctcss_freq": _F(-1.0), "bank": tone_bank_state()}


def squelch_step(state, rssi_ch_f32, cfg):
    """One call of the squelch / selector state machine on the float32 RSSI of every channel; updates `state` (rx_state())
    in place and returns the events (1 tuned, 2 channel changed, 4 detuned).  cfg: squelch (float32), mask, lock_mode.

    Bit-exact to squelch_kernel and oracle/receiver.c: the sum over the enabled channels in channel order and
    top - sum / enabled in float32, the first enabled channel wins ties and -- with every RSSI NaN (a call with no
    frame) -- counts as the strongest; a NaN spread neither tunes nor detunes; the detune test in double.  A detune
    clears the discriminator's previous sample (the caller's business: the selected stream restarts from 0) and the tone
    bank, not the CTCSS DC blocker."""
    r = np.asarray(rssi_ch_f32, np.float32)
    best, enabled, top, total = -1, 0, _F(0.0), _F(0.0)
    for i in range(r.shape[0]):
        if not (int(cfg["mask"]) >> i) & 1:
            continue
        enabled += 1
        total = _F(total + r[i])
        if best < 0 or r[i] > top:
            top, best = r[i], i
    spread = _F(top - _F(total / _F(enabled)))
    ev = 0
    state["rssi"] = spread
    sq = _F(cfg["squelch"])
    if state["state"] == 0:
        if spread > sq:
            state["active"], state["state"] = best, 1
            ev |= EV_TUNED
    else:
        if cfg["lock_mode"] == 1 and state["active"] != best:
            state["active"] = best
            ev |= EV_CHANGED
        if float(spread) < float(sq) - 5.0:
            state["active"], state["state"], state["ctcss_freq"] = -1, 0, _F(0.0)
            state["bank"] = tone_bank_state()
            ev |= EV_DETUNED
    return ev


def ctcss_bank(x_f32, coef, block, bank):
    """ctcss_detector_analyze over one call's DC-blocked CTCSS branch (float32), bit-exact to ctcss_kernel: the 38
    Goertzel recurrences u0 <- (x + coef u0) - u1, and at the end of every `block` samples the powers
    (u0 u0 + u1 u1) - (coef u0) u1, their float32 sum in tone order over 38, the first strict maximum above 0 (the index is
    kept when none is) and tone = avg > 120 and max / avg > 10.  Updates `bank` (tone_bank_state()) in place and
    returns the CTCSS events of the call (8 acquired, 16 code changed, 32 lost)."""
    x = np.asarray(x_f32, np.float32)
    coef = np.asarray(coef, np.float32)
    had_tone, had_code = bank["tone"], bank["index"]
    u0, u1, samp = bank["u0"].copy(), bank["u1"].copy(), bank["samp"]
    i, n = 0, x.shape[0]
    while i < n:
        e = min(n, i + block - samp)
        for k in range(i, e):
            u0, u1 = (x[k] + coef * u0) - u1, u0
        samp += e - i
        i = e
        if samp == block:
            p = ((u0 * u0) + (u1 * u1)) - ((coef * u0) * u1)
            bank["power"] = p
            u0, u1 = np.zeros_like(u0), np.zeros_like(u1)
            avg = _F(np.cumsum(p, dtype=np.float32)[-1] / _F(len(p)))   # cumsum: sequential, in tone order
            j = int(np.argmax(p))
            mx = p[j] if p[j] > 0 else _F(0.0)
            if p[j] > 0:
                bank["index"] = j
            bank["max_power"] = mx
            bank["tone"] = int(bool(avg > _F(120.0)) and bool(_F(mx / avg) > _F(10.0)))
            samp = 0
    bank["u0"], bank["u1"], bank["samp"] = u0, u1, samp
    ev = 0
    if bank["tone"]:
        if not had_tone:
            ev |= EV_CTCSS_ACQUIRED
        elif had_code != bank["index"]:
            ev |= EV_CTCSS_CHANGED
    elif had_tone:
        ev |= EV_CTCSS_LOST
    return ev


def selected_stream(chan_calls, active_per_call, kf=0.5, wrong_first=False):
    """The discriminator output the selected chain sees over a run of calls from a fresh (or reset) receiver, float64.

    chan_calls: per call the channel samples [M][ns] (ns may be 0); active_per_call: the active channel after that call's
    squelch step (-1 = none).  The active channel's samples of every tuned call, sample 0 of a call discriminated
    against the last sample of the previous tuned call's then-active channel -- 0 at start and after a detune (a call
    with no active channel) -- with the component-wise products of `discriminator`, so the sign-of-zero cases match.
    wrong_first: discriminate sample 0 against the NEW channel's own previous frame instead (what an append that ignores
    channel changes and resets would play; a self-check of the tests' bounds).  Returns (stream, call_starts)."""
    parts, starts, pos = [], [], 0
    prev = 0j
    own_prev = {}
    for ch, a in zip(chan_calls, active_per_call):
        ch = np.asarray(ch, np.complex128)
        ns = ch.shape[-1]
        starts.append(pos)
        if a < 0:
            prev = 0j
        elif ns:
            p0 = own_prev.get(a, 0j) if wrong_first else prev
            y = ch[a]
            parts.append(discriminator(np.concatenate([[p0], y])[None, :], kf)[0, 1:])
            pos += ns
            prev = y[-1]
        for c in range(ch.shape[0]):
            if ns:
                own_prev[c] = ch[c, -1]
    return (np.concatenate(parts) if parts else np.zeros(0)), starts


def dc_block_real(x, alpha):
    """iirfilt_rrrf_create_dc_blocker(alpha) in float64: v0 = x - a1 v1, y = v0 - v1, a1 = fl32(-1 + alpha), zero state."""
    a1 = float(_F(_F(-1.0) + _F(alpha)))
    return signal.lfilter([1.0, -1.0], [1.0, a1], np.asarray(x, np.float64))


def rx_cfg(squelch_level=18.0, channel_mask=2 ** 64 - 1, lock_mode=0, **_):
    return {"squelch": np.float32(squelch_level), "mask": int(channel_mask), "lock_mode": int(lock_mode)}


def same_f32(a, b):
    """Bitwise equality of float32 values (every NaN equal to every NaN: their payloads are not part of the contract)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def replay_rx(rows, rssi_ch, ctcss_in, cfg, block=2441, coef=None):
    """squelch_step + ctcss_bank over a run of calls from a fresh receiver, fed `rssi_ch[k]` and `ctcss_in[k]` (the
    implementation's own float32 values).  Yields per call (state dict snapshot, events)."""
    coef = ctcss_coef() if coef is None else coef
    st = rx_state()
    for k in range(len(rows)):
        ev = squelch_step(st, rssi_ch[k], cfg)
        if st["active"] >= 0:
            ev |= ctcss_bank(ctcss_in[k], coef, block, st["bank"])
            st["ctcss_freq"] = CTCSS_FREQS[st["bank"]["index"]]
        yield st, ev


def check_replay(rows, cfg, block):
    """The replay of squelch_step / ctcss_bank from the rows' own rssi_ch and ctcss_in reproduces every status field, the
    events and the Goertzel powers bitwise.  Returns the events seen."""
    seen = 0
    rs = [r["rssi_ch"] for r in rows]
    cs = [r["ctcss_in"][:int(r["n_audio"])] for r in rows]
    for k, (st, ev) in enumerate(replay_rx(rows, rs, cs, cfg, block)):
        r, b = rows[k], st["bank"]
        want = {"state": st["state"], "active_chan": st["active"], "events": ev, "n_audio": r["ns"] if st["active"] >= 0 else 0,
                "ctcss_index": b["index"], "tone_detected": b["tone"]}
        for f, v in want.items():
            assert int(r[f]) == int(v), (k, f, int(r[f]), int(v))
        for f, v in (("rssi", st["rssi"]), ("max_power", b["max_power"]), ("ctcss_freq", st["ctcss_freq"]), ("ctcss_power", b["power"])):
            assert same_f32(r[f], v), (k, f, r[f], v)
        seen |= ev
    return seen
