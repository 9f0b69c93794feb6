"""GPU stage sweep: every kernel the configuration can select, stage by stage, against the float64 references of
tests/stage_ref.py.

Each case runs 3 streams with distinct seeds (unless it varies the stream count on purpose) and checks every stream and
every channel.  The reference of a stage is fed the GPU's own float32 input to that stage (the `res` or `demod` output
requested alongside, concatenated over the calls), so the bounds only have to cover the rounding of the stage itself and
can be far tighter than the whole-chain parity tests.  Chunk sizes are uneven and include chunks shorter than a kernel
tile.

Bounds (about ten times the largest error measured on a B200, never looser than 1e-4 relative RMS / +-1 LSB):
  chan    per channel, error RMS <= CHAN_TOL_CH of the channel's RMS + CHAN_TOL_STAGE of the stage's RMS
  demod   |wrapped angle error| < DEMOD_TOL_RAD against the float64 discriminator of the GPU's own channel samples, and
          within twice the channel error cone of the reference's samples where that cone is below 1e-3 rad
  audio   AUDIO_TOL relative RMS per row; lpcomp LPCOMP_TOL of the row's discriminator RMS
  pcm     equal to the float64 value's s16, except +-1 where it lies within the audio error of an integer
  psd     PSD_TOL_DB on bins within 60 dB of the row peak; peak and characters as stage_ref.check_asgram
"""
import functools

import numpy as np
import pytest

import stage_ref
from util import design_asgram_window, design_dtheta, design_pfbch, rel_rms

pytestmark = pytest.mark.gpu

S = 3
CHAN_TOL_CH, CHAN_TOL_STAGE = 1e-5, 1e-6
DEMOD_TOL_RAD = 4e-6
AUDIO_TOL = 1e-5
LPCOMP_TOL = 4e-6
PSD_TOL_DB = 1e-3


def _execute(b, iq, sizes, want, bps):
    """Runs the chunks of `sizes` samples through batch `b`; returns the per-call results."""
    assert sum(sizes) * bps == iq.shape[1]
    parts, o = [], 0
    for k in sizes:
        parts.append(b.execute(iq[:, o * bps:(o + k) * bps], want=want))
        o += k
    return parts


def _cat(parts, k):
    return np.concatenate([p[k] for p in parts], axis=-1)


# ---- channelizer ------------------------------------------------------------------------------------------------------
def _chan_case(M, frames=100, pfb_m=13, pfb_as=80.0, kf=0.5, seed0=500):
    from sdr_pmr446_b200 import chain, synth
    fs = M * 12500
    n = M * frames + M // 2 + 3
    car = (synth.Carrier(1, 0.2, 1000.0, 67.0), synth.Carrier(max(1, M // 2), 0.1, 600.0, 88.5), synth.Carrier(M, 0.05, 2400.0, 0.0))
    iq = np.stack([synth.make_cf32(synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=car), n, seed0 + s) for s in range(S)])
    # uneven calls, one shorter than a channelizer tile (8 frames of the generic kernels)
    sizes = [n // 3 + 7, 3 * M + 5, 1, n - (n // 3 + 7) - (3 * M + 5) - 1]
    b = chain.PmrBatch(n_streams=S, fs_in=fs, in_fmt=0, num_channels=M, pfb_m=pfb_m, pfb_as=pfb_as, kf=kf, max_chunk=max(sizes))
    parts = _execute(b, iq, sizes, ("res", "chan", "demod"), 1)
    b.close()
    res, chan, demod = _cat(parts, "res"), _cat(parts, "chan"), _cat(parts, "demod")
    taps, dtheta = design_pfbch(M, pfb_m, pfb_as), design_dtheta(M)
    worst_c = worst_d = 0.0
    for s in range(S):
        rc, _ = stage_ref.channelize(res[s], M, taps, dtheta, kf)
        assert rc.shape == chan[s].shape, (rc.shape, chan[s].shape)
        worst_c = max(worst_c, stage_ref.check_chan(chan[s], rc, CHAN_TOL_CH, CHAN_TOL_STAGE))
        worst_d = max(worst_d, stage_ref.check_demod(demod[s], chan[s], rc, kf, DEMOD_TOL_RAD))
    print("MEASURED chan M=%d pfb_m=%d as=%g kf=%g: chan %.3g of bound, demod %.3g rad" % (M, pfb_m, pfb_as, kf, worst_c, worst_d))


@pytest.mark.parametrize("M", [2, 3, 4, 7, 8, 12, 17, 32, 97, 210, 509, 1024, 1828])
def test_channelizer_generic_tile(M):
    """channelize_generic_tile_kernel<26> (pfb_m = 13): radices 2, 3, 4, 5, 7, large primes (97, 509), up to its
    shared-memory limit."""
    _chan_case(M)


@pytest.mark.parametrize("pfb_m", [1, 4, 32])
def test_channelizer_generic_pfb_m(pfb_m):
    """channelize_generic_kernel: 16 channels with a prototype other than 2 x 13 taps per branch."""
    _chan_case(16, pfb_m=pfb_m)


@pytest.mark.parametrize("M", [1829, 2048, 2075, 2076, 3657, 3658, 4096])
def test_channelizer_generic_large(M):
    """Channel counts around the two shared-memory limits (tile kernel: 112 M bytes, generic kernel: 56 M bytes) up to the
    4096 channels pmr446_b200.h promises."""
    _chan_case(M, frames=64)


@pytest.mark.parametrize("pfb_as", [60.0, 100.0])
def test_channelizer16_stopband(pfb_as):
    """channelize16_kernel (16 x 26 taps in registers) with the prototype designed for another stop-band attenuation."""
    _chan_case(16, frames=400, pfb_as=pfb_as)


@pytest.mark.parametrize("M", [16, 12])
def test_channelizer_kf(M):
    """The discriminator scale 1 / (2 pi kf) with kf != 0.5, in the 16-channel and the generic kernel."""
    _chan_case(M, frames=300, kf=0.3)


# ---- audio ------------------------------------------------------------------------------------------------------------
AUDIO_FS, AUDIO_N = 2400000, 960000
AUDIO_SIZES = [240000, 1000, 333333, 385667]   # 1000 inputs = 5 audio samples: shorter than any audio tile


@functools.lru_cache(maxsize=None)
def _audio_capture():
    from sdr_pmr446_b200 import synth
    return np.stack([synth.make_cu8(synth.CaptureSpec(fs=float(AUDIO_FS), carriers=synth.rotated_carriers(s)), AUDIO_N, 520 + s)
                     for s in range(S)])


def _taps(n, seed):
    """A seeded odd-length FIR: the stage reference does not care what the filter is, only that it is applied right."""
    rng = np.random.Generator(np.random.PCG64(seed))
    return (rng.standard_normal(n) / np.sqrt(n)).astype(np.float32)


def _audio_case(iq=None, fs=AUDIO_FS, sizes=AUDIO_SIZES, num_channels=16, in_fmt=1, hp=None, lp=None, lowpass=0, gain=1.0, deemph=None):
    from liquid_api import reference_taps
    from sdr_pmr446_b200 import chain
    iq = _audio_capture() if iq is None else iq
    kw = dict(n_streams=iq.shape[0], fs_in=fs, in_fmt=in_fmt, num_channels=num_channels, lowpass=lowpass, audio_gain=gain,
              max_chunk=max(sizes))
    keep = []
    if hp is not None:
        keep.append(hp)
        kw.update(hp_taps=hp.ctypes.data, hp_len=hp.size)
    if lp is not None:
        keep.append(lp)
        kw.update(lp_taps=lp.ctypes.data, lp_len=lp.size)
    if deemph is not None:
        kw.update(deemph_b0=deemph[0], deemph_b1=deemph[1], deemph_a1=deemph[2])
    b = chain.PmrBatch(**kw)
    cfg = b.cfg
    parts = _execute(b, iq, sizes, ("demod", "lpcomp", "audio", "pcm"), 2 if in_fmt == 1 else 1)
    b.close()
    demod, lpcomp, audio, pcm = (_cat(parts, k) for k in ("demod", "lpcomp", "audio", "pcm"))
    ref_hp, ref_lp = reference_taps()
    hp = ref_hp if hp is None else hp
    lp = ref_lp if lp is None else lp
    f32 = lambda v: np.float32(v)  # noqa: E731  the coefficients as the library holds them
    rows = demod.shape[0] * demod.shape[1]
    lpc64, au64, _ = stage_ref.audio(demod.reshape(rows, -1), hp, lp if lowpass else None, f32(cfg.audio_gain), f32(cfg.deemph_b0),
                                     f32(cfg.deemph_b1), f32(cfg.deemph_a1))
    au32, lpc32, dm = audio.reshape(rows, -1), lpcomp.reshape(rows, -1), demod.reshape(rows, -1).astype(np.float64)
    worst_a = worst_l = 0.0
    for r in range(rows):
        e = rel_rms(au32[r], au64[r])
        worst_a = max(worst_a, e)
        assert e < AUDIO_TOL, ("audio", r, e)
        el = np.sqrt(np.mean((lpc32[r] - lpc64[r]) ** 2)) / np.sqrt(np.mean(dm[r] ** 2))
        worst_l = max(worst_l, el)
        assert el < LPCOMP_TOL, ("lpcomp", r, el)
    flips = stage_ref.check_pcm(pcm.reshape(rows, -1), au64, float(np.max(np.abs(au32 - au64))))
    print("MEASURED audio rows=%d hp=%d lp=%d lowpass=%d a1=%g: audio %.3g rel rms, lpcomp %.3g, pcm +-1 at %d samples"
          % (rows, hp.size, lp.size, lowpass, cfg.deemph_a1, worst_a, worst_l, flips))


def test_audio_default():
    """The reference's configuration (audio gain 4, FFT audio kernel)."""
    _audio_case(gain=4.0)


@pytest.mark.parametrize("hp_len,lp_len,lowpass", [(1, 1, 1), (3, 103, 0), (383, 1, 1), (377, 112, 1), (383, 112, 1)])
def test_audio_custom_filters(hp_len, lp_len, lowpass):
    """Custom CTCSS-removal and low-pass FIRs: composite responses of 25 .. 518 taps (both FFT tile overlaps, AF_HALO and
    AF_HALO_LONG), a one-tap high-pass (no delay) and a one-tap low-pass."""
    _audio_case(hp=_taps(hp_len, hp_len), lp=_taps(lp_len, 1000 + lp_len), lowpass=lowpass)


@pytest.mark.parametrize("a1", [-0.3, -0.9, 0.5])
@pytest.mark.parametrize("lowpass", [0, 1])
def test_audio_deemphasis_pole(a1, lowpass):
    """A one-pole de-emphasis y = b0 x + b1 x[-1] - a1 y[-1] with unit DC gain, pole far from the reference's 0.0146
    (a1 = -0.9 is a conventional 750 us NBFM de-emphasis at 12.5 kHz)."""
    b = (1.0 + a1) / 2.0
    _audio_case(deemph=(b, b, a1), lowpass=lowpass)


def test_audio_odd_row_count():
    """7 channels x 3 streams = 21 rows: the four-row FFT audio blocks end with a partial block (generic channelizer at
    resampler rate 1.0)."""
    from sdr_pmr446_b200 import synth
    M, n = 7, 87500 * 2
    iq = np.stack([synth.make_cf32(synth.CaptureSpec(fs=M * 12500.0, num_channels=M, carriers=synth.rotated_carriers(s, M, (
        synth.Carrier(1, 0.2, 1000.0, 67.0), synth.Carrier(5, 0.1, 600.0, 88.5)))), n, 530 + s) for s in range(S)])
    _audio_case(iq=iq, fs=M * 12500, sizes=[60000, 99, 40001, n - 100100], num_channels=M, in_fmt=0)
    _audio_case(iq=iq, fs=M * 12500, sizes=[60000, 99, 40001, n - 100100], num_channels=M, in_fmt=0, deemph=(0.05, 0.05, -0.9))


def test_receiver_deemphasis_pole():
    """The receiver's direct-form audio chain with a1 = -0.9: a carrier keyed from t = 0 opens the squelch in the first chunk,
    so the played audio is the whole audio chain applied to the batch discriminator output of that channel."""
    from liquid_api import reference_taps
    from sdr_pmr446_b200 import chain, synth
    import rx_scenarios as sc
    a1 = -0.9
    de = dict(deemph_b0=(1 + a1) / 2, deemph_b1=(1 + a1) / 2, deemph_a1=a1)
    chans = (5, 9, 14)
    iq = np.stack([sc.capture((synth.Carrier(c, 0.2, 1000.0, 67.0),), 540 + s, seconds=0.8) for s, c in enumerate(chans)])
    rx = chain.PmrReceiver(n_streams=S, fs_in=sc.FS, in_fmt=1, max_chunk=sc.CHUNK, audio_gain=1.0, **de)
    rows = rx.run(iq, sc.CHUNK)
    rx.close()
    b = chain.PmrBatch(n_streams=S, fs_in=sc.FS, in_fmt=1, max_chunk=sc.CHUNK, audio_gain=1.0, **de)
    g = b.run(iq, sc.CHUNK, want=("demod",))
    b.close()
    hp, _ = reference_taps()
    worst = 0.0
    for s, c in enumerate(chans):
        assert all(int(r["active_chan"][s]) == c - 1 for r in rows)
        assert [int(r["n_audio"][s]) for r in rows] == [r["ns"] for r in rows]
        played = np.concatenate([r["audio"][s] for r in rows])
        pcm = np.concatenate([r["pcm"][s] for r in rows])
        _, au64, _ = stage_ref.audio(g["demod"][s, c - 1], hp, None, np.float32(1.0), np.float32(de["deemph_b0"]),
                                     np.float32(de["deemph_b1"]), np.float32(a1))
        e = rel_rms(played, au64)
        worst = max(worst, e)
        assert e < 1e-4, ("receiver audio", s, e)
        assert np.abs(pcm.astype(np.int32) - stage_ref.to_pcm(au64).astype(np.int32)).max() <= 1
    print("MEASURED receiver a1=-0.9: audio %.3g rel rms" % worst)


# ---- waterfall --------------------------------------------------------------------------------------------------------
def _waterfall_case(W, streams=S):
    from sdr_pmr446_b200 import chain, synth
    fs, n = 200000, 60000
    iq = np.stack([synth.make_cf32(synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(s)), n, 560 + s) for s in range(streams)])
    sizes = [20000, 700, 9000, 3, max(W // 2 - 1, 1), 15000]
    sizes.append(n - sum(sizes))
    b = chain.PmrBatch(n_streams=streams, fs_in=fs, in_fmt=0, waterfall=W, max_chunk=max(sizes))
    parts = _execute(b, iq, sizes, ("res", "ascii"), 1)
    b.close()
    w = design_asgram_window(W)
    worst, rows = 0.0, 0
    for p in parts:
        for s in range(streams):
            psd, peak, ascii, nt = stage_ref.asgram_row(p["res"][s], W, w)
            if nt == 0:
                assert np.all(p["ascii"][s] == ord(" ")) and np.all(p["peak"][s] == 0)
                continue
            worst = max(worst, stage_ref.check_asgram(p["psd"][s], p["peak"][s], p["ascii"][s], psd, peak, PSD_TOL_DB))
            rows += 1
    assert rows >= 4 * streams
    print("MEASURED waterfall W=%d S=%d: psd %.3g dB over %d rows" % (W, streams, worst, rows))


@pytest.mark.parametrize("W", [64, 80, 96, 120, 128, 160])
def test_waterfall_fast(W):
    """wf_accumulate_fast_kernel<P>, W = 8 P for every P it is instantiated for."""
    _waterfall_case(W)


@pytest.mark.parametrize("W", [2, 3, 17, 63, 65, 67, 127, 129, 251, 256])
def test_waterfall_warp(W):
    """wf_accumulate_warp_kernel<8 / 16 / 32> (nfft <= 256 / 512 / 1024), odd widths (hop = floor(W / 2))."""
    _waterfall_case(W)


@pytest.mark.parametrize("W", [257, 512, 1021, 1025, 1600, 2047, 2048])
def test_waterfall_block(W):
    """wf_accumulate_kernel with 256 (nfft <= 4096) and 512 threads per transform, up to nfft = 8192."""
    _waterfall_case(W)


@pytest.mark.parametrize("W", [120, 512, 1600])
@pytest.mark.parametrize("streams", [1, 5])
def test_waterfall_stream_count(W, streams):
    """The stream count sets how many blocks share a stream's transforms (`parts`)."""
    _waterfall_case(W, streams)
