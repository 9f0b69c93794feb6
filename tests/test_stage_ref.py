"""The float64 stage references of tests/stage_ref.py against the float32 CPU oracle (no GPU).

Each reference is fed the oracle's own input to that stage and must reproduce the oracle's output of the stage to
float32 rounding.  This pins the conventions the GPU stage sweep (test_gpu_stage_sweep.py) relies on -- commutator
order, tap order, frame alignment, NCO sign, discriminator start, FIR delay, de-emphasis form, s16 conversion,
asgram hop and row rules -- before any GPU result is judged by them.
"""
import numpy as np
import pytest

import stage_ref
from util import design_asgram_window, design_dtheta, design_pfbch, nco_offset, rel_rms


@pytest.mark.parametrize("M", [16, 20])
def test_channelize_matches_oracle(M):
    from oracle import oracle as orc
    from sdr_pmr446_b200 import synth
    fs = 1024000 if M == 16 else M * 12500
    car = (synth.Carrier(2, 0.2, 1000.0, 67.0), synth.Carrier(M - 3, 0.1, 600.0, 88.5), synth.Carrier(M, 0.05, 2400.0, 250.3))
    iq = synth.make_cf32(synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=car), 250000, 446)
    o = orc.PmrOracle(fs_in=fs, in_fmt=0, num_channels=M, chunk=50000)
    r = o.run(iq, 50000, want=("res", "chan", "demod"))
    o.close()
    dtheta = design_dtheta(M)
    nco = orc.lib().nco_crcf_create(0)
    orc.lib().nco_crcf_set_frequency(nco, nco_offset(M))
    assert orc.lib().oracle_nco_crcf_get_dtheta_u32(nco) == dtheta
    orc.lib().nco_crcf_destroy(nco)
    chan, demod = stage_ref.channelize(r["res"], M, design_pfbch(M), dtheta, 0.5)
    assert chan.shape == r["chan"].shape == (M, r["ny"] // M)
    stage_ref.check_chan(r["chan"], chan, 2e-5, 2e-6)
    stage_ref.check_demod(r["demod"], r["chan"], chan, 0.5, 1e-5)


@pytest.mark.parametrize("lowpass", [0, 1])
def test_audio_matches_oracle(lowpass):
    from liquid_api import reference_taps
    from oracle import oracle as orc
    from sdr_pmr446_b200 import synth
    iq = synth.make_cu8(synth.CaptureSpec(fs=1024000.0), 400000, 447)
    o = orc.PmrOracle(fs_in=1024000, in_fmt=1, audio_gain=1.0, lowpass=lowpass, chunk=100000)
    r = o.run(iq, 100000, want=("demod", "lpcomp", "audio", "pcm"))
    o.close()
    hp, lp = reference_taps()
    b0, b1, a1 = (np.float32(v) for v in (0.507301437230636, 0.507301437230636, 0.014602874461272194))
    lpc, au, pcm = stage_ref.audio(r["demod"], hp, lp if lowpass else None, 1.0, b0, b1, a1)
    for c in range(16):
        assert rel_rms(r["audio"][c], au[c]) < 1e-5, (c, rel_rms(r["audio"][c], au[c]))
        # lpcomp is the difference of two nearly equal signals: measured against the discriminator's level
        e = np.sqrt(np.mean((r["lpcomp"][c] - lpc[c]) ** 2)) / np.sqrt(np.mean(r["demod"][c].astype(np.float64) ** 2))
        assert e < 1e-6, (c, e)
    stage_ref.check_pcm(r["pcm"], au, np.max(np.abs(r["audio"] - au)))


@pytest.mark.parametrize("W", [67, 120])
def test_asgram_matches_oracle(W):
    from oracle import oracle as orc
    from sdr_pmr446_b200 import synth
    iq = synth.make_cu8(synth.CaptureSpec(fs=1024000.0), 300000, 448)
    o = orc.PmrOracle(fs_in=1024000, in_fmt=1, waterfall=W, chunk=100000)
    parts = [o.execute(iq[2 * k:2 * (k + n)], want=("res",)) for k, n in ((0, 100000), (100000, 313), (100313, 99687), (200000, 100000))]
    o.close()
    w = design_asgram_window(W)
    for p in parts:
        psd, peak, ascii, nt = stage_ref.asgram_row(p["res"], W, w)
        if nt == 0:
            assert np.all(p["ascii"] == ord(" ")) and np.all(p["peak"] == 0)
            continue
        stage_ref.check_asgram(p["psd"], p["peak"], p["ascii"], psd, peak, 1e-3)


# ---- front end and dsd_in back end --------------------------------------------------------------------------------------
FE_TOL_RMS, FE_TOL_MAX = 2e-5, 6e-5      # ~3x the float32 oracle's own distance from float64 (1.4e-6 .. 6.3e-6 / 1.8e-5)
ALPHA = 0.0005


def _capture(fs, fmt, n, seed, dsd=False):
    from sdr_pmr446_b200 import synth
    if dsd:   # dsd_in: one carrier at 0 Hz
        spec = synth.CaptureSpec(fs=float(fs), carriers=(synth.Carrier(1, 0.3, 1000.0, 0.0),), offset_hz=-synth.channel_offset_hz(1))
    else:
        spec = synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(seed))
    return synth.make_cu8(spec, n, seed) if fmt == stage_ref.FMT_CU8 else synth.make_cf32(spec, n, seed)


def _uneven(n, chunk):
    """Chunk sizes (at most `chunk`) covering n samples: a long call, 1 and 7 samples, one off a multiple of 16, the rest."""
    sizes = [chunk - 5, 1, 7, 4095, 333]
    while sum(sizes) < n:
        sizes.append(min(chunk, n - sum(sizes)))
    sizes[-1] -= sum(sizes) - n
    return [k for k in sizes if k > 0]


def _oracle_calls(o, iq, sizes, bps, **kw):
    parts, p = [], 0
    for k in sizes:
        parts.append(o.execute(iq[p * bps:(p + k) * bps], **kw))
        p += k
    return parts


@pytest.mark.parametrize("fs,fmt,fs_out", [(2400000, 1, 200000), (1024000, 1, 200000), (3200000, 0, 200000), (4800000, 0, 200000),
                                           (20000000, 0, 200000), (500000, 0, 200000), (250000, 0, 200000), (200000, 0, 200000),
                                           (2400000, 1, 12500), (1024000, 0, 12500)])
def test_front_end_matches_oracle(fs, fmt, fs_out):
    """stage_ref.front_end (conversion, DC blocker, half-band cascade, arbitrary resampler) against the oracle's `res`, fed
    in uneven chunks; every sample, not only the RMS."""
    from oracle import oracle as orc
    from util import design_msresamp
    n, chunk = fs // 2, fs // 10
    iq = _capture(fs, fmt, n, 600 + fmt, dsd=fs_out == 12500)
    bps = 2 if fmt == stage_ref.FMT_CU8 else 1
    if fs_out == 12500:   # the dsd_in chain is the oracle's only front end into 12.5 kHz
        o = orc.DsdOracle(fs_in=fs, in_fmt=fmt, chunk=chunk)
        parts = _oracle_calls(o, iq, _uneven(n, chunk), bps)
    else:
        o = orc.PmrOracle(fs_in=fs, in_fmt=fmt, num_channels=fs_out // 12500, chunk=chunk)
        parts = _oracle_calls(o, iq, _uneven(n, chunk), bps, want=("res",))
    o.close()
    res = np.concatenate([p["res"] for p in parts])
    ref = stage_ref.front_end(iq, fmt, design_msresamp(np.float32(fs_out) / np.float32(fs)), ALPHA)
    stage_ref.check_res(res, ref, FE_TOL_RMS, FE_TOL_MAX)


@pytest.mark.parametrize("fmt", [0, 1])
def test_dc_block_matches_oracle(fmt):
    from oracle import oracle as orc
    n, chunk = 300000, 100000
    iq = _capture(1024000, fmt, n, 610 + fmt)
    bps = 2 if fmt == stage_ref.FMT_CU8 else 1
    o = orc.PmrOracle(fs_in=1024000, in_fmt=fmt, chunk=chunk)
    parts = _oracle_calls(o, iq, _uneven(n, chunk), bps, want=("dcblocked",))
    o.close()
    ref = stage_ref.dc_block(stage_ref.convert(iq, fmt), ALPHA)
    stage_ref.check_res(np.concatenate([p["dcblocked"] for p in parts]), ref, FE_TOL_RMS, FE_TOL_MAX)


def test_convert_integer_formats():
    """cs16 x 2^-15 and cs8 x 2^-7 at the extremes; cu8 (u8 - 127.4f) / 128 rounded as float32 arithmetic rounds it."""
    v16 = np.array([-32768, 32767, 0, 1, -1, 12345], np.int16)
    assert np.array_equal(stage_ref.convert(v16, stage_ref.FMT_CS16), (v16[0::2] + 1j * v16[1::2]) / 32768.0)
    v8 = np.array([-128, 127, 0, -1], np.int8)
    assert np.array_equal(stage_ref.convert(v8, stage_ref.FMT_CS8), (v8[0::2] + 1j * v8[1::2]) / 128.0)
    u8 = np.arange(256, dtype=np.uint8)
    x = stage_ref.convert(u8, stage_ref.FMT_CU8)
    want = ((u8.astype(np.float32) - np.float32(127.4)) * np.float32(1 / 128)).astype(np.float64)
    assert np.array_equal(x.real, want[0::2]) and np.array_equal(x.imag, want[1::2])


@pytest.mark.parametrize("fs,fmt", [(2400000, 1), (1024000, 0)])
def test_msresamp_interp_matches_oracle(fs, fmt):
    """stage_ref.msresamp_interp_real (msresamp_rrrf x 3.84) against the dsd_in oracle's audio given its own discriminator
    output, and its s16 cast (dsd_in truncates and does not saturate: only samples inside +-1 are compared)."""
    from oracle import oracle as orc
    from util import design_msresamp
    n, chunk = 600000, 200000
    iq = _capture(fs, fmt, n, 620 + fmt, dsd=True)
    o = orc.DsdOracle(fs_in=fs, in_fmt=fmt, chunk=chunk)
    parts = _oracle_calls(o, iq, _uneven(n, chunk), 2 if fmt == stage_ref.FMT_CU8 else 1)
    o.close()
    fm, audio, pcm = (np.concatenate([p[k] for p in parts]) for k in ("fm", "audio", "pcm"))
    au = stage_ref.msresamp_interp_real(fm, design_msresamp(np.float32(48000) / np.float32(12500)))
    stage_ref.check_res(audio, au, 1e-6, 1e-5)
    inside = np.abs(au) < 0.999
    assert np.mean(inside) > 0.95
    stage_ref.check_pcm(pcm[inside], au[inside], float(np.max(np.abs(audio - au))))


# ---- receiver: squelch / selector, tone bank, RSSI, selected stream ------------------------------------------------------
RX_CASES = {"keyed_two_calls": ({}, "keyed_two_calls"), "stronger_later_lock_max": ({"lock_mode": 1}, "stronger_later"),
            "ctcss_change": ({}, "ctcss_change")}


def _rx_oracle_rows(case, block=2441, alpha=0.0005):
    import rx_scenarios as sc
    from oracle import oracle as orc
    kw, scen = RX_CASES[case]
    car = getattr(sc, scen)()
    iq = sc.capture(car)
    o = orc.RxOracle(fs_in=sc.FS, in_fmt=1, chunk=sc.CHUNK, audio_gain=1.0, ctcss_block=block, ctcss_dc_alpha=alpha, **kw)
    rows, p = [], 0
    for k in sc.rx_sizes(iq.shape[0] // 2, sc.CHUNK):
        rows.append(o.execute(iq[2 * p:2 * (p + k)]))
        p += k
    o.close()
    return rows, kw


@pytest.mark.parametrize("block", [2441, 1, 5000])
@pytest.mark.parametrize("case", sorted(RX_CASES))
def test_squelch_and_tone_bank_replay_oracle(case, block):
    """stage_ref.squelch_step and stage_ref.ctcss_bank replayed from the oracle's own rssi_ch and ctcss_in reproduce its
    state, active channel, spread, events, tone flag, code, maximum and every Goertzel power bitwise in every call."""
    rows, kw = _rx_oracle_rows(case, block)
    seen = stage_ref.check_replay(rows, stage_ref.rx_cfg(**kw), block)
    assert seen & 1 and (seen & 8 or block == 1)
    if case == "keyed_two_calls":
        assert seen & 4
    if case == "stronger_later_lock_max":
        assert seen & 2
    if case == "ctcss_change" and block == 2441:
        assert seen & 16 and seen & 32


# ~3x the float32 oracle's own distance from float64, measured on these three runs: rssi 1.5e-5 dB (a float32 running
# sum of ~1 221 magnitudes), audio 3.0e-7 relative RMS / 2.9e-6 of the RMS per sample, ctcss_in 3.8e-6 of the
# discriminator RMS per sample
RX_RSSI_TOL_DB = 5e-5
RX_AUDIO_TOL_RMS, RX_AUDIO_TOL_MAX = 1e-6, 1e-5
RX_CTCSS_TOL = 1.2e-5


@pytest.mark.parametrize("case", sorted(RX_CASES))
def test_receiver_stages_match_oracle(case):
    """stage_ref.rssi of the oracle's channel samples against its rssi_ch; selected_stream -> stage_ref.audio ->
    dc_block_real against its audio, s16 and ctcss_in, per sample over everything it played (every call, key-up,
    detune, retune and channel changes included)."""
    from liquid_api import reference_taps
    rows, kw = _rx_oracle_rows(case)
    d_rssi = 0.0
    for r in rows:
        want = stage_ref.rssi(r["chan"])
        if r["ns"] == 0:
            assert np.all(np.isnan(r["rssi_ch"])) and np.all(np.isnan(want))
            continue
        d_rssi = max(d_rssi, float(np.max(np.abs(r["rssi_ch"] - want))))
    x, _ = stage_ref.selected_stream([r["chan"] for r in rows], [r["active_chan"] for r in rows])
    hp, lp = reference_taps()
    b0, b1, a1 = (np.float32(v) for v in (0.507301437230636, 0.507301437230636, 0.014602874461272194))
    lpc, au, pcm = stage_ref.audio(x, hp, None, 1.0, b0, b1, a1)
    audio = np.concatenate([r["audio"] for r in rows])
    ctin = np.concatenate([r["ctcss_in"] for r in rows])
    assert audio.shape == au.shape
    rms, worst = stage_ref.check_res(audio, au, RX_AUDIO_TOL_RMS, RX_AUDIO_TOL_MAX)
    stage_ref.check_pcm(np.concatenate([r["pcm"] for r in rows]), au, float(np.max(np.abs(audio - au))))
    ct = stage_ref.dc_block_real(lpc, 0.0005)
    e_ct = float(np.max(np.abs(ctin - ct)) / np.sqrt(np.mean(x ** 2)))
    print("MEASURED oracle %s: rssi %.2e dB, audio %.2e rms / %.2e sample, ctcss_in %.2e" % (case, d_rssi, rms, worst, e_ct))
    assert d_rssi < RX_RSSI_TOL_DB and e_ct < RX_CTCSS_TOL
