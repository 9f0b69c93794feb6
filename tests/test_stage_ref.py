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
