"""GPU parity of the batched receiver (pmr446_receiver_*, host buffers through the C ABI) against oracle/receiver.c.

Discrete outputs (state, active channel, audio sample counts, CTCSS code, tone flag, events) must match exactly in
every chunk; RSSI within 1e-3 dB; Goertzel powers within 1e-3 of the block maximum; selected-channel audio within
BASELINE.json's 1e-4 relative RMS / +-1 LSB on the chunks where the active channel's carrier is keyed on (on
noise-only spans the discriminator is ill-conditioned, SURVEY.md 7, and only a loose bound is asserted).
"""
import numpy as np
import pytest

import rx_scenarios as sc
from util import PCM_TOL_LSB, REL_RMS_TOL, rel_rms

pytestmark = pytest.mark.gpu

EXACT = ("state", "active_chan", "n_audio", "tone_detected", "ctcss_index", "events")


def _pair(carrier_sets, chunk=sc.CHUNK, fs=sc.FS, **kw):
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain
    iq = np.stack([sc.capture(c, 446 + s, fs=fs, num_channels=kw.get("num_channels", 16)) for s, c in enumerate(carrier_sets)])
    rx = chain.PmrReceiver(n_streams=len(carrier_sets), fs_in=fs, in_fmt=1, max_chunk=chunk, audio_gain=1.0, **kw)
    g = rx.run(iq, chunk)
    rx.close()
    refs = []
    for s in range(len(carrier_sets)):
        o = orc.RxOracle(fs_in=fs, in_fmt=1, chunk=chunk, audio_gain=1.0, **kw)
        refs.append(o.run(iq[s], chunk))
        o.close()
    return g, refs


def _check(g, refs, carrier_sets, chunk=sc.CHUNK, fs=sc.FS):
    for s, (rows, car) in enumerate(zip(refs, carrier_sets)):
        assert len(g) == len(rows)
        for k, (a, r) in enumerate(zip(g, rows)):
            for f in EXACT:
                assert int(a[f][s]) == int(r[f]), (f, s, k, int(a[f][s]), int(r[f]))
            assert a["ns"] == r["ns"]
            assert abs(float(a["rssi"][s]) - r["rssi"]) < 1e-3, ("rssi", s, k)
            assert np.max(np.abs(a["rssi_ch"][s] - r["rssi_ch"])) < 1e-3, ("rssi_ch", s, k)
            assert float(a["ctcss_freq"][s]) == r["ctcss_freq"], ("ctcss_freq", s, k)
            scale = max(float(np.max(r["ctcss_power"])), 1.0)
            assert np.max(np.abs(a["ctcss_power"][s] - r["ctcss_power"])) / scale < 1e-3, ("ctcss_power", s, k)
            assert abs(float(a["max_power"][s]) - r["max_power"]) / scale < 1e-3, ("max_power", s, k)
        good = sc.steady_chunks(rows, car, chunk, fs)
        assert len(good) >= 8, good
        ga = np.concatenate([g[k]["audio"][s, :rows[k]["n_audio"]] for k in good])
        ra = np.concatenate([rows[k]["audio"] for k in good])
        assert rel_rms(ga, ra) < REL_RMS_TOL, ("audio", s, rel_rms(ga, ra))
        gp = np.concatenate([g[k]["pcm"][s, :rows[k]["n_audio"]] for k in good]).astype(np.int32)
        rp = np.concatenate([rows[k]["pcm"] for k in good]).astype(np.int32)
        assert np.abs(gp - rp).max() <= PCM_TOL_LSB
        gc = np.concatenate([g[k]["ctcss_in"][s, :rows[k]["n_audio"]] for k in good])
        rc = np.concatenate([rows[k]["ctcss_in"] for k in good])
        # the CTCSS branch is a small difference of two nearly equal signals: scale by the discriminator level (0.28 rms)
        assert np.sqrt(np.mean((gc - rc) ** 2)) / 0.28 < REL_RMS_TOL, ("ctcss_in", s)
        # everything that was played, including key-up / key-down transients and noise-only tails
        n_all = sum(r["n_audio"] for r in rows)
        ga = np.concatenate([g[k]["audio"][s, :rows[k]["n_audio"]] for k in range(len(rows))])
        ra = np.concatenate([r["audio"] for r in rows])
        assert ga.shape[0] == n_all and rel_rms(ga, ra) < 5e-2


def test_tune_detune_retune_two_streams():
    """Stream 0: two calls on different channels with a pause (tune, detune with freqdem/CTCSS reset, retune).
    Stream 1: a steady carrier joined by a stronger one that lock_mode_start ignores."""
    sets = (sc.keyed_two_calls(), sc.stronger_later())
    g, refs = _pair(sets)
    _check(g, refs, sets)
    assert any(int(r["events"][0]) & 4 for r in g) and int(g[-1]["active_chan"][0]) == 6
    assert all(int(r["active_chan"][1]) == 7 for r in g)


def test_lock_mode_max_follows_the_strongest_channel():
    sets = (sc.stronger_later(),)
    g, refs = _pair(sets, lock_mode=1)
    _check(g, refs, sets)
    assert int(g[0]["active_chan"][0]) == 7 and int(g[-1]["active_chan"][0]) == 14
    assert int(g[-1]["ctcss_index"][0]) == 37 and int(g[-1]["tone_detected"][0]) == 1


def test_channel_mask_and_lowpass():
    sets = (sc.stronger_later(),)
    g, refs = _pair(sets, lock_mode=1, channel_mask=(2 ** 64 - 1) & ~(1 << 14), lowpass=1)
    _check(g, refs, sets)
    assert all(int(r["active_chan"][0]) == 7 for r in g)


def test_uneven_chunks_and_reset():
    """Chunks that are not the reference's size (RSSI windows move with them) and a reset back to scanning."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain
    car = sc.keyed_two_calls()
    iq = sc.capture(car, seconds=1.0)
    rx = chain.PmrReceiver(n_streams=1, fs_in=sc.FS, in_fmt=1, max_chunk=70001, audio_gain=1.0)
    first = rx.run(iq, 70001)
    rx.reset()
    again = rx.run(iq, 70001)
    rx.close()
    o = orc.RxOracle(fs_in=sc.FS, in_fmt=1, chunk=70001, audio_gain=1.0)
    rows = o.run(iq, 70001)
    o.close()
    for a, b, r in zip(first, again, rows):
        for f in EXACT:
            assert int(a[f][0]) == int(b[f][0]) == int(r[f]), f
        assert np.array_equal(a["audio"][0, :r["n_audio"]], b["audio"][0, :r["n_audio"]])
        assert np.array_equal(a["rssi_ch"], b["rssi_ch"])


def test_receiver_on_2400k_captures():
    """The same scenarios from 2.4 Msps captures (tiled front-end kernels, 240 000-sample chunks = 1250 frames)."""
    sets = (sc.keyed_two_calls(), sc.stronger_later())
    g, refs = _pair(sets, chunk=240000, fs=2400000, lock_mode=1)
    _check(g, refs, sets, chunk=240000, fs=2400000)
    assert int(g[-1]["active_chan"][0]) == 6 and int(g[-1]["active_chan"][1]) == 14


def test_eight_channel_receiver():
    """num_channels = 8: the receiver's non-fused path (channel samples of every channel, rssi_kernel, rx_demod_kernel) behind
    the generic channelizer, on a 100 kHz grid of 8 channels."""
    sets = (sc.keyed_two_calls(), sc.stronger_later()[:1])
    g, refs = _pair(sets, num_channels=8)
    _check(g, refs, sets)
    assert int(g[0]["active_chan"][0]) == 1 and int(g[-1]["active_chan"][0]) == 6 and int(g[0]["active_chan"][1]) == 7
