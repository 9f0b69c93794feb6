"""GPU tests of the batch chain's per-channel DSD feed (dsd_audio / dsd_pcm, dsd_backend_kernel over every row): bitwise
equal to the msresamp_rrrf shim fed each concatenated discriminator row, within the float64 bounds of DESIGN 4, on every channelizer
path, and without moving any other output."""
import ctypes as C

import numpy as np
import pytest

import stage_ref
from util import design_msresamp

pytestmark = pytest.mark.gpu

ALL = ("res", "chan", "demod", "lpcomp", "audio", "pcm")


def _capture(fs, n, fmt, seed, streams=1, M=16, carriers=None):
    from sdr_pmr446_b200 import synth
    rows = []
    for s in range(streams):
        kw = {} if carriers is None else {"carriers": carriers}
        spec = synth.CaptureSpec(fs=float(fs), num_channels=M, **kw)
        rows.append(synth.make_cu8(spec, n, seed + s) if fmt == 1 else synth.make_cf32(spec, n, seed + s))
    return np.stack(rows)


def _run(b, iq, calls, want):
    """calls: sample counts or "reset".  Returns one dict per stretch between resets: outputs concatenated along time, and
    the (n, ns, last_dsd) of every call."""
    from sdr_pmr446_b200 import chain
    segs, cur, off = [], {"calls": []}, 0
    for c in calls:
        if c == "reset":
            b.reset()
            segs.append(cur)
            cur = {"calls": []}
            continue
        step = chain._columns(c, iq, b.bytes_per_sample)
        r = b.execute(iq[:, off:off + step], want)
        off += step
        cur["calls"].append((c, r["ns"], b.last_dsd))
        for k, v in r.items():
            if k in ("ny", "ns"):
                continue
            if k in ("ascii", "peak", "psd", "rssi", "chan_edge"):
                cur.setdefault(k, []).append(v)
            else:
                cur[k] = np.concatenate([cur[k], v], axis=-1) if k in cur else v
    segs.append(cur)
    return segs


def _shim():
    import liquid_api
    from sdr_pmr446_b200 import _lib
    return liquid_api.bind(C.CDLL(_lib.LIB_PATH))


def _shim_up(G, x, rate, as_db=60.0):
    q = G.msresamp_rrrf_create(np.float32(rate), as_db)
    assert q
    x = np.ascontiguousarray(x, np.float32)
    y = np.zeros(4 * x.size + 64, np.float32)
    ny = C.c_uint()
    assert G.msresamp_rrrf_execute(q, x.ctypes.data, x.size, y.ctypes.data, C.byref(ny)) == 0
    G.msresamp_rrrf_destroy(q)
    return y[:ny.value]


def _pcm_of(a):
    v = np.asarray(a, np.float32) * np.float32(32767.0)
    return np.trunc(np.clip(v, -32768.0, 32767.0)).astype(np.int16)


def _check_rows(seg, rate, rows=None, f64=True, as_db=60.0):
    """Every (stream, channel) row: dsd_audio bitwise the shim's msresamp_rrrf of the concatenated demod row, dsd_pcm its
    saturated s16, and (f64) within the float64 bounds of DESIGN 4.  Returns the number of saturated samples."""
    G = _shim()
    plan = design_msresamp(np.float32(rate), as_db)
    demod, au, pcm = seg["demod"], seg["dsd_audio"], seg["dsd_pcm"]
    S, M = demod.shape[:2]
    sat = 0
    for s, c in (rows if rows is not None else [(s, c) for s in range(S) for c in range(M)]):
        ref = _shim_up(G, demod[s, c], rate, as_db)
        assert ref.shape == au[s, c].shape, (s, c, ref.shape, au[s, c].shape)
        assert np.array_equal(ref.view(np.int32), au[s, c].view(np.int32)), (s, c, int(np.argmax(ref != au[s, c])))
        assert np.array_equal(pcm[s, c], _pcm_of(ref)), (s, c)
        sat += int(np.sum(np.abs(ref.astype(np.float64)) * 32767.0 > 32767.0))
        if f64:
            stage_ref.check_res(au[s, c], stage_ref.msresamp_interp_real(demod[s, c], plan), 1e-6, 1.5e-5)
    return sat


UNEVEN = [0, 1, 7, 100, "max", 5000, 77777, "reset", 3, "max", 12345]


@pytest.mark.parametrize("fs,fmt,max_chunk", [(2400000, 1, 240000), (1024000, 1, 100000), (1024000, 0, 600000)])
def test_bitwise_against_the_shim_uneven_calls(fs, fmt, max_chunk):
    """Uneven calls (0, 1, 7 samples, one that completes no frame, max_chunk, a reset part-way) on the fused 2.4 Msps cu8
    front end, 1.024 Msps cu8 and cf32 (max_chunk 600000: the host-buffer call runs in time slices)."""
    from sdr_pmr446_b200 import chain
    calls = [max_chunk if c == "max" else c for c in UNEVEN]
    n = sum(c for c in calls if c != "reset")
    iq = _capture(fs, n, fmt, 900 + fmt, streams=2)
    b = chain.PmrBatch(n_streams=2, fs_in=fs, in_fmt=fmt, max_chunk=max_chunk, dsd_rate=48000)
    segs = _run(b, iq, calls, ("demod", "dsd_audio", "dsd_pcm"))
    b.close()
    assert any(c > 0 and ns == 0 for seg in segs for c, ns, _ in seg["calls"])   # a call that completes no frame
    assert all(d == 0 for seg in segs for c, ns, d in seg["calls"] if ns == 0)
    sat = sum(_check_rows(seg, 48000 / 12500) for seg in segs)
    assert sat > 0   # empty channels swing to +-1 and the interpolator overshoots: the saturating cast is exercised


@pytest.mark.parametrize("M,cw,rate,fs,fmt,as_db", [(8, 12500, 48000, 1024000, 1, 60.0), (64, 12500, 48000, 1024000, 0, 60.0),
                                                   (16, 16000, 48000, 1024000, 1, 60.0), (16, 12500, 44100, 2400000, 1, 60.0),
                                                   (16, 12500, 48000, 250000, 1, 40.0)])
def test_shapes_and_rates(M, cw, rate, fs, fmt, as_db):
    """The generic channelizers (M = 8; M = 64, the tiled kernel), channel_width 16000 (x3.0), dsd_rate 44100 (x3.528), and
    resamp_as 40 dB (half-band m = 6: the kernel's run-time m path; fs_in 250 kHz keeps the front end to its arbitrary stage)."""
    from sdr_pmr446_b200 import chain
    if as_db != 60.0:
        assert design_msresamp(np.float32(rate) / np.float32(cw), as_db)["m"][0] < 10
    n = 303000
    iq = _capture(fs, n, fmt, 930 + M, streams=2, M=M)
    b = chain.PmrBatch(n_streams=2, fs_in=fs, in_fmt=fmt, num_channels=M, channel_width=cw, max_chunk=60000, dsd_rate=rate,
                       resamp_as=as_db)
    segs = _run(b, iq, [60000, 1, 59999, 60000, 37000, 60000, 63000 - 37000], ("demod", "dsd_audio", "dsd_pcm"))
    b.close()
    rows = [(s, c) for s in range(2) for c in range(M)] if M <= 16 else [(s, c) for s in range(2) for c in range(0, M, 7)]
    _check_rows(segs[0], np.float32(rate) / np.float32(cw), rows, as_db=as_db)


def test_cfg4_wideband_6400_rows():
    """configs[3]'s shape: 20 Msps cf32, M = 1600 (4 streams: 6400 rows), in two calls."""
    from sdr_pmr446_b200 import chain, synth
    n = 1000000
    carriers = tuple(synth.Carrier(c, 0.1, 1000.0, 0.0) for c in (3, 800, 1599))
    iq = _capture(20000000, n, 0, 950, streams=4, M=1600, carriers=carriers)
    b = chain.PmrBatch(n_streams=4, fs_in=20000000, num_channels=1600, max_chunk=600000, dsd_rate=48000)
    segs = _run(b, iq, [600000, 400000], ("demod", "dsd_audio", "dsd_pcm"))
    b.close()
    assert segs[0]["dsd_pcm"].shape[:2] == (4, 1600)
    rows = [(s, c) for s in range(4) for c in (0, 2, 799, 1023, 1598, 1599)]
    _check_rows(segs[0], 48000 / 12500, rows)


def test_130_equal_streams():
    """130 streams (2080 rows: one warp past a multiple of the 256-row block) with equal input give bitwise equal rows."""
    from sdr_pmr446_b200 import chain
    n, chunk = 512000, 128000
    iq = np.repeat(_capture(1024000, n, 1, 960), 130, axis=0)
    b = chain.PmrBatch(n_streams=130, fs_in=1024000, in_fmt=1, max_chunk=chunk, dsd_rate=48000)
    seg = _run(b, iq, [chunk] * (n // chunk), ("demod", "dsd_audio", "dsd_pcm"))[0]
    b.close()
    for k in ("dsd_audio", "dsd_pcm"):
        assert all(np.array_equal(seg[k][0], seg[k][s]) for s in range(1, 130))
    _check_rows(seg, 48000 / 12500, [(0, c) for c in range(16)] + [(129, 1), (129, 14)])


def test_ring_wraps_three_times():
    """4 s of 1.024 Msps in 20000-sample calls: the discriminator ring (at most 16384 frames at this max_chunk) wraps more
    than three times under the feed."""
    from sdr_pmr446_b200 import chain
    n, chunk = 4096000, 20000
    iq = _capture(1024000, n, 1, 965, streams=2)
    b = chain.PmrBatch(n_streams=2, fs_in=1024000, in_fmt=1, max_chunk=chunk, dsd_rate=48000)
    seg = _run(b, iq, [chunk] * (n // chunk), ("demod", "dsd_audio", "dsd_pcm"))[0]
    b.close()
    assert seg["demod"].shape[-1] > 3 * 16384
    _check_rows(seg, 48000 / 12500)


def test_nothing_else_moves():
    """dsd_rate 0, dsd_rate 48000 without the tap, and with it: every other output bitwise equal, waterfall and the
    selector taps included."""
    from sdr_pmr446_b200 import chain
    calls = [0, 7, 100000, 33333, 100000, "reset", 50000]
    iq = _capture(1024000, 283340, 1, 970, streams=2)
    want = ALL + ("ascii", "rssi", "chan_edge")
    outs = []
    for rate, tap in ((0, False), (48000, False), (48000, True)):
        b = chain.PmrBatch(n_streams=2, fs_in=1024000, in_fmt=1, max_chunk=100000, waterfall=64, dsd_rate=rate)
        outs.append(_run(b, iq, calls, want + (("dsd_audio", "dsd_pcm") if tap else ())))
        b.close()
    for segs in outs[1:]:
        for a, g in zip(outs[0], segs):
            for k in want + ("peak", "psd"):
                va, vg = np.asarray(a[k]), np.asarray(g[k])
                assert va.dtype == vg.dtype and np.array_equal(va.view(np.uint8), vg.view(np.uint8)), k


def test_host_call_time_slices_equal_the_device_call():
    """The host-buffer call (600000 samples: eight time slices of 75008) against device calls of the same slices, bitwise, dsd
    outputs included: each slice's columns land at the offset its k(F) gives."""
    import torch
    from sdr_pmr446_b200 import chain
    n = 600000
    iq = _capture(2400000, 2 * n, 1, 980, streams=2)
    want = ("demod", "pcm", "dsd_audio", "dsd_pcm")
    h = chain.PmrBatch(n_streams=2, fs_in=2400000, in_fmt=1, max_chunk=n, dsd_rate=48000)
    d = chain.PmrBatch(n_streams=2, fs_in=2400000, in_fmt=1, max_chunk=n, dsd_rate=48000)
    S, M = 2, 16
    for c in range(2):
        part = np.ascontiguousarray(iq[:, c * 2 * n:(c + 1) * 2 * n])
        rh = h.execute(part, want)
        dev = torch.from_numpy(part).cuda()
        o = {"ld": d.max_ns, "dsd_ld": d.max_dsd,
             "demod": torch.zeros((S, M, d.max_ns), dtype=torch.float32, device="cuda"),
             "pcm": torch.zeros((S, M, d.max_ns), dtype=torch.int16, device="cuda"),
             "dsd_audio": torch.zeros((S, M, d.max_dsd), dtype=torch.float32, device="cuda"),
             "dsd_pcm": torch.zeros((S, M, d.max_dsd), dtype=torch.int16, device="cuda")}
        parts = {k: [] for k in want}
        launches = 0
        for a in range(0, n, 75008):
            m = min(75008, n - a)
            _, ns = d.execute_device(dev[:, 2 * a:2 * (a + m)], m, o)
            torch.cuda.synchronize()
            launches += d.last_launches
            for k, cnt in (("demod", ns), ("pcm", ns), ("dsd_audio", d.last_dsd), ("dsd_pcm", d.last_dsd)):
                parts[k].append(o[k][:, :, :cnt].cpu().numpy())
        assert h.last_dsd == rh["dsd_pcm"].shape[-1] > 0 and h.last_launches == launches
        for k in want:
            assert np.array_equal(np.concatenate(parts[k], axis=-1), rh[k]), k
    h.close()
    d.close()


def test_refused_calls_leave_state_untouched():
    from sdr_pmr446_b200 import _lib, chain
    for rate in (24000, 60000):   # x1.92 (no half-band stage) and x4.8 (two)
        with pytest.raises(_lib.Pmr446Error) as e:
            chain.PmrBatch(dsd_rate=rate)
        assert e.value.code == _lib.EINVAL
    with pytest.raises(_lib.Pmr446Error) as e:
        chain.PmrReceiver(dsd_rate=48000)
    assert e.value.code == _lib.EINVAL
    iq = _capture(1024000, 300000, 1, 990, streams=2)
    calls = [100000, 100000, 100000]
    # dsd_* requested with dsd_rate = 0
    a, t = (chain.PmrBatch(n_streams=2, in_fmt=1, max_chunk=100000) for _ in range(2))
    with pytest.raises(_lib.Pmr446Error) as e:
        a.execute(iq[:, :200000], ("demod", "dsd_pcm"))
    assert e.value.code == _lib.EINVAL
    ra, rt = _run(a, iq, calls, ALL)[0], _run(t, iq, calls, ALL)[0]
    for k in ALL:
        assert np.array_equal(ra[k], rt[k]), k
    # dsd_ld one short
    a, t = (chain.PmrBatch(n_streams=2, in_fmt=1, max_chunk=100000, dsd_rate=48000) for _ in range(2))
    want = ("demod", "dsd_audio", "dsd_pcm")
    first = t.execute(iq[:, :200000], want)
    need = t.last_dsd
    out = _lib.Outputs()
    pcm = np.zeros((2, 16, need), np.int16)
    out.dsd_pcm, out.dsd_ld = pcm.ctypes.data, need - 1
    chunk = np.ascontiguousarray(iq[:, :200000])
    assert _lib.lib().pmr446_batch_execute(a.h, chunk.ctypes.data, chunk.strides[0], 100000, C.byref(out), None, None) == _lib.ERANGE
    got = a.execute(iq[:, :200000], want)
    for k in want:
        assert np.array_equal(got[k], first[k]), k
    ra, rt = _run(a, iq[:, 200000:], calls[:2], want)[0], _run(t, iq[:, 200000:], calls[:2], want)[0]
    for k in want:
        assert np.array_equal(ra[k], rt[k]), k
    for x in (a, t):
        x.close()


def _tone_db(x, f, fs):
    """Amplitude (dB) of the sinusoid at f in x (least squares against cos / sin)."""
    t = np.arange(x.size) / fs
    A = np.stack([np.cos(2 * np.pi * f * t), np.sin(2 * np.pi * f * t)], axis=1)
    c = np.linalg.lstsq(A, np.asarray(x, np.float64), rcond=None)[0]
    return 20 * np.log10(np.hypot(*c))


def test_it_is_a_dsd_in_for_channel_k():
    """cfg1: FM carriers with tones on channels 2, 7, 8 and 15.  Channel k's feed against dsd446_batch on the same capture
    shifted so that channel k sits at DC: the tone at its frequency within 0.05 dB (600, 1000 Hz) or 1 dB (1700, 2400 Hz, where
    the two chains' channel filters differ), and channel 7 free of channel 8's 1700 Hz tone (>= 40 dB below its own)."""
    from sdr_pmr446_b200 import chain, synth
    fs, n, fa = 1024000, 1024000, 48000.0
    b = chain.PmrBatch(fs_in=fs, in_fmt=1, max_chunk=200000, dsd_rate=48000)
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(fs)), n, 446)[None, :]
    tap = b.run(iq, 200000, ("dsd_audio",))["dsd_audio"][0]
    b.close()
    skip = 4800   # 0.1 s: filters and de-emphasis of the synthetic modulation settle
    for car in synth.CFG1_CARRIERS:
        k = car.channel
        spec = synth.CaptureSpec(fs=float(fs), offset_hz=-synth.channel_offset_hz(k))
        d = chain.DsdBatch(fs_in=fs, in_fmt=1, max_chunk=200000)
        ref = d.run(synth.make_cu8(spec, n, 446)[None, :], 200000)["audio"][0]
        d.close()
        own = tap[k - 1][skip:]
        m = min(own.size, ref.size - skip)
        g, r = _tone_db(own[:m], car.audio_hz, fa), _tone_db(ref[skip:skip + m], car.audio_hz, fa)
        print("MEASURED channel %d: %.0f Hz tone %.3f dB (tap) vs %.3f dB (dsd446), diff %.3f dB" % (k, car.audio_hz, g, r, g - r))
        # the channelizer's prototype and dsd_in's decimator shape the FM sidebands differently: measured on a B200 (1000 W)
        # 0.010 dB at 1000 Hz, 0.002 dB at 600 Hz, 0.69 dB at 1700 Hz, 0.57 dB at 2400 Hz (DESIGN 4); bounds about 1.5x those
        assert abs(g - r) < (0.05 if car.audio_hz <= 1000.0 else 1.0), (k, g, r)
    ch7 = tap[6][skip:]
    rej = _tone_db(ch7, 600.0, fa) - _tone_db(ch7, 1700.0, fa)
    print("MEASURED channel 7: channel 8's 1700 Hz tone %.1f dB below its own 600 Hz tone" % rej)
    assert rej >= 40.0, rej
