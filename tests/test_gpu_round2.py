"""Round-2 GPU parity cases (VERDICT r01 "next round" item 1, ADVICE r01):

 * the block-per-transform waterfall kernel (nfft > 1024, /root/reference/src/sdr_pmr446.c:473-477, :910-913 with the
   terminal width W as asgramcf_create's argument) for W in {300, 512, 1600}, the warp kernel's largest plan (W = 250,
   nfft = 1000 = 4 * 2 * 5^3), and a width whose nfft has a large prime factor (W = 67);
 * BASELINE configs[3] as written: 20 Msps cf32, 1600 channels AND the W = 1600 waterfall in the same run;
 * BASELINE configs[0] and configs[1] at their stated length (10 s captures, the reference's chunk sizes);
 * the saturating s16 conversion at the reference's default audio_gain = 4;
 * a failed execute (ld too small) leaves the stream state untouched.
"""
import numpy as np
import pytest

from util import PCM_TOL_LSB, REL_RMS_TOL, active_channels, rel_rms

pytestmark = pytest.mark.gpu


def _waterfall_pair(fs, n, chunk, W, fmt_cu8=True, M=16, carriers=None, seed=446):
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    spec = synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=carriers) if carriers else synth.CaptureSpec(fs=float(fs), num_channels=M)
    iq = synth.make_cu8(spec, n, seed) if fmt_cu8 else synth.make_cf32(spec, n, seed)
    fmt = 1 if fmt_cu8 else 0
    gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=fmt, num_channels=M, audio_gain=1.0, max_chunk=chunk, waterfall=W)
    g = gpu.run(iq[None, :], chunk, want=("res", "ascii"))
    gpu.close()
    o = orc.PmrOracle(fs_in=fs, in_fmt=fmt, num_channels=M, audio_gain=1.0, chunk=chunk, waterfall=W)
    r = o.run(iq, chunk, want=("res", "ascii"))
    o.close()
    return g, r


def _check_waterfall(g, r, W):
    assert g["ny"] == r["ny"]
    assert g["psd"].shape[1:] == r["psd"].shape and r["psd"].shape[-1] == 4 * W
    # dB values of every bin of every row, the peak (value, frequency) and the characters; a character may flip only
    # where the 4-bin column value sits on a 2 dB level edge
    assert np.max(np.abs(g["psd"][0] - r["psd"])) < 0.02
    assert np.max(np.abs(g["peak"][0] - r["peak"])) < 0.02
    mism = int(np.sum(g["ascii"][0] != r["ascii"]))
    assert mism <= max(2, r["ascii"].size // 200), mism


@pytest.mark.parametrize("W", [250, 300, 512, 1600])
def test_waterfall_large_widths(W):
    """W = 250 is the warp kernel's largest mixed-radix plan; 300 / 512 / 1600 (nfft 1200 / 2048 / 6400) run the
    block-per-transform kernel, 6400 with its 1024-thread launch and the radix-4 lead stage folded into the load."""
    g, r = _waterfall_pair(1024000, 300000, 100000, W)
    _check_waterfall(g, r, W)


def test_waterfall_width_with_large_prime_factor():
    """asgramcf_create accepts any width: W = 67 gives nfft = 268 = 4 * 67 (generic radix-67 butterfly)."""
    g, r = _waterfall_pair(1024000, 200000, 100000, 67)
    _check_waterfall(g, r, 67)


def test_cfg4_wideband_1600_channels_with_waterfall_1600():
    """BASELINE configs[3] as written (shortened to 0.04 s): 20 Msps cf32 -> 1600-channel PFB + per-channel NBFM demod
    AND the W = 1600 waterfall (nfft 6400) on the same resampled stream."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    M, fs, n, W = 1600, 20_000_000, 800_000, 1600
    car = (synth.Carrier(3, 0.2, 1000.0, 67.0), synth.Carrier(800, 0.1, 600.0, 88.5),
           synth.Carrier(801, 0.15, 1700.0, 123.0), synth.Carrier(1599, 0.05, 2400.0, 250.3))
    iq = synth.make_cf32(synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=car), n, 446)
    want = ("chan", "demod", "pcm", "ascii")
    gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=0, num_channels=M, max_chunk=400000, waterfall=W)
    g = gpu.run(iq[None, :], 400000, want)
    gpu.close()
    o = orc.PmrOracle(fs_in=fs, in_fmt=0, num_channels=M, chunk=400000, waterfall=W)
    r = o.run(iq, 400000, want)
    o.close()
    assert g["ns"] == r["ns"] == n // M
    assert rel_rms(g["chan"][0], r["chan"]) < REL_RMS_TOL
    for c in active_channels(car):
        sl = slice(1, None) if g["demod"][0, c, 0] == r["demod"][c, 0] else slice(500, None)
        assert rel_rms(g["demod"][0, c, sl], r["demod"][c, sl]) < REL_RMS_TOL, ("demod", c)
    _check_waterfall(g, r, W)


def test_cfg1_full_length_10s_1024k():
    """BASELINE configs[0] at its stated length: 10 s of 1.024 Msps cu8 (10 240 000 samples, 103 chunks of 100 000 like
    SDR_INPUT_CHUNK, src/sdr_pmr446.c:30), 4 FM carriers + CTCSS: counts, channelizer output and s16 audio."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    fs, n, chunk = 1024000, 10_240_000, 100000
    car = synth.CFG1_CARRIERS
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(fs), carriers=car), n, 446)
    gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=chunk)
    g = gpu.run(iq[None, :], chunk, want=("chan", "pcm"))
    gpu.close()
    o = orc.PmrOracle(fs_in=fs, in_fmt=1, audio_gain=1.0, chunk=chunk)
    r = o.run(iq, chunk, want=("chan", "pcm"))
    o.close()
    assert g["ny"] == r["ny"] and abs(g["ny"] - 2_000_000) <= 1 and g["ns"] == r["ns"] == 125_000     # SURVEY.md Appendix B
    assert rel_rms(g["chan"][0], r["chan"]) < REL_RMS_TOL
    for c in active_channels(car):
        assert rel_rms(g["chan"][0, c], r["chan"][c]) < REL_RMS_TOL, ("chan", c)
        dp = np.abs(g["pcm"][0, c, 700:].astype(np.int32) - r["pcm"][c, 700:].astype(np.int32))
        assert dp.max() <= PCM_TOL_LSB, ("pcm", c, int(dp.max()))


def test_cfg2_full_length_10s_dsd_2400k():
    """BASELINE configs[1] at its stated length: 10 s of 2.4 Msps cu8 through the dsd_in chain in the reference's
    200 000-sample chunks (src/dsd_in.c:25) -> 48 kHz s16."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    fs, n, chunk = 2400000, 24_000_000, 200000
    iq = synth.cfg2_capture(n=n)
    gpu = chain.DsdBatch(n_streams=1, fs_in=fs, in_fmt=1, max_chunk=chunk)
    g = gpu.run(iq[None, :], chunk)
    gpu.close()
    o = orc.DsdOracle(fs_in=fs, in_fmt=1, chunk=chunk)
    r = o.run(iq, chunk)
    o.close()
    assert g["ny"] == r["ny"] and g["nz"] == r["nz"]
    assert abs(g["nz"] - 480_000) <= 8
    assert rel_rms(g["res"][0], r["res"]) < REL_RMS_TOL
    sl = slice(1, None) if g["fm"][0, 0] == r["fm"][0] else slice(64, None)
    assert rel_rms(g["fm"][0, sl], r["fm"][sl]) < REL_RMS_TOL
    dp = np.abs(g["pcm"][0, 256:].astype(np.int32) - r["pcm"][256:].astype(np.int32))
    assert dp.max() <= PCM_TOL_LSB, int(dp.max())


def test_default_gain_saturates_instead_of_wrapping():
    """audio_gain = 4 is the reference's default (src/sdr_pmr446.c:33): a +-2.5 kHz deviation tone reaches +-1.6 of full
    scale.  The s16 output must clip (like the audio device clips RtAudio's float32), never wrap, and still equal the
    oracle's within 1 LSB."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    fs, n = 1024000, 300000
    car = synth.CFG1_CARRIERS
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(fs), carriers=car), n, 446)
    gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=1, max_chunk=100000)           # default gain
    assert gpu.cfg.audio_gain == 4.0
    g = gpu.run(iq[None, :], 100000, want=("audio", "pcm"))
    gpu.close()
    o = orc.PmrOracle(fs_in=fs, in_fmt=1, audio_gain=4.0, chunk=100000)
    r = o.run(iq, 100000, want=("audio", "pcm"))
    o.close()
    clipped = 0
    for c in active_channels(car):
        a, p = g["audio"][0, c, 700:], g["pcm"][0, c, 700:].astype(np.int32)
        over = np.abs(a) > 1.001
        clipped += int(over.sum())
        assert np.all(p[over] == np.where(a[over] > 0, 32767, -32768))                   # clipped, same sign as the audio
        dp = np.abs(p - r["pcm"][c, 700:].astype(np.int32))
        assert dp.max() <= PCM_TOL_LSB, (c, int(dp.max()))
    assert clipped > 1000


def test_failed_execute_leaves_state_untouched():
    """A call rejected for a too-small leading dimension must not consume the chunk (ADVICE r01): the same data fed
    again with a valid `ld` gives exactly what an undisturbed handle gives."""
    import ctypes as C

    from sdr_pmr446_b200 import chain, synth
    from sdr_pmr446_b200._lib import ERANGE, Outputs, lib
    fs, n = 2400000, 240000
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(fs)), 2 * n, 446)[None, :]
    a = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=n)
    b = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=n)
    first_a = a.execute(iq[:, :2 * n], want=("pcm",))
    first_b = b.execute(iq[:, :2 * n], want=("pcm",))
    assert np.array_equal(first_a["pcm"], first_b["pcm"])
    # rejected call on b: pcm requested with ld = 10
    bad = Outputs()
    pcm = np.zeros((1, 16, 10), np.int16)
    bad.pcm, bad.ld = pcm.ctypes.data, 10
    chunk2 = np.ascontiguousarray(iq[:, 2 * n:])
    rc = lib().pmr446_batch_execute(b.h, chunk2.ctypes.data, chunk2.strides[0], n, C.byref(bad), None, None)
    assert rc == ERANGE
    second_a = a.execute(chunk2, want=("pcm",))
    second_b = b.execute(chunk2, want=("pcm",))
    a.close()
    b.close()
    assert second_a["ns"] == second_b["ns"]
    assert np.array_equal(second_a["pcm"], second_b["pcm"])
    # dsd_in path
    da = chain.DsdBatch(n_streams=1, fs_in=fs, in_fmt=1, max_chunk=n)
    db = chain.DsdBatch(n_streams=1, fs_in=fs, in_fmt=1, max_chunk=n)
    da.execute(iq[:, :2 * n])
    db.execute(iq[:, :2 * n])
    from sdr_pmr446_b200._lib import DsdOutputs
    dbad = DsdOutputs()
    small = np.zeros((1, 8), np.int16)
    dbad.pcm, dbad.out_ld, dbad.res_ld = small.ctypes.data, 8, 0
    rc = lib().dsd446_batch_execute(db.h, chunk2.ctypes.data, chunk2.strides[0], n, C.byref(dbad), None, None)
    assert rc == ERANGE
    ra, rb = da.execute(chunk2), db.execute(chunk2)
    da.close()
    db.close()
    assert ra["nz"] == rb["nz"] and np.array_equal(ra["pcm"], rb["pcm"])
    # receiver path
    xa = chain.PmrReceiver(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=n)
    xb = chain.PmrReceiver(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=n)
    xa.execute(iq[:, :2 * n])
    xb.execute(iq[:, :2 * n])
    from sdr_pmr446_b200._lib import RxOutputs
    xbad = RxOutputs()
    audio, pcm = np.zeros((1, 10), np.float32), np.zeros((1, 10), np.int16)
    xbad.audio, xbad.pcm, xbad.ld = audio.ctypes.data, pcm.ctypes.data, 10
    rc = lib().pmr446_receiver_execute(xb.h, chunk2.ctypes.data, chunk2.strides[0], n, C.byref(xbad), None)
    assert rc == ERANGE
    ra, rb = xa.execute(chunk2), xb.execute(chunk2)
    xa.close()
    xb.close()
    assert ra["ns"] == rb["ns"]
    for k in chain.PmrReceiver.STATUS_FIELDS:
        assert np.array_equal(ra[k], rb[k]), k
    assert np.array_equal(ra["audio"], rb["audio"]) and np.array_equal(ra["pcm"], rb["pcm"])


@pytest.mark.parametrize("fs,M,fmt_cu8", [(3200000, 16, True), (1024000, 20, True), (500000, 16, False), (4800000, 16, True)])
def test_other_resampler_plans(fs, M, fmt_cu8):
    """msresamp_crcf_create accepts any rate (src/sdr_pmr446.c:425-426).  3.2 Msps -> 200 kHz ([3,5] | [10] + resampler
    at rate 1/2), 250 kHz output (20 channels from 1.024 Msps), a single half-band (500 kHz -> 200 kHz) and a four-stage
    plan (4.8 Msps): resampler, channelizer and s16 audio against the oracle."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    n = int(fs * 0.15)
    chunk = n // 3 + 17
    car = (synth.Carrier(2, 0.2, 1000.0, 67.0), synth.Carrier(M - 1, 0.1, 600.0, 88.5))
    spec = synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=car)
    iq = synth.make_cu8(spec, n, 446) if fmt_cu8 else synth.make_cf32(spec, n, 446)
    fmt = 1 if fmt_cu8 else 0
    gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=fmt, num_channels=M, audio_gain=1.0, max_chunk=chunk)
    g = gpu.run(iq[None, :], chunk, want=("res", "chan", "demod", "pcm"))
    gpu.close()
    o = orc.PmrOracle(fs_in=fs, in_fmt=fmt, num_channels=M, audio_gain=1.0, chunk=chunk)
    r = o.run(iq, chunk, want=("res", "chan", "demod", "pcm"))
    o.close()
    assert g["ny"] == r["ny"] and g["ns"] == r["ns"]
    assert rel_rms(g["res"][0], r["res"]) < REL_RMS_TOL
    assert rel_rms(g["chan"][0], r["chan"]) < REL_RMS_TOL
    for c in active_channels(car):
        sl = slice(1, None) if g["demod"][0, c, 0] == r["demod"][c, 0] else slice(500, None)
        assert rel_rms(g["demod"][0, c, sl], r["demod"][c, sl]) < REL_RMS_TOL, ("demod", c)
        dp = np.abs(g["pcm"][0, c, 600:].astype(np.int32) - r["pcm"][c, 600:].astype(np.int32))
        assert dp.max() <= PCM_TOL_LSB, ("pcm", c, int(dp.max()))


def test_deferred_dc_correction_path_float_parity():
    """2.4 Msps cu8 WITHOUT the `res` output and without a waterfall: the fused front end leaves the zero-input part of its
    DC blocker to channelize16_kernel (added while it stages its tiles; the ring's tail is then finished in place).  Channelizer
    and discriminator outputs at 1e-4, s16 within 1 LSB, over chunk sizes that split tiles, batches and segments, including
    chunks smaller than a tile, and the stream start (DC state zero) as well as a DC offset 10x the default."""
    from oracle import oracle as orc
    from sdr_pmr446_b200 import chain, synth
    fs, n = 2400000, 900000
    for dc in (0.02 - 0.015j, 0.2 - 0.15j):
        car = synth.rotated_carriers(4)
        spec = synth.CaptureSpec(fs=float(fs), carriers=car, dc=dc)
        iq = synth.make_cu8(spec, n, 455)
        gpu = chain.PmrBatch(n_streams=1, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=300000)
        sizes = [300000, 1, 47, 6143, 6145, 73729, 200000, 13, 300000, 13922]
        assert sum(sizes) == n
        parts, o = [], 0
        for k in sizes:
            parts.append(gpu.execute(iq[None, 2 * o:2 * (o + k)], want=("chan", "demod", "pcm")))
            o += k
        gpu.close()
        g = {"ns": sum(p["ns"] for p in parts)}
        for k in ("chan", "demod", "pcm"):
            g[k] = np.concatenate([p[k] for p in parts], axis=-1)
        ref = orc.PmrOracle(fs_in=fs, in_fmt=1, audio_gain=1.0, chunk=300000)
        r = ref.run(iq, 300000, want=("chan", "demod", "pcm"))
        ref.close()
        assert g["ns"] == r["ns"]
        assert rel_rms(g["chan"][0], r["chan"]) < REL_RMS_TOL
        for c in active_channels(car):
            assert rel_rms(g["chan"][0, c], r["chan"][c]) < REL_RMS_TOL, ("chan", c)
            sl = slice(1, None) if g["demod"][0, c, 0] == r["demod"][c, 0] else slice(500, None)
            assert rel_rms(g["demod"][0, c, sl], r["demod"][c, sl]) < REL_RMS_TOL, ("demod", c)
            dp = np.abs(g["pcm"][0, c, 600:].astype(np.int32) - r["pcm"][c, 600:].astype(np.int32))
            assert dp.max() <= PCM_TOL_LSB, ("pcm", c, int(dp.max()))


def test_unaligned_device_buffer_takes_the_guarded_path():
    """pmr446_batch_execute_device / dsd446_batch_execute_device with a device pointer that is only sample-aligned (2 bytes): no
    32-byte vector loads, no cp.async of whole sub-blocks -- every sample goes through the guarded loader, and the result must be
    the aligned run's (same arithmetic, same segment grid: at most the 1 LSB the s16 tolerance allows)."""
    import torch
    from sdr_pmr446_b200 import chain, synth
    fs, n, S = 2400000, 240000, 2
    caps = [synth.make_cu8(synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(s)), n, 446 + s) for s in range(S)]
    iq = torch.from_numpy(np.stack(caps)).cuda()
    pad = torch.zeros((S, 2 * n + 64), dtype=torch.uint8, device="cuda")
    shifted = pad[:, 2:2 + 2 * n]
    shifted.copy_(iq)
    assert shifted.data_ptr() % 32 == 2
    res = []
    for buf in (iq, shifted):
        b = chain.PmrBatch(n_streams=S, fs_in=fs, in_fmt=1, audio_gain=1.0, max_chunk=n)
        pcm = torch.zeros((S, 16, b.max_ns), dtype=torch.int16, device="cuda")
        ny, ns = b.execute_device(buf, n, {"ld": b.max_ns, "pcm": pcm})
        torch.cuda.synchronize()
        res.append((ny, ns, pcm[:, :, :ns].cpu().numpy()))
        b.close()
    assert res[0][:2] == res[1][:2]
    assert np.abs(res[0][2].astype(np.int32) - res[1][2].astype(np.int32)).max() <= PCM_TOL_LSB
    res = []
    for buf in (iq, shifted):
        d = chain.DsdBatch(n_streams=S, fs_in=fs, in_fmt=1, max_chunk=n)
        pcm = torch.zeros((S, d.max_out), dtype=torch.int16, device="cuda")
        r = d.execute_device(buf, n, pcm=pcm)
        torch.cuda.synchronize()
        res.append((r, pcm.cpu().numpy()))
        d.close()
    assert res[0][0] == res[1][0]
    assert np.abs(res[0][1].astype(np.int32) - res[1][1].astype(np.int32)).max() <= PCM_TOL_LSB
