"""Golden fixtures (tests/golden/*.npz, made by tools/make_golden.py from the oracle).
CPU: the oracle reproduces them bit for bit (guards the checker against drift).
GPU: the CUDA path matches them within the north-star tolerances."""
import glob
import hashlib
import os

import numpy as np
import pytest

from util import PCM_TOL_LSB, REL_RMS_TOL, rel_rms

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    """Where a fixture does not store its capture (it would take the file over 1 MB), the capture is regenerated from its
    seed as tools/make_golden.py made it, and must match the stored SHA-256."""
    g = dict(np.load(os.path.join(GOLD, name)))
    if "iq" not in g:
        from sdr_pmr446_b200 import synth
        sid = int(g["stream_id"])
        g["iq"] = synth.make_cu8(synth.CaptureSpec(fs=float(g["fs"]), carriers=synth.rotated_carriers(sid)), int(g["n"]), 446 + sid)
        assert hashlib.sha256(g["iq"].tobytes()).hexdigest() == str(g["iq_sha256"]), "synth no longer makes the capture of " + name
    return g


def test_fixtures_present():
    files = glob.glob(os.path.join(GOLD, "*.npz"))
    assert len(files) >= 4
    assert all(os.path.getsize(f) < 1_000_000 for f in files)


@pytest.mark.parametrize("name", ["pmr_1024k_cu8.npz", "pmr_2400k_cu8_lowpass.npz"])
def test_oracle_reproduces_pmr_golden(name):
    from oracle import oracle as orc
    g = _load(name)
    o = orc.PmrOracle(fs_in=int(g["fs"]), in_fmt=1, audio_gain=1.0, lowpass=int(g["lowpass"]), chunk=int(g["chunk"]),
                      waterfall=int(g["waterfall"]))
    r = o.run(g["iq"], int(g["chunk"]))
    o.close()
    assert r["ny"] == int(g["ny"]) and r["ns"] == int(g["ns"])
    for k in ("res", "chan", "demod", "lpcomp", "audio", "pcm"):
        assert np.array_equal(r[k], g[k]), k
    if int(g["waterfall"]):
        assert np.array_equal(r["ascii"], g["ascii"]) and np.array_equal(r["psd"], g["psd"])


@pytest.mark.parametrize("name", ["dsd_1024k_cu8.npz", "dsd_2400k_cu8.npz"])
def test_oracle_reproduces_dsd_golden(name):
    from oracle import oracle as orc
    g = _load(name)
    o = orc.DsdOracle(fs_in=int(g["fs"]), in_fmt=1, chunk=int(g["chunk"]))
    r = o.run(g["iq"], int(g["chunk"]))
    o.close()
    assert r["ny"] == int(g["ny"]) and r["nz"] == int(g["nz"])
    for k in ("res", "fm", "audio", "pcm"):
        assert np.array_equal(r[k], g[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pmr_1024k_cu8.npz", "pmr_2400k_cu8_lowpass.npz"])
def test_gpu_matches_pmr_golden(name):
    from sdr_pmr446_b200 import chain, synth
    g = _load(name)
    b = chain.PmrBatch(n_streams=1, fs_in=int(g["fs"]), in_fmt=1, audio_gain=1.0, lowpass=int(g["lowpass"]), max_chunk=int(g["chunk"]),
                       waterfall=int(g["waterfall"]))
    want = ("res", "chan", "demod", "lpcomp", "audio", "pcm") + (("ascii",) if int(g["waterfall"]) else ())
    r = b.run(g["iq"], int(g["chunk"]), want)
    b.close()
    assert r["ny"] == int(g["ny"]) and r["ns"] == int(g["ns"])
    assert rel_rms(r["res"][0], g["res"]) < REL_RMS_TOL
    assert rel_rms(r["chan"][0], g["chan"]) < REL_RMS_TOL
    for c in sorted({x.channel - 1 for x in synth.rotated_carriers(int(g["stream_id"]))}):
        k = 1 if r["demod"][0, c, 0] == g["demod"][c, 0] else 500
        assert rel_rms(r["chan"][0, c], g["chan"][c]) < REL_RMS_TOL
        assert rel_rms(r["demod"][0, c, k:], g["demod"][c, k:]) < REL_RMS_TOL
        assert rel_rms(r["audio"][0, c, k:], g["audio"][c, k:]) < REL_RMS_TOL
        d = np.abs(r["pcm"][0, c, k:].astype(np.int32) - g["pcm"][c, k:].astype(np.int32))
        assert d.max() <= PCM_TOL_LSB
    if int(g["waterfall"]):
        assert np.max(np.abs(r["psd"][0] - g["psd"])) < 0.02
        assert np.sum(r["ascii"][0] != g["ascii"]) <= 2


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dsd_1024k_cu8.npz", "dsd_2400k_cu8.npz"])
def test_gpu_matches_dsd_golden(name):
    from sdr_pmr446_b200 import chain
    g = _load(name)
    b = chain.DsdBatch(n_streams=1, fs_in=int(g["fs"]), in_fmt=1, max_chunk=int(g["chunk"]))
    r = b.run(g["iq"], int(g["chunk"]))
    b.close()
    assert r["ny"] == int(g["ny"]) and r["nz"] == int(g["nz"])
    assert rel_rms(r["res"][0], g["res"]) < REL_RMS_TOL
    assert rel_rms(r["fm"][0, 1:], g["fm"][1:]) < REL_RMS_TOL
    k = 0 if r["fm"][0, 0] == g["fm"][0] else 200
    assert rel_rms(r["audio"][0, k:], g["audio"][k:]) < REL_RMS_TOL
    d = np.abs(r["pcm"][0, k:].astype(np.int32) - g["pcm"][k:].astype(np.int32))
    assert d.max() <= PCM_TOL_LSB
