"""The CUDA receiver against THE REFERENCE PROGRAM ITSELF: oracle/_ref/sdr_pmr446_ref is the unmodified upstream
src/sdr_pmr446.c + shared.c (file-backed SoapySDR / RtAudio stand-ins, oracle/ref.mk) -- its played audio,
tune / detune / channel-change and CTCSS log lines are compared DIRECTLY with pmr446_receiver_execute()'s outputs, without
oracle/receiver.c in between.  The same for dsd_in: its stdout s16 stream against dsd446_batch_execute().

The repository does not contain the reference's sources: build the binaries with `make -f oracle/ref.mk REF=<checkout>`;
the tests skip while they are missing."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import rx_scenarios as sc
from util import PCM_TOL_LSB, REL_RMS_TOL, rel_rms

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _exe(name):
    path = os.path.join(REF, name)
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/%s is not built (make -f oracle/ref.mk REF=<checkout of the upstream sdr_pmr446>)" % name)
    return path


def _run_reference(iq, args):
    with tempfile.TemporaryDirectory() as d:
        p_iq, p_au, p_cn = (os.path.join(d, n) for n in ("iq.cu8", "audio.f32", "counts.txt"))
        iq.tofile(p_iq)
        env = dict(os.environ, REF_IQ=p_iq, REF_IQ_FMT="cu8", REF_AUDIO=p_au, REF_AUDIO_COUNTS=p_cn)
        p = subprocess.run([_exe("sdr_pmr446_ref"), *args], env=env, capture_output=True, timeout=600)
        assert p.returncode == 0, p.stderr.decode(errors="replace")[-1500:]
        return np.fromfile(p_au, np.float32), np.loadtxt(p_cn, dtype=np.int64, ndmin=1), p.stderr.decode(errors="replace").splitlines()


@pytest.mark.parametrize("scenario,lock,extra", [("keyed_two_calls", 0, ()), ("stronger_later", 1, ("-p", "max"))])
def test_receiver_equals_the_reference_program(scenario, lock, extra):
    from sdr_pmr446_b200 import chain
    carriers = getattr(sc, scenario)()
    iq = sc.capture(carriers)
    audio, counts, log = _run_reference(iq, ("-a", "1.0", *extra))
    rx = chain.PmrReceiver(n_streams=1, fs_in=sc.FS, in_fmt=1, max_chunk=sc.CHUNK, audio_gain=1.0, lock_mode=lock)
    rows = rx.run(iq[None, :], sc.CHUNK)
    rx.close()
    n = len(rows)
    # samples handed to the audio device per chunk: identical
    assert np.array_equal(counts[1:n + 1], np.array([int(r["n_audio"][0]) for r in rows]))
    # log lines of the reference in order = event bits of the GPU receiver
    got = []
    for ln in log:
        m = re.search(r"Tuned to channel (\d+)", ln)
        if m:
            got.append(("tuned", int(m.group(1))))
        m = re.search(r"Changed active channel from (\d+) to (\d+)", ln)
        if m:
            got.append(("changed", int(m.group(2))))
        if "Detuned from channel" in ln:
            got.append(("detuned", None))
        m = re.search(r"(?:Acquired CTCSS code|CTCSS code change): (\d+) \(frequency: (\d+\.\d+)Hz\)", ln)
        if m:
            got.append(("ctcss", int(m.group(1))))
        if "Lost CTCSS code" in ln:
            got.append(("ctcss_lost", None))
    want = []
    for r in rows:
        e = int(r["events"][0])
        if e & 1:
            want.append(("tuned", int(r["active_chan"][0]) + 1))
        if e & 2:
            want.append(("changed", None if e & 4 else int(r["active_chan"][0]) + 1))
        if e & 4:
            want.append(("detuned", None))
        if e & (8 | 16):
            want.append(("ctcss", int(r["ctcss_index"][0]) + 1))
        if e & 32:
            want.append(("ctcss_lost", None))
    assert [k for k, _ in got] == [k for k, _ in want], (got, want)
    for (k, a), (_, b) in zip(got, want):
        if b is not None:
            assert a == b, (got, want)
    assert ("tuned" in [k for k, _ in got]) and ("ctcss" in [k for k, _ in got])
    # the played audio on chunks where the active channel's carrier is keyed on (noise-only spans: the discriminator is
    # ill-conditioned, SURVEY.md 7)
    rows1 = [{k: (v[0] if isinstance(v, np.ndarray) and v.ndim >= 1 and k not in ("audio", "pcm", "ctcss_in", "rssi_ch", "ctcss_power") else v) for k, v in r.items()} for r in rows]
    good = sc.steady_chunks(rows1, carriers)
    assert len(good) >= 8
    off = np.concatenate([[0], np.cumsum(counts[1:n + 1])])
    ref_a = np.concatenate([audio[off[k]:off[k + 1]] for k in good])
    gpu_a = np.concatenate([rows[k]["audio"][0, :int(rows[k]["n_audio"][0])] for k in good])
    assert rel_rms(gpu_a, ref_a) < REL_RMS_TOL, rel_rms(gpu_a, ref_a)


def test_dsd_chain_equals_the_reference_program():
    from sdr_pmr446_b200 import chain, synth
    fs, n = 1024000, 700000
    spec = synth.CaptureSpec(fs=float(fs), carriers=(synth.Carrier(1, 0.3, 1000.0, 0.0),), offset_hz=-synth.channel_offset_hz(1))
    iq = synth.make_cu8(spec, n, 446)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "iq.cu8")
        iq.tofile(path)
        p = subprocess.run([_exe("dsd_in_ref")], env=dict(os.environ, REF_IQ=path, REF_IQ_FMT="cu8"), capture_output=True, timeout=600)
    assert p.returncode == 0, p.stderr.decode(errors="replace")[-1500:]
    ref = np.frombuffer(p.stdout, np.int16)
    gpu = chain.DsdBatch(n_streams=1, fs_in=fs, in_fmt=1, max_chunk=200000)
    g = gpu.run(iq[None, :], 200000)
    gpu.close()
    assert g["nz"] == ref.size
    assert np.abs(g["pcm"][0, 256:].astype(np.int32) - ref[256:].astype(np.int32)).max() <= PCM_TOL_LSB
