"""The reference ITSELF: oracle/ref.mk compiles the UNMODIFIED upstream src/sdr_pmr446.c, dsd_in.c and
shared.c (file-backed stand-ins for SoapySDR / RtAudio / dlg, oracle/ref_stubs/) into oracle/_ref/.  Without liquid-dsp
in the image the DSP objects come from oracle/liquid_subset.c (LIQUID=oracle), so this pins everything the reference has
IN TREE -- main-loop order, ring-buffer carry, RSSI / squelch / selector state machine, demodulation chain wiring, CTCSS
detector, waterfall call sequence, dsd_in's loop -- against oracle/chains.c and oracle/receiver.c sample for sample.
With liquid-dsp v1.7.0 installed the same recipe links the real library (tests/test_oracle_vs_liquid.py).

The repository does not contain the reference's sources: build the binaries with `make -f oracle/ref.mk REF=<checkout>`;
the tests skip while they are missing."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

import rx_scenarios as sc
from oracle import oracle as orc
from sdr_pmr446_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _binary(name):
    path = os.path.join(REF, name)
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/%s is not built (make -f oracle/ref.mk REF=<checkout of the upstream sdr_pmr446>)" % name)
    return path


def _liquid_kind():
    p = os.path.join(REF, "LIQUID")
    return open(p).read().strip() if os.path.exists(p) else "oracle"


def _run_ref_pmr(iq_cu8, args=()):
    """Runs the reference receiver on a cu8 capture -> (audio float32, per-chunk counts, stderr log lines, stdout)."""
    exe = _binary("sdr_pmr446_ref")
    with tempfile.TemporaryDirectory() as d:
        iq, au, cn = (os.path.join(d, n) for n in ("iq.cu8", "audio.f32", "counts.txt"))
        iq_cu8.tofile(iq)
        env = dict(os.environ, REF_IQ=iq, REF_IQ_FMT="cu8", REF_AUDIO=au, REF_AUDIO_COUNTS=cn)
        p = subprocess.run([exe, *args], env=env, capture_output=True, timeout=600)
        assert p.returncode == 0, p.stderr.decode(errors="replace")[-2000:]
        audio = np.fromfile(au, np.float32)
        counts = np.loadtxt(cn, dtype=np.int64, ndmin=1)
        return audio, counts, p.stderr.decode(errors="replace").splitlines(), p.stdout.decode(errors="replace")


def _events_from_log(lines):
    """(kind, channel or tone) tuples in order of appearance, from the reference's own LOG lines (:616-622, :845, :861)."""
    ev = []
    for ln in lines:
        m = re.search(r"Tuned to channel (\d+)", ln)
        if m:
            ev.append(("tuned", int(m.group(1))))
        m = re.search(r"Changed active channel from (\d+) to (\d+)", ln)
        if m:
            ev.append(("changed", int(m.group(2))))
        m = re.search(r"Detuned from channel (\d+)", ln)
        if m:
            ev.append(("detuned", int(m.group(1))))
        m = re.search(r"(?:Acquired CTCSS code|CTCSS code change): (\d+) \(frequency: (\d+\.\d+)Hz\)", ln)
        if m:
            ev.append(("ctcss", (int(m.group(1)), round(float(m.group(2)), 1))))
        if "Lost CTCSS code" in ln:
            ev.append(("ctcss_lost", None))
    return ev


@pytest.mark.parametrize("scenario,lock,extra", [("keyed_two_calls", 0, ()), ("stronger_later", 1, ("-p", "max")),
                                                 ("keyed_two_calls", 0, ("-l",))])
def test_reference_receiver_audio_equals_oracle_receiver(scenario, lock, extra):
    """What the reference plays (selected channel through ONE demodulator chain, squelch, CTCSS) vs oracle/receiver.c."""
    carriers = getattr(sc, scenario)()
    iq = sc.capture(carriers)
    lowpass = 1 if "-l" in extra else 0
    audio, counts, log, _ = _run_ref_pmr(iq, ("-a", "1.0", *extra))
    o = orc.RxOracle(lock_mode=lock, fs_in=sc.FS, in_fmt=1, audio_gain=1.0, lowpass=lowpass, chunk=sc.CHUNK)
    rows = o.run(iq, sc.CHUNK)
    o.close()
    n_chunks = len(rows)
    # the stub drains once per readStream call: call 0 precedes the first chunk, call n_chunks hits end of file, and
    # rtaudio_stop_stream drains once more (nothing left)
    assert len(counts) == n_chunks + 2 and counts[0] == 0 and counts[-1] == 0
    want_counts = np.array([r["n_audio"] for r in rows])
    assert np.array_equal(counts[1:n_chunks + 1], want_counts)
    want = np.concatenate([r["audio"] for r in rows]) if want_counts.sum() else np.zeros(0, np.float32)
    assert audio.size == want.size and audio.size > 10000
    if _liquid_kind() == "oracle":
        assert np.array_equal(audio, want)                      # same DSP objects underneath: bit for bit
    else:
        assert np.sqrt(np.mean((audio - want) ** 2)) / np.sqrt(np.mean(want ** 2)) < 1e-4
    # tune / detune / CTCSS events in the reference's log = the oracle's event bits, in order
    ev = _events_from_log(log)
    want_ev = []
    prev_active = -1
    for r in rows:
        e = int(r["events"])
        if e & 1:
            want_ev.append(("tuned", int(r["active_chan"]) + 1))
        if e & 2:
            want_ev.append(("changed", int(r["active_chan"]) + 1 if not e & 4 else None))
        if e & 4:
            want_ev.append(("detuned", None))
        prev_active = int(r["active_chan"])
    got = [(k, c) for k, c in ev if k in ("tuned", "changed", "detuned")]
    assert [k for k, _ in got] == [k for k, _ in want_ev], (got, want_ev)
    for (k, c), (_, wc) in zip(got, want_ev):
        if wc is not None:
            assert c == wc, (got, want_ev)
    assert any(k == "tuned" for k, _ in got)
    tones = [f for k, f in ev if k == "ctcss"]
    want_tones = [(int(r["ctcss_index"]) + 1, round(float(r["ctcss_freq"]), 1)) for r in rows if int(r["events"]) & (8 | 16)]
    assert tones == want_tones and len(tones) >= 1, (tones, want_tones)
    assert sum(1 for k, _ in ev if k == "ctcss_lost") == sum(1 for r in rows if int(r["events"]) & 32)


def test_reference_waterfall_rows_equal_oracle_asgram():
    """`-w 120`: the rows the reference prints (asgramcf_write / asgramcf_execute per chunk, :910-918) vs the oracle chain."""
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(sc.FS), carriers=synth.CFG1_CARRIERS), 5 * sc.CHUNK, 446)
    _, _, _, out = _run_ref_pmr(iq, ("-a", "1.0", "-w", "120"))
    rows = re.findall(r" > (.{120}) < pk\s*(-?\d+\.\d)dB \[\s*(-?\d+\.\d\d)\]", out)
    o = orc.PmrOracle(fs_in=sc.FS, in_fmt=1, audio_gain=1.0, chunk=sc.CHUNK, waterfall=120)
    r = o.run(iq, sc.CHUNK, want=("res", "ascii"))
    o.close()
    assert len(rows) == 5
    for k, (txt, pk, pf) in enumerate(rows):
        assert txt == bytes(r["ascii"][k]).decode("ascii"), k
        assert abs(float(pk) - float(r["peak"][k][0])) <= 0.051 and abs(float(pf) - float(r["peak"][k][1])) <= 0.0051


def test_reference_dsd_in_equals_oracle_dsd_chain():
    """dsd_in (1.024 Msps is hard-coded, include/dsd_in.h:11) on a cu8 capture: its stdout s16 stream vs oracle chains.c."""
    exe = _binary("dsd_in_ref")
    fs, n = 1024000, 700000
    spec = synth.CaptureSpec(fs=float(fs), carriers=(synth.Carrier(1, 0.3, 1000.0, 0.0),), offset_hz=-synth.channel_offset_hz(1))
    iq = synth.make_cu8(spec, n, 446)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "iq.cu8")
        iq.tofile(path)
        p = subprocess.run([exe], env=dict(os.environ, REF_IQ=path, REF_IQ_FMT="cu8"), capture_output=True, timeout=600)
    assert p.returncode == 0, p.stderr.decode(errors="replace")[-2000:]
    got = np.frombuffer(p.stdout, np.int16)
    o = orc.DsdOracle(fs_in=fs, in_fmt=1, chunk=200000)
    r = o.run(iq, 200000)
    o.close()
    assert got.size == r["nz"]
    if _liquid_kind() == "oracle":
        assert np.array_equal(got, r["pcm"])
    else:
        assert np.abs(got[256:].astype(np.int32) - r["pcm"][256:].astype(np.int32)).max() <= 1
