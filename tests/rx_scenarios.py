"""Keyed-carrier scenarios for the receiver tests (squelch / selector / CTCSS, SURVEY.md 8f rows 1-2).

Times are in seconds of a 1.024 Msps capture processed in the reference's 100 000-sample chunks
(/root/reference/src/sdr_pmr446.c:30), i.e. 97.66 ms and 1220-1221 audio samples per chunk.
"""
import numpy as np

from sdr_pmr446_b200 import synth

FS = 1024000
CHUNK = 100000
SECONDS = 3.0


def keyed_two_calls():
    """Channel 2 (67.0 Hz) keys up at t = 0 and drops at 1.0 s; channel 7 (88.5 Hz) talks from 1.5 s on."""
    return (synth.Carrier(2, 0.20, 1000.0, 67.0, t_off=1.0), synth.Carrier(7, 0.10, 600.0, 88.5, t_on=1.5))


def stronger_later():
    """Channel 8 (123.0 Hz) from the start; a stronger channel 15 (250.3 Hz) joins at 1.2 s (lock_mode_max follows it)."""
    return (synth.Carrier(8, 0.08, 1700.0, 123.0), synth.Carrier(15, 0.25, 2400.0, 250.3, t_on=1.2))


def capture(carriers, seed=446, seconds=SECONDS, fs=FS, num_channels=16):
    spec = synth.CaptureSpec(fs=float(fs), num_channels=num_channels, carriers=carriers)
    return synth.make_cu8(spec, int(seconds * fs), seed)


def chunk_times(n_chunks, chunk=CHUNK, fs=FS):
    """[start, end) time of every chunk."""
    k = np.arange(n_chunks)
    return k * chunk / fs, (k + 1) * chunk / fs


def steady_chunks(rows, carriers, chunk=CHUNK, fs=FS):
    """Indices of chunks whose active channel's carrier is keyed on for the whole chunk and has been for at least
    two chunks of selected audio (so the 377-tap FIR no longer holds noise-only discriminator output)."""
    good = []
    run = 0
    for k, r in enumerate(rows):
        t0, t1 = k * chunk / fs, (k + 1) * chunk / fs
        act = int(r["active_chan"])
        on = any(c.channel - 1 == act and c.t_on <= t0 and t1 <= c.t_off for c in carriers) if act >= 0 else False
        run = run + 1 if on else 0
        if run >= 3:
            good.append(k)
    return good
