#!/usr/bin/env python3
"""Generates tests/golden/*.npz: seeded synthetic inputs and the CPU oracle's outputs for them.

The reference ships no golden vectors (SURVEY.md 4) and cannot be built here, so these fixtures are produced by the
oracle restatement (PARITY UNPINNED, see oracle/liquid_subset.h).  They freeze the oracle's behaviour: a later
change to oracle/ that alters any sample fails tests/test_golden.py, and the CUDA path is checked against the same
files on the GPU box.  Run from the repo root:  python tools/make_golden.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as orc  # noqa: E402
from sdr_pmr446_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def pmr(name, fs, n, chunk, stream_id, lowpass, waterfall, store_iq=True):
    """store_iq=False keeps a fixture under 1 MB: tests/test_golden.py regenerates the capture from its seed and checks it
    against the stored SHA-256."""
    iq = synth.make_cu8(synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(stream_id)), n, 446 + stream_id)
    o = orc.PmrOracle(fs_in=fs, in_fmt=1, audio_gain=1.0, lowpass=lowpass, chunk=chunk, waterfall=waterfall)
    r = o.run(iq, chunk)
    o.close()
    d = dict(fs=fs, chunk=chunk, stream_id=stream_id, lowpass=lowpass, waterfall=waterfall, ny=r["ny"], ns=r["ns"],
             res=r["res"], chan=r["chan"], demod=r["demod"], lpcomp=r["lpcomp"], audio=r["audio"], pcm=r["pcm"])
    if store_iq:
        d.update(iq=iq)
    else:
        d.update(n=n, iq_sha256=hashlib.sha256(iq.tobytes()).hexdigest())
    if waterfall:
        d.update(ascii=r["ascii"], peak=r["peak"], psd=r["psd"])
    np.savez_compressed(os.path.join(OUT, name), **d)
    print(name, r["ny"], r["ns"])


def dsd(name, fs, n, chunk):
    spec = synth.CaptureSpec(fs=float(fs), carriers=(synth.Carrier(1, 0.3, 1000.0, 0.0),), offset_hz=-synth.channel_offset_hz(1))
    iq = synth.make_cu8(spec, n, 446)
    o = orc.DsdOracle(fs_in=fs, in_fmt=1, chunk=chunk)
    r = o.run(iq, chunk)
    o.close()
    np.savez_compressed(os.path.join(OUT, name), iq=iq, fs=fs, chunk=chunk, ny=r["ny"], nz=r["nz"], res=r["res"], fm=r["fm"],
                        audio=r["audio"], pcm=r["pcm"])
    print(name, r["ny"], r["nz"])


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    pmr("pmr_1024k_cu8.npz", 1024000, 150000, 100000, 0, 0, 120, store_iq=False)
    pmr("pmr_2400k_cu8_lowpass.npz", 2400000, 240000, 120000, 3, 1, 0)
    dsd("dsd_1024k_cu8.npz", 1024000, 300000, 200000)
    dsd("dsd_2400k_cu8.npz", 2400000, 480000, 200000)
