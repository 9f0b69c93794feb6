"""CPU checks of the batch chain's per-channel DSD feed: the new C ABI symbols and fields, their ctypes mirrors against the
header as a C compiler lays it out, and the float64 msresamp_rrrf reference the GPU tests use, pinned to the oracle at every
rate they run."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import stage_ref
from util import design_msresamp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_new_symbols_are_exported_and_off_by_default():
    from sdr_pmr446_b200 import _lib, chain
    L = _lib.lib()
    for name in ("pmr446_batch_max_dsd", "pmr446_batch_last_dsd"):
        assert hasattr(L, name) and name in _lib.EXPORTS
    assert chain.default_config().dsd_rate == 0
    assert L.pmr446_batch_max_dsd(None) == 0 and L.pmr446_batch_last_dsd(None) == 0
    assert chain.PmrBatch.TIMING_TAGS[10] == "dsd" and len(chain.PmrBatch.TIMING_TAGS) == 11


def test_ctypes_layouts_match_the_header(tmp_path):
    from sdr_pmr446_b200 import _lib
    structs = {"pmr446_config": _lib.Config, "pmr446_outputs": _lib.Outputs, "pmr446_rx_config": _lib.RxConfig}
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "pmr446_b200.h"', "int main(void) {"]
    for cname, py in structs.items():
        lines.append('  printf("%s sizeof %%zu\\n", sizeof(%s));' % (cname, cname))
        for f, _ in py._fields_:
            lines.append('  printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, f, cname, f))
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict(line.rsplit(" ", 1) for line in subprocess.check_output([str(exe)], text=True).splitlines())
    for cname, py in structs.items():
        assert int(got[cname + " sizeof"]) == C.sizeof(py), cname
        for f, _ in py._fields_:
            assert int(got["%s %s" % (cname, f)]) == getattr(py, f).offset, (cname, f)


@pytest.mark.parametrize("rate", [48000 / 12500, 48000 / 16000, 44100 / 12500, 4.0])
def test_msresamp_interp_real_matches_the_oracle(rate):
    """stage_ref.msresamp_interp_real against the oracle's own msresamp_rrrf fed the same input, at x3.84 (12.5 kHz -> 48 kHz),
    x3.0 (16 kHz channels), x3.528 (44.1 kHz) and x4.0 (the edge of the accepted range)."""
    from oracle import oracle as orc
    O = orc.lib()
    rng = np.random.default_rng(446)
    n = 30000
    x = (0.3 * np.sin(2 * np.pi * 1000.0 / 12500.0 * np.arange(n)) + 0.3 * rng.standard_normal(n)).astype(np.float32)
    q = O.msresamp_rrrf_create(np.float32(rate), 60.0)
    ys = []
    for a, b in ((0, 1), (1, 7777), (7777, n)):
        blk = np.ascontiguousarray(x[a:b])
        y = np.zeros(4 * blk.size + 64, np.float32)
        ny = C.c_uint()
        assert O.msresamp_rrrf_execute(q, blk.ctypes.data, blk.size, y.ctypes.data, C.byref(ny)) == 0
        ys.append(y[:ny.value])
    O.msresamp_rrrf_destroy(q)
    ref = stage_ref.msresamp_interp_real(x, design_msresamp(np.float32(rate)))
    stage_ref.check_res(np.concatenate(ys), ref, 1e-6, 1.5e-5)
