"""GPU front-end sweep: the DC blocker, the half-band cascade and the arbitrary resampler of every plan the configuration
selects, and the dsd_in back end, against the float64 references of tests/stage_ref.py.

The front end's reference is fed the raw capture: the conversion to float32 is exact, so conversion, DC blocker,
half-bands and resampler are one stage, and `res` is compared sample by sample (stage_ref.check_res): the error RMS over
the whole output AND every single sample against the output's RMS.  An RMS alone lets sparse errors through, and segment
starts, tile edges, chunk edges, ring wrap and halo warm-up produce exactly those.

Each case runs 3 streams with distinct seeds (unless it varies the stream count on purpose) and checks every stream.
Chunk lists are uneven: 0-, 1- and 7-sample calls, calls shorter than a 16-sample group, a 48-sample fused iteration or
a tile, calls one off the fused kernel's 1536- and 6144-sample segments and off 4096, and calls that are not multiples
of 16.  Cases are named by the plan string pmr446_describe_frontend gives; test_cases_reach_every_frontend_kernel (no
GPU) checks that they reach every front-end kernel the library instantiates.

Bounds (about ten times the largest error measured on a B200 at 1000 W, DESIGN.md 4; the float32 oracle itself sits at
1.4e-6 .. 6.7e-6 relative RMS of the same references):
  res     FE_TOL_RMS relative RMS, FE_TOL_MAX of the output's RMS per sample
  fm      DSD_FM_TOL_RAD per sample against the float64 discriminator of the GPU's own res
  audio   DSD_AUDIO_TOL_RMS relative RMS, DSD_AUDIO_TOL_MAX of the RMS per sample, against msresamp_rrrf of the GPU's fm
  pcm     stage_ref.check_pcm on the samples inside +-1 (dsd_in's cast truncates and does not saturate)
  chan    (correction deferred to the channelizer) bitwise equal to the chan of the same capture with the correction
          applied in place, and stage_ref.check_chan against the float64 channelizer of the float64 front end
"""
import functools
import os
import re

import numpy as np
import pytest

import stage_ref
from util import describe_frontend, design_dtheta, design_msresamp, design_pfbch

GPU = pytest.mark.gpu
S = 3
ALPHA = 0.0005
FE_TOL_RMS, FE_TOL_MAX = 3e-6, 1e-5
DSD_FM_TOL_RAD = 2.5e-6
DSD_AUDIO_TOL_RMS, DSD_AUDIO_TOL_MAX = 1e-6, 1.5e-5
CHAN_TOL_CH, CHAN_TOL_STAGE = 1e-5, 1e-6
CU8, CF32, CS16, CS8 = stage_ref.FMT_CU8, stage_ref.FMT_CF32, stage_ref.FMT_CS16, stage_ref.FMT_CS8
FMT_NAME = {CU8: "cu8", CF32: "cf32", CS16: "cs16", CS8: "cs8"}
BPS = {CU8: 2, CF32: 1, CS16: 2, CS8: 2}   # array columns per IQ sample of the synth captures


def _rate(fs_in, fs_out):
    return float(np.float32(fs_out) / np.float32(fs_in))


# ---- the cases and the kernels they reach -------------------------------------------------------------------------------
# (chain, fs_in, fmt, fs_out): "batch" = PmrBatch into 16 x 12.5 kHz, "dsd" = DsdBatch into 12.5 kHz, "shim" = the liquid
# shim's msresamp_crcf (cf32, no DC blocker)
def _all(fs_in, fs_out=200000, chain="batch"):
    return [(chain, fs_in, f, fs_out) for f in (CU8, CF32, CS16, CS8)]


FE_CASES = (_all(2400000) + _all(1024000) + _all(3200000) + _all(4800000) + _all(1200000) + _all(20000000) + _all(500000) +
            _all(250000) + [("batch", 6400000, CF32, 200000), ("batch", 9600000, CF32, 200000), ("batch", 800000, CF32, 200000),
                            ("batch", 400000, CF32, 200000), ("batch", 200000, CF32, 200000)] +
            _all(2400000, 12500, "dsd") + [("dsd", 1024000, CU8, 12500), ("dsd", 2048000, CU8, 12500), ("dsd", 20000000, CU8, 12500),
                                                                 ("dsd", 4800000, CF32, 12500)])
SHIM_CASES = [("shim", fs, CF32, 200000) for fs in (2400000, 20000000, 4800000, 1024000, 500000, 1200000, 250000)]


def _plan(case):
    chain, fs_in, fmt, fs_out = case
    return describe_frontend(_rate(fs_in, fs_out), fmt, 0 if chain == "shim" else 1)


def _case_id(case):
    chain, fs_in, fmt, fs_out = case
    return "%s-%s-%g-%g-%s" % (chain, FMT_NAME[fmt], fs_in / 1e6, fs_out / 1e3, _plan(case).replace(" ", ""))


def _kernels(plan, fmt, with_dc):
    """The kernels a plan string launches, keyed the way Frontend::init assigns levels: ("fused",), ("front6", m5, m6),
    ("tile",), ("cascade", src, dc, stages, arb), ("dc_local", src)."""
    levels = plan.split(" | ")
    out = set()
    for l, lv in enumerate(levels):
        kind, ms, arb = re.fullmatch(r"(\w+)\[([\d,]*)\](\+arb)?", lv).groups()
        ms = tuple(int(v) for v in ms.split(",")) if ms else ()
        src = FMT_NAME[fmt] if l == 0 else "ring"
        dc = ("zsr" if len(levels) >= 2 or kind == "fused" else "scan") if l == 0 and with_dc else "none"
        if kind == "fused":
            out.add(("fused",))
        elif kind == "front6":
            out.add(("front6",) + ms[4:6])
        elif kind == "tile":
            out.add(("tile",))
        else:
            out.add(("cascade", src, dc, ms, bool(arb)))
        if dc == "scan":
            out.add(("dc_local", src))
    return out


def _instantiated():
    """Every front-end kernel instantiation in frontend_host.hpp, read from the source."""
    txt = open(os.path.join(os.path.dirname(__file__), "..", "sdr_pmr446_b200", "csrc", "frontend_host.hpp")).read()
    body = txt[txt.index("inline cascade_fn pick_cascade"):txt.index("#undef PMR_GROUPS")]
    groups = [tuple(int(v) for v in g if v != "0") for g in re.findall(r"if \(is\((\d+), (\d+), (\d+), (\d+)\)\) return cfn<SRC, DC,", body)]
    out = set()
    for dc, src in re.findall(r"if \(dc == DC_(\w+) && src == SRC_(\w+)\) \{ PMR_GROUPS\(", body):
        out |= {("cascade", src.lower(), dc.lower(), g, False) for g in groups}
    for dc, src, *g in re.findall(r"if \(dc == DC_(\w+) && src == SRC_(\w+) && is\((\d+), (\d+), (\d+), (\d+)\)\)", body):
        out.add(("cascade", src.lower(), dc.lower(), tuple(int(v) for v in g if v != "0"), True))
    out |= {("front6", int(a), int(b)) for a, b in re.findall(r"front6_kernel<(\d+), (\d+)><<<", txt)}
    out |= {("dc_local", s.lower()) for s in re.findall(r"dc_local_kernel<SRC_(\w+)><<<", txt)}
    if "fused_frontend_kernel<<<" in txt:
        out.add(("fused",))
    if "hbarb_tile_kernel<10, 2, 3><<<" in txt:
        out.add(("tile",))
    return out


def test_cases_reach_every_frontend_kernel():
    """The case list reaches every front-end kernel that some rate selects, and the instantiations no rate selects are
    exactly the known ones: a group that becomes reachable, or a new instantiation, fails here until it has a case."""
    inst = _instantiated()
    assert len(inst) > 40
    reach = set()
    rates = sorted(set(np.exp(np.linspace(np.log(1e-4), 0.0, 600)).tolist() + [_rate(c[1], c[3]) for c in FE_CASES + SHIM_CASES]))
    for r in rates:
        for fmt in (CU8, CF32, CS16, CS8):
            reach |= _kernels(describe_frontend(r, fmt, 1), fmt, True)
        reach |= _kernels(describe_frontend(r, CF32, 0), CF32, False)
    assert reach <= inst, reach - inst
    # the half-band list of a decimating plan is 3, ..., 3, 5, 10 in execution order and the last stage goes with the
    # resampler unless the plan is [5, 10] with a non-periodic phase or a single stage: a lone [3] is never cut, and a ring
    # never feeds [5, 10] or [10] without the resampler
    unreachable = {("cascade", s, d, (3,), False) for s, d in (("cu8", "zsr"), ("cf32", "zsr"), ("cs16", "zsr"), ("cs8", "zsr"),
                                                               ("cf32", "none"), ("ring", "none"))}
    unreachable |= {("cascade", "ring", "none", (5, 10), False), ("cascade", "ring", "none", (10,), False)}
    assert inst - reach == unreachable, (inst - reach) ^ unreachable
    covered = set()
    for c in FE_CASES + SHIM_CASES:
        covered |= _kernels(_plan(c), c[2], c[0] != "shim")
    assert covered == reach, reach - covered


def test_case_plans():
    """The plan strings the case list was chosen for."""
    want = {("batch", 2400000, CU8, 200000): "fused[3,5,10]+arb", ("batch", 2400000, CS16, 200000): "cascade[3,5] | tile[10]+arb",
            ("batch", 1024000, CS8, 200000): "cascade[5,10] | cascade[]+arb",
            ("batch", 3200000, CF32, 200000): "cascade[3,5] | cascade[10]+arb",
            ("batch", 4800000, CU8, 200000): "cascade[3,3] | cascade[5] | tile[10]+arb",
            ("batch", 6400000, CF32, 200000): "cascade[3,3] | cascade[5] | cascade[10]+arb",
            ("batch", 9600000, CF32, 200000): "cascade[3,3] | cascade[3,5] | tile[10]+arb",
            ("batch", 20000000, CF32, 200000): "cascade[3,3,3,3] | cascade[5] | cascade[10]+arb",
            ("batch", 20000000, CU8, 200000): "front6[3,3,3,3,5,10] | cascade[]+arb",
            ("batch", 500000, CU8, 200000): "cascade[10] | cascade[]+arb", ("batch", 250000, CS8, 200000): "cascade[]+arb",
            ("dsd", 2400000, CU8, 12500): "front6[3,3,3,3,3,5] | tile[10]+arb",
            ("dsd", 2400000, CF32, 12500): "cascade[3,3,3,3] | cascade[3,5] | tile[10]+arb",
            ("dsd", 20000000, CU8, 12500): "cascade[3,3,3,3] | cascade[3,3,3,3] | cascade[5] | cascade[10]+arb"}
    for c, p in want.items():
        assert c in FE_CASES and _plan(c) == p, (c, _plan(c))


# ---- captures, calls, references ----------------------------------------------------------------------------------------
def _capture(fs, fmt, n, seed, dc_scale=1.0, dsd=False):
    from sdr_pmr446_b200 import synth
    if dsd:   # dsd_in: one carrier at 0 Hz
        spec = synth.CaptureSpec(fs=float(fs), carriers=(synth.Carrier(1, 0.3, 1000.0 + 150.0 * (seed % 3), 0.0),),
                                 offset_hz=-synth.channel_offset_hz(1))
    else:
        spec = synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(seed))
    spec.dc = spec.dc * dc_scale
    return {CU8: synth.make_cu8, CF32: synth.make_cf32, CS16: synth.make_cs16, CS8: synth.make_cs8}[fmt](spec, n, seed)


def _captures(fs, fmt, n, seed0, streams=S, dc_scale=1.0, dsd=False):
    return np.stack([_capture(fs, fmt, n, seed0 + s, dc_scale, dsd) for s in range(streams)])


# awkward calls: empty, 1 and 7 samples, shorter than a 48-sample fused iteration, not multiples of 16, one off the fused
# kernel's 1536 / 6144-sample segments and off 4096
EDGE_SIZES = [0, 1, 7, 47, 49, 333, 1535, 1537, 4095, 4097, 6143, 6145, 0, 15]


def _sizes(n):
    head = (n - sum(EDGE_SIZES)) // 2 + 5
    sizes = [head] + EDGE_SIZES
    sizes.append(n - sum(sizes))
    assert min(sizes) >= 0 and sum(sizes) == n
    return sizes


def _calls(run, iq, sizes, bps):
    parts, o = [], 0
    for k in sizes:
        parts.append(run(iq[:, o * bps:(o + k) * bps]))
        o += k
    return parts


def _cat(parts, k):
    return np.concatenate([p[k] for p in parts], axis=-1)


def _ref(iq, fmt, fs_in, fs_out, with_dc=True):
    return stage_ref.front_end(iq, fmt, design_msresamp(_rate(fs_in, fs_out)), ALPHA, with_dc)


def _check_streams(res, iq, fmt, fs_in, fs_out, streams, label, with_dc=True, tol_scale=1.0):
    rms = worst = 0.0
    for s in streams:
        r, w = stage_ref.check_res(res[s], _ref(iq[s], fmt, fs_in, fs_out, with_dc), tol_scale * FE_TOL_RMS, tol_scale * FE_TOL_MAX)
        rms, worst = max(rms, r), max(worst, w)
    print("MEASURED fe %s: res %.3g rel rms, %.3g of rms worst sample" % (label, rms, worst))
    return rms, worst


def _run_batch(iq, fmt, fs, sizes, want=("res",)):
    from sdr_pmr446_b200 import chain
    b = chain.PmrBatch(n_streams=iq.shape[0], fs_in=fs, in_fmt=fmt, max_chunk=max(sizes))
    parts = _calls(lambda x: b.execute(x, want=want), iq, sizes, BPS[fmt])
    b.close()
    return parts


def _run_dsd(iq, fmt, fs, sizes):
    from sdr_pmr446_b200 import chain
    b = chain.DsdBatch(n_streams=iq.shape[0], fs_in=fs, in_fmt=fmt, max_chunk=max(sizes))
    parts = _calls(b.execute, iq, sizes, BPS[fmt])
    b.close()
    return parts


# ---- every plan shape x every source ------------------------------------------------------------------------------------
@GPU
@pytest.mark.parametrize("case", FE_CASES, ids=_case_id)
def test_frontend_plan(case):
    chain_name, fs, fmt, fs_out = case
    n = max(fs // 10, 120000)
    iq = _captures(fs, fmt, n, 700 + 10 * fmt, dsd=chain_name == "dsd")
    sizes = _sizes(n)
    parts = (_run_dsd if chain_name == "dsd" else _run_batch)(iq, fmt, fs, sizes)
    _check_streams(_cat(parts, "res"), iq, fmt, fs, fs_out, range(S), _case_id(case))


@GPU
@pytest.mark.parametrize("case", [("batch", 2400000, CU8, 200000), ("batch", 1024000, CU8, 200000), ("batch", 20000000, CF32, 200000),
                                  ("batch", 250000, CF32, 200000), ("batch", 500000, CS16, 200000), ("dsd", 2400000, CU8, 12500)],
                         ids=_case_id)
def test_frontend_large_dc(case):
    """A DC offset ten times the default: the DC blocker's zero-input correction (E table, rho powers, v_seg) then carries
    real weight in every segment.  The blocker's state v ~ DC / alpha is ten times larger and so is its float32 rounding
    (the oracle's own error grows from 1.6e-6 to 1.5e-5 relative RMS at 2.4 Msps cu8; the GPU's from at most 2.9e-7 to
    5.1e-7 on a B200): the bounds are doubled."""
    chain_name, fs, fmt, fs_out = case
    n = max(fs // 10, 120000)
    iq = _captures(fs, fmt, n, 760, dc_scale=10.0, dsd=chain_name == "dsd")
    parts = (_run_dsd if chain_name == "dsd" else _run_batch)(iq, fmt, fs, _sizes(n))
    _check_streams(_cat(parts, "res"), iq, fmt, fs, fs_out, range(S), "dc x10 " + _case_id(case), tol_scale=2.0)


# ---- the bench shape ----------------------------------------------------------------------------------------------------
@GPU
def test_frontend_bench_shape():
    """2.4 Msps cu8, 1024 streams, a 240 000-sample call and then uneven ones: the only shape that gets the fused kernel's
    6144-sample segments (small batches get 1536) and the most segments per dc_scan_kernel.  The batch repeats 4 captures:
    streams with the same input must give bitwise the same res."""
    fs, streams, distinct = 2400000, 1024, 4
    sizes = [240000, 0, 1, 7, 47, 6143, 6145, 3001, 1535]
    caps = _captures(fs, CU8, sum(sizes), 780, streams=distinct)
    iq = np.tile(caps, (streams // distinct, 1))
    res = _cat(_run_batch(iq, CU8, fs, sizes), "res")
    for s in range(distinct, streams):
        assert np.array_equal(res[s].view(np.uint64), res[s % distinct].view(np.uint64)), s
    picks = (0, streams // 2 + 1, streams - 1)
    _check_streams(res[list(picks)], iq[list(picks)], CU8, fs, 200000, range(3), "bench shape 1024 x 2.4 Msps cu8 " + _case_id(
        ("batch", fs, CU8, 200000)))


@GPU
def test_frontend_dc_scan_block():
    """Few streams with more than 128 DC segments in one call: dc_scan_block_kernel (rate 1.0, DC_SCAN, a 2 M-sample call),
    and dc_scan_kernel for the short calls after it."""
    fs, fmt = 200000, CF32
    sizes = [2000000, 1, 7, 4097, 333]
    iq = _captures(fs, fmt, sum(sizes), 790)
    res = _cat(_run_batch(iq, fmt, fs, sizes), "res")
    _check_streams(res, iq, fmt, fs, 200000, range(S), "dc_scan_block " + _case_id(("batch", fs, fmt, 200000)))


# ---- deferred zero-input correction -------------------------------------------------------------------------------------
@GPU
@pytest.mark.parametrize("dc_scale", [1.0, 10.0])
def test_deferred_correction_in_channelizer(dc_scale):
    """Without `res` the fused front end leaves the DC blocker's zero-input correction to channelize16_kernel's staging;
    with `res` it is applied in place.  Both channel outputs must be bitwise equal (the same float32 operations in the
    same order), and match the float64 channelizer of the float64 front end within the composed bound."""
    fs, fmt, M = 2400000, CU8, 16
    n = 480000
    iq = _captures(fs, fmt, n, 800, dc_scale=dc_scale)
    sizes = _sizes(n)
    a = _run_batch(iq, fmt, fs, sizes, want=("res", "chan"))
    b = _run_batch(iq, fmt, fs, sizes, want=("chan",))
    chan_a, chan_b = _cat(a, "chan"), _cat(b, "chan")
    taps, dtheta = design_pfbch(M), design_dtheta(M)
    assert np.array_equal(chan_a.view(np.uint64), chan_b.view(np.uint64))
    worst_64 = 0.0
    for s in range(S):
        ref, _ = stage_ref.channelize(_ref(iq[s], fmt, fs, 200000), M, taps, dtheta, 0.5)
        worst_64 = max(worst_64, stage_ref.check_chan(chan_b[s], ref, CHAN_TOL_CH, CHAN_TOL_STAGE + FE_TOL_RMS))
    print("MEASURED fe deferred correction dc x%g: chan bitwise equal to in-place, vs float64 %.3g of bound" % (dc_scale, worst_64))


# ---- dsd_in back end ----------------------------------------------------------------------------------------------------
def _dsd_sizes(fs, n):
    """Calls that give the back end no input, one input sample, a few (fewer than 48 outputs) and many (more than 1536)."""
    from sdr_pmr446_b200._lib import lib
    rate = np.float32(_rate(fs, 12500))
    sizes = [n // 3 + 11, 0, 7]

    def shortest(want):   # the shortest call from the current position that gives `want` res samples
        pos, k = sum(sizes), 1
        while lib().pmr446_count_resampled(rate, 60.0, pos + k) - lib().pmr446_count_resampled(rate, 60.0, pos) < want:
            k += 1
        return k
    sizes.append(shortest(1))
    sizes.append(shortest(9))
    sizes.append(n - sum(sizes))
    return sizes


@GPU
@pytest.mark.parametrize("fs,fmt", [(2400000, CU8), (1024000, CU8), (1024000, CF32), (2400000, CS16)])
def test_dsd_backend(fs, fmt):
    """dsd_in: res against the float64 front end, fm against the float64 discriminator of the GPU's res, audio against
    msresamp_rrrf x 3.84 in float64 of the GPU's fm (dsd_backend_kernel's tiles and the 19 recomputed outputs in front of a
    block), pcm against the s16 cast of that audio."""
    n = 600000
    iq = _captures(fs, fmt, n, 820 + fmt, dsd=True)
    sizes = _dsd_sizes(fs, n)
    parts = _run_dsd(iq, fmt, fs, sizes)
    ny, nz = [p["ny"] for p in parts], [p["nz"] for p in parts]
    assert 1 in ny and 0 in nz and max(nz) > 1536 and any(0 < z < 48 for z in nz), (ny, nz)
    res, fm, audio, pcm = (_cat(parts, k) for k in ("res", "fm", "audio", "pcm"))
    _check_streams(res, iq, fmt, fs, 12500, range(S), "dsd %s %g Msps %s" % (FMT_NAME[fmt], fs / 1e6, _plan(("dsd", fs, fmt, 12500))))
    up = design_msresamp(_rate(12500, 48000))
    fm_err = rms = worst = 0.0
    for s in range(S):
        own = stage_ref.discriminator(res[s], 0.5)
        d = np.abs(stage_ref.wrapped((fm[s].astype(np.float64) - own) * np.pi))[1:]
        fm_err = max(fm_err, float(d.max()))
        assert fm_err < DSD_FM_TOL_RAD, fm_err
        au = stage_ref.msresamp_interp_real(fm[s], up)
        r, w = stage_ref.check_res(audio[s], au, DSD_AUDIO_TOL_RMS, DSD_AUDIO_TOL_MAX)
        rms, worst = max(rms, r), max(worst, w)
        inside = np.abs(au) < 0.999
        assert np.mean(inside) > 0.95
        stage_ref.check_pcm(pcm[s][inside], au[inside], float(np.max(np.abs(audio[s] - au))))
    print("MEASURED dsd backend %s %g Msps: fm %.3g rad, audio %.3g rel rms, %.3g of rms worst sample, calls nz=%s"
          % (FMT_NAME[fmt], fs / 1e6, fm_err, rms, worst, nz[:8]))


# ---- liquid shim --------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _shim():
    import ctypes as C

    import liquid_api
    from sdr_pmr446_b200 import _lib
    return liquid_api.bind(C.CDLL(_lib.LIB_PATH))


@GPU
@pytest.mark.parametrize("case", SHIM_CASES, ids=_case_id)
def test_shim_msresamp_crcf(case):
    """msresamp_crcf on the shim (cf32, DC_NONE groups, no DC blocker) in uneven blocks against the float64 msresamp."""
    import ctypes as C
    _, fs, fmt, fs_out = case
    L = _shim()
    n = max(fs // 10, 120000)
    x = _capture(fs, CF32, n, 840)
    q = L.msresamp_crcf_create(np.float32(_rate(fs, fs_out)), 60.0)
    assert q
    ys, o = [], 0
    for k in _sizes(n):
        blk = np.ascontiguousarray(x[o:o + k])
        y = np.zeros(k + 16, np.complex64)
        ny = C.c_uint()
        assert L.msresamp_crcf_execute(q, blk.ctypes.data, k, y.ctypes.data, C.byref(ny)) == 0
        ys.append(y[:ny.value])
        o += k
    L.msresamp_crcf_destroy(q)
    _check_streams(np.concatenate(ys)[None], x[None], CF32, fs, fs_out, range(1), _case_id(case), with_dc=False)


@GPU
def test_shim_msresamp_rrrf():
    """msresamp_rrrf x 3.84 on the shim (dsd_arb_kernel / dsd_interp_kernel) in uneven blocks against the float64 msresamp."""
    import ctypes as C
    L = _shim()
    rng = np.random.default_rng(850)
    n = 60000
    x = (0.4 * np.sin(2 * np.pi * 1000.0 / 12500.0 * np.arange(n)) + 0.05 * rng.standard_normal(n)).astype(np.float32)
    q = L.msresamp_rrrf_create(np.float32(48000.0 / 12500.0), 60.0)
    assert q
    ys, o = [], 0
    for k in [0, 1, 7, 12, 1000, 47, 4097, 1] + [n - 5165]:
        blk = np.ascontiguousarray(x[o:o + k])
        y = np.zeros(4 * k + 16, np.float32)
        ny = C.c_uint()
        assert L.msresamp_rrrf_execute(q, blk.ctypes.data, k, y.ctypes.data, C.byref(ny)) == 0
        ys.append(y[:ny.value])
        o += k
    assert o == n
    L.msresamp_rrrf_destroy(q)
    r, w = stage_ref.check_res(np.concatenate(ys), stage_ref.msresamp_interp_real(x, design_msresamp(_rate(12500, 48000))),
                               DSD_AUDIO_TOL_RMS, DSD_AUDIO_TOL_MAX)
    print("MEASURED shim msresamp_rrrf x3.84: %.3g rel rms, %.3g of rms worst sample" % (r, w))
