#!/usr/bin/env python3
"""Speed of the four input formats (cu8, cf32, cs16, cs8) on the same synthetic signal: the batch chain (16 channels ->
s16) at 1024 x 1.024 Msps and 1024 x 2.4 Msps, and dsd_in at 1024 x 2.4 Msps.  For each, two numbers:

  device_ms   ms per step with the input already on the GPU (pmr446_batch_execute_device / dsd446_batch_execute_device);
  e2e_msps    Msamples/s through the host-buffer call (pmr446_batch_execute / dsd446_batch_execute) from pinned memory,
              i.e. including the host -> device copy of 2 (cu8, cs8), 4 (cs16) or 8 (cf32) bytes per sample.

Formats alternate within each round so that a drift of the clocks or of the shared host hits all of them alike.
Every input is larger than the 126 MB L2.  Prints the GPU's name, power limit and maximum SM clock with the numbers as one
JSON object.  usage: bench_formats.py [--rounds R] [--steps K] [--warmup W]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sdr_pmr446_b200 import _lib, chain, synth

FORMATS = (("cu8", _lib.FMT_CU8), ("cf32", _lib.FMT_CF32), ("cs16", _lib.FMT_CS16), ("cs8", _lib.FMT_CS8))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3] if q.returncode == 0 else (torch.cuda.get_device_name(), "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def inputs(fs, S, n):
    """The same capture in every format, tiled over S streams: pinned host copies and device copies ([S, row] uint8)."""
    x = synth.make_cf64(synth.CaptureSpec(fs=float(fs)), n, 446)
    rows = {"cu8": synth.to_cu8(x), "cf32": x.astype(np.complex64), "cs16": synth.to_cs16(x), "cs8": synth.to_cs8(x)}
    out = {}
    for name, row in rows.items():
        b = torch.from_numpy(np.ascontiguousarray(row).view(np.uint8))
        host = torch.empty((S, b.numel()), dtype=torch.uint8, pin_memory=True)
        host.copy_(b.unsqueeze(0).expand(S, -1))
        out[name] = (host, host.cuda())
    return out


def measure(make, host, dev, n, steps, warmup):
    obj = make()
    if isinstance(obj, chain.DsdBatch):
        pcm = torch.empty((obj.S, obj.max_out), dtype=torch.int16, device="cuda")
        dev_step = lambda: obj.execute_device(dev, n, pcm=pcm)  # noqa: E731
        pcm_h = torch.empty((obj.S, obj.max_out), dtype=torch.int16, pin_memory=True).numpy()
        o = _lib.DsdOutputs(None, None, obj.max_res, None, pcm_h.ctypes.data, obj.max_out)
        call = lambda ptr, stride: _lib.lib().dsd446_batch_execute(obj.h, ptr, stride, n, C.byref(o), None, None)  # noqa: E731
    else:
        pcm = torch.empty((obj.S, obj.M, obj.max_ns), dtype=torch.int16, device="cuda")
        dev_step = lambda: obj.execute_device(dev, n, {"pcm": pcm, "ld": obj.max_ns})  # noqa: E731
        pcm_h = torch.empty((obj.S, obj.M, obj.max_ns), dtype=torch.int16, pin_memory=True).numpy()
        o = _lib.Outputs()
        o.ld, o.res_ld, o.pcm = obj.max_ns, obj.max_res, pcm_h.ctypes.data
        call = lambda ptr, stride: _lib.lib().pmr446_batch_execute(obj.h, ptr, stride, n, C.byref(o), None, None)  # noqa: E731
    for _ in range(warmup):
        dev_step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        dev_step()
    e1.record()
    torch.cuda.synchronize()
    device_ms = e0.elapsed_time(e1) / steps
    hp, hs = host.data_ptr(), host.stride(0)
    for _ in range(warmup):
        _lib.check(call(hp, hs), "execute")
    t0 = time.perf_counter()
    for _ in range(steps):
        _lib.check(call(hp, hs), "execute")
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / steps
    S = obj.S
    obj.close()
    return {"device_ms": round(device_ms, 4), "device_msps": round(S * n / device_ms / 1e3, 1), "e2e_ms": round(e2e_s * 1e3, 3),
            "e2e_msps": round(S * n / e2e_s / 1e6, 1), "h2d_gb_per_step": round(host.numel() / 1e9, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--streams", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_formats.py needs a CUDA device")
    S = args.streams
    # samples per stream per step: at least 2^19, so that the host-buffer call of the batch chain overlaps its copy with the kernels
    workloads = [("pmr_1024k", 1024000, 524288, "pmr"), ("pmr_2400k", 2400000, 600000, "pmr"), ("dsd_2400k", 2400000, 600000, "dsd")]
    result = dict(gpu_info(), streams=S, steps=args.steps, rounds=args.rounds, workloads={})
    for wname, fs, n, kind in workloads:
        data = inputs(fs, S, n)
        runs = {f: [] for f, _ in FORMATS}
        for _ in range(args.rounds):
            for f, code in FORMATS:
                if kind == "pmr":
                    make = lambda: chain.PmrBatch(n_streams=S, fs_in=fs, in_fmt=code, audio_gain=1.0, max_chunk=n)  # noqa: E731
                else:
                    make = lambda: chain.DsdBatch(n_streams=S, fs_in=fs, in_fmt=code, max_chunk=n)  # noqa: E731
                runs[f].append(measure(make, data[f][0], data[f][1], n, args.steps, args.warmup))
        result["workloads"][wname] = {"fs_in": fs, "samples_per_stream_per_step": n, "runs": runs}
        del data
        torch.cuda.empty_cache()
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
