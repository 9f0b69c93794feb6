#!/usr/bin/env python3
"""Cost of the batch chain's per-channel DSD feed (dsd_pcm, dsd_backend_kernel) at the benchmark's shapes, device-resident input:

  bench   1024 streams x 2.4 Msps cu8, 16 channels, 1 s steps (the flagship workload)
  cfg4    4 streams x 20 Msps cf32, 1600 channels, 0.1 s steps

Within each round it measures, alternately: the step without the feed (pcm only), the step with dsd_pcm as well, and the
kernel time of the feed from timing tag 10 ("dsd").  The feed's floors are computed from the shapes: 34 FMA per resampler
output z (14 taps of the arbitrary stage, 20 of the half-band) at the FP32 FMA rate pmr446_measure_fp32_peak measures on this
GPU, and the discriminator ring read once (4 bytes per frame per row) plus the s16 written (4 bytes per z per row) at 6.5 TB/s.
Every input is larger than the 126 MB L2.  Prints the GPU's name, power limit and maximum SM clock with the numbers as one
JSON object.  usage: bench_dsd_tap.py [--rounds R] [--steps K] [--warmup W]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sdr_pmr446_b200 import chain, synth
from tools.bench_formats import gpu_info

HBM_TBPS = 6.5
WORKLOADS = (("bench", dict(S=1024, fs=2400000, fmt=1, M=16, n=2400000)),
             ("cfg4", dict(S=4, fs=20000000, fmt=0, M=1600, n=2000000)))


def device_input(fs, fmt, S, n):
    x = synth.make_cf64(synth.CaptureSpec(fs=float(fs)), n, 446)
    row = synth.to_cu8(x) if fmt == 1 else x.astype(np.complex64)
    b = torch.from_numpy(np.ascontiguousarray(row).view(np.uint8)).cuda()
    return b.unsqueeze(0).expand(S, -1).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_dsd_tap.py needs a CUDA device")
    peak = chain.measure_fp32_peak()
    result = dict(gpu_info(), fp32_peak_tflops=round(peak, 1), hbm_tbps_floor=HBM_TBPS, rounds=args.rounds, steps=args.steps, workloads={})
    for name, w in WORKLOADS:
        S, M, n = w["S"], w["M"], w["n"]
        iq = device_input(w["fs"], w["fmt"], S, n)
        b = chain.PmrBatch(n_streams=S, fs_in=w["fs"], in_fmt=w["fmt"], num_channels=M, audio_gain=1.0, max_chunk=n, dsd_rate=48000)
        pcm = torch.empty((S, M, b.max_ns), dtype=torch.int16, device="cuda")
        dsd = torch.empty((S, M, b.max_dsd), dtype=torch.int16, device="cuda")
        arms = {"without": {"pcm": pcm}, "with_dsd_pcm": {"pcm": pcm, "dsd_pcm": dsd}}
        runs = {a: [] for a in arms}
        kernel_ms, z_per_row, frames_per_row = [], 0, 0
        for a in arms:
            for _ in range(args.warmup):
                b.execute_device(iq, n, arms[a])
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for a, outs in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    _, ns = b.execute_device(iq, n, outs)
                e1.record()
                torch.cuda.synchronize()
                runs[a].append(round(e0.elapsed_time(e1) / args.steps, 4))
            b.timing(True)
            for _ in range(args.steps):
                _, ns = b.execute_device(iq, n, arms["with_dsd_pcm"])
                z_per_row, frames_per_row = b.last_dsd // 2, ns
            t = b.get_timings()
            b.timing(False)
            kernel_ms.append(round(t["dsd"][0] / t["dsd"][1], 4))
        b.close()
        del iq
        torch.cuda.empty_cache()
        rows = S * M
        z = rows * z_per_row
        flop = 2.0 * 34 * z
        nbytes = 4.0 * rows * frames_per_row + 4.0 * z
        t_flop, t_mem = flop / (peak * 1e12) * 1e3, nbytes / (HBM_TBPS * 1e12) * 1e3
        best = min(kernel_ms)
        result["workloads"][name] = {
            "streams": S, "channels": M, "fs_in": w["fs"], "samples_per_stream_per_step": n, "rows": rows,
            "z_per_row_per_step": z_per_row, "dsd_pcm_per_row_per_step": 2 * z_per_row,
            "step_ms_without": runs["without"], "step_ms_with_dsd_pcm": runs["with_dsd_pcm"], "dsd_kernel_ms": kernel_ms,
            "flop_floor_ms": round(t_flop, 4), "bytes_floor_ms": round(t_mem, 4),
            "achieved_fraction_of_flop_floor": round(t_flop / best, 3), "achieved_fraction_of_bytes_floor": round(t_mem / best, 3),
            "achieved_tflops": round(flop / (best * 1e-3) / 1e12, 2), "achieved_tbps": round(nbytes / (best * 1e-3) / 1e12, 3)}
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
