#!/usr/bin/env python3
"""Benchmark of the PMR446 receive chain on B200 (BASELINE.json metric: IQ Msamples/s through the
full chain + roofline fraction).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[2]; configs[4] is the same shard per GPU at N = 8): a batch of
STREAMS = 1024 independent 2.4 Msps cu8 PMR446 captures per GPU, all 16 channels demodulated to s16
audio.  One step = one second of signal of every stream (2.4 M samples x 1024 streams = 2.46 G
samples, 4.9 GB of input per GPU -- far larger than the 126 MB L2, so no L2 flush is needed between
steps).  Filter state carries from step to step exactly as in streaming use.

  value     device-resident throughput: inputs already in HBM, s16 audio left in HBM; K steps timed with
            CUDA events on the launch stream between barriers, max over ranks.
  e2e       K more steps through the host-buffer C-ABI call pmr446_batch_execute(): pinned host IQ
            -> H2D -> chain -> D2H of the s16 audio, copies inside the timed region.
  roofline  the kernel with the longest launch, timed live with CUDA events inside the timed steps: algorithmic
            bytes / measured HBM peak and algorithmic flop / measured FP32 FFMA peak, reported for the roofline that
            binds (the larger fraction); "kernels" carries the same numbers for every launch of the step.
  cpu_baseline  the CPU oracle (port of the reference chain, all 16 channels) on all host cores.

--impl reference times the reference's CPU chain (the oracle port -- the reference itself cannot be
built here, see DESIGN.md) on the host cores with the same config/metric.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned as DIR/<name>.npy in float32
(see dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FS = 2400000
CHUNK = 2400000            # one second of signal per step
STREAMS = int(os.environ.get("PMR446_BENCH_STREAMS", "1024"))
METRIC = "IQ Msamples/s through full PMR446 chain"
UNIT = "Msamples/s"
# SURVEY.md 8d: algorithmic work of the 2.4 Msps / 16-channel chain
FLOP_PER_SAMPLE = 122.1
BYTES_PER_SAMPLE = 2.17
# per kernel launch: algorithmic flop and HBM bytes per INPUT sample (SURVEY.md 8d table, 2.4 Msps column, divided
# by 2.4e6; direct-form FIR counts = the CREDIT; bytes = what the launch must read + write once), and what it replaces.
# The EXECUTED flop of the same launch (ncu source page, tools/ncu_kernel_report.py -> profiles/kernel_exec.json) is
# reported beside the credit: the audio kernel executes ~10x fewer flop than the direct-form count it is credited with.
KERNELS_FUSED = {
    "cascade0": {"what": "fused_frontend_kernel: cu8 load, DC blocker, half-bands m=3, 5, 10 and the 14-tap x2/3 resampler in one pass "
                         "-> 200 kHz ring (no intermediate ring)",
                 "flop": (19.2 + 31.2 + 25.2 + 24.6 + 11.2) / 2.4, "bytes": 2.0 + 0.2e6 * 8 / 2.4e6},
    "channelize": {"what": "channelize16_kernel: DC zero-input correction, NCO mix, 16 x 26-tap polyphase bank, 16-point DFT, FM discriminator",
                   "flop": (1.2 + 20.8 + 4.0 + 3.8) / 2.4, "bytes": 0.2e6 * 8 / 2.4e6 + 0.2e6 * 4 / 2.4e6},
    "audio": {"what": "audio_fft4_kernel: 377-tap CTCSS high-pass FIR + gain + de-emphasis + s16 by 4096-point overlap-save, four channel rows per block "
                      "(credit = direct-form count of SURVEY 8d; see executed_*)",
              "flop": (150.8 + 1.0) / 2.4, "bytes": 0.2e6 * 4 / 2.4e6 + 0.2e6 * 2 / 2.4e6},
}
KERNELS_SPLIT = {   # PMR446_FRONTEND=split: round 1's two-launch front end
    "cascade0": {"what": "cascade_kernel<cu8, DC, m=3, m=5>: cu8 load, DC blocker, two half-band decimators -> 600 kHz ring",
                 "flop": (19.2 + 31.2 + 25.2) / 2.4, "bytes": 2.0 + 0.6e6 * 8 / 2.4e6},
    "cascade1": {"what": "hbarb_tile_kernel<10, 2, 3>: m=10 half-band decimator + 14-tap arbitrary resampler -> 200 kHz ring",
                 "flop": (24.6 + 11.2) / 2.4, "bytes": 0.6e6 * 8 / 2.4e6 + 0.2e6 * 8 / 2.4e6},
    "channelize": KERNELS_FUSED["channelize"],
    "audio": KERNELS_FUSED["audio"],
}
WORKLOAD = "configs[2]: %d independent 2.4 Msps cu8 PMR446 captures x 16 channels per GPU, 1 s of signal per step" % STREAMS


emit = None   # set by main(): prints the one JSON line on the real stdout


def config_dict(n_gpus):
    return {"workload": WORKLOAD, "streams_per_gpu": STREAMS, "fs_in": FS, "samples_per_stream_per_step": CHUNK,
            "channels": 16, "in_fmt": "cu8", "out": "s16 audio, 16 x 12.5 kHz per stream", "parallelism": "streams sharded, %d GPU(s)" % n_gpus,
            "l2": "inputs (4.9 GB/step/GPU) larger than L2; no flush needed"}


# ------------------------------------------------------------------------------------------------
def make_base_captures(count, n):
    from sdr_pmr446_b200 import synth
    return [synth.make_cu8(synth.CaptureSpec(fs=float(FS), carriers=synth.rotated_carriers(s)), n, 446 + s) for s in range(count)]


def cpu_chain_rate(threads, seconds_of_signal, active_only=-1, last=None):
    """Oracle (CPU port of the reference chain) on `threads` host threads, one stream each.  Returns
    (Msamples/s aggregate, wall seconds); `last`, a dict, receives each thread's s16 audio of its last chunk."""
    from oracle import oracle as orc
    base = make_base_captures(min(threads, 4), CHUNK)
    objs = [orc.PmrOracle(fs_in=FS, in_fmt=1, audio_gain=1.0, chunk=CHUNK, active_only=active_only) for _ in range(threads)]

    def work(i):
        for _ in range(seconds_of_signal):
            r = objs[i].execute(base[i % len(base)], want=("pcm",))
        if last is not None:
            last[i] = r["pcm"]

    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    for o in objs:
        o.close()
    return threads * seconds_of_signal * CHUNK / dt / 1e6, dt


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, reasons = [], None, set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        top = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (top[len(top) // 2] if top else None), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
def reference_binary_rate(cores):
    """The UNMODIFIED reference program (oracle/_ref/sdr_pmr446_ref, built by `make -f oracle/ref.mk REF=<checkout>` with
    file-backed SoapySDR / RtAudio stand-ins) on `cores` processes, each on a 10 s capture at the ONE configuration it
    supports: 1.024 Msps hard-coded, one squelch-selected channel demodulated.  Informational (another config than the
    bench line); None when the binary was not built."""
    exe = os.path.join(ROOT, "oracle", "_ref", "sdr_pmr446_ref")
    if not os.path.exists(exe):
        return None
    import tempfile
    from sdr_pmr446_b200 import synth
    n = 10_240_000
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "iq.cu8")
        synth.make_cu8(synth.CaptureSpec(fs=1024000.0, carriers=synth.CFG1_CARRIERS), n, 446).tofile(path)
        env = dict(os.environ, REF_IQ=path, REF_IQ_FMT="cu8")
        t0 = time.perf_counter()
        ps = [subprocess.Popen([exe, "-a", "1.0"], env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for _ in range(cores)]
        ok = all(p.wait() == 0 for p in ps)
        dt = time.perf_counter() - t0
    if not ok:
        return None
    with open(os.path.join(ROOT, "oracle", "_ref", "LIQUID")) as f:
        dsp = f.read().strip()
    return {"value": cores * n / dt / 1e6, "unit": UNIT, "cores": cores, "config": "1.024 Msps cu8, 16 channels channelized, 1 demodulated (the reference's own operating point)",
            "dsp_objects": "liquid-dsp" if dsp == "system" else "oracle restatement of liquid-dsp (liquid-dsp is not installed)", "wall_s": dt}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    secs = 4
    vals = []
    last = {}
    for it in range(args.warmup + args.steps):
        v, dt = cpu_chain_rate(cores, secs, last=last)
        if it >= args.warmup:
            vals.append((v, dt))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pcm": np.stack([last[i] for i in range(cores)])})
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    sample = "%d host threads x %d s of one 2.4 Msps stream each per step (all 16 channels demodulated)" % (cores, secs)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_dict(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference = CPU oracle port of the liquid-dsp chain at the bench configuration (2.4 Msps, all 16 channels); the "
                    "reference's own programs compile (oracle/ref.mk) but are hard-wired to 1.024 Msps / one demodulated channel: reference_binary",
            "reference_binary": reference_binary_rate(cores)}
    emit(line)


def bind_near_gpu(local_rank):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the
    end-to-end arm are allocated next to the GPU's PCIe root (first-touch).  Returns the node or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        pass
    return None


def pcie_probe(dev, pinned_u8, reps=3):
    """Host<->device copy bandwidth of THIS rank while every rank runs the same probe (called between barriers): the
    end-to-end arm moves 4.9 GB in and 0.4 GB out per step, so this is its ceiling.  Returns (h2d GB/s, d2h GB/s)."""
    import torch
    nbytes = min(pinned_u8.numel(), 1 << 30)
    src = pinned_u8.view(-1)[:nbytes]
    dst = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = []
    for a, b in ((src, dst), (dst, src)):
        b.copy_(a, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            b.copy_(a, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        out.append(nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del dst
    return out[0], out[1]


def pcie_topology(local_rank):
    """PCIe link of this rank's GPU (generation, width, NUMA node, bus id) from nvidia-smi / sysfs, for the SCALE line."""
    info = {}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id,pcie.link.gen.current,pcie.link.width.current,pcie.link.gen.max",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout.strip().split(",")
        info = {"bus_id": q[0].strip(), "pcie_gen": int(q[1]), "pcie_width": int(q[2]), "pcie_gen_max": int(q[3])}
        bdf = info["bus_id"].lower()[-12:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            info["numa_node"] = int(f.read().strip())
    except Exception:
        pass
    return info


DUMP_STREAMS = 64   # the largest dump, 64 streams x 16 channels x 12500 samples of audio in float32, is 51 MB


def dump_outputs(out_dir, arrays):
    """Writes each array (numpy or torch, one stream per row) as out_dir/<name>.npy in float32, reduced to a fixed sample
    of DUMP_STREAMS rows drawn with seed 0, in increasing order (every row when there are fewer)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        S = a.shape[0]
        pick = np.sort(np.random.default_rng(0).choice(S, min(S, DUMP_STREAMS), replace=False))
        a = a[torch.from_numpy(pick).to(a.device)].cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)[pick]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from sdr_pmr446_b200 import chain

    torch.cuda.set_device(local_rank)
    numa_node = bind_near_gpu(local_rank) if world > 1 else None
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        dist.init_process_group("nccl", device_id=dev)

    # weak scaling (default): STREAMS per GPU.  --scaling strong: configs[4] as written, 8192 streams in total sharded
    # over the GPUs (capped at 2048 per GPU = 9.8 GB of input per step, so N = 1, 2 run 2048 per GPU and say so).
    S, n = STREAMS, CHUNK
    strong_total = None
    if args.scaling == "strong":
        strong_total = int(os.environ.get("PMR446_BENCH_TOTAL_STREAMS", "8192"))
        S = min(2048, strong_total // world)
    # synthetic captures: 8 distinct seeded captures, circularly shifted per stream
    base = make_base_captures(8, n)
    base_t = [torch.from_numpy(b) for b in base]
    iq_host = torch.empty((S, 2 * n), dtype=torch.uint8).pin_memory()
    for s in range(S):
        sh = 2 * 16 * ((s // 8) + rank * (S // 8))
        iq_host[s, :2 * n - sh] = base_t[s % 8][sh:]
        iq_host[s, 2 * n - sh:] = base_t[s % 8][:sh]
    iq_dev = iq_host.to(dev, non_blocking=True)
    batch = chain.PmrBatch(n_streams=S, device=local_rank, fs_in=FS, in_fmt=1, audio_gain=1.0, max_chunk=n)
    ld = batch.max_ns
    pcm_dev = torch.empty((S, 16, ld), dtype=torch.int16, device=dev)
    outs = {"pcm": pcm_dev, "ld": ld}
    torch.cuda.synchronize()
    fp32_peak = chain.measure_fp32_peak()

    def barrier():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm ("value") ----------------
    launches = 0
    ns = 0
    # ranks finish their set-up (synthetic captures, pinned buffers) seconds apart: meet BEFORE the warm-up, so that no GPU sits idle --
    # and drops its clocks -- between its warm-up steps and the timed region (seen at 8 GPUs: three ranks at 4.2-4.4 ms, five at 4.10)
    barrier()
    for _ in range(args.warmup):
        batch.execute_device(iq_dev, n, outs)
    batch.timing(True)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        _, ns = batch.execute_device(iq_dev, n, outs)
        launches += batch.last_launches
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    timings = batch.get_timings()
    batch.timing(False)
    checksum = int(pcm_dev[:, :, :12500].to(torch.int64).abs().sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pcm": pcm_dev[:, :, :ns]})

    # ---------------- PCIe probe: what the end-to-end arm can at best reach on this rank, all ranks copying at once ----
    barrier()
    h2d_gbs, d2h_gbs = pcie_probe(dev, iq_host)
    barrier()
    topo = pcie_topology(local_rank)
    # ---------------- end-to-end arm ("e2e"): host buffers through the C ABI ----------------
    pcm_host = np.zeros((S, 16, ld), np.int16)
    pcm_host_t = torch.from_numpy(pcm_host).pin_memory()
    pcm_host = pcm_host_t.numpy()
    iq_np = iq_host.numpy()
    import ctypes as C
    from sdr_pmr446_b200._lib import Outputs, check, lib
    o = Outputs()
    o.ld, o.res_ld, o.pcm = ld, batch.max_res, pcm_host.ctypes.data
    ny, ns = C.c_uint(0), C.c_uint(0)
    e2e_steps = args.steps

    def e2e_step():
        check(lib().pmr446_batch_execute(batch.h, iq_np.ctypes.data, iq_np.strides[0], n, C.byref(o), C.byref(ny), C.byref(ns)),
              "pmr446_batch_execute")

    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_ns = ns.value
    clocks = sampler.stop()   # sampled across both timed regions

    # ---------------- reduce over ranks ----------------
    # NCCL is used for statistics only; the data path has no collective (streams are independent)
    from sdr_pmr446_b200 import shard
    rank_stats = shard.gather_stats({"samples": float(S) * n * args.steps, "elapsed_ms": ms_total, "e2e_ms": e2e_s * 1e3,
                                     "checksum": float(checksum % (1 << 40)), "sm_mhz": float(clocks.get("sm_mhz") or 0),
                                     "h2d_gbs_all_ranks_copying": h2d_gbs, "d2h_gbs_all_ranks_copying": d2h_gbs,
                                     "e2e_input_gbs": float(S) * n * 2 * e2e_steps / e2e_s / 1e9,
                                     "pcie_gen": float(topo.get("pcie_gen", 0)), "pcie_width": float(topo.get("pcie_width", 0)),
                                     "numa_node": float(topo.get("numa_node", -1))}, device=dev)
    ms_total = shard.max_over_ranks(ms_total, device=dev)
    e2e_ms = shard.max_over_ranks(e2e_s * 1e3, device=dev)
    total_samples = float(world) * S * n * args.steps
    value = total_samples / (ms_total * 1e-3) / 1e6
    e2e_value = float(world) * S * n * e2e_steps / (e2e_ms * 1e-3) / 1e6

    if rank == 0:
        peaks, peak_src = measured_peaks()
        step_ms = ms_total / args.steps
        shares = {k: round(v[0] / max(v[1], 1) / step_ms, 4) for k, v in timings.items()}
        hbm_peak = peaks.get("hbm_gbs")
        traffic_all, exec_all = {}, {}
        for fn, dst in (("kernel_traffic.json", traffic_all), ("kernel_exec.json", exec_all)):
            tpath = os.path.join(ROOT, "profiles", fn)
            if os.path.exists(tpath):
                with open(tpath) as f:
                    dst.update(json.load(f))
        split = "cascade1" in timings
        KERNELS = KERNELS_SPLIT if split else KERNELS_FUSED
        if split:
            traffic_all = traffic_all.get("_r01_split", {})
            exec_all = {}
        per_kernel = {}
        exec_total = 0.0
        for name, k in KERNELS.items():
            ms, cnt = timings.get(name, (0.0, 0))
            if not cnt:
                continue
            avg = ms / cnt                                  # one launch = one step's samples of this rank
            tf = k["flop"] * float(S) * n / (avg * 1e-3) / 1e12
            gbs = k["bytes"] * float(S) * n / (avg * 1e-3) / 1e9
            per_kernel[name] = {"avg_launch_ms": avg, "share_of_step": shares.get(name), "credited_tflops": tf, "credited_fp32_frac": tf / fp32_peak,
                                "gbs": gbs, "hbm_frac": gbs / hbm_peak}
            ex = exec_all.get(name)
            if ex:   # executed flop of one launch at 1024 streams, from the committed ncu capture
                ef = ex["executed_flop_per_launch"] * (float(S) / 1024.0)
                exec_total += ef
                per_kernel[name].update({"executed_tflops": ef / (avg * 1e-3) / 1e12, "executed_fp32_frac": ef / (avg * 1e-3) / 1e12 / fp32_peak,
                                         "ncu_fma_pipe_active_pct": ex.get("fma_pipe_active_pct"), "ncu_issue_active_pct": ex.get("issue_active_pct"),
                                         "executed_source": ex.get("source")})
        dom = max(per_kernel, key=lambda q: per_kernel[q]["avg_launch_ms"])
        dk = per_kernel[dom]
        # the dominant launch is graded on EXECUTED flop when the capture exists (never above the credit), else on the credit
        dom_fp = dk.get("executed_fp32_frac", dk["credited_fp32_frac"])
        dom_tf = dom_fp * fp32_peak
        dom_hbm = dk["hbm_frac"] >= dom_fp
        tr = traffic_all.get(dom)
        roofline = {"kernel": dom + " -- " + KERNELS[dom]["what"], "bound": "hbm" if dom_hbm else "fp32",
                    "achieved": dk["gbs"] if dom_hbm else dom_tf, "peak": hbm_peak if dom_hbm else fp32_peak,
                    "unit": "GB/s" if dom_hbm else "TFLOP/s", "frac": dk["hbm_frac"] if dom_hbm else dom_fp,
                    "traffic": tr * (float(S) / 1024.0) if tr else None,
                    "algorithmic_bytes_per_launch": KERNELS[dom]["bytes"] * float(S) * n,
                    "algorithmic_flop_per_launch": KERNELS[dom]["flop"] * float(S) * n,
                    "flop_basis": "executed (ncu source page)" if "executed_fp32_frac" in dk else "credited (SURVEY 8d direct-form count)",
                    "credited_fp32_frac": dk["credited_fp32_frac"],
                    "peak_source": (peak_src if dom_hbm else "FFMA issue peak measured live by pmr446_measure_fp32_peak "
                                    "(MEASURED_PEAKS.json has no FP32 figure)"),
                    "other_roofline_frac": dom_fp if dom_hbm else dk["hbm_frac"],
                    "avg_launch_ms": dk["avg_launch_ms"], "share_of_step": dk["share_of_step"]}
        cores = os.cpu_count() or 1
        cpu_v, cpu_dt = cpu_chain_rate(cores, 8)
        cpu_f, cpu_fdt = cpu_chain_rate(cores, 8, active_only=1)   # what the reference executes: one demodulated channel
        cpu_1, _ = cpu_chain_rate(1, 8)                             # one stream on one core (SURVEY 8d (i))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(config_dict(world), streams_per_gpu=S, **({"total_streams": S * world, "strong_target_total": strong_total} if strong_total else {})),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": S * n * 2, "d2h_bytes_per_step": S * 16 * int(e2e_ns) * 2,
                    "steps": e2e_steps, "api": "pmr446_batch_execute (host buffers, pinned)",
                    "numa_bound": numa_node is not None,
                    "pcie_ceiling": {"h2d_gbs_sum_over_ranks": sum(r["h2d_gbs_all_ranks_copying"] for r in rank_stats),
                                     "h2d_gbs_min_rank": min(r["h2d_gbs_all_ranks_copying"] for r in rank_stats),
                                     "e2e_input_gbs_sum_over_ranks": sum(r["e2e_input_gbs"] for r in rank_stats),
                                     "note": "measured in this run with every rank copying 1 GiB pinned <-> device at the same time; "
                                             "e2e moves 2 B per input sample in, so its ceiling is h2d_gbs / 2 samples per second per rank"}},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "kernels": per_kernel,
            "chain_roofline": {"fp32": {"flop_per_sample": FLOP_PER_SAMPLE, "achieved_tflops": value * 1e6 * FLOP_PER_SAMPLE / 1e12 / world,
                                        "peak_tflops": fp32_peak, "frac": value * 1e6 * FLOP_PER_SAMPLE / 1e12 / world / fp32_peak,
                                        "basis": "credited: SURVEY 8d direct-form flop per input sample"},
                               "fp32_executed": ({"flop_per_step": exec_total, "achieved_tflops": exec_total / (step_ms * 1e-3) / 1e12,
                                                  "peak_tflops": fp32_peak, "frac": exec_total / (step_ms * 1e-3) / 1e12 / fp32_peak,
                                                  "basis": "executed: FFMA2/FFMA/FADD/FMUL thread instructions of the step's kernels (ncu, profiles/kernel_exec.json)"}
                                                 if exec_total and len([q for q in per_kernel.values() if "executed_tflops" in q]) == len(per_kernel) else None),
                               "hbm": {"bytes_per_sample": BYTES_PER_SAMPLE, "achieved_gbs": value * 1e6 * BYTES_PER_SAMPLE / 1e9 / world,
                                       "peak_gbs": hbm_peak, "frac": value * 1e6 * BYTES_PER_SAMPLE / 1e9 / world / hbm_peak,
                                       "peak_source": peak_src}},
            "kernel_share_of_step": shares,
            "cpu_baseline": {"value": cpu_v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d host threads x 8 s of one 2.4 Msps stream each (all 16 channels demodulated), %.1f s wall" % (cores, cpu_dt),
                             "single_core_value": cpu_1,
                             "reference_faithful_value": cpu_f,
                             "reference_faithful_sample": "same, only one channel demodulated as the reference does (SURVEY 8d), %.1f s wall" % cpu_fdt},
            "checksum": checksum,
            "per_rank": rank_stats,
        }
        emit(line)
    batch.close()
    if distributed:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# The other BASELINE.json configurations (parity-test cases, not the judged line): same JSON fields, chain-level
# roofline from SURVEY.md 8d's per-sample work of THAT configuration.
OTHER = {
    "cfg1": {"workload": "configs[0] scaled out: 1024 x 1.024 Msps cu8 PMR446 captures x 16 channels, 1 000 000 samples per stream per step "
                         "(the reference's own rate)", "streams": 1024, "fs": 1024000, "n": 1000000, "flop": 237.8, "bytes": 2.39, "kind": "pmr", "fmt": 1},
    "cfg2": {"workload": "configs[1] scaled out: 1024 x 2.4 Msps cu8 captures through the dsd_in chain -> 48 kHz s16, 1 s of signal (2 400 000 samples) per stream per step",
             "streams": 1024, "fs": 2400000, "n": 2400000, "flop": 35.6, "bytes": 2.094, "kind": "dsd", "fmt": 1},
    "cfg4": {"workload": "configs[3]: 4 x 20 Msps cf32 captures, 1600-channel 12.5 kHz PFB + per-channel NBFM demod + W=1600 waterfall, 0.1 s per step",
             "streams": 4, "fs": 20000000, "n": 2000000, "flop": 1539.0, "bytes": 10.0, "kind": "wide", "fmt": 0},
    "receiver": {"workload": "reference receiver mode: 1024 x 2.4 Msps cu8, RSSI + squelch/selector + selected-channel audio + CTCSS detector per stream",
                 "streams": 1024, "fs": 2400000, "n": 2400000, "flop": (19.2 + 81.0 + 11.2 + 1.2 + 20.8 + 4.0 + (3.8 + 150.8 + 1.0) / 16) / 2.4, "bytes": 2.0 + 0.0104,
                 "kind": "rx", "fmt": 1},
}


def run_other(args, name):
    import ctypes as C

    import torch
    from sdr_pmr446_b200 import _lib, chain, synth
    cfg = OTHER[name]
    S, fs, n, kind = cfg["streams"], cfg["fs"], cfg["n"], cfg["kind"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    if kind == "wide":
        M = 1600
        car = tuple(synth.Carrier(int(c), 0.05, 1000.0, 67.0) for c in np.random.default_rng(446).choice(np.arange(1, M + 1), 64, replace=False))
        base = synth.make_cf32(synth.CaptureSpec(fs=float(fs), num_channels=M, carriers=car), n, 446)
        host = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(base, (S, n)))).pin_memory()
    elif kind == "dsd":
        base = synth.cfg2_capture(n=n)
        host = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(base, (S, 2 * n)))).pin_memory()
    else:
        caps = [synth.make_cu8(synth.CaptureSpec(fs=float(fs), carriers=synth.rotated_carriers(s)), n, 446 + s) for s in range(4)]
        host = torch.empty((S, 2 * n), dtype=torch.uint8).pin_memory()
        for s in range(S):
            host[s] = torch.from_numpy(np.roll(caps[s % 4], 2 * 16 * (s // 4)))
    iq_dev = host.to(dev)
    fp32_peak = chain.measure_fp32_peak()
    if kind in ("pmr", "wide"):
        kw = dict(num_channels=1600, waterfall=1600) if kind == "wide" else {}
        obj = chain.PmrBatch(n_streams=S, fs_in=fs, in_fmt=cfg["fmt"], audio_gain=1.0, max_chunk=n, **kw)
        M = obj.M
        outs = {"ld": obj.max_ns, "pcm": torch.empty((S, M, obj.max_ns), dtype=torch.int16, device=dev)}
        if kind == "wide":
            outs.update(ascii=torch.empty((S, 1600), dtype=torch.uint8, device=dev), peak=torch.empty((S, 2), dtype=torch.float32, device=dev))
        view = iq_dev.view(torch.float32).view(S, -1) if kind == "wide" else iq_dev
        dev_step = lambda: obj.execute_device(view, n, outs)
        dump = lambda r: dict(pcm=outs["pcm"][:, :, :r[1]], **{k: outs[k] for k in ("ascii", "peak") if k in outs})
        pcm_host = torch.zeros((S, M, obj.max_ns), dtype=torch.int16).pin_memory()
        o = _lib.Outputs()
        o.ld, o.res_ld, o.pcm = obj.max_ns, obj.max_res, pcm_host.data_ptr()
        if kind == "wide":
            asc_h, pk_h = np.zeros((S, 1600), np.uint8), np.zeros((S, 2), np.float32)
            o.ascii, o.peak = asc_h.ctypes.data, pk_h.ctypes.data
        ny, ns = C.c_uint(0), C.c_uint(0)
        host_np = host.numpy()
        host_step = lambda: _lib.check(_lib.lib().pmr446_batch_execute(obj.h, host_np.ctypes.data, host_np.strides[0], n, C.byref(o), C.byref(ny), C.byref(ns)),
                                       "pmr446_batch_execute")
        d2h = lambda: S * M * int(ns.value) * 2
        api = "pmr446_batch_execute"
    elif kind == "dsd":
        obj = chain.DsdBatch(n_streams=S, fs_in=fs, in_fmt=1, max_chunk=n)
        pcm = torch.empty((S, obj.max_out), dtype=torch.int16, device=dev)
        dev_step = lambda: obj.execute_device(iq_dev, n, pcm=pcm)
        dump = lambda r: {"pcm": pcm[:, :r[1]]}
        pcm_host = torch.zeros((S, obj.max_out), dtype=torch.int16).pin_memory()
        o = _lib.DsdOutputs()
        o.res_ld, o.out_ld, o.pcm = obj.max_res, obj.max_out, pcm_host.data_ptr()
        ny, nz = C.c_uint(0), C.c_uint(0)
        host_np = host.numpy()
        host_step = lambda: _lib.check(_lib.lib().dsd446_batch_execute(obj.h, host_np.ctypes.data, host_np.strides[0], n, C.byref(o), C.byref(ny), C.byref(nz)),
                                       "dsd446_batch_execute")
        d2h = lambda: S * int(nz.value) * 2
        api = "dsd446_batch_execute"
    else:
        obj = chain.PmrReceiver(n_streams=S, fs_in=fs, in_fmt=1, max_chunk=n, audio_gain=1.0)
        ro = {"ld": obj.max_ns, "pcm": torch.empty((S, obj.max_ns), dtype=torch.int16, device=dev),
              "status": torch.empty((S, C.sizeof(_lib.RxStatus)), dtype=torch.uint8, device=dev),
              "rssi": torch.empty((S, 16), dtype=torch.float32, device=dev)}
        dev_step = lambda: obj.execute_device(iq_dev, n, ro)

        def dump(ns):
            st = (_lib.RxStatus * S).from_buffer_copy(ro["status"].cpu().numpy().tobytes())
            fields = {"status_" + k: np.array([getattr(x, k) for x in st]) for k in chain.PmrReceiver.STATUS_FIELDS}
            pcm = ro["pcm"][:, :ns].cpu().numpy()
            pcm[np.arange(ns)[None, :] >= fields["status_n_audio"][:, None]] = 0   # a stream's audio ends at its n_audio
            return dict(pcm=pcm, rssi=ro["rssi"], **fields)
        pcm_host = torch.zeros((S, obj.max_ns), dtype=torch.int16).pin_memory()
        status = (_lib.RxStatus * S)()
        rssi_h = np.zeros((S, 16), np.float32)
        o = _lib.RxOutputs()
        o.ld, o.pcm, o.status, o.rssi = obj.max_ns, pcm_host.data_ptr(), C.addressof(status), rssi_h.ctypes.data
        nsr = C.c_uint(0)
        host_np = host.numpy()
        host_step = lambda: _lib.check(_lib.lib().pmr446_receiver_execute(obj.h, host_np.ctypes.data, host_np.strides[0], n, C.byref(o), C.byref(nsr)),
                                       "pmr446_receiver_execute")
        d2h = lambda: S * int(nsr.value) * 2 + S * (C.sizeof(_lib.RxStatus) + 64)
        api = "pmr446_receiver_execute"
    for _ in range(args.warmup):
        dev_step()
    sampler = ClockSampler(0)
    torch.cuda.synchronize()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = dev_step()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / args.steps
    launches = getattr(obj, "last_launches", 0) * args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dump(last))
    e2e_steps = args.steps
    host_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    clocks = sampler.stop()
    value = S * n / (step_ms * 1e-3) / 1e6
    peaks, peak_src = measured_peaks()
    hbm_peak = peaks.get("hbm_gbs")
    bps = 2 if cfg["fmt"] == 1 else 8
    tf, gbs = value * 1e6 * cfg["flop"] / 1e12, value * 1e6 * cfg["bytes"] / 1e9
    fp_bound = tf / fp32_peak >= gbs / hbm_peak
    # CPU oracle of the same configuration, bounded sample, all host threads (one stream each)
    from oracle import oracle as orc
    cores = os.cpu_count() or 1
    secs = {"pmr": 4, "dsd": 8, "wide": 1, "rx": 4}[kind]

    def cpu_work(i):
        if kind == "dsd":
            q = orc.DsdOracle(fs_in=fs, in_fmt=1, chunk=n)
            for _ in range(secs):
                q.execute(host_np[0])
        elif kind == "rx":
            q = orc.RxOracle(fs_in=fs, in_fmt=1, audio_gain=1.0, chunk=n)
            for _ in range(secs):
                q.execute(host_np[i % S])
        else:
            kw2 = dict(num_channels=1600, waterfall=1600) if kind == "wide" else {}
            q = orc.PmrOracle(fs_in=fs, in_fmt=cfg["fmt"], audio_gain=1.0, chunk=n, **kw2)
            for _ in range(secs):
                q.execute(host_np[i % S], want=("pcm",) + (("ascii",) if kind == "wide" else ()))
        q.close()
    threads = min(cores, 8) if kind == "wide" else cores
    ths = [threading.Thread(target=cpu_work, args=(i,)) for i in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    cpu_dt = time.perf_counter() - t0
    cpu_v = threads * secs * n / cpu_dt / 1e6
    emit({"metric": METRIC if kind != "dsd" else "IQ Msamples/s through the dsd_in chain", "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": {"workload": cfg["workload"], "streams_per_gpu": S, "fs_in": fs, "samples_per_stream_per_step": n, "in_fmt": "cu8" if cfg["fmt"] else "cf32",
                     "l2": "inputs (%.1f GB/step) larger than L2; no flush needed" % (S * n * bps / 1e9), "bench_config": name},
          "e2e": {"value": S * n / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": S * n * bps, "d2h_bytes_per_step": d2h(), "steps": e2e_steps,
                  "api": api + " (host buffers, pinned)"},
          "gpu_launches": launches, "clocks": clocks,
          "roofline": {"kernel": "whole chain of this configuration (per-kernel captures: profiles/)", "bound": "fp32" if fp_bound else "hbm",
                       "achieved": tf if fp_bound else gbs, "peak": fp32_peak if fp_bound else hbm_peak, "unit": "TFLOP/s" if fp_bound else "GB/s",
                       "frac": tf / fp32_peak if fp_bound else gbs / hbm_peak, "traffic": None,
                       "flop_basis": "credited: SURVEY 8d direct-form flop per input sample (%.1f) and algorithmic bytes (%.3f)" % (cfg["flop"], cfg["bytes"]),
                       "other_roofline_frac": gbs / hbm_peak if fp_bound else tf / fp32_peak,
                       "peak_source": peak_src if not fp_bound else "FFMA issue peak measured live by pmr446_measure_fp32_peak"},
          "cpu_baseline": {"value": cpu_v, "unit": UNIT, "cores": threads, "kind": "port",
                           "sample": "%d host threads x %d steps of one stream each, %.1f s wall" % (threads, secs, cpu_dt)}})
    obj.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default): 1024 streams per GPU; strong: 8192 streams in total sharded over the GPUs (BASELINE configs[4])")
    ap.add_argument("--config", default="cfg3", choices=["cfg3"] + sorted(OTHER),
                    help="cfg3 (default) = BASELINE configs[2], the judged line; the others are the remaining BASELINE configurations (1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (the s16 audio; for --config cfg4 also the waterfall, for "
                         "--config receiver also the status and RSSI) to DIR/<name>.npy as float32: a fixed sample of %d streams, rank 0's "
                         "with several GPUs" % DUMP_STREAMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything libraries print meanwhile (NCCL's version banner, ...) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global emit

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif args.config != "cfg3":
        if rank == 0:
            run_other(args, args.config)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
