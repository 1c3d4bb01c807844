#!/usr/bin/env python
"""The matrix convolver (b200conv_mx_*) against today's composition of the same workload.

Rank 11, one-frame (1024-sample) device-resident calls on one stream, timed with CUDA events over
--reps calls after a warm-up of at least the longest route's partition count (the ring is full and
the IR spectra have been streamed once).  Configs:
  A  16 true-stereo reverbs: 32 in x 32 out, 64 routes (block-diagonal 2 x 2), 480 000 taps
  B  4 sources x 16 ambisonic channels: 64 routes (full 4 x 16), 480 000 taps
  C  binaural decoder: 16 in x 2 out, 32 routes, 48 000 taps (L2-resident, latency-bound)
The composition is what a caller does without the matrix object: a ConvolverBatch with one
instance per route, the inputs gathered into per-route rows and the outputs summed with index_add_,
gather and sum inside the timed region.  Both see the same seeded inputs and IRs; the outputs of
every call are compared.  A separate profiled pass (torch.profiler) gives per-kernel device times.
One JSON line per config (and --out FILE gets the same lines)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import __graft_entry__ as ge
import synth

RG = 4          # routes per k_mx_mac CTA (MX_RG in csrc/matrix.cuh): a group reads its input's ring once


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return out[0].strip(), out[1].strip()


def configs():
    a = [(2 * b + i, 2 * b + o) for b in range(16) for i in range(2) for o in range(2)]
    b = [(i, o) for i in range(4) for o in range(16)]
    c = [(i, o) for i in range(16) for o in range(2)]
    return [("A", "16 true-stereo reverbs, 32 x 32 block-diagonal", 32, 32, a, 480000),
            ("B", "4 sources x 16 ambisonic channels, full 4 x 16", 4, 16, b, 480000),
            ("C", "binaural decoder, 16 x 2", 16, 2, c, 48000)]


def algo_bytes(F, I, O, pairs, taps):
    """8F (sum_r nq_r + sum_i groups_i nq_i + I) + 4F (I + O): IR rows, ring rows (once per group of
    up to RG routes leaving an input), the new spectrum of each input; input and output samples."""
    nq = (taps + F - 1) // F + 1
    leaving = np.bincount([i for i, _ in pairs], minlength=I)
    groups = int(np.sum((leaving + RG - 1) // RG))
    return 8 * F * (len(pairs) * nq + groups * nq + I) + 4 * F * (I + O)


def composition_bytes(F, pairs, taps):
    bins = (taps + F - 1) // F
    return len(pairs) * (16 * F * bins + 24 * F)        # the engine's per instance-frame count (DESIGN 4)


def run(pkg, cfg, reps, peak):
    key, what, I, O, pairs, taps = cfg
    rank = 11
    F = 1 << (rank - 1)
    nq = (taps + F - 1) // F + 1
    warm = nq + 8
    blocks = warm + reps
    irs = [synth.decaying_ir(5000 + r, taps) for r in range(len(pairs))]
    gen = torch.Generator(device="cuda").manual_seed(0xB200 + ord(key))
    x = torch.rand((I, blocks * F), device="cuda", generator=gen) * 2 - 1
    y_mx = torch.empty((O, blocks * F), device="cuda")
    y_cp = torch.zeros((O, blocks * F), device="cuda")
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream

    mx = pkg.MatrixConvolver(I, O, rank, device=0)
    mx.set_routes([(i, o, h) for (i, o), h in zip(pairs, irs)])
    batch = pkg.ConvolverBatch(len(pairs), device=0)
    assert batch.init_many(list(range(len(pairs))), irs, rank)
    gidx = torch.tensor([i for i, _ in pairs], device="cuda")
    oidx = torch.tensor([o for _, o in pairs], device="cuda")
    rows_in = torch.empty((len(pairs), F), device="cuda")
    rows_out = torch.empty((len(pairs), F), device="cuda")

    def mx_call(k):
        mx.process_device(y_mx.data_ptr() + 4 * k * F, y_mx.stride(0), x.data_ptr() + 4 * k * F, x.stride(0), F,
                          stream=sp)

    def comp_call(k):
        torch.index_select(x[:, k * F:(k + 1) * F], 0, gidx, out=rows_in)
        batch.process_device(rows_out.data_ptr(), rows_in.data_ptr(), F, F, stream=sp)
        y_cp[:, k * F:(k + 1) * F].index_add_(0, oidx, rows_out)

    def timed(call):
        with torch.cuda.stream(stream):
            for k in range(warm):
                call(k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for k in range(warm, blocks):
                call(k)
            e1.record(stream)
        stream.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    torch.cuda.synchronize()
    us_mx = timed(mx_call)
    us_cp = timed(comp_call)
    ref = y_cp.abs().max().item()
    diff = (y_mx - y_cp).abs().max().item() / ref

    # per-kernel device time, in a pass of its own (the profiler slows the host)
    mx.clear()
    kern = {}
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(stream):
            for k in range(warm + 50):
                mx_call(k)
        stream.synchronize()
    n_prof = warm + 50
    for ev in prof.key_averages():
        name = ev.key
        for short in ("k_mx_mac", "k_fwd", "k_inv"):
            if short in name:
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                kern[short] = kern.get(short, 0.0) + t / n_prof
    mx.close()
    batch.close()

    b = algo_bytes(F, I, O, pairs, taps)
    bc = composition_bytes(F, pairs, taps)
    return {"config": key, "what": what, "inputs": I, "outputs": O, "routes": len(pairs), "taps": taps,
            "rank": rank, "call_samples": F, "timed_calls": reps, "warmup_calls": warm,
            "us_per_block": us_mx, "algo_bytes_per_block": b, "bytes_per_s": b / (us_mx * 1e-6),
            "end_to_end_share_of_hbm_peak": b / (us_mx * 1e-6) / (peak * 1e9),
            "composition_us_per_block": us_cp, "composition_algo_bytes_per_block": bc,
            "ratio_us_mx_over_composition": us_mx / us_cp, "ratio_bytes_mx_over_composition": b / bc,
            "max_abs_mx_minus_composition_over_peak": diff,
            "kernel_us_per_block_profiled": {k: round(v, 2) for k, v in sorted(kern.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=400)
    ap.add_argument("--configs", default="ABC")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 200:
        raise SystemExit("--reps must be at least 200")
    if not torch.cuda.is_available():
        raise SystemExit("bench_mx: no CUDA device")
    pkg = ge.load()
    pkg.lib()
    peak = 6546.2
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    name, power = gpu_info()
    lines = []
    for cfg in configs():
        if cfg[0] not in args.configs:
            continue
        res = run(pkg, cfg, args.reps, peak)
        res.update({"gpu": name, "power_limit": power, "hbm_peak_gbs": peak})
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
