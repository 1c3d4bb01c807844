#!/usr/bin/env python
"""k_frame lookahead (DESIGN 4.1c) at the headline shape: 64 instances x 480 000-tap IRs, rank 11,
one 1024-sample device-resident call per block on one stream.

For lookahead off, K = 2, 4, 8 and the automatic choice: microseconds per block (CUDA events over
--blocks calls after a warm-up of --warmup calls), the bytes the launches stream per block (the
engine's mac_stream_bytes counter) and their share of HBM peak at the measured block rate.  Then a
profiled pass (launches serialised, one pair of events around each call) gives every launch's
duration: the priming group (full sums plus the next group's tails) is reported apart from the
steady state.  One JSON line per setting, the card's name and power limit in every line."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

import __graft_entry__ as ge
import synth

N, TAPS, RANK = 64, 480000, 11
F = 1 << (RANK - 1)
BINS = (TAPS + F - 1) // F
DATASHEET_HBM_GBS = 7700.0


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return out[0].strip(), out[1].strip()


def run(pkg, la, args, irs, src, dst):
    b = pkg.ConvolverBatch(N, 0)
    b.set_option("lookahead", la)
    assert b.init_many(list(range(N)), [irs[c % len(irs)] for c in range(N)], RANK)
    stream = torch.cuda.Stream()
    total = src.shape[1] // F
    sp, dp = src.data_ptr(), dst.data_ptr()

    def calls(first, count):
        for i in range(first, first + count):
            k = i % total
            b.process_device(dp + 4 * k * F, sp + 4 * k * F, src.shape[1], F, stream.cuda_stream)

    with torch.cuda.stream(stream):
        calls(0, args.warmup)
        torch.cuda.synchronize()
        b.reset_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        calls(args.warmup, args.blocks)
        e1.record(stream)
        torch.cuda.synchronize()
        us = 1e3 * e0.elapsed_time(e1) / args.blocks
        st = b.stats()
        # profiled pass: serialised launches, events around each call
        b.set_profiling(True)
        n_prof = args.profiled
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_prof + 1)]
        first = args.warmup + args.blocks
        for i in range(n_prof):
            evs[i].record(stream)
            calls(first + i, 1)
        evs[n_prof].record(stream)
        torch.cuda.synchronize()
        b.profile()
        b.set_profiling(False)
    b.close()
    launch_us = [1e3 * evs[i].elapsed_time(evs[i + 1]) for i in range(n_prof)]
    return us, st, launch_us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=600)
    ap.add_argument("--profiled", type=int, default=64)
    ap.add_argument("--settings", default="0,2,4,8,-1")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = gpu_info()
    pkg = ge.load()
    pkg.lib()
    irs = [synth.decaying_ir(c, TAPS) for c in range(8)]
    g = torch.Generator(device="cuda").manual_seed(0x5EED)
    src = torch.rand((N, 1000 * F), generator=g, device="cuda") * 2 - 1
    dst = torch.empty_like(src)
    algo = N * (16 * F * BINS + 24 * F)
    lines = []
    for la in [int(x) for x in args.settings.split(",")]:
        us, st, launch_us = run(pkg, la, args, irs, src, dst)
        streamed = st["mac_stream_bytes"] / max(1, st["mac_launches"])
        k = la if la > 0 else (8 if la < 0 else 0)      # the automatic choice at this shape (engine.cu, lookahead_k)
        prime = launch_us[:k] if k else []
        steady = launch_us[k:] if k else launch_us
        line = {"gpu": name, "power_limit": power, "lookahead": la, "us_per_block": us,
                "launches_per_block": st["launches"] / args.blocks,
                "algorithmic_bytes_per_block": algo, "streamed_bytes_per_block": streamed,
                "streamed_share_of_datasheet_hbm": streamed / (us * 1e-6) / (DATASHEET_HBM_GBS * 1e9),
                "profiled_launch_us": {"steady_mean": sum(steady) / len(steady), "steady_max": max(steady),
                                       "priming_max": max(prime) if prime else None, "launches": len(launch_us)},
                "shape": "%d x %d taps, rank %d, one %d-sample call per block, %d blocks after %d warm-up"
                         % (N, TAPS, RANK, F, args.blocks, args.warmup)}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
