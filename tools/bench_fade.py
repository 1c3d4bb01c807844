#!/usr/bin/env python
"""Cost of replacing instances' impulse responses while a convolver batch runs (b200conv_set_irs).

  cfg3  64 instances x 480 000 taps, rank 11, one-frame (1024-sample) process_device calls on the
        batch's own stream, CUDA events around --blocks blocks after a warm-up of 600 blocks (the ring
        holds 502).  Reports us per block in steady state, while 1 instance fades and while all 64
        fade (fades longer than the timed window), and the host time of the set_irs calls that start
        those fades (new IRs of the same length).
  cfg1  1 instance x 65 536 taps, rank 11, synchronous 1024-sample process calls from host memory:
        the host-visible call time (median, p90) in steady state and during a fade.
One JSON line per result, each with the card's name and power limit; --out FILE gets the same lines."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import __graft_entry__ as ge
import synth

RANK = 11
F = 1 << (RANK - 1)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return out[0].strip(), out[1].strip()


def cfg3(pkg, blocks, emit):
    n, taps = 64, 480000
    b = pkg.ConvolverBatch(n, 0)
    assert b.init_many(list(range(n)), [synth.decaying_ir(c, taps) for c in range(n)], RANK)
    ring = 1200
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.rand((n, ring * F), device="cuda", generator=gen) * 2 - 1
    y = torch.empty_like(x)
    st = torch.cuda.ExternalStream(b.stream())
    at = [0]

    def calls(k):
        for _ in range(k):
            o = 4 * (at[0] % ring) * F
            b.process_device(y.data_ptr() + o, x.data_ptr() + o, ring * F, F)
            at[0] += 1

    def timed():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        calls(blocks)
        e1.record(st)
        e1.synchronize()
        return 1000.0 * e0.elapsed_time(e1) / blocks

    calls(600)
    b.sync()
    base = dict(config="cfg3", instances=n, taps=taps, rank=RANK, call_samples=F, timed_blocks=blocks)
    emit(dict(base, what="steady state", us_per_block=timed()))
    new = [synth.decaying_ir(1000 + c, taps) for c in range(n)]
    for k in (1, n):
        calls(20)
        t0 = time.perf_counter()
        b.set_irs(list(range(k)), new[:k], fade=(blocks + 40) * F)
        t_set = 1000.0 * (time.perf_counter() - t0)
        calls(20)
        emit(dict(base, what="during a fade of %d instance(s)" % k, fading=k, us_per_block=timed(),
                  set_irs_host_ms=t_set))
        while b.fade_remaining(0) > 0:
            calls(1)
        b.sync()
    calls(20)
    emit(dict(base, what="steady state after the fades", us_per_block=timed()))
    b.close()


def cfg1(pkg, calls_n, emit):
    taps = 65536
    b = pkg.ConvolverBatch(1, 0)
    assert b.init(0, synth.decaying_ir(1, taps), RANK, 0.0)
    x = synth.noise(2, F)[None, :]
    out = np.empty_like(x)

    def timed(k):
        ts = []
        for _ in range(k):
            t0 = time.perf_counter()
            b.process(x, out=out)
            ts.append(1e6 * (time.perf_counter() - t0))
        return float(np.median(ts)), float(np.percentile(ts, 90))

    timed(200)
    base = dict(config="cfg1", instances=1, taps=taps, rank=RANK, call_samples=F, timed_calls=calls_n, entry="process")
    med, p90 = timed(calls_n)
    emit(dict(base, what="steady state", host_us_median=med, host_us_p90=p90))
    b.set_irs([0], [synth.decaying_ir(3, taps)], fade=(calls_n + 10) * F)
    med, p90 = timed(calls_n)
    emit(dict(base, what="during a fade", host_us_median=med, host_us_p90=p90))
    b.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=300)
    ap.add_argument("--calls", type=int, default=500)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = ge.load()
    name, power = gpu_info()
    lines = []

    def emit(d):
        d = dict(d, gpu=name, power_limit=power)
        print(json.dumps(d), flush=True)
        lines.append(d)

    cfg3(pkg, args.blocks, emit)
    cfg1(pkg, args.calls, emit)
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
