#!/usr/bin/env python
"""Cost of replacing routes' impulse responses while the matrix convolver runs (b200conv_mx_set_irs).

Rank 11, one-frame (1024-sample) device-resident calls on one stream, CUDA events, a warm-up of at
least the longest route's partition count.  Workloads:
  binaural  16 in x 2 out, 32 routes of 48 000 taps (bench_mx.py config C).  Every 8 blocks all 32
            routes take the next set of a bank of 8 pre-generated IR sets, fade = 2048.  Reports
            us per block over --blocks blocks against the same object with no updates (alternated),
            and the host time spent inside set_irs (median, p99) against set_routes on the same shape.
  bandwidth 32 in x 32 out, 64 routes of 480 000 taps (block-diagonal 2 x 2, config A).  8 routes change
            every 32 blocks, fade = 4096.  Reports us per block in steady state and while a fade runs
            (events around every block), and the device time of the ingest.
  regress   --parent DIR: tools/bench_mx.py configs A, B and C, run alternately from DIR (a checkout of
            the parent commit with its library built) and from this tree.
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


class Run:
    """An object, its input and output on the device, and one-frame calls on one stream."""

    def __init__(self, pkg, I, O, pairs, irs, blocks, seed):
        self.mx = pkg.MatrixConvolver(I, O, RANK, device=0)
        self.mx.set_routes([(i, o, h) for (i, o), h in zip(pairs, irs)])
        gen = torch.Generator(device="cuda").manual_seed(seed)
        self.x = torch.rand((I, blocks * F), device="cuda", generator=gen) * 2 - 1
        self.y = torch.empty((O, blocks * F), device="cuda")
        self.stream = torch.cuda.Stream()
        self.sp = self.stream.cuda_stream
        self.blocks = blocks

    def call(self, k):
        k %= self.blocks
        self.mx.process_device(self.y.data_ptr() + 4 * k * F, self.y.stride(0), self.x.data_ptr() + 4 * k * F,
                               self.x.stride(0), F, stream=self.sp)

    def close(self):
        self.mx.close()


def pct(v, q):
    return float(np.percentile(np.asarray(v), q))


def binaural(pkg, blocks, rounds):
    I, O, taps = 16, 2, 48000
    pairs = [(i, o) for i in range(I) for o in range(O)]
    bank = [[synth.decaying_ir(7000 + 100 * s + r, taps) for r in range(len(pairs))] for s in range(8)]
    warm = (taps + F - 1) // F + 1 + 8
    run = Run(pkg, I, O, pairs, bank[0], warm + blocks, 0xFADE)
    host_irs = []
    at = [0, 1]                             # next block, next IR set

    def timed(updates):
        with torch.cuda.stream(run.stream):
            for k in range(warm):
                run.call(k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(run.stream)
            for k in range(blocks):
                if updates and k % 8 == 0:
                    changes = list(enumerate(bank[at[1] % 8]))
                    t0 = time.perf_counter()
                    run.mx.set_irs(changes, fade=2048, stream=run.sp)
                    host_irs.append(time.perf_counter() - t0)
                    at[1] += 1
                run.call(warm + k)
            e1.record(run.stream)
        run.stream.synchronize()
        return e0.elapsed_time(e1) * 1e3 / blocks

    torch.cuda.synchronize()
    plain, upd = [], []
    for _ in range(rounds):                 # alternate, so that drift hits both alike
        plain.append(timed(False))
        upd.append(timed(True))
    host_routes = []
    routes = [(i, o, h) for (i, o), h in zip(pairs, bank[0])]
    for _ in range(20):
        t0 = time.perf_counter()
        run.mx.set_routes(routes)
        host_routes.append(time.perf_counter() - t0)
    run.close()
    return {"workload": "binaural", "what": "16 x 2, 32 routes of 48 000 taps; all 32 routes replaced every 8 "
            "blocks from a bank of 8 IR sets, fade 2048", "rank": RANK, "call_samples": F, "blocks": blocks,
            "rounds": rounds, "warmup_calls": warm,
            "us_per_block_no_updates": [round(v, 2) for v in plain],
            "us_per_block_with_updates": [round(v, 2) for v in upd],
            "set_irs_host_us_median": pct(host_irs, 50) * 1e6, "set_irs_host_us_p99": pct(host_irs, 99) * 1e6,
            "set_irs_calls": len(host_irs),
            "set_routes_host_us_median": pct(host_routes, 50) * 1e6,
            "set_routes_host_us_p99": pct(host_routes, 99) * 1e6, "set_routes_calls": len(host_routes)}


def bandwidth(pkg, cycles):
    I, O, taps = 32, 32, 480000
    pairs = [(2 * b + i, 2 * b + o) for b in range(16) for i in range(2) for o in range(2)]
    irs = [synth.decaying_ir(5000 + r, taps) for r in range(len(pairs))]
    alt = [synth.decaying_ir(9000 + r, taps) for r in range(len(pairs))]
    warm = (taps + F - 1) // F + 1 + 8
    blocks = cycles * 32
    run = Run(pkg, I, O, pairs, irs, warm + blocks, 0xBA4D)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(blocks + 1)]
    ing = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(cycles)]
    fading = []
    torch.cuda.synchronize()
    with torch.cuda.stream(run.stream):
        for k in range(warm):
            run.call(k)
        for k in range(blocks):
            if k % 32 == 0:
                c = k // 32
                routes = [(8 * c + j) % len(pairs) for j in range(8)]
                src = alt if c % 2 == 0 else irs
                ing[c][0].record(run.stream)
                run.mx.set_irs([(r, src[r]) for r in routes], fade=4096, stream=run.sp)
                ing[c][1].record(run.stream)
            fading.append(run.mx.fade_remaining() > 0)
            ev[k].record(run.stream)
            run.call(warm + k)
        ev[blocks].record(run.stream)
    run.stream.synchronize()
    per = [ev[k].elapsed_time(ev[k + 1]) * 1e3 for k in range(blocks)]
    # the block after a set_irs starts behind the ingest, whose time is reported on its own
    steady = [t for k, t in enumerate(per) if not fading[k] and k % 32 >= 8]
    during = [t for k, t in enumerate(per) if fading[k]]
    ingest = [a.elapsed_time(b) * 1e3 for a, b in ing]
    run.close()
    return {"workload": "bandwidth", "what": "32 x 32 block-diagonal, 64 routes of 480 000 taps; 8 routes "
            "replaced every 32 blocks, fade 4096", "rank": RANK, "call_samples": F, "blocks": blocks,
            "warmup_calls": warm, "us_per_block_steady_median": pct(steady, 50),
            "us_per_block_steady_mean": float(np.mean(steady)), "steady_blocks": len(steady),
            "us_per_block_fading_median": pct(during, 50), "us_per_block_fading_mean": float(np.mean(during)),
            "fading_blocks": len(during), "ingest_device_us_median": pct(ingest, 50)}


def regress(parent, reps, rounds):
    out = []
    for r in range(rounds):
        for build, tree in (("parent", parent), ("new", ROOT)):
            res = subprocess.run([sys.executable, os.path.join(tree, "tools", "bench_mx.py"), "--reps", str(reps)],
                                 capture_output=True, text=True, cwd=tree)
            if res.returncode != 0:
                raise SystemExit("bench_mx.py (%s) failed:\n%s" % (build, res.stderr[-3000:]))
            for line in res.stdout.splitlines():
                if line.startswith("{"):
                    d = json.loads(line)
                    out.append({"workload": "regress", "build": build, "round": r, "config": d["config"],
                                "us_per_block": d["us_per_block"],
                                "composition_us_per_block": d["composition_us_per_block"],
                                "max_abs_mx_minus_composition_over_peak": d["max_abs_mx_minus_composition_over_peak"]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=480)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cycles", type=int, default=16)
    ap.add_argument("--regress-rounds", type=int, default=2)
    ap.add_argument("--parent", default=None, help="tree of the parent commit, library built: run the no-regression A/B")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.blocks < 400:
        raise SystemExit("--blocks must be at least 400")
    if not torch.cuda.is_available():
        raise SystemExit("bench_mx_fade: no CUDA device")
    pkg = ge.load()
    pkg.lib()
    name, power = gpu_info()
    results = [binaural(pkg, args.blocks, args.rounds), bandwidth(pkg, args.cycles)]
    if args.parent:
        results += regress(os.path.abspath(args.parent), 400, args.regress_rounds)
    lines = []
    for res in results:
        res.update({"gpu": name, "power_limit": power})
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
