#!/usr/bin/env python
"""Cost of the batched SpectralProcessor's spectral-function path (b200conv_sp_set_function /
bind_function) against the table path (bind_gain), on device-resident calls of the bench_sp shapes.

Per shape, three objects with the same input: every instance bound to a gain table; every instance
bound to an identity function; every instance bound to a torch function that multiplies by the same
gains.  Their calls are timed with CUDA events on each object's stream, alternating between the
three for several rounds; the median round is reported.  The function paths include the host
callback of every sub-call.  Outputs of the gain function and of the gain table are compared.
One JSON line per shape with the card's name and power limit; --out FILE gets the same lines."""
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


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().split(",")
    return out[0].strip(), out[1].strip()


def span(rank, bound):
    N = 1 << rank
    return (N // 2) * max(1, (1 << 25) // (bound * N))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sp_function: no CUDA device")
    pkg = ge.load()
    name, power = card()
    lines = []
    for rank, n, call in ((10, 4096, 8192), (12, 2048, 16384)):
        N = 1 << rank
        gain = np.linspace(0.5, 1.0, N).astype(np.float32)
        g_dev = torch.tensor(gain, device="cuda")
        calls = {"fn_identity": 0, "fn_gain": 0}

        def identity(X, instances, positions, r):
            calls["fn_identity"] += 1

        def multiply(X, instances, positions, r):
            calls["fn_gain"] += 1
            X.mul_(g_dev)

        objs = {}
        for key, fn in (("table_gain", None), ("fn_identity", identity), ("fn_gain", multiply)):
            sp = pkg.SpectralProcessorBatch(n, rank, device=0)
            if fn is not None:
                sp.set_function(fn)
            for c in range(n):
                sp.set_phase(c, (c % 5) / 5.0)
                if fn is None:
                    sp.bind_gain(c, gain)
                else:
                    sp.bind_function(c)
            objs[key] = sp
        src = torch.rand((n, call), device="cuda") * 2 - 1
        dst = {k: torch.empty_like(src) for k in objs}
        streams = {k: torch.cuda.ExternalStream(sp.stream()) for k, sp in objs.items()}
        torch.cuda.synchronize()
        # same input from the same state: the gain function must reproduce the gain table
        for k, sp in objs.items():
            for _ in range(3):
                sp.process_device(dst[k].data_ptr(), call, src.data_ptr(), call, call)
            sp.sync()
        ref = dst["table_gain"].abs().max().item()
        agree = (dst["fn_gain"] - dst["table_gain"]).abs().max().item() / max(1.0, ref)
        times = {k: [] for k in objs}
        for _ in range(args.rounds):
            for k, sp in objs.items():
                if k in calls:
                    calls[k] = 0
                st = streams[k]
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                with torch.cuda.stream(st):
                    for _ in range(args.reps):
                        sp.process_device(dst[k].data_ptr(), call, src.data_ptr(), call, call)
                e1.record(st)
                e1.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.reps)
        ms = {k: float(np.median(v)) for k, v in times.items()}
        frames = n * call / (N / 2)
        line = {"what": "SpectralProcessor batch: spectral function vs gain table", "gpu": name, "power_limit": power,
                "rank": rank, "instances": n, "call": call, "sub_call_samples": span(rank, n),
                "invocations_per_call": calls["fn_gain"] / args.reps,
                "ms_per_call": ms, "samples_per_s": {k: n * call / (v * 1e-3) for k, v in ms.items()},
                "frames_per_call": frames,
                "fn_over_table": {k: ms[k] / ms["table_gain"] for k in ("fn_identity", "fn_gain")},
                "fn_gain_vs_table_max_err_of_peak": agree,
                "spectrum_bytes_per_frame_by_construction": 4 * N * 8,
                "timing": "CUDA events on each object's stream, %d calls per round, median of %d rounds alternating "
                          "table / identity / gain" % (args.reps, args.rounds)}
        lines.append(json.dumps(line))
        print(lines[-1], flush=True)
        for sp in objs.values():
            sp.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
