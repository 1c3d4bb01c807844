#!/usr/bin/env python
"""Developer tool: where does a steady-state k_frame lookahead launch spend its time?  The headline
shape of bench.py (64 instances x 480 000-tap IRs, rank 11, one 1024-sample device-resident call per
block on one stream, K chosen automatically).  Uses a library built with -DB200CONV_TIMING (built
under tools/ab/ when missing, or --lib PATH).  Stamps (%globaltimer, thread 0 of each CTA):
0 start, 4 end of the tail stages, 5 tail rows published (la_prod), 6 end of the head stages, 1 after
the last stage (split 0: after the input transform and the q = 0 stage), 2 ticket, 7 T rows acquired
(la_prod wait, last CTA of a job), 3 end of the inverse transform.

After `--calls` calls the stream is drained and the stamps of the LAST launch are read (CTAs of the
launch before it may have left a few stale stamps: a stamp older than the CTA's own start is
dropped).  Repeated for --reps different final group positions.  Prints per-phase percentiles over
the CTAs and the CTA-time split; --out FILE also writes the raw stamps (µs from the launch's first
CTA start) as text."""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ap = argparse.ArgumentParser()
ap.add_argument("--lib", default=os.path.join(ROOT, "tools", "ab", "libb200conv_timing.so"))
ap.add_argument("--build", action="store_true", help="(re)build --lib and exit")
ap.add_argument("--calls", type=int, default=200)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--lookahead", type=int, default=-1)
ap.add_argument("--out", default=None)
args = ap.parse_args()

if args.build or not os.path.exists(args.lib):
    os.makedirs(os.path.dirname(args.lib), exist_ok=True)
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler",
                           "-fPIC", "-shared", "-DB200CONV_TIMING", "-I", os.path.join(ROOT, "include"), "-o", args.lib,
                           os.path.join(ROOT, "lsp-dsp-units_b200", "csrc", "engine.cu")])
    if args.build:
        sys.exit(0)

import torch
import __graft_entry__ as ge
import synth

pkg = ge.load()
pkg.LIB_PATH = args.lib
pkg._lib = None
lib = pkg.lib()
lib.b200conv_debug_frame_times.argtypes = [ctypes.c_void_p, ctypes.c_size_t]

N, TAPS, RANK = 64, 480000, 11
F = 1 << (RANK - 1)
name, power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.strip().split(",")
lines = ["# %s, power limit %s; %d x %d taps, rank %d, 1024-sample calls, lookahead option %d" % (
    name.strip(), power.strip(), N, TAPS, RANK, args.lookahead)]


def say(s):
    print(s, flush=True)
    lines.append(s)


b = pkg.ConvolverBatch(N, 0)
b.set_option("lookahead", args.lookahead)
irs = [synth.decaying_ir(c, TAPS) for c in range(4)]
assert b.init_many(list(range(N)), [irs[c % 4] for c in range(N)], RANK)
total = 64
src = torch.rand((N, total * F), device="cuda") * 2 - 1
dst = torch.empty_like(src)
stream = torch.cuda.Stream()
ncta = 8192
done = 0
raw = []
for rep in range(args.reps):
    with torch.cuda.stream(stream):
        for i in range(args.calls + rep):
            k = (done + i) % total
            b.process_device(dst.data_ptr() + 4 * k * F, src.data_ptr() + 4 * k * F, total * F, F, stream.cuda_stream)
        done += args.calls + rep
    torch.cuda.synchronize()
    buf = (ctypes.c_ulonglong * (ncta * 8))()
    assert lib.b200conv_debug_frame_times(buf, ncta * 8) == 0
    t = np.array(buf[:], dtype=np.float64).reshape(ncta, 8)
    live = t[:, 0] > t[:, 0].max() - 1e6            # CTAs of the last launch (all within 1 ms)
    t = t[live]
    t0 = t[:, 0].min()
    stale = t < t[:, :1]
    r = (t - t0) / 1e3
    r[stale] = np.nan
    raw.append(r)
    say("call %d: %d CTAs, start spread %.1f us, launch span %.1f us" % (
        done - 1, live.sum(), np.nanmax(r[:, 0]), np.nanmax(r[:, 3]) - np.nanmin(r[:, 0])))

    def pct(x, label):
        x = x[~np.isnan(x)]
        if x.size:
            say("   %-34s n %4d  min %6.1f  median %6.1f  p90 %6.1f  max %6.1f us" % (
                label, x.size, x.min(), np.median(x), np.percentile(x, 90), x.max()))

    pct(r[:, 4] - r[:, 0], "tail stages (start -> 4)")
    pct(r[:, 5] - r[:, 4], "tail rows out (4 -> 5)")
    pct(r[:, 6] - r[:, 5], "head stages (5 -> 6)")
    pct(r[:, 1] - r[:, 6], "last stage / transform (6 -> 1)")
    pct(r[:, 2] - r[:, 1], "slot + pdl wait, rows, ticket (1 -> 2)")
    last = ~np.isnan(r[:, 7])
    pct(r[last, 7] - r[last, 2], "T wait, last CTAs (2 -> 7)")
    pct(r[last, 3] - r[last, 7], "inverse transform (7 -> 3)")
    pct(r[:, 2], "ticket, from launch start")
    pct(r[last, 3], "end, from launch start")
    # CTA-time split: sum over CTAs of each phase, as a share of the summed CTA lifetimes
    life = np.where(last, r[:, 3], r[:, 2]) - r[:, 0]
    parts = [("tail", r[:, 4] - r[:, 0]), ("tail rows", r[:, 5] - r[:, 4]), ("head", r[:, 6] - r[:, 5]),
             ("last stage/fwd", r[:, 1] - r[:, 6]), ("wait+ticket", r[:, 2] - r[:, 1]),
             ("T wait", np.where(last, r[:, 7] - r[:, 2], 0.0)), ("inverse", np.where(last, r[:, 3] - r[:, 7], 0.0))]
    tot = np.nansum(life)
    say("   CTA-time split: " + ", ".join("%s %.1f %%" % (k, 100.0 * np.nansum(v) / tot) for k, v in parts))
b.close()
if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
        f.write("# raw stamps per CTA (us from the launch's first start; nan = stale): "
                "rep cta start tail_end tail_rows head_end last_stage ticket T_acquired end\n")
        for rep, r in enumerate(raw):
            for c in range(r.shape[0]):
                f.write("%d %d %s\n" % (rep, c, " ".join("%.2f" % r[c, k] for k in (0, 4, 5, 6, 1, 2, 7, 3))))
