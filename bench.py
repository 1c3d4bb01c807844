#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 batched Convolver (BASELINE.json, config 3).

    python bench.py --gpus N --steps K --warmup W            # the CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's output

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): 64 independent
dspu::Convolver instances per GPU, 480 000-tap (10 s @ 48 kHz) synthetic exponentially-decaying
noise IRs, rank 11 (1024-sample frames), fed white noise in 1024-sample process() calls.  One
"step" is `frames_per_step` (default 469 = one full IR length, so every ring slot is rewritten)
consecutive process calls on all instances.  Multi-GPU: one process per GPU (torchrun), each
rank owns its own 64 instances -- independent channels, no collective on the data path
("scaling": "weak"); `value` = samples of all ranks / max-over-ranks device time.

One JSON line on rank 0; see the task contract for the keys.  `roofline` is for the dominant
kernel -- k_frame<11>, the one launch per block: algorithmic bytes per launch
(64 x (16*F*bins + 24*F), DESIGN.md) / its average launch duration.  The timed region consists of
nothing but those launches, back to back on one stream (CUDA events on that stream), so its
duration / launches is the kernel's launch duration as deployed; `isolated_*` repeats the
measurement with every launch bracketed by its own event pair (no overlap between blocks) in an
extra pass right after the timed steps.  peak = MEASURED_PEAKS.json hbm_gbs (fallback 6650 GB/s);
`e2e` = synchronous b200conv_process_planar calls on pinned host buffers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TAPS, RANK, BLOCK, INSTANCES = 480000, 11, 1024, 64
F = 1 << (RANK - 1)
BINS = (TAPS + F - 1) // F                      # 469
BYTES_PER_INSTANCE_FRAME = 16 * F * BINS + 24 * F
METRIC = "Convolver output samples/s (64ch x 10s IR, 1024-sample blocks)"
UNIT = "samples/s"
FALLBACK_HBM_GBS = 6650.0
DUMP_ROWS, DUMP_BYTES = 16, 60_000_000


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md, 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms during the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, smax = [], set(), None
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    smax = float(p[2])
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), p[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            busy = [v for v in sm if v >= 0.5 * sm[-1]] or sm
            out.update(sm_mhz=busy[len(busy) // 2], sm_max_mhz=smax, reasons=sorted(reasons),
                       samples=len(sm))
        return out


def cpu_reference_rate(threads, blocks, warm=4):
    """The reference's CPU path on `threads` host cores: one Convolver per thread, `blocks`
    process() calls of 1024 samples each after `warm` untimed ones.  Uses oracle/_ref (the
    reference's Convolver.cpp compiled verbatim over restated dsp:: kernels) when it was built,
    else the plain-C oracle port."""
    from oracle import bindings
    kind = "reference" if bindings.CpuConvolver.available("reference") else "port"
    impl = "reference" if kind == "reference" else "oracle"
    rate, sec = bindings.cpu_bench(impl, threads, TAPS, RANK, BLOCK, warm, blocks, threads)
    return rate, sec, kind


def dump_outputs(path, dst):
    """Saves what the last timed step returned to its caller, ``dst`` = [64 instances][frames * 1024]
    float32, as ``path/convolver_dst.npy``: the rows of a fixed, seeded choice of 16 instances, in
    instance order, every sample of the step (a seeded, sorted choice of columns when a longer step
    would exceed DUMP_BYTES).  The inputs are seeded too, so two builds can be compared sample for sample."""
    import numpy as np
    import torch
    rng = np.random.default_rng(0)
    rows = np.sort(rng.choice(dst.shape[0], DUMP_ROWS, replace=False))
    out = dst[torch.as_tensor(rows, device=dst.device)]
    limit = DUMP_BYTES // (4 * DUMP_ROWS)
    if out.shape[1] > limit:
        cols = np.sort(rng.choice(out.shape[1], limit, replace=False))
        out = out[:, torch.as_tensor(cols, device=dst.device)]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "convolver_dst.npy"), out.cpu().numpy())


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, all host threads."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    threads = min(cores, INSTANCES)
    # bounded sample per step: a few seconds of CPU work (one convolver per thread, 192 blocks each)
    blocks = args.cpu_blocks
    rates = []
    t0 = time.time()
    for s in range(args.warmup + args.steps):
        rate, sec, kind = cpu_reference_rate(threads, blocks)
        if s >= args.warmup:
            rates.append((rate, sec))
    total_samples = sum(r * s for r, s in rates)
    total_sec = sum(s for _, s in rates)
    value = total_samples / total_sec
    sample = ("%d of the 64 instances (one per host thread), 480000-tap IR, rank 11, %d process() "
              "calls of 1024 samples per step after 4 warm calls; reference Convolver.cpp compiled "
              "verbatim over restated scalar dsp:: kernels (lsp-dsp-lib AVX/SSE is not available "
              "offline)" % (threads, blocks)) if kind == "reference" else \
             ("%d instances of the plain-C oracle port, %d calls of 1024 samples per step" % (threads, blocks))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_sec / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "cfg3: 64 ch x 480000-tap IR (10 s @ 48 kHz), rank 11, 1024-sample blocks",
                   "cpu_sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t0,
    }
    print(json.dumps(line), flush=True)


def timed_blocks(batch_call, blocks, stream, barrier):
    """Device time (ms, CUDA events on `stream`) of `blocks` back-to-back one-frame process calls."""
    import torch
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for t in range(blocks):
        batch_call(t)
    e1.record(stream)
    barrier()
    return e0.elapsed_time(e1)


def max_over_ranks(x, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_latency_configs(pkg, args, rank, local_rank, world, barrier, peak):
    """BASELINE configs[0] and [1] -- the latency-bound shapes (mono 65 536 taps in 1024-sample calls;
    stereo 192 000 taps, rank 9, 256-sample calls, phases 0 / 0.5: the job-list path) on ONE GPU:
    device time per call back to back, and what a synchronous host call on page-locked buffers sees
    when the host comes back once per millisecond."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import synth
    out = {}
    for key, n, taps, rnk, block, phases in (("cfg1", 1, 65536, 11, 1024, (0.0,)), ("cfg2", 2, 192000, 9, 256, (0.0, 0.5))):
        b = pkg.ConvolverBatch(n, local_rank)
        for c in range(n):
            assert b.init(c, synth.decaying_ir(c, taps), rnk, phases[c % len(phases)])
        calls = 512
        src = torch.rand((n, calls * block), device="cuda") * 2 - 1
        dst = torch.empty_like(src)
        st = torch.cuda.ExternalStream(b.stream())
        torch.cuda.synchronize()

        def run():
            for i in range(calls):
                b.process_device(dst.data_ptr() + 4 * i * block, src.data_ptr() + 4 * i * block, calls * block, block, None)
        run()
        b.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            for _ in range(4):
                run()
            e1.record(st)
        torch.cuda.synchronize()
        dev_us = e0.elapsed_time(e1) * 1e3 / (4 * calls)
        hs = torch.rand((n, block)).pin_memory()
        hd = torch.empty((n, block)).pin_memory()
        a, o = hs.numpy(), hd.numpy()
        lat = []
        for i in range(260):
            t_wait = time.perf_counter() + 1e-3
            while time.perf_counter() < t_wait:
                pass
            t0 = time.perf_counter()
            b.process(a, o)
            lat.append((time.perf_counter() - t0) * 1e6)
        lat = np.sort(np.array(lat[60:]))
        out[key] = {"instances": n, "taps": taps, "rank": rnk, "call_samples": block,
                    "device_us_per_call": dev_us, "host_call_us_median": float(lat[len(lat) // 2]),
                    "host_call_us_p99": float(lat[int(len(lat) * 0.99)]),
                    "block_period_us_at_48k": block / 48000.0 * 1e6}
        b.close()
    out["note"] = ("device: back-to-back calls on the batch's stream, CUDA events; host: synchronous calls on page-locked "
                   "buffers, one per millisecond, wall clock around the call (python ctypes included)")
    return out


def run_strong_cfg3(pkg, args, rank, local_rank, world, barrier, peak):
    """BASELINE configs[2] read literally: the 64-channel batch sharded by channel over the ranks
    (64 / N channels per GPU, fixed total work), no collective."""
    import torch
    import synth
    from lsp_dsp_units_b200 import sharding
    lo, hi = sharding.channel_shard(INSTANCES, world, rank)
    n = hi - lo
    b = pkg.ConvolverBatch(n, device=local_rank)
    irs = [synth.decaying_ir(c, TAPS) for c in range(4)]
    for c in range(n):
        assert b.init(c, irs[(lo + c) % 4], RANK, 0.0)
    frames = BINS
    g = torch.Generator(device="cuda").manual_seed(0x5EED1000 + rank)
    src = torch.rand((n, 64 * BLOCK), generator=g, device="cuda") * 2.0 - 1.0
    dst = torch.empty_like(src)
    # the batch's OWN stream: there the engine knows every enqueued operation and may run a block's
    # input transform ahead of the previous block's tail (option "early_src", include/b200conv.h)
    stream = torch.cuda.ExternalStream(b.stream())
    sp, dp = src.data_ptr(), dst.data_ptr()

    def call(t):
        o = 4 * (t % 64) * BLOCK
        b.process_device(dp + o, sp + o, 64 * BLOCK, BLOCK, None)

    torch.cuda.synchronize()                    # the buffers were filled on torch's current stream
    with torch.cuda.stream(stream):
        for t in range(frames):                 # fill the ring
            call(t)
        reps = 4
        ms = timed_blocks(call, reps * frames, stream, barrier)
    ms = max_over_ranks(ms, world)
    b.close()
    us = ms * 1e3 / (reps * frames)
    rate = INSTANCES * BLOCK / (us * 1e-6)
    per_gpu_bytes = n * BYTES_PER_INSTANCE_FRAME
    return {
        "workload": "cfg3 strong: 64 ch x 480000 taps TOTAL, %d ch per GPU, rank 11, 1024-sample calls" % n,
        "n_gpus": world, "channels_per_gpu": n, "samples_per_s": rate, "us_per_block": us,
        "algorithmic_bytes_per_block_per_gpu": per_gpu_bytes,
        "share_of_hbm_roofline_per_gpu": per_gpu_bytes / (us * 1e-6) / 1e9 / peak,
        "working_set_mb_per_gpu": 2 * n * (BINS + 1) * F * 8 / 1e6,
        "note": "working set per GPU (IR spectra + ring) below ~126 MB sits in L2: a share > 1 of the HBM "
                "roofline is then L2 traffic, not DRAM (see profiles/ for the ncu dram__bytes of this shape)",
        "collective": "none (independent channels)",
    }


def run_cfg5(pkg, args, rank, local_rank, world, barrier, peak):
    """BASELINE configs[4]: ONE 8-channel convolver with a 120 s IR (5.76 M taps, 5625 partitions of
    1024 taps) split by partition range over the ranks; the partial output blocks are summed inside
    the kernel tails, all-to-all over NVLink peer memory (no collective call per block).  Parity:
    channel 0 against float64 FFT convolution over the WHOLE impulse-response length."""
    import numpy as np
    import torch
    import synth
    from lsp_dsp_units_b200 import sharding
    C5, TAPS5 = 8, 5760000
    bins5 = (TAPS5 + F - 1) // F
    irs = [synth.decaying_ir(100 + c, TAPS5) for c in range(C5)]
    conv = sharding.PartitionShardedConvolver(pkg, C5, RANK, local_rank, reduce="fused")
    assert conv.init(irs), "device allocation failed"
    init_ms, connect_ms = conv.init_ms, conv.connect_ms
    p_lo, p_hi, _, _ = sharding.partition_shard(TAPS5, F, world, rank)
    stream = torch.cuda.ExternalStream(conv.batch.stream())    # the batch's own stream (see run_strong_cfg3)

    # ---- parity over the whole IR length: 16 blocks of noise, then silence --------------------
    nz = 16
    total = bins5 + nz
    g = torch.Generator(device="cuda").manual_seed(0x5EED5000)     # the same input on every rank
    head = torch.rand((C5, nz * BLOCK), generator=g, device="cuda") * 2.0 - 1.0
    zeros = torch.zeros((C5, BLOCK), device="cuda")
    out = torch.empty((C5, total * BLOCK), device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        for t in range(total):
            src = head[:, t * BLOCK:(t + 1) * BLOCK] if t < nz else zeros
            conv.process_device(out[:, t * BLOCK:(t + 1) * BLOCK], src, BLOCK, None)
        stream.synchronize()
    err = None
    if rank == 0:
        from scipy.signal import fftconvolve
        x = head[0].cpu().numpy().astype(np.float64)
        full = fftconvolve(x, irs[0].astype(np.float64))
        want = np.zeros(total * BLOCK)
        want[:min(full.size, want.size)] = full[:want.size]
        got = out[0].cpu().numpy().astype(np.float64)
        err = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
    same = True
    if world > 1:
        import torch.distributed as dist
        ref0 = out[:, -64 * BLOCK:].clone()
        dist.broadcast(ref0, src=0)
        same = bool(torch.equal(ref0, out[:, -64 * BLOCK:]))
    del out

    # ---- throughput: back-to-back 1024-sample blocks ------------------------------------------
    g = torch.Generator(device="cuda").manual_seed(0x5EED5001)
    src = torch.rand((C5, 64 * BLOCK), generator=g, device="cuda") * 2.0 - 1.0
    dst = torch.empty_like(src)

    sp, dp, raw = src.data_ptr(), dst.data_ptr(), conv.batch

    def call(t):                                # lean host path: the block period is ~15 us at 8 GPUs
        o = 4 * (t % 64) * BLOCK
        raw.process_device(dp + o, sp + o, 64 * BLOCK, BLOCK, None)

    blocks = 2000
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        for t in range(256):
            call(t)
        ms = timed_blocks(call, blocks, stream, barrier)
    ms = max_over_ranks(ms, world)
    timed_out = conv.timed_out()
    flags = max_over_ranks(float(timed_out) + 2.0 * float(not same), world)
    conv.close()
    us = ms * 1e3 / blocks
    per_gpu_bytes = C5 * (16 * F * (p_hi - p_lo) + 24 * F)
    return {
        "workload": "cfg5: ONE 8-ch convolver, 5760000-tap IR (120 s), rank 11, 1024-sample blocks, "
                    "partition range split over %d GPU(s)" % world,
        "n_gpus": world, "partitions_total": bins5, "partitions_this_gpu": p_hi - p_lo,
        "samples_per_s": C5 * BLOCK / (us * 1e-6), "us_per_block": us, "blocks_timed": blocks,
        "realtime_factor": C5 * BLOCK / (us * 1e-6) / (C5 * 48000.0),
        "algorithmic_bytes_per_block_per_gpu": per_gpu_bytes,
        "share_of_hbm_roofline_per_gpu": per_gpu_bytes / (us * 1e-6) / 1e9 / peak,
        "max_err_vs_float64_of_peak": err,
        "init_ms": init_ms, "init_bytes_h2d_this_gpu": C5 * (min(TAPS5, p_hi * F) - p_lo * F) * 4,
        "reduce_connect_ms": connect_ms,
        "parity_span": "%d blocks = the whole IR length + %d (every partition of every rank contributes)" % (total, nz),
        "all_ranks_bit_identical": bool(int(flags) & 2 == 0),
        "peer_wait_timed_out": bool(int(flags) & 1),
        "reduce": ("fused into the k_frame tails: all-to-all over NVLink peer memory, every rank ends with "
                   "the sum, %d blocks in flight" % 4) if world > 1 else "none (one GPU holds every partition)",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=BINS)
    ap.add_argument("--e2e-frames", type=int, default=BINS)
    ap.add_argument("--cpu-blocks", type=int, default=192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--splits", type=int, default=0)
    ap.add_argument("--stages", type=int, default=0)
    ap.add_argument("--fused", type=int, default=1)
    ap.add_argument("--bias", type=int, default=6)
    ap.add_argument("--pdl", type=int, default=1)
    ap.add_argument("--zero-copy", type=int, default=1)
    ap.add_argument("--eager", type=int, default=1)
    ap.add_argument("--no-facade", action="store_true", help="skip the C++ facade / pointer-table e2e legs")
    ap.add_argument("--extras-timeout", type=int, default=420)
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra multi-GPU shapes (cfg3 strong scaling, cfg5 partition split)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step (rank 0, a seeded sample of 16 instances) "
                         "to DIR/convolver_dst.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pkg = ge.load()
    pkg.lib()
    batch = pkg.ConvolverBatch(INSTANCES, device=local_rank)
    batch.set_option("mac_splits", args.splits)
    batch.set_option("mac_stages", args.stages)
    batch.set_option("fused", args.fused)
    batch.set_option("fft_bias", args.bias)
    batch.set_option("pdl", args.pdl)
    batch.set_option("zero_copy", args.zero_copy)
    batch.set_option("eager", args.eager)

    # ---- synthetic data (SURVEY 8d): decaying-noise IRs, white-noise input --------------------
    # A handful of distinct seeded IRs/inputs are cycled over the 64 instances: timing does not
    # depend on the values, parity at full size is covered by tests/.
    base = rank * INSTANCES
    irs = [synth.decaying_ir(base + c, TAPS) for c in range(8)]
    t_init = time.perf_counter()
    ok = batch.init_many(list(range(INSTANCES)), [irs[c % 8] for c in range(INSTANCES)], RANK)
    assert ok, "device allocation failed"
    init_ms = (time.perf_counter() - t_init) * 1e3      # 64 x Convolver::init: upload + 30 016 partition transforms
    frames = args.frames_per_step
    n = frames * BLOCK
    g = torch.Generator(device="cuda").manual_seed(0x5EED0000 + rank)
    src = torch.rand((INSTANCES, n), generator=g, device="cuda", dtype=torch.float32) * 2.0 - 1.0
    dst = torch.empty_like(src)
    stream = torch.cuda.Stream()
    sp, dp = src.data_ptr(), dst.data_ptr()

    def step():
        # `frames` consecutive Convolver::process calls of 1024 samples on all 64 instances
        for f in range(frames):
            batch.process_device(dp + 4 * f * BLOCK, sp + 4 * f * BLOCK, n, BLOCK, stream.cuda_stream)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step()
        barrier()
        batch.reset_stats()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps - 1)]
        ev0.record(stream)
        for s_i in range(args.steps):
            step()
            if s_i < args.steps - 1:
                marks[s_i].record(stream)        # per-step durations (min / median), SURVEY 8d
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        edges = [ev0] + marks + [ev1]
        step_ms = sorted(edges[i].elapsed_time(edges[i + 1]) for i in range(args.steps))
        clocks = sampler.stop() if rank == 0 else None
        stats = batch.stats()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, dst)

        # ---- roofline pass: per-launch duration of k_mac, CUDA events on the launching stream ---
        batch.set_profiling(True)
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        mac_ms, mac_n = batch.profile()
        batch.set_profiling(False)

    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    samples_per_rank = args.steps * frames * BLOCK * INSTANCES
    value = world * samples_per_rank / (ms_max * 1e-3)

    # ---- end-to-end through the host-pointer C ABI (pinned host buffers, H2D + D2H inside) -----
    e2e_frames = args.e2e_frames
    hsrc = torch.empty((INSTANCES, BLOCK), dtype=torch.float32).pin_memory()
    hsrc.copy_(src[:, :BLOCK].cpu())
    hdst = torch.empty((INSTANCES, BLOCK), dtype=torch.float32).pin_memory()
    hs, hd = hsrc.numpy(), hdst.numpy()
    for _ in range(8):
        batch.process(hs, hd)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for f in range(e2e_frames):
            batch.process(hs, hd)       # b200conv_process_planar: H2D, kernels, D2H, sync
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * e2e_frames * BLOCK * INSTANCES / float(t.item())
    io_bytes = e2e_frames * INSTANCES * BLOCK * 4

    # ---- the reference-facing call itself: 64 x lsp::dspu::Convolver::process (C++ facade, pageable
    #      buffers, serial loop) and the explicit coalescing API b200conv_process (pointer table) -----
    facade = None
    exe = os.path.join(ROOT, "lsp-dsp-units_b200", "host", "bench_facade")
    if rank == 0 and world == 1 and os.path.exists(exe) and not args.no_facade:
        try:
            env = dict(os.environ, B200CONV_DEVICE=str(local_rank))
            out = subprocess.run([exe, str(INSTANCES), str(TAPS), str(RANK), str(BLOCK), "200"],
                                 capture_output=True, text=True, timeout=300, env=env)
            facade = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as exc:
            facade = {"error": "%s: %s" % (type(exc).__name__, exc)}

    peak, peak_src = hbm_peak()
    extras = {}
    batch.close()
    del src, dst
    torch.cuda.empty_cache()
    extras_hung = False
    if not args.no_extras:
        # the multi-GPU shapes that CAN fail: fixed total work, and the one real exchange step.
        # They run on a worker thread with a deadline: whatever happens to them (an exception on
        # one rank, a peer that never answers), the headline line above is still printed.
        import threading

        def run_extras():
            torch.cuda.set_device(local_rank)
            legs = [("strong_cfg3", run_strong_cfg3), ("cfg5_split", run_cfg5)]
            if world == 1:
                legs.append(("latency_configs", run_latency_configs))
            for name, fn in legs:
                try:
                    extras[name] = fn(pkg, args, rank, local_rank, world, barrier, peak)
                except Exception as exc:
                    extras[name] = {"error": "%s: %s" % (type(exc).__name__, exc)}
                    break                               # the ranks may be out of step now

        th = threading.Thread(target=run_extras, daemon=True)
        th.start()
        th.join(timeout=args.extras_timeout)
        extras_hung = th.is_alive()
        if extras_hung:
            extras.setdefault("error", "extra shapes did not finish within %d s" % args.extras_timeout)

    if rank == 0:
        bytes_per_launch = INSTANCES * BYTES_PER_INSTANCE_FRAME
        iso_ms = mac_ms / max(1, mac_n)             # event-bracketed launches (no overlap between them)
        if args.fused:
            # the timed region is nothing but k_frame launches, back to back on one stream with
            # programmatic dependent launch: its duration / launches is the kernel's average
            # launch duration as deployed (tail of block t overlaps the stream of block t+1)
            mac_avg_ms = ms / (args.steps * frames)
        else:
            mac_avg_ms = iso_ms
        achieved = bytes_per_launch / (mac_avg_ms * 1e-3) / 1e9 if mac_avg_ms > 0 else None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "mac_traffic.json")) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": "cfg3: 64 ch x 480000-tap IR (10 s @ 48 kHz) per GPU, rank 11, "
                            "1024-sample process() calls, %d calls per step" % frames,
                "instances_per_gpu": INSTANCES, "taps": TAPS, "rank": RANK, "block": BLOCK,
                "partitions": BINS, "frames_per_step": frames,
                "l2": "working set 2 x 246 MB (IR spectra + input-spectrum ring) per GPU streams "
                      "once per call: inputs larger than the 126 MB L2, no flush needed",
                "sharding": "independent channels per rank, no collective",
                "init_ms": init_ms, "init_bytes_h2d": INSTANCES * TAPS * 4,
                "value_share_of_hbm_roofline": value / world * (16 * BINS + 24) / (peak * 1e9),
            },
            "clocks": clocks,
            "step_ms": {"min": step_ms[0], "median": step_ms[len(step_ms) // 2], "max": step_ms[-1]},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": io_bytes,
                    "d2h_bytes_per_step": io_bytes,
                    "api": "b200conv_process_planar (pinned host buffers, synchronous per 1024-sample call; %s; "
                           "the next block's partitions q >= 1 are summed while the host is away)"
                           % ("kernels read/write the pinned buffers over PCIe" if args.zero_copy else "staged H2D/D2H copies")},
            "gpu_launches": stats["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "kernel": "k_frame<11>" if args.fused else "k_mac", "launch_ms": mac_avg_ms,
                         "launches_timed": (args.steps * frames) if args.fused else mac_n,
                         "isolated_launch_ms": iso_ms, "isolated_launches_timed": mac_n,
                         "isolated_frac": bytes_per_launch / (iso_ms * 1e-3) / 1e9 / peak if iso_ms > 0 else None,
                         "algorithmic_bytes_per_launch": bytes_per_launch, "peak_source": peak_src},
        }
        if facade is not None:
            for k in ("facade_64x_process", "pointer_table_pageable", "error"):
                if k in facade:
                    line["e2e"][k] = facade[k]
        line.update(extras)
        if (world == 1) and (not args.no_cpu_baseline):
            cores = min(os.cpu_count() or 1, INSTANCES)
            rate, sec, kind = cpu_reference_rate(cores, 192)
            one_rate, _, _ = cpu_reference_rate(1, 96)
            line["cpu_baseline"] = {
                "value": rate, "unit": UNIT, "cores": cores, "kind": kind, "one_core_value": one_rate,
                "sample": "%d of the 64 instances (one per host thread), 480000-tap IR, rank 11, 192 "
                          "process() calls of 1024 samples each after 4 warm calls (%.1f s); reference "
                          "Convolver.cpp compiled verbatim over restated scalar dsp:: kernels "
                          "(lsp-dsp-lib AVX/SSE is not available offline)" % (cores, sec)}
        print(json.dumps(line), flush=True)

    if extras_hung:
        sys.stdout.flush()
        os._exit(0)                 # a stuck collective cannot be unwound; the line is out
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
