"""The batched Equalizer, SpectralProcessor and SpectralSplitter at batch sizes where every CTA
processes two or three instances (k_eq, k_sp and the function kernels, k_ss all loop
`for (inst = blockIdx.x; inst < n_inst; inst += gridDim.x)`), and at the shapes the throughput
tools measure (tools/bench_eq.py, tools/bench_sp.py).  What k_eq carries from one instance to the
next -- the TMA prefetch of the next instance's block, the state read ahead, the barrier phases --
and the per-instance offsets of k_sp / k_ss only run when a CTA gets a second instance.

Every row is checked against the vectorised float64 models of tests/batch_models.py (held to the
per-instance models by tests/test_batch_models.py), with the tolerances of the per-object files:
1e-5 of the row's peak for the equalizer, 2e-5 for the spectral objects.  Every instance has its
own kernel / tables / phase / input, so output from the wrong instance cannot pass.  Rows
{0, 1, g-1, g, g+1, 2g-1, 2g, n-1} are then run alone in a batch of 8 (one instance per CTA) and
must come out bit-identical: an instance's arithmetic does not depend on which CTA runs it, or in
which round."""
import numpy as np
import pytest

import batch_models

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOL_EQ = 1e-5
TOL_SPECTRAL = 2e-5
HOST_BYTES = 512 << 20          # model working set per slab of instances


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# launch geometry, restated from the sources

def fft_cfg(rank):
    """FftCfg<RANK> (csrc/kernels.cuh:366-397): threads and shared memory of a transform."""
    N = 1 << rank
    M, P = N // 2, N // 4
    logp = rank - 2
    nh = 1 if rank >= 16 else 2
    bf = nh * P // 4
    T = 512 if bf >= 512 else (32 if bf < 32 else bf)
    pp = tws = rank <= 12
    work = nh * P
    ns0 = 2 if (logp & 1) else 1
    tw_total = (P - ns0) + P + M // 2 + 1
    twc_n = (P - ns0) // 3
    smem = (work * (2 if pp else 1) + (tw_total if tws else twc_n)) * 8
    return {"N": N, "M": M, "T": T, "PP": pp, "SMEM": smem}


def eq_smem(rank):
    """EqCfg<RANK>::SMEM (csrc/equalizer.cuh:149-161), RANK = fir_rank + 1."""
    c = fft_cfg(rank)
    if not c["PP"]:
        return c["SMEM"]
    off_h = (c["SMEM"] + 127) & ~127
    return off_h + c["M"] * 8 + c["M"] * 4 + 16


def resident_grid(jobs, threads, smem, sms):
    """resident_grid (csrc/engine.cu:78-94)."""
    per_sm = min((227 * 1024) // (smem + 1024), 2048 // threads)
    per_sm = min(max(per_sm, 1), 16)
    return min(jobs, per_sm * sms)


def eq_grid(n, fir_rank, sms):
    """k_eq's launch (csrc/equalizer.cuh:381): resident_grid(n_inst, C::T, EqCfg::SMEM)."""
    return resident_grid(n, fft_cfg(fir_rank + 1)["T"], eq_smem(fir_rank + 1), sms)


def spectral_grid(n, sms):
    """k_sp (csrc/spectral_host.cuh:507) and k_ss (csrc/splitter.cuh:583): min(n, 8 SMs)."""
    return min(n, 8 * sms)


def wide(g):
    """2 g + 37 instances: every CTA gets two or three of them and the last round is ragged."""
    n = 2 * g + 37
    assert n >= 2 * g + 1 and n % g != 0, (n, g)
    return n


def solo_rows(n, g):
    return sorted({0, 1, g - 1, g, g + 1, 2 * g - 1, 2 * g, n - 1})


def test_launch_geometry_on_148_sms():
    """The restatement gives the grids of the design notes on a 148-SM B200."""
    assert [eq_grid(10 ** 6, r, 148) for r in range(7, 16)] == [2368, 2368, 1480, 740, 296, 592, 444, 148, 148]
    assert [fft_cfg(r + 1)["T"] for r in range(7, 16)] == [32, 64, 128, 256, 512, 512, 512, 512, 512]
    assert spectral_grid(10 ** 6, 148) == 1184 and wide(1184) == 2405


# ---------------------------------------------------------------------------------------------
# per-row data: distinct for every instance, regenerated for any subset of rows

_BASE = np.random.Generator(np.random.PCG64(0xB47C4)).uniform(-1.0, 1.0, (67, 1 << 15))


def row_curves(rows, length, salt):
    """[len(rows), length] float64: two of 67 seeded curves mixed with weights unique to the row."""
    rows = np.asarray(rows, dtype=np.int64)
    a = _BASE[(7 * rows + salt) % 67, :length]
    b = _BASE[(11 * rows + 3 * salt + 1) % 67, :length]
    wa = 1.0 + rows / 8191.0
    wb = 0.5 + ((rows * 2654435761 + salt) % 1000) / 1000.0
    return a * wa[:, None] + b * wb[:, None]


def row_kernels(rows, F, salt):
    k = row_curves(rows, F, salt) * np.exp(-np.arange(F) / (F / 4.0))
    return (k / np.sqrt(np.sum(k * k, axis=1, keepdims=True))).astype(np.float32)


def row_gains(rows, N, salt):
    return (0.85 + 0.3 * row_curves(rows, N, salt)).astype(np.float32)


def row_tables(rows, N, salt):
    return (row_curves(rows, N, salt) + 1j * row_curves(rows, N, salt + 1)).astype(np.complex64)


def dev_input(n, T, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand((n, T), generator=g, device="cuda") * 2.0 - 1.0


def slabs(n, bytes_per_row):
    step = max(1, HOST_BYTES // bytes_per_row)
    return [np.arange(a, min(n, a + step)) for a in range(0, n, step)]


def assert_rows_close(got, want, tol, what, floor=1.0):
    """Every row within tol x its own peak (at least `floor`)."""
    err = np.max(np.abs(got.astype(np.float64) - want), axis=-1)
    peak = np.maximum(floor, np.max(np.abs(want), axis=-1))
    bad = np.argwhere(err > tol * peak)
    assert bad.size == 0, "%s: %d rows off, first %s: err %.3e peak %.3e" % (
        what, len(bad), bad[0].tolist(), err[tuple(bad[0])], peak[tuple(bad[0])])


def assemble(n, T, calls, bufs):
    """The output of every call from the buffer that call wrote (device)."""
    out = torch.empty((n, T), device="cuda")
    pos = 0
    for size, mode in calls:
        out[:, pos:pos + size] = bufs[mode][:, pos:pos + size]
        pos += size
    return out


def io_buffers(X, T):
    """'even': its own [n][T] matrix; 'odd': rows T + 1 floats apart (every other row 4 bytes off
    8-byte alignment); 'inplace': a copy of the input the calls overwrite."""
    n = X.shape[0]
    odd = torch.full((n * (T + 1),), float("nan"), device="cuda")
    return {"even": torch.full_like(X, float("nan")), "odd": odd.view(n, T + 1), "inplace": X.clone()}


def io_pointers(X, bufs, pos, mode, T):
    src = (bufs["inplace"] if mode == "inplace" else X).data_ptr() + 4 * pos
    dst = bufs[mode].data_ptr() + 4 * pos
    return dst, (T + 1 if mode == "odd" else T), src, T


# ---------------------------------------------------------------------------------------------
# Equalizer

def eq_events(n, g):
    """Row masks of the hand-overs, in terms of the CTA b = i mod g and the round r = i div g: the
    same CTA sees hand-over -> hand-over (b, b + g), hand-over -> ordinary and ordinary -> hand-over."""
    i = np.arange(n)
    b, r = i % g, i // g
    smooth = ((r == 0) & (b % 3 != 2)) | ((r == 1) & (b % 3 != 1)) | ((r == 2) & (b % 2 == 0))
    now = ~smooth & (b % 5 == 0)
    pending = smooth & (b % 7 == 0)                 # replaced at once while its cross-fade is pending
    smooth2 = (b + r) % 4 == 1
    return smooth, now, pending, smooth2


def eq_schedule(F, n, g):
    smooth, now, pending, smooth2 = eq_events(n, g)
    return [("call", F, "even"), ("call", F, "odd"),
            ("set", smooth, 1, True), ("set", now, 2, False), ("set", pending, 3, False),
            ("call", F, "inplace"),                 # a hand-over block taken by a whole-block call
            ("call", 37, "even"), ("call", 2 * F + 11, "odd"), ("call", F - 48, "inplace"),
            ("clear",),
            ("call", F, "even"), ("set", smooth2, 4, True), ("call", F, "odd"),
            ("call", F, "even"), ("call", F, "inplace")]


def eq_run_gpu(pkg, fir_rank, rows, X, schedule):
    F = 1 << fir_rank
    n, T = X.shape
    eq = pkg.EqualizerBatch(n, fir_rank, device=0)
    k0 = row_kernels(rows, F, 0)
    for j in range(n):
        eq.set_kernel(j, k0[j])
    bufs = io_buffers(X, T)
    torch.cuda.synchronize()
    calls, pos = [], 0
    for step in schedule:
        if step[0] == "call":
            _, size, mode = step
            eq.process_device(*io_pointers(X, bufs, pos, mode, T), size)
            calls.append((size, mode))
            pos += size
        elif step[0] == "set":
            _, mask, salt, smooth = step
            sel = np.flatnonzero(mask[rows])
            ks = row_kernels(rows[sel], F, salt)
            for j, k in zip(sel, ks):
                eq.set_kernel(int(j), k, smooth)
        else:
            eq.clear()
    eq.sync()
    assert pos == T
    out = assemble(n, T, calls, bufs)
    eq.close()
    return out


def eq_check_model(fir_rank, out, X, schedule):
    F = 1 << fir_rank
    n, T = X.shape
    for rows in slabs(n, 8 * (8 * F + 3 * T)):
        m = batch_models.BatchEqualizer(rows.size, fir_rank)
        m.set_kernel(np.arange(rows.size), row_kernels(rows, F, 0))
        x = X[rows[0]:rows[-1] + 1].cpu().numpy().astype(np.float64)
        want = np.empty_like(x)
        pos = 0
        for step in schedule:
            if step[0] == "call":
                want[:, pos:pos + step[1]] = m.process(x[:, pos:pos + step[1]])
                pos += step[1]
            elif step[0] == "set":
                _, mask, salt, smooth = step
                sel = np.flatnonzero(mask[rows])
                m.set_kernel(sel, row_kernels(rows[sel], F, salt), smooth)
            else:
                m.clear()
        got = out[rows[0]:rows[-1] + 1].cpu().numpy()
        assert_rows_close(got, want, TOL_EQ, "equalizer rows %d..%d" % (rows[0], rows[-1]), floor=0.0)


@pytest.mark.parametrize("fir_rank", list(range(7, 16)))
def test_equalizer_every_row_of_a_wide_batch(pkg, fir_rank):
    F = 1 << fir_rank
    g = eq_grid(1 << 30, fir_rank, sm_count())
    n = wide(g)
    print("equalizer fir_rank %d: n = %d, g = %d" % (fir_rank, n, g))
    assert eq_grid(n, fir_rank, sm_count()) == g
    schedule = eq_schedule(F, n, g)
    T = sum(s[1] for s in schedule if s[0] == "call")
    assert T % 2 == 0
    X = dev_input(n, T, 1000 + fir_rank)
    rows = np.arange(n)
    out = eq_run_gpu(pkg, fir_rank, rows, X, schedule)
    eq_check_model(fir_rank, out, X, schedule)
    # the same rows alone, one instance per CTA: bit-identical.  (Under the odd stride a uniform
    # row pitch cannot give these rows their big-batch 8-byte alignment; the direct store of a
    # whole-block call and the store through vOutBuffer write the same float.)
    solo = solo_rows(n, g)
    small = eq_run_gpu(pkg, fir_rank, np.array(solo), X[solo].contiguous(), schedule)
    assert torch.equal(small, out[solo])


@pytest.mark.parametrize("n,fir_rank", [(4096, 10), (4096, 12), (1024, 13), (256, 15)])
def test_equalizer_bench_shapes(pkg, n, fir_rank):
    """tools/bench_eq.py's cases: whole-block device calls on contiguous rows."""
    F = 1 << fir_rank
    print("equalizer bench %d:%d: g = %d" % (n, fir_rank, eq_grid(n, fir_rank, sm_count())))
    schedule = [("call", F, "even")] * 5
    X = dev_input(n, 5 * F, 2000 + fir_rank)
    out = eq_run_gpu(pkg, fir_rank, np.arange(n), X, schedule)
    eq_check_model(fir_rank, out, X, schedule)


# ---------------------------------------------------------------------------------------------
# SpectralProcessor

PHASES = np.array([0.0, 0.25, 0.37, 0.5, 1.0])
SP_NONE, SP_GAIN, SP_COMPLEX, SP_FUNCTION = 0, 1, 2, 3


def sp_setup(n, g):
    """Kinds and phases interleaved so that the instances one CTA walks differ in both."""
    i = np.arange(n)
    b, r = i % g, i // g
    return (b + r) % 4, PHASES[(b + 2 * r) % 5]


def sp_calls(rank, seed, T):
    """Sizes below, at and above the hop, and random ones; modes rotate over the three layouts."""
    F = 1 << (rank - 1)
    rng = np.random.default_rng(seed)
    sizes, pos = [], 0
    for j in range(10 ** 6):
        s = [F - 1, F, F + 1, 1, int(rng.integers(2, 4 * F))][j % 5]
        s = min(s, T - pos)
        if s == 0:
            break
        sizes.append(s)
        pos += s
    return [(s, ("even", "odd", "inplace")[j % 3]) for j, s in enumerate(sizes)]


def sp_run_gpu(pkg, rank, rows, X, calls, kind, phases, spread=()):
    N = 1 << rank
    n, T = X.shape
    sp = pkg.SpectralProcessorBatch(n, rank, device=0)
    fi = np.flatnonzero(kind[rows] == SP_FUNCTION)
    if fi.size:
        G = torch.from_numpy(row_gains(rows[fi], N, 7)).cuda()
        lut = torch.full((n,), -1, dtype=torch.long, device="cuda")
        lut[torch.from_numpy(fi).cuda()] = torch.arange(fi.size, device="cuda")

        def fn(X, instances, positions, rank):
            X.mul_(G[lut[instances]])
        sp.set_function(fn)
    for j, i in enumerate(rows):
        sp.set_phase(j, float(phases[i]))
        if kind[i] == SP_GAIN:
            sp.bind_gain(j, row_gains([i], N, 5)[0])
        elif kind[i] == SP_COMPLEX:
            sp.bind_complex(j, row_tables([i], N, 6)[0])
        elif kind[i] == SP_FUNCTION:
            sp.bind_function(j)
    bufs = io_buffers(X, T)
    torch.cuda.synchronize()
    pos, rem = 0, []
    for size, mode in calls:
        dst, dst_stride, src, src_stride = io_pointers(X, bufs, pos, mode, T)
        sp.process_device(dst, dst_stride, src, src_stride, size)
        rem.append([sp.remaining(j) for j in spread])
        pos += size
    sp.sync()
    out = assemble(n, T, calls, bufs)
    sp.close()
    return out, np.array(rem)


def sp_check_model(rank, out, X, calls, kind, phases, spread=(), rem=None):
    N = 1 << rank
    n, T = X.shape
    spread = np.asarray(spread, dtype=np.int64)
    for rows in slabs(n, 8 * (12 * N + 3 * T)):
        k = kind[rows]
        tables = np.zeros((rows.size, N), dtype=np.complex128)
        sel = k == SP_GAIN
        tables[sel] = row_gains(rows[sel], N, 5)
        sel = k == SP_COMPLEX
        tables[sel] = row_tables(rows[sel], N, 6)
        sel = k == SP_FUNCTION
        gf = np.zeros((rows.size, N))
        gf[sel] = row_gains(rows[sel], N, 7)
        m = batch_models.BatchSpectralProcessor(rank, phases[rows], np.select(
            [k == SP_NONE, (k == SP_GAIN) | (k == SP_COMPLEX)], [0, 1], 2), tables, lambda X, r: X * gf[r])
        x = X[rows[0]:rows[-1] + 1].cpu().numpy().astype(np.float64)
        want = np.empty_like(x)
        here = np.flatnonzero((spread >= rows[0]) & (spread <= rows[-1]))
        pos = 0
        for c, (size, mode) in enumerate(calls):
            want[:, pos:pos + size] = m.process(x[:, pos:pos + size])
            pos += size
            if rem is not None and here.size:
                assert np.array_equal(rem[c, here], m.remaining()[spread[here] - rows[0]]), (c, spread[here])
        got = out[rows[0]:rows[-1] + 1].cpu().numpy()
        assert_rows_close(got, want, TOL_SPECTRAL, "spectral processor rows %d..%d" % (rows[0], rows[-1]))


@pytest.mark.parametrize("rank", list(range(7, 16)))
def test_spectral_processor_every_row_of_a_wide_batch(pkg, rank):
    N, F = 1 << rank, 1 << (rank - 1)
    g = spectral_grid(1 << 30, sm_count())
    n = wide(g)
    print("spectral processor rank %d: n = %d, g = %d" % (rank, n, g))
    kind, phases = sp_setup(n, g)
    T = N + 5 * F
    calls = sp_calls(rank, 3000 + rank, T)
    X = dev_input(n, T, 3000 + rank)
    spread = np.unique(np.concatenate([solo_rows(n, g), np.linspace(0, n - 1, 41).astype(np.int64)]))
    out, rem = sp_run_gpu(pkg, rank, np.arange(n), X, calls, kind, phases, spread)
    sp_check_model(rank, out, X, calls, kind, phases, spread, rem)
    solo = solo_rows(n, g)
    small, _ = sp_run_gpu(pkg, rank, np.array(solo), X[solo].contiguous(), calls, kind, phases)
    assert torch.equal(small, out[solo])


@pytest.mark.parametrize("rank,n,call", [(8, 4096, 4096), (10, 4096, 8192), (12, 2048, 16384), (14, 512, 65536)])
def test_spectral_processor_bench_shapes(pkg, rank, n, call):
    """tools/bench_sp.py's cases: every instance gain-bound, phase 0, device calls of `call` samples."""
    print("spectral processor bench rank %d: n = %d, g = %d" % (rank, n, spectral_grid(n, sm_count())))
    kind, phases = np.full(n, SP_GAIN), np.zeros(n)
    calls = [(call, "even")] * 2
    X = dev_input(n, 2 * call, 4000 + rank)
    out, _ = sp_run_gpu(pkg, rank, np.arange(n), X, calls, kind, phases)
    sp_check_model(rank, out, X, calls, kind, phases)


# ---------------------------------------------------------------------------------------------
# SpectralSplitter

SS_UNBOUND, SS_COMPLEX, SS_GAIN, SS_SINK = 0, 1, 2, 3
SENTINEL = 1234.5


def ss_setup(n, g, H):
    """Handler kinds and phases per instance, mixed within every CTA; some instances bind nothing."""
    i = np.arange(n)
    b, r = i % g, i // g
    kinds = (b + 2 * r + np.arange(H)[:, None]).T % 4
    kinds[(b + r) % 9 == 4] = SS_UNBOUND
    return kinds, PHASES[(b + 3 * r) % 5]


def ss_run_gpu(pkg, rank, chunk, rows, X, sizes, kinds, phases):
    N = 1 << rank
    n, T = X.shape
    H = kinds.shape[1]
    ss = pkg.SpectralSplitterBatch(n, rank, H, device=0)
    if chunk:
        ss.set_chunk_rank(chunk)
    for j, i in enumerate(rows):
        ss.set_phase(j, float(phases[i]))
        for h in range(H):
            if kinds[i, h] == SS_COMPLEX:
                ss.bind_complex(j, h, row_tables([i], N, 10 + 2 * h)[0])
            elif kinds[i, h] == SS_GAIN:
                ss.bind_gain(j, h, row_gains([i], N, 10 + 2 * h)[0])
            elif kinds[i, h] == SS_SINK:
                ss.bind_sink(j, h)
    dst_stride = T + 3
    band_stride = n * dst_stride + 17
    D = torch.full((H * band_stride,), SENTINEL, device="cuda")
    torch.cuda.synchronize()
    pos = 0
    for size in sizes:
        ss.process_device(D.data_ptr() + 4 * pos, band_stride, dst_stride, X.data_ptr() + 4 * pos, T, size)
        pos += size
    ss.sync()
    assert pos == T
    out = torch.stack([D[h * band_stride:h * band_stride + n * dst_stride].view(n, dst_stride)[:, :T] for h in range(H)])
    ss.close()
    return out


def ss_check_model(rank, chunk, out, X, sizes, kinds, phases):
    N = 1 << rank
    n, T = X.shape
    H = kinds.shape[1]
    for rows in slabs(n, 8 * H * (4 * N + 3 * T)):
        k = kinds[rows]
        tables = np.zeros((rows.size, H, N), dtype=np.complex128)
        for h in range(H):
            sel = k[:, h] == SS_COMPLEX
            tables[sel, h] = row_tables(rows[sel], N, 10 + 2 * h)
            sel = k[:, h] == SS_GAIN
            tables[sel, h] = row_gains(rows[sel], N, 10 + 2 * h)
        mk = np.select([k == SS_UNBOUND, k == SS_SINK], [0, 2], 1)
        m = batch_models.BatchSpectralSplitter(rank, mk, tables, phases[rows], chunk)
        x = X[rows[0]:rows[-1] + 1].cpu().numpy().astype(np.float64)
        want = np.concatenate([m.process(x[:, a:a + s]) for a, s in zip(np.cumsum([0] + sizes[:-1]), sizes)], axis=2)
        got = out[:, rows[0]:rows[-1] + 1].cpu().numpy()
        unbound = (k == SS_UNBOUND).T
        assert np.all(got[unbound] == SENTINEL), "an unbound handler's row was written"
        assert_rows_close(got[~unbound], want[~unbound], TOL_SPECTRAL, "splitter rows %d..%d" % (rows[0], rows[-1]))


def ss_sizes(rank, chunk, seed, T):
    F = 1 << ((chunk or rank) - 1)
    rng = np.random.default_rng(seed)
    sizes, pos = [], 0
    while pos < T:
        s = min(int(rng.integers(1, 3 * F)), T - pos)
        sizes.append(s)
        pos += s
    return sizes


@pytest.mark.parametrize("rank", list(range(7, 15)))
def test_spectral_splitter_every_row_of_a_wide_batch(pkg, rank):
    N = 1 << rank
    H = 1 + rank % 4
    chunk = rank - 1
    F = 1 << (chunk - 1)
    g = spectral_grid(1 << 30, sm_count())
    n = wide(g)
    print("spectral splitter rank %d, chunk rank %d, %d handlers: n = %d, g = %d" % (rank, chunk, H, n, g))
    kinds, phases = ss_setup(n, g, H)
    T = N + 4 * F
    sizes = ss_sizes(rank, chunk, 5000 + rank, T)
    X = dev_input(n, T, 5000 + rank)
    out = ss_run_gpu(pkg, rank, chunk, np.arange(n), X, sizes, kinds, phases)
    ss_check_model(rank, chunk, out, X, sizes, kinds, phases)
    solo = solo_rows(n, g)
    small = ss_run_gpu(pkg, rank, chunk, np.array(solo), X[solo].contiguous(), sizes, kinds, phases)
    assert torch.equal(small, out[:, solo])


@pytest.mark.parametrize("rank,n,call", [(10, 2048, 8192), (12, 1024, 16384)])
def test_spectral_splitter_crossover_bench_shapes(pkg, rank, n, call):
    """tools/bench_sp.py's three-way crossover: three real-gain bands per instance, phase 0."""
    print("spectral splitter bench rank %d: n = %d, g = %d" % (rank, n, spectral_grid(n, sm_count())))
    kinds, phases = np.full((n, 3), SS_GAIN), np.zeros(n)
    X = dev_input(n, 2 * call, 6000 + rank)
    out = ss_run_gpu(pkg, rank, 0, np.arange(n), X, [call, call], kinds, phases)
    ss_check_model(rank, 0, out, X, [call, call], kinds, phases)
