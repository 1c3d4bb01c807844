"""The batched SpectralProcessor with the caller's own spectral function (b200conv_sp_set_function /
bind_function): every frame of a function-bound instance is transformed on the device, handed to a
torch function, folded to its Hermitian part, transformed back and overlap-added -- the reference's
loop (SpectralProcessor.cpp:154-198) with pFunc bound.  Checked against the float64 model of the
reference class (tests/spectral_model.py) with the same function written in numpy."""
import numpy as np
import pytest

import spectral_model
import spectral_cases as cases
import synth

pytestmark = pytest.mark.gpu
TOL = 2e-5


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def span(rank, bound):
    """Samples of one sub-call: L = P * max(1, floor(2^25 / (B * N)))."""
    N = 1 << rank
    return (N // 2) * max(1, (1 << 25) // (bound * N))


def expected_invocations(rank, refs, count, L):
    """Per invocation, the (instance, pos) table the function must receive for one call of `count`
    samples: frames of instance i at remaining(), + P, ... (refs: {instance: model} before the call)."""
    F = 1 << (rank - 1)
    out = []
    for s0 in range(0, count, L):
        tab = [(i, p) for i in sorted(refs) for p in range(refs[i].remaining(), count, F) if s0 <= p < s0 + L]
        if tab:
            out.append(tab)
    return out


def peak_err(got, want):
    return float(np.max(np.abs(got - want))) / max(1.0, float(np.max(np.abs(want))))


class Recorder:
    """A spectral function that applies `op` (torch, in place or returning the new spectrum) and
    records what every invocation received."""

    def __init__(self, torch, op=None):
        self.torch, self.op, self.calls = torch, op, []

    def __call__(self, X, instances, positions, rank):
        t = self.torch
        self.calls.append({"n": X.shape[0], "rank": rank, "stream": t.cuda.current_stream().cuda_stream,
                           "frames": list(zip(instances.tolist(), positions.tolist()))})
        assert X.dtype == t.complex64 and X.is_cuda and X.shape[1] == 1 << rank
        if self.op is not None:
            self.op(X)


def soft_gate_np(X, c=1.0):
    return X * np.abs(X) / (np.abs(X) + c)


def soft_gate_torch(X, c=1.0):
    a = X.abs()
    X.mul_(a / (a + c))


def rotation(rank):
    N = 1 << rank
    return 0.3 + 2.1 * np.arange(N) / N          # theta_k, not odd-symmetric


@pytest.mark.parametrize("rank", [7, 8, 9, 10, 11, 12, 13, 14, 15])
def test_identity_against_the_model(pkg, torch, rank):
    N, P = 1 << rank, 1 << (rank - 1)
    phases = [0.0, 0.37, 0.5, 1.0]
    n = len(phases)
    sp = pkg.SpectralProcessorBatch(n, 15, device=0)
    sp.set_rank(rank)
    rec = Recorder(torch)
    sp.set_function(rec)
    refs = {}
    for c, ph in enumerate(phases):
        sp.set_phase(c, ph)
        sp.bind_function(c)
        refs[c] = spectral_model.ModelSpectralProcessor(rank, ph, lambda X: X)
    sizes = [1, 7, P - 1, P, P + 1, 3 * N + 5]
    x = np.stack([synth.noise(300 + c, sum(sizes)) for c in range(n)])
    L = span(rank, n)
    at, want_calls = 0, []
    for size in sizes:
        want_calls += expected_invocations(rank, refs, size, L)
        got = sp.process(x[:, at:at + size])
        for c in range(n):
            want = refs[c].process(x[c, at:at + size])
            assert peak_err(got[c], want) <= TOL, (c, size)
            assert sp.remaining(c) == refs[c].remaining()
        at += size
    assert [r["frames"] for r in rec.calls] == want_calls
    assert all(r["rank"] == rank for r in rec.calls)
    sp.close()


def test_identity_long_call_invocations(pkg, torch):
    """One device call long enough for several sub-calls: 2048 bound instances at rank 7 make L = 8192."""
    rank, n = 7, 2048
    N = 1 << rank
    L = span(rank, n)
    assert L == 8192
    count = 3 * L + 5
    sp = pkg.SpectralProcessorBatch(n, rank, device=0)
    rec = Recorder(torch)
    sp.set_function(rec)
    refs = {}
    for c in range(n):
        sp.set_phase(c, (c % 7) / 7.0)
        sp.bind_function(c)
        refs[c] = spectral_model.ModelSpectralProcessor(rank, (c % 7) / 7.0, lambda X: X)
    g = torch.Generator(device="cuda").manual_seed(5)
    src = torch.rand((n, count), device="cuda", generator=g) * 2 - 1
    dst = torch.empty_like(src)
    want_calls = expected_invocations(rank, refs, count, L)
    sp.process_device(dst.data_ptr(), count, src.data_ptr(), count, count)
    sp.sync()
    assert len(rec.calls) == len(want_calls) >= 3
    assert [r["frames"] for r in rec.calls] == want_calls
    assert max(r["n"] for r in rec.calls) * N <= max(1 << 25, n * N)
    out, x = dst.cpu().numpy(), src.cpu().numpy()
    for c in (0, 1, 6, 1000, n - 1):
        assert peak_err(out[c], refs[c].process(x[c])) <= TOL, c
    sp.close()


@pytest.mark.parametrize("rank", [8, 11, 15])
@pytest.mark.parametrize("kind", ["soft_gate", "rotation"])
def test_nonlinear_functions(pkg, torch, rank, kind):
    N = 1 << rank
    if kind == "soft_gate":
        op_t, op_np = soft_gate_torch, soft_gate_np
    else:
        theta = rotation(rank)
        rot = torch.tensor(np.exp(1j * theta).astype(np.complex64), device="cuda")
        op_t, op_np = (lambda X: X.mul_(rot)), (lambda X: X * np.exp(1j * theta))
    phases = [0.0, 0.25, 0.9]
    n = len(phases)
    sp = pkg.SpectralProcessorBatch(n, 15, device=0)
    sp.set_rank(rank)
    sp.set_function(Recorder(torch, op_t))
    refs = []
    for c, ph in enumerate(phases):
        sp.set_phase(c, ph)
        sp.bind_function(c)
        refs.append(spectral_model.ModelSpectralProcessor(rank, ph, op_np))
    total, step = 5 * N + 123, 1000 if rank < 15 else 20000
    x = np.stack([synth.noise(400 + c, total) for c in range(n)])
    got = np.concatenate([sp.process(x[:, i:i + step]) for i in range(0, total, step)], axis=1)
    for c in range(n):
        assert peak_err(got[c], refs[c].process(x[c])) <= TOL, c
    sp.close()


def test_function_equals_table(pkg, torch):
    rank = 10
    N = 1 << rank
    _, H = cases.tables(rank, 77)
    Ht = torch.tensor(H, device="cuda")
    x = np.stack([synth.noise(500 + c, 6 * N + 17) for c in range(2)])
    a = pkg.SpectralProcessorBatch(2, rank, device=0)
    b = pkg.SpectralProcessorBatch(2, rank, device=0)
    a.set_function(Recorder(torch, lambda X: X.mul_(Ht)))
    for c, ph in enumerate((0.0, 0.6)):
        a.set_phase(c, ph)
        b.set_phase(c, ph)
        a.bind_function(c)
        b.bind_complex(c, H)
    for i in range(0, x.shape[1], 777):
        ya, yb = a.process(x[:, i:i + 777]), b.process(x[:, i:i + 777])
        assert peak_err(ya, yb) <= TOL
    a.close()
    b.close()


def test_frame_table_planar_positions_across_staging(pkg, torch):
    """process_planar stages 2^24 / instances samples at a time (here 4096 = L): positions still
    count from the first sample of the caller's call."""
    rank, n = 7, 4096
    L = span(rank, n)
    count = 10000
    sp = pkg.SpectralProcessorBatch(n, rank, device=0)
    rec = Recorder(torch)
    sp.set_function(rec)
    refs = {}
    for c in range(n):
        sp.set_phase(c, (c % 3) / 3.0)
        sp.bind_function(c)
        refs[c] = spectral_model.ModelSpectralProcessor(rank, (c % 3) / 3.0, lambda X: X)
    x = np.stack([synth.noise(c % 16, count) for c in range(n)])
    want_calls = expected_invocations(rank, refs, count, L)
    got = sp.process(x)
    assert len(want_calls) == 3
    assert [r["frames"] for r in rec.calls] == want_calls
    for c in (0, 1, 2, n - 1):
        assert peak_err(got[c], refs[c].process(x[c])) <= TOL
    sp.close()


def test_mixed_batch_bit_identical_and_unbind(pkg, torch):
    rank = 9
    N = 1 << rank
    kinds = ["table", "none", "fn", "gain", "fn", "none"]
    phases = [0.0, 0.5, 0.37, 1.0, 0.0, 0.2]
    n = len(kinds)
    gain, H = cases.tables(rank, 9)
    mixed = pkg.SpectralProcessorBatch(n, rank, device=0)
    plain = pkg.SpectralProcessorBatch(n, rank, device=0)
    mixed.set_function(Recorder(torch, soft_gate_torch))
    refs = {}
    for c, (k, ph) in enumerate(zip(kinds, phases)):
        for sp in (mixed, plain):
            sp.set_phase(c, ph)
            if k == "table":
                sp.bind_complex(c, H)
            elif k == "gain":
                sp.bind_gain(c, gain)
        if k == "fn":
            mixed.bind_function(c)
            refs[c] = spectral_model.ModelSpectralProcessor(rank, ph, soft_gate_np)
    total, step = 8 * N + 31, 333
    x = np.stack([synth.noise(600 + c, total) for c in range(n)])
    got, base, want = np.empty_like(x), np.empty_like(x), {c: np.empty(total) for c in refs}
    for i in range(0, total, step):
        if i >= 4 * N and refs[4].hook is not None:
            mixed.unbind(4)                         # the model's hook switched off at the same sample
            refs[4].hook = None
        got[:, i:i + step] = mixed.process(x[:, i:i + step])
        base[:, i:i + step] = plain.process(x[:, i:i + step])
        for c in refs:
            want[c][i:i + step] = refs[c].process(x[c, i:i + step])
    for c, k in enumerate(kinds):
        if k == "fn":
            assert peak_err(got[c], want[c]) <= TOL, c
        else:
            assert np.array_equal(got[c], base[c]), c
    mixed.close()
    plain.close()


def test_device_stream_in_place_and_strided_rows(pkg, torch):
    rank, n = 10, 5
    N = 1 << rank
    count, stride_src, stride_dst = 3 * N + 11, 4 * N, 4 * N + 64
    sp = pkg.SpectralProcessorBatch(n, rank, device=0)
    sp2 = pkg.SpectralProcessorBatch(n, rank, device=0)
    rec, rec2 = Recorder(torch, soft_gate_torch), Recorder(torch, soft_gate_torch)
    sp.set_function(rec)
    sp2.set_function(rec2)
    for c in range(n):
        for s in (sp, sp2):
            s.set_phase(c, c / n)
            s.bind_function(c)
    g = torch.Generator(device="cuda").manual_seed(11)
    src = torch.rand((n, stride_src), device="cuda", generator=g) * 2 - 1
    dst = torch.full((n, stride_dst), 7.0, device="cuda")
    buf = src.clone()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        for i in range(0, count, 1000):
            m = min(1000, count - i)
            sp.process_device(dst.data_ptr() + 4 * i, stride_dst, src.data_ptr() + 4 * i, stride_src, m, st.cuda_stream)
            sp2.process_device(buf.data_ptr() + 4 * i, stride_src, buf.data_ptr() + 4 * i, stride_src, m, st.cuda_stream)
    st.synchronize()
    assert rec.calls and all(r["stream"] == st.cuda_stream for r in rec.calls)
    x, y, z = src.cpu().numpy(), dst.cpu().numpy(), buf.cpu().numpy()
    for c in range(n):
        want = spectral_model.ModelSpectralProcessor(rank, c / n, soft_gate_np).process(x[c, :count])
        assert peak_err(y[c, :count], want) <= TOL, c
        assert peak_err(z[c, :count], want) <= TOL, c
        assert np.all(y[c, count:] == 7.0) and np.array_equal(z[c, count:], x[c, count:])
    sp.close()
    sp2.close()


def test_set_rank_keeps_functions_drops_tables_phase_and_reset(pkg, torch):
    rank = 9
    gain, _ = cases.tables(rank, 3)
    sp = pkg.SpectralProcessorBatch(3, 12, device=0)
    sp.set_rank(rank)
    sp.set_function(Recorder(torch, soft_gate_torch))
    sp.bind_gain(0, gain)
    sp.bind_function(1)
    sp.bind_function(2)
    sp.set_phase(2, 0.3)
    refs = [spectral_model.ModelSpectralProcessor(rank, 0.0, lambda X: X * gain.astype(np.float64)),
            spectral_model.ModelSpectralProcessor(rank, 0.0, soft_gate_np),
            spectral_model.ModelSpectralProcessor(rank, 0.3, soft_gate_np)]

    def run(seed, total, step=700):
        x = np.stack([synth.noise(seed + c, total) for c in range(3)])
        for i in range(0, total, step):
            got = sp.process(x[:, i:i + step])
            for c in range(3):
                assert peak_err(got[c], refs[c].process(x[c, i:i + step])) <= TOL, (seed, c, i)

    run(700, 5000)
    sp.set_phase(1, 0.8)                            # update_settings: buffers cleared, new offset
    refs[1] = spectral_model.ModelSpectralProcessor(rank, 0.8, soft_gate_np)
    run(710, 3000)
    sp.reset()
    for r in refs:
        r.reset()
    run(720, 3000)
    sp.set_rank(rank + 2)                           # the table goes, the function binding stays
    refs = [spectral_model.ModelSpectralProcessor(rank + 2, 0.0, None),
            spectral_model.ModelSpectralProcessor(rank + 2, 0.8, soft_gate_np),
            spectral_model.ModelSpectralProcessor(rank + 2, 0.3, soft_gate_np)]
    run(730, 9000, 2500)
    sp.close()


def test_state_errors_and_reentry(pkg, torch):
    sp = pkg.SpectralProcessorBatch(2, 8, device=0)
    with pytest.raises(pkg.B200ConvError) as e:
        sp.bind_function(0)
    assert e.value.code == pkg.ERR_STATE
    codes = []

    def fn(X, instances, positions, rank):
        lib = pkg.lib()
        codes.append(lib.b200conv_sp_reset(sp._h))
        codes.append(lib.b200conv_sp_bind_function(sp._h, 1))
        codes.append(lib.b200conv_sp_set_phase(sp._h, 0, 0.5))
        codes.append(lib.b200conv_sp_process_planar(sp._h, None, None, 4, 4))

    sp.set_function(fn)
    sp.bind_function(0)
    with pytest.raises(pkg.B200ConvError) as e:
        sp.set_function(None)
    assert e.value.code == pkg.ERR_STATE
    sp.set_function(fn)                             # replacing a non-NULL function is allowed
    x = synth.noise(800, 1000)[None, :].repeat(2, 0)
    got = sp.process(x)
    assert codes and all(c == pkg.ERR_STATE for c in codes)
    want = spectral_model.ModelSpectralProcessor(8, 0.0, lambda X: X).process(x[0])
    assert peak_err(got[0], want) <= TOL
    sp.unbind(0)
    sp.set_function(None)
    sp.close()


def test_exception_is_reraised_and_the_object_keeps_matching(pkg, torch):
    rank = 8
    N = 1 << rank
    sp = pkg.SpectralProcessorBatch(1, rank, device=0)
    count = {"n": 0}

    def fn(X, instances, positions, r):
        count["n"] += 1
        if count["n"] == 2:
            raise KeyError("boom")                  # before touching X: this call's frames pass unchanged
        soft_gate_torch(X)

    sp.set_function(fn)
    sp.bind_function(0)
    ref = spectral_model.ModelSpectralProcessor(rank, 0.0, soft_gate_np)
    x = synth.noise(900, 6 * N)
    step = 2 * N
    for k, i in enumerate(range(0, x.size, step)):
        chunk = x[None, i:i + step]
        if k == 1:
            with pytest.raises(KeyError):
                sp.process(chunk)
            ref.hook = None
            ref.process(chunk[0])
            ref.hook = soft_gate_np
            continue
        sp_out = sp.process(chunk)[0]
        assert peak_err(sp_out, ref.process(chunk[0])) <= TOL, k
    sp.close()
