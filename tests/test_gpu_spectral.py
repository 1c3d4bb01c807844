"""Scope-table row f4 on the GPU: the batched SpectralProcessor (b200conv_sp_*) against the outputs
of the reference's own class frozen in tests/golden/spectral_golden.npz, the reference's unit test
shape (src/test/utest/util/spectral_proc.cpp:33-66) and the float64 model of the reference class
(tests/spectral_model.py, held to the frozen outputs by tests/test_oracle_spectral_golden.py)."""
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


def test_reference_utest_simple(pkg):
    # spectral_proc.cpp:33-62 : 440 Hz sine, init(14), phase 0, rank 8, one call of 8192 samples
    n = 8192
    src = np.sin(2 * np.pi * 440.0 / 48000.0 * np.arange(n)).astype(np.float32)
    sp = pkg.SpectralProcessorBatch(1, 14, device=0)
    sp.set_phase(0, 0.0)
    sp.set_rank(8)
    dst = sp.process(src[None, :])[0]
    lat = sp.latency()
    assert lat == 256
    assert np.max(np.abs(src[:n - lat] - dst[lat:])) <= 1e-5
    sp.close()


@pytest.mark.parametrize("rank,step", [(7, 31), (8, 77), (9, 256), (10, 1000), (11, 4096), (12, 333), (13, 10000), (14, 8192), (15, 50000)])
def test_batch_against_the_reference_class(pkg, rank, step):
    """Instances with different phases and spectral operations (none / real gains / complex table)
    in one batch, arbitrary call sizes: every instance against the model of the reference class,
    output and remaining() after every call."""
    N = 1 << rank
    n = 5 * N + 123
    kinds = [0, 2, 1, 2, 0, 1]
    phases = [0.0, 0.5, 0.37, 1.0, 0.25, 0.0]
    x = np.stack([synth.noise(200 + c, n) for c in range(len(kinds))])
    sp = pkg.SpectralProcessorBatch(len(kinds), 15, device=0)
    sp.set_rank(rank)
    refs = []
    for c, (kind, ph) in enumerate(zip(kinds, phases)):
        gain, H = cases.tables(rank, 10 * rank + c)
        sp.set_phase(c, ph)
        hook = None
        if kind == 1:
            sp.bind_complex(c, H)
            hook = lambda X, H=H: X * H.astype(np.complex128)
        elif kind == 2:
            sp.bind_gain(c, gain)
            hook = lambda X, gain=gain: X * gain.astype(np.float64)
        refs.append(spectral_model.ModelSpectralProcessor(rank, ph, hook))
    out, want = np.empty_like(x), np.empty((len(kinds), n))
    for i in range(0, n, step):
        out[:, i:i + step] = sp.process(x[:, i:i + step])
        for c in range(len(kinds)):
            want[c, i:i + step] = refs[c].process(x[c, i:i + step])
            assert sp.remaining(c) == refs[c].remaining(), (c, i)
    for c in range(len(kinds)):
        assert np.max(np.abs(out[c] - want[c])) <= TOL * max(1.0, float(np.max(np.abs(want[c])))), (c, kinds[c])
    assert sp.latency() == N
    sp.close()


@pytest.mark.parametrize("name", [c[0] for c in cases.SP_CASES])
def test_frozen_reference_outputs(pkg, name):
    """The cases of tests/golden/spectral_golden.npz: what the reference class itself produced."""
    g = np.load(cases.GOLDEN)
    rank, phase, step, kind, latency, seed, n = g[name + ".meta"]
    rank, step, kind, seed, n = int(rank), int(step), int(kind), int(seed), int(n)
    src = synth.noise(seed, n)
    gain, H = cases.tables(rank, seed)
    sp = pkg.SpectralProcessorBatch(1, 14, device=0)
    sp.set_rank(rank)
    sp.set_phase(0, float(phase))
    if kind == 1:
        sp.bind_complex(0, H)
    elif kind == 2:
        sp.bind_gain(0, gain)
    got = np.concatenate([sp.process(src[None, i:i + step])[0] for i in range(0, n, step)])
    want = g[name + ".dst"]
    assert np.max(np.abs(got - want)) <= TOL * max(1.0, float(np.max(np.abs(want))))
    assert sp.latency() == int(latency)
    sp.close()


def test_rank_change_reset_and_model(pkg):
    rank = 9
    N = 1 << rank
    x = synth.noise(7, 7 * N)
    gain, _ = cases.tables(rank, 3)
    sp = pkg.SpectralProcessorBatch(2, 12, device=0)
    sp.set_rank(rank)
    sp.bind_gain(0, gain)
    got = sp.process(np.stack([x, x]))
    want = spectral_model.ModelSpectralProcessor(rank, 0.0, lambda X: X * gain.astype(np.float64)).process(x)
    assert np.max(np.abs(got[0] - want)) <= TOL * float(np.max(np.abs(want)))
    ident = spectral_model.ModelSpectralProcessor(rank, 0.0, None).process(x)
    assert np.max(np.abs(got[1] - ident)) <= TOL
    # reset(): buffers cleared, offset kept -> the next N samples come out as if the past were silence
    sp.reset()
    ref = spectral_model.ModelSpectralProcessor(rank, 0.0, None)
    ref.process(x)
    ref.reset()
    y = synth.noise(8, 3 * N)
    assert np.max(np.abs(sp.process(np.stack([y, y]))[1] - ref.process(y))) <= TOL
    # a rank change drops history and tables (update_settings, :107-125)
    sp.set_rank(rank + 1)
    z = synth.noise(9, 4 * N)
    got = sp.process(np.stack([z, z]))
    ident = spectral_model.ModelSpectralProcessor(rank + 1, 0.0, None).process(z)
    assert np.max(np.abs(got[0] - ident)) <= TOL and np.max(np.abs(got[1] - ident)) <= TOL
    assert sp.latency() == 2 * N
    sp.close()


def test_device_pointers_in_place_and_many_instances(pkg):
    torch = pytest.importorskip("torch")
    rank, n = 10, 3000
    N = 1 << rank
    count = 6 * N
    src = torch.rand((n, count), device="cuda") * 2 - 1
    sp = pkg.SpectralProcessorBatch(n, 10, device=0)
    for c in range(n):
        sp.set_phase(c, (c % 5) / 5.0)
    gain = np.linspace(0.5, 1.0, N).astype(np.float32)
    sp.bind_gain(17, gain)
    buf = src.clone()
    for i in range(0, count, 1536):                                     # in place, device pointers
        sp.process_device(buf.data_ptr() + 4 * i, count, buf.data_ptr() + 4 * i, count, 1536)
    sp.sync()
    out = buf.cpu().numpy()
    for c in (0, 1, 17, 2999):
        hook = (lambda X: X * gain.astype(np.float64)) if c == 17 else None
        want = spectral_model.ModelSpectralProcessor(rank, (c % 5) / 5.0, hook).process(src[c].cpu().numpy())
        assert np.max(np.abs(out[c] - want)) <= TOL * max(1.0, float(np.max(np.abs(want))))
    sp.close()
