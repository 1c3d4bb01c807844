"""Scope-table row f4, second sibling, on the GPU: the batched SpectralSplitter (b200conv_ss_*)
against the outputs of the reference's own class frozen in tests/golden/spectral_golden.npz, the
float64 model of the reference class (tests/splitter_model.py, held to the frozen outputs by
tests/test_oracle_spectral_golden.py) and, where oracle/_ref has been built, the reference class
itself (SpectralSplitter.cpp compiled verbatim, host callbacks in oracle/ref_wrap_splitter.cpp)."""
import numpy as np
import pytest

import splitter_model
import spectral_cases as cases
import synth
from oracle.bindings import CpuSpectralSplitter

pytestmark = pytest.mark.gpu
TOL = 2e-5


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


def _close(got, want):
    return np.max(np.abs(got.astype(np.float64) - want)) <= TOL * max(1.0, np.max(np.abs(want)))


@pytest.mark.parametrize("rank,chunk,step", [(7, 0, 31), (8, 6, 77), (9, 0, 256), (10, 8, 1000), (11, 5, 4096), (12, 0, 333),
                                             (13, 11, 10000), (14, 0, 8192), (14, 9, 3000)])
def test_batch_against_the_reference_class(pkg, rank, chunk, step):
    """Instances with different phases and handler sets (real gains / complex table / sink only /
    unbound) in one batch, arbitrary call sizes: every band of every instance against the model of
    the reference class."""
    N = 1 << rank
    n = 5 * N + 123
    H4 = 4
    setups = [((2, 1, 0, 3), 0.0), ((3, 0, 0, 2), 0.5), ((0, 0, 0, 0), 0.3), ((1, 1, 2, 2), 0.37), ((0, 2, 0, 0), 1.0)]
    x = np.stack([synth.noise(400 + c, n) for c in range(len(setups))])
    ss = pkg.SpectralSplitterBatch(len(setups), 14, H4, device=0)
    ss.set_rank(rank)
    if chunk:
        ss.set_chunk_rank(chunk)
    refs = []
    for c, (kinds, ph) in enumerate(setups):
        ref = splitter_model.ModelSpectralSplitter(rank, H4, chunk, ph)
        ss.set_phase(c, ph)
        for h, kind in enumerate(kinds):
            gain, H = cases.tables(rank, 100 * rank + 10 * c + h)
            if kind == 1:
                ref.bind(h, lambda X, H=H: X * H.astype(np.complex128))
                ss.bind_complex(c, h, H)
            elif kind == 2:
                ref.bind(h, lambda X, gain=gain: X * gain.astype(np.float64))
                ss.bind_gain(c, h, gain)
            elif kind == 3:
                ref.bind(h, "copy")
                ss.bind_sink(c, h)
        assert ss.bindings(c) == sum(kind != 0 for kind in kinds)
        refs.append(ref)
    got = np.concatenate([ss.process(x[:, i:i + step]) for i in range(0, n, step)], axis=2)
    assert ss.latency() == refs[0].latency() and 1 << ss.chunk_rank() == refs[0].latency()
    for c, (kinds, ph) in enumerate(setups):
        want = refs[c].process(x[c])
        for h, kind in enumerate(kinds):
            if kind == 0:
                assert np.all(got[h, c] == 0.0)
            else:
                assert _close(got[h, c], want[h]), (c, h, kind)
    ss.close()


@pytest.mark.parametrize("name", [c[0] for c in cases.SS_CASES])
def test_frozen_reference_outputs(pkg, name):
    """The cases of tests/golden/spectral_golden.npz: what the reference class itself produced."""
    g = np.load(cases.GOLDEN)
    rank, chunk, phase, step, latency, seed, n = g[name + ".meta"]
    rank, chunk, step, seed, n = int(rank), int(chunk), int(step), int(seed), int(n)
    kinds = [int(k) for k in g[name + ".kinds"]]
    src = synth.noise(seed, n)
    ss = pkg.SpectralSplitterBatch(1, 13, len(kinds), device=0)
    ss.set_rank(rank)
    if chunk:
        ss.set_chunk_rank(chunk)
    ss.set_phase(0, float(phase))
    for h, kind in enumerate(kinds):
        gain, H = cases.tables(rank, 10 * seed + h)
        if kind == 1:
            ss.bind_complex(0, h, H)
        elif kind == 2:
            ss.bind_gain(0, h, gain)
        elif kind == 3:
            ss.bind_sink(0, h)
    got = np.concatenate([ss.process(src[None, i:i + step])[:, 0] for i in range(0, n, step)], axis=1)
    want = g[name + ".dst"].astype(np.float64)
    bound = [h for h, kind in enumerate(kinds) if kind != 0]
    assert _close(got[bound], want)
    assert np.all(got[[h for h, kind in enumerate(kinds) if kind == 0]] == 0.0)
    assert ss.latency() == int(latency)
    ss.close()


def test_crossover_bands_add_up_to_the_delayed_input_and_match_the_model(pkg):
    # FFTCrossover's use: real gains per band that sum to one
    rank, n, inst = 11, 20000, 3
    N = 1 << rank
    x = np.stack([synth.noise(30 + c, n) for c in range(inst)])
    k = np.minimum(np.arange(N), N - np.arange(N)) / (N / 2)
    lo = (1.0 / (1.0 + (k / 0.05) ** 4)).astype(np.float32)
    mid = ((1.0 - lo) * (1.0 / (1.0 + (k / 0.4) ** 4))).astype(np.float32)
    hi = (1.0 - lo - mid).astype(np.float32)
    ss = pkg.SpectralSplitterBatch(inst, rank, 3, device=0)
    for c in range(inst):
        for h, g in enumerate((lo, mid, hi)):
            ss.bind_gain(c, h, g)
    out = np.concatenate([ss.process(x[:, i:i + 777]) for i in range(0, n, 777)], axis=2)
    lat = ss.latency()
    assert lat == N
    assert np.max(np.abs(out[:, :, lat:].sum(axis=0) - x[:, :n - lat])) <= 3e-5
    m = splitter_model.ModelSpectralSplitter(rank, 3)
    for h, g in enumerate((lo, mid, hi)):
        m.bind(h, lambda X, g=g: X * g.astype(np.float64))
    want = m.process(x[1])
    for h in range(3):
        assert _close(out[h, 1], want[h])
    ss.close()


def test_settings_rebinding_device_api_and_errors(pkg):
    torch = pytest.importorskip("torch")
    rank, inst, hn, n = 9, 4, 2, 5000
    N = 1 << rank
    x = np.stack([synth.noise(60 + c, n) for c in range(inst)])
    ss = pkg.SpectralSplitterBatch(inst, 12, hn, device=0)
    with pytest.raises(Exception):
        ss.unbind(0, 0)                                 # STATUS_NOT_BOUND
    with pytest.raises(Exception):
        ss.bind_sink(0, 5)                              # STATUS_OVERFLOW
    with pytest.raises(Exception):
        pkg.SpectralSplitterBatch(1, 15, 1, device=0)   # ranks 7..14
    ss.set_rank(rank)
    gain, H = cases.tables(rank, 9)
    for c in range(inst):
        ss.bind_gain(c, 0, gain)
        ss.bind_complex(c, 1, H)
    src = torch.from_numpy(x).cuda()
    dst = torch.zeros((hn, inst, n), device="cuda")
    st = torch.cuda.Stream()
    pos = 0
    for step in (100, 1000, 37, 2000, 1863):
        ss.process_device(dst.data_ptr() + 4 * pos, inst * n, n, src.data_ptr() + 4 * pos, n, step, st.cuda_stream)
        pos += step
    st.synchronize()
    assert pos == n
    got = dst.cpu().numpy()
    m = splitter_model.ModelSpectralSplitter(rank, hn)
    m.bind(0, lambda X: X * gain.astype(np.float64))
    m.bind(1, lambda X: X * H.astype(np.complex128))
    want = m.process(x[2])
    for h in range(hn):
        assert _close(got[h, 2], want[h])
    # a phase change restarts that instance only (update_settings clears its buffers); a chunk rank
    # change restarts all; unbinding one band leaves its row untouched
    ss.set_phase(1, 0.5)
    ss.unbind(3, 1)
    y = ss.process(x[:, :3000])
    m0 = splitter_model.ModelSpectralSplitter(rank, hn, 0, 0.5)
    m0.bind(0, lambda X: X * gain.astype(np.float64))
    m0.bind(1, lambda X: X * H.astype(np.complex128))
    w1 = m0.process(x[1, :3000])
    assert _close(y[0, 1], w1[0]) and _close(y[1, 1], w1[1])
    assert np.all(y[1, 3] == 0.0) and ss.bindings(3) == 1
    w2 = m.process(x[2, :3000])                          # instance 2 simply carried on
    assert _close(y[0, 2], w2[0])
    ss.set_chunk_rank(7)
    assert ss.latency() == 128
    y = ss.process(x[:, :2000])
    m7 = splitter_model.ModelSpectralSplitter(rank, hn, 7, 0.0)
    m7.bind(0, lambda X: X * gain.astype(np.float64))
    m7.bind(1, lambda X: X * H.astype(np.complex128))
    w0 = m7.process(x[0, :2000])
    assert _close(y[0, 0], w0[0]) and _close(y[1, 0], w0[1])
    ss.close()


def test_fft_crossover_with_the_reference_band_curves(pkg):
    """lsp::dspu::FFTCrossover = SpectralSplitter + one real curve per band (FFTCrossover.cpp:124-140).
    The curves come from the reference's own crossover::*_fft_* functions (misc/fft_crossover.cpp
    compiled verbatim, combined as FFTCrossover::update_band does, :458-480); the device splits a
    stereo signal into three bands with them, in 1024-sample blocks, and must agree with the
    reference splitter running the same curves."""
    if not CpuSpectralSplitter.available():
        pytest.skip("oracle/_ref has not been built")
    from oracle.bindings import crossover_band_curve
    rank, sr, n, ch = 12, 48000, 40000, 2
    curves = [crossover_band_curve(rank, sr, lpf=(250.0, -24.0)),
              crossover_band_curve(rank, sr, hpf=(250.0, -24.0), lpf=(4000.0, -48.0), gain=0.8),
              crossover_band_curve(rank, sr, hpf=(4000.0, -48.0), flatten=0.9)]
    x = np.stack([synth.noise(90 + c, n) for c in range(ch)])
    ss = pkg.SpectralSplitterBatch(ch, rank, 3, device=0)
    ss.set_phase(1, 0.5)                                # FFTCrossover::set_phase: channels de-phased
    refs = []
    for c in range(ch):
        ref = CpuSpectralSplitter(rank, 3)
        ref.set_phase(0.5 * c)
        for h, curve in enumerate(curves):
            ss.bind_gain(c, h, curve)
            ref.bind_gain(h, curve)
        refs.append(ref)
    got = np.concatenate([ss.process(x[:, i:i + 1024]) for i in range(0, n, 1024)], axis=2)
    assert ss.latency() == 1 << rank
    for c in range(ch):
        want = refs[c].run(x[c], 1024)
        for h in range(3):
            assert _close(got[h, c], want[h].astype(np.float64)), (c, h)
    ss.close()
