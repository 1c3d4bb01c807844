"""The vectorised float64 models of tests/batch_models.py against the per-instance models they
restate (held to the reference by test_oracle_equalizer.py, test_oracle_spectral_golden.py and
test_oracle_splitter.py): a mixed batch, random call sizes, mid-stream hand-overs and mixed
bindings; a handful of random instances must agree to ~1e-12 of their peak."""
import numpy as np
import pytest

import batch_models
from equalizer_model import ModelEqualizer
from spectral_model import ModelSpectralProcessor
from splitter_model import ModelSpectralSplitter

TOL = 1e-12


def _rel(a, b):
    return float(np.max(np.abs(a - b))) / max(1e-300, float(np.max(np.abs(b))))


def _calls(rng, total, hi):
    sizes = []
    while sum(sizes) < total:
        sizes.append(int(rng.integers(1, hi)))
    return sizes


@pytest.mark.parametrize("fir_rank", [7, 9])
def test_equalizer_matches_the_per_instance_model(fir_rank):
    rng = np.random.default_rng(fir_rank)
    F, n = 1 << fir_rank, 23
    x = rng.uniform(-1, 1, (n, 9 * F))
    kern = lambda: rng.uniform(-1, 1, (n, F)) * np.exp(-np.arange(F) / (F / 4))
    k0, k1, k2, k3 = kern(), kern(), kern(), kern()
    smooth = rng.random(n) < 0.5
    now = (~smooth) & (rng.random(n) < 0.5)
    pending = smooth & (rng.random(n) < 0.4)
    bm = batch_models.BatchEqualizer(n, fir_rank)
    bm.set_kernel(np.arange(n), k0)
    pick = rng.choice(n, 5, replace=False)
    ms = {c: ModelEqualizer(fir_rank) for c in pick}
    for c in pick:
        ms[c].set_kernel(k0[c])
    sizes = _calls(rng, x.shape[1], 2 * F + 40)
    got = np.empty_like(x)
    want = {c: np.empty(x.shape[1]) for c in pick}
    pos = 0
    for j, size in enumerate(sizes):
        size = min(size, x.shape[1] - pos)
        events = []
        if j == len(sizes) // 3:
            events = [(np.flatnonzero(smooth), k1, True), (np.flatnonzero(now), k2, False),
                      (np.flatnonzero(pending), k3, False)]                     # replace while a fade is pending
        if j == len(sizes) // 2:
            bm.clear()
            for c in pick:
                ms[c].clear()
        if j == 2 * len(sizes) // 3:
            events = [(np.flatnonzero(~smooth), k3, True)]
        for rows, k, sm in events:
            bm.set_kernel(rows, k[rows], sm)
            for c in set(pick) & set(rows.tolist()):
                ms[c].set_kernel(k[c], sm)
        got[:, pos:pos + size] = bm.process(x[:, pos:pos + size])
        for c in pick:
            want[c][pos:pos + size] = ms[c].process(x[c, pos:pos + size])
        pos += size
    for c in pick:
        assert _rel(got[c], want[c]) <= TOL, c


def _spectral_batch(rng, rank, n):
    N = 1 << rank
    phases = rng.choice([0.0, 0.25, 0.37, 0.5, 1.0], n)
    kind = rng.integers(0, 3, n)
    tables = rng.uniform(-1, 1, (n, N)) + 1j * rng.uniform(-1, 1, (n, N))
    tables[::2] = rng.uniform(0.2, 1.5, (len(tables[::2]), N))         # real gains on every other row
    ramp = 0.5 + np.arange(N) / N
    fn = lambda X, rows: X * ramp * (1.0 + rows[:, None] / n)          # a function of the spectrum and the instance
    return phases, kind, tables, fn


@pytest.mark.parametrize("rank", [7, 10])
def test_spectral_processor_matches_the_per_instance_model(rank):
    rng = np.random.default_rng(100 + rank)
    N, n = 1 << rank, 31
    phases, kind, tables, fn = _spectral_batch(rng, rank, n)
    x = rng.uniform(-1, 1, (n, 6 * N + 17))
    bm = batch_models.BatchSpectralProcessor(rank, phases, kind, tables, fn)
    pick = rng.choice(n, 6, replace=False)
    hooks = {0: lambda c: None, 1: lambda c: (lambda X: X * tables[c]),
             2: lambda c: (lambda X: fn(X[None, :], np.array([c]))[0])}
    ms = {c: ModelSpectralProcessor(rank, phases[c], hooks[int(kind[c])](c)) for c in pick}
    pos = 0
    for size in _calls(rng, x.shape[1], N + N // 3) + [x.shape[1]]:
        size = min(size, x.shape[1] - pos)
        if size == 0:
            break
        got = bm.process(x[:, pos:pos + size])
        rem = bm.remaining()
        for c in pick:
            want = ms[c].process(x[c, pos:pos + size])
            assert _rel(got[c], want) <= TOL or np.max(np.abs(want)) == 0.0 and np.all(got[c] == 0.0), (c, pos)
            assert rem[c] == ms[c].remaining()
        pos += size


@pytest.mark.parametrize("rank,chunk", [(7, 0), (10, 8), (9, 6)])
def test_spectral_splitter_matches_the_per_instance_model(rank, chunk):
    rng = np.random.default_rng(200 + rank)
    N, n, H = 1 << rank, 29, 3
    phases = rng.choice([0.0, 0.3, 0.5, 0.37, 1.0], n)
    kinds = rng.integers(0, 3, (n, H))
    kinds[3] = 0                                                       # nothing bound
    kinds[4] = 2                                                       # sinks only
    tables = rng.uniform(-1, 1, (n, H, N)) + 1j * rng.uniform(-1, 1, (n, H, N))
    tables[:, 1] = rng.uniform(0.2, 1.5, (n, N))                       # handler 1: real gains
    bm = batch_models.BatchSpectralSplitter(rank, kinds, tables, phases, chunk)
    pick = np.concatenate([[3, 4], rng.choice(np.arange(5, n), 5, replace=False)])
    ms = {}
    for c in pick:
        m = ModelSpectralSplitter(rank, H, chunk, phases[c])
        for h in range(H):
            if kinds[c, h] == 1:
                m.bind(h, lambda X, t=tables[c, h]: X * t)
            elif kinds[c, h] == 2:
                m.bind(h, "copy")
        ms[c] = m
    assert bm.latency() == ms[pick[0]].latency()
    x = rng.uniform(-1, 1, (n, 5 * N + 33))
    pos = 0
    for size in _calls(rng, x.shape[1], N) + [x.shape[1]]:
        size = min(size, x.shape[1] - pos)
        if size == 0:
            break
        got = bm.process(x[:, pos:pos + size])
        for c in pick:
            want = ms[c].process(x[c, pos:pos + size])
            for h in range(H):
                if np.max(np.abs(want[h])) == 0.0:
                    assert np.all(got[h, c] == 0.0), (c, h, pos)
                else:
                    assert _rel(got[h, c], want[h]) <= TOL, (c, h, pos)
        pos += size
    assert bm.fill[3] == int(np.float32(bm.F) * (np.float32(phases[3]) * np.float32(0.5)))     # never advanced
