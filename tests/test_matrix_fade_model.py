"""The float64 fade model (tests/matrix_fade_model.py) against direct sums, and its identities."""
import numpy as np
import pytest

from matrix_fade_model import FadeInProgress, MatrixFadeModel
from matrix_model import MatrixModel


def _ir(seed, n):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(n) * np.exp(-np.arange(n) / max(n / 4, 1.0))


def _feed(model, x, sizes):
    out, at, k = [], 0, 0
    while at < x.shape[1]:
        n = min(sizes[k % len(sizes)], x.shape[1] - at)
        out.append(model.process(x[:, at:at + n]))
        at += n
        k += 1
    return np.concatenate(out, axis=1)


def _direct(x, routes, changed, start, fade):
    """y by np.convolve over the whole input: `changed` maps route -> (old, new); the weights are
    written out sample by sample from the definition."""
    n = x.shape[1]
    outputs = 1 + max(o for _, o, _ in routes)
    y = np.zeros((outputs, n))
    w = np.array([1.0 if fade == 0 else min(1.0, max(0.0, (k - start + 1) / fade)) for k in range(n)])
    for r, (i, o, h) in enumerate(routes):
        if r in changed:
            old, new = changed[r]
            yo = np.convolve(x[i], old)[:n]
            yn = np.convolve(x[i], new)[:n]
            y[o] += np.where(np.arange(n) < start, yo, (1.0 - w) * yo + w * yn)
        else:
            y[o] += np.convolve(x[i], h)[:n]
    return y


@pytest.mark.parametrize("fade", [0, 1, 7, 100])
@pytest.mark.parametrize("new_len", [5, 40, 130])          # shorter than, between and longer than the old IRs
def test_model_matches_direct_sums(fade, new_len):
    rng = np.random.default_rng(fade * 1000 + new_len)
    routes = [(0, 0, _ir(1, 60)), (1, 0, _ir(2, 25)), (1, 1, _ir(3, 90)), (0, 1, _ir(4, 12))]
    x = rng.standard_normal((2, 700))
    m = MatrixFadeModel(2, 2)
    m.set_routes(routes)
    start = 96
    first = _feed(m, x[:, :start], [32])
    changes = [(0, _ir(10, new_len)), (2, _ir(11, new_len + 3))]
    m.set_irs(changes, fade=fade)
    rest = _feed(m, x[:, start:], [32, 96, 256])
    got = np.concatenate([first, rest], axis=1)
    want = _direct(x, routes, {0: (routes[0][2], changes[0][1]), 2: (routes[2][2], changes[1][1])}, start, fade)
    assert np.max(np.abs(got - want)) <= 1e-9 * np.max(np.abs(want))


def test_fade_zero_equals_routing_with_new_irs_from_the_start():
    rng = np.random.default_rng(5)
    routes = [(0, 0, _ir(20, 50)), (1, 0, _ir(21, 80))]
    new = _ir(22, 70)
    x = rng.standard_normal((2, 512))
    m = MatrixFadeModel(2, 1)
    m.set_routes(routes)
    m.set_irs([(1, new)], fade=0)
    ref = MatrixModel(2, 1)
    ref.set_routes([routes[0], (1, 0, new)])
    assert np.allclose(_feed(m, x, [64, 128]), ref.process(x), rtol=0, atol=1e-12)


def test_after_the_fade_output_equals_routing_with_new_irs():
    rng = np.random.default_rng(6)
    routes = [(0, 0, _ir(30, 50)), (0, 1, _ir(31, 80))]
    new = [_ir(32, 100), _ir(33, 20)]
    x = rng.standard_normal((1, 1024))
    m = MatrixFadeModel(1, 2)
    m.set_routes(routes)
    _feed(m, x[:, :128], [64])
    m.set_irs([(0, new[0]), (1, new[1])], fade=300)
    assert m.fade_remaining() == 300
    got = _feed(m, x[:, 128:], [64])
    assert m.fade_remaining() == 0
    ref = MatrixModel(1, 2)
    ref.set_routes([(0, 0, new[0]), (0, 1, new[1])])
    want = ref.process(x)[:, 128:]
    assert np.allclose(got[:, 300:], want[:, 300:], rtol=0, atol=1e-12)
    assert not np.allclose(got[:, :300], want[:, :300], rtol=0, atol=1e-12)


def test_state_rules():
    m = MatrixFadeModel(1, 1)
    m.set_routes([(0, 0, _ir(40, 30))])
    m.set_irs([(0, _ir(41, 30))], fade=100)
    m.process(np.zeros((1, 64)))
    assert m.fade_remaining() == 36
    with pytest.raises(FadeInProgress):
        m.set_irs([(0, _ir(42, 30))], fade=10)
    m.clear()                               # ends the fade with the new IR in place
    assert m.fade_remaining() == 0
    m.set_irs([(0, _ir(42, 30))], fade=10)
    m.set_routes([(0, 0, _ir(43, 10))])     # discards the fade
    assert m.fade_remaining() == 0
