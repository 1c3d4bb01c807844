"""The float64 model of b200conv_set_irs (tests/batch_fade_model.py) against np.convolve of the
explicit blend: fades that end inside a call, chains of fades, hard switches, and the error rules."""
import numpy as np
import pytest

from batch_fade_model import ArgError, BatchFadeModel, StateError


def _sig(seed, n):
    return np.random.Generator(np.random.PCG64(seed)).uniform(-1.0, 1.0, n)


def _run(model, x, sizes):
    out, at, k = [], 0, 0
    while at < x.size:
        n = min(sizes[k % len(sizes)], x.size - at)
        out.append(model.process(x[at:at + n]))
        at += n
        k += 1
    return np.concatenate(out) if out else np.zeros(0)


def _blend(x, stages):
    """stages: [(start sample, fade, ir)], the first one the IR from init; direct np.convolve"""
    y = np.convolve(x, stages[0][2])[:x.size]
    k = np.arange(x.size)
    for start, fade, h in stages[1:]:
        new = np.convolve(x, h)[:x.size]
        w = np.where(k < start, 0.0, np.minimum(1.0, (k - start + 1) / fade) if fade > 1 else 1.0)
        y = (1.0 - w) * y + w * new
    return y


@pytest.mark.parametrize("sizes", [(64,), (17, 64, 5), (200,)])
@pytest.mark.parametrize("fade", [0, 1, 7, 64, 250])
def test_one_fade_matches_explicit_blend(sizes, fade):
    F = 64
    x, h0, h1 = _sig(1, 1500), _sig(2, 3 * F + 1), _sig(3, 2 * F)
    m = BatchFadeModel(F)
    m.init(h0)
    y0 = _run(m, x[:300], sizes)
    m.set_irs(h1, fade=fade)
    assert m.fade_remaining() == (fade if fade > 1 else 0)
    y1 = _run(m, x[300:], sizes)
    assert m.fade_remaining() == 0
    want = _blend(x, [(0, 0, h0), (300, fade, h1)])
    assert np.allclose(np.concatenate([y0, y1]), want, atol=1e-9)
    assert m.state() == {"conv_size": h1.size, "bins": 2, "partitions": 3}


def test_fade_ends_inside_a_call_and_counts_down():
    F = 32
    m = BatchFadeModel(F)
    m.init(_sig(4, 2 * F))
    m.process(_sig(5, 3 * F))
    m.set_irs(_sig(6, F), fade=50)
    assert m.fade_remaining() == 50
    m.process(_sig(7, 30))
    assert m.fade_remaining() == 20
    m.process(_sig(8, 30))                  # ends 10 samples before the end of this call
    assert m.fade_remaining() == 0 and m.fade is None


def test_chain_of_fades():
    F = 32
    x = _sig(10, 2000)
    irs = [_sig(11, 4 * F + 3), _sig(12, 3 * F), _sig(13, 2 * F - 5), _sig(14, 1), np.zeros(1)]
    fades = [40, 0, 3 * F + 5, 100]
    m = BatchFadeModel(F)
    m.init(irs[0])
    ys, stages, at = [], [(0, 0, irs[0])], 0
    for h, f in zip(irs[1:], fades):
        ys.append(_run(m, x[at:at + 150], (23, F)))
        at += 150
        m.set_irs(h, fade=f)
        stages.append((at, f, h))
        ys.append(_run(m, x[at:at + 250], (F, 7)))
        at += 250
        assert m.fade_remaining() == 0
    ys.append(_run(m, x[at:], (F,)))
    assert np.allclose(np.concatenate(ys), _blend(x, stages), atol=1e-9)
    assert not np.any(ys[-1])               # faded out by a one-tap zero IR


def test_error_rules_change_nothing():
    F = 32
    m = BatchFadeModel(F)
    with pytest.raises(StateError):
        m.set_irs(_sig(20, 10))             # not initialised
    m.init(_sig(21, 2 * F))                 # 3 partitions
    with pytest.raises(ArgError):
        m.set_irs(np.zeros(0))
    with pytest.raises(ArgError):
        m.set_irs(_sig(22, 2 * F + 1))      # 4 partitions
    with pytest.raises(StateError):
        m.set_irs(_sig(23, F), lends=True)
    m.set_irs(_sig(24, 2 * F), fade=10)
    with pytest.raises(StateError):
        m.set_irs(_sig(25, F))              # already fading
    assert m.fade_remaining() == 10
    m.process(_sig(26, 10))
    m.set_irs(_sig(27, F), fade=0)          # the fade has ended: allowed, and the reach shrinks
    with pytest.raises(ArgError):
        m.set_irs(_sig(28, 2 * F))
    m.init(_sig(29, 2 * F))                 # init restores it and ends any fade
    m.set_irs(_sig(30, 2 * F), fade=5)
    m.init(_sig(31, F))
    assert m.fade_remaining() == 0
