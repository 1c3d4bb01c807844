"""CPU checks of the matrix convolver's float64 model (tests/matrix_model.py): against direct
np.convolve sums, and a 1 x 1 matrix against the restated convolver and direct_convolve."""
import numpy as np
import pytest

from matrix_model import MatrixModel


def _routes(rng, inputs, outputs, density, max_len):
    routes = []
    for i in range(inputs):
        for o in range(outputs):
            if rng.random() < density:
                routes.append((i, o, rng.standard_normal(int(rng.integers(1, max_len + 1)))))
    return routes


@pytest.mark.parametrize("inputs,outputs", [(1, 1), (2, 2), (3, 5), (6, 2)])
def test_model_matches_direct_sums_across_calls(inputs, outputs):
    rng = np.random.default_rng(100 + 10 * inputs + outputs)
    routes = _routes(rng, inputs, outputs, 0.7, 90)
    model = MatrixModel(inputs, outputs)
    model.set_routes(routes)
    x = rng.standard_normal((inputs, 400))
    got = np.concatenate([model.process(x[:, a:b]) for a, b in ((0, 17), (17, 200), (200, 400))], axis=1)
    want = np.zeros((outputs, 400))
    for i, o, h in routes:
        want[o] += np.convolve(x[i], h)[:400]
    assert np.max(np.abs(got - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


def test_model_clear_and_set_routes_discard_history():
    rng = np.random.default_rng(7)
    model = MatrixModel(2, 1)
    model.set_routes([(0, 0, rng.standard_normal(50)), (1, 0, rng.standard_normal(30))])
    x = rng.standard_normal((2, 120))
    first = model.process(x)
    model.process(rng.standard_normal((2, 64)))
    model.clear()
    assert np.array_equal(model.process(x), first)
    model.set_routes([])
    assert not np.any(model.process(x))


@pytest.mark.parametrize("rank", [8, 9])
def test_one_by_one_matches_the_restated_convolver(rank):
    from oracle.bindings import CpuConvolver, direct_convolve
    rng = np.random.default_rng(rank)
    F = 1 << (rank - 1)
    h = rng.uniform(-1, 1, 3 * F + 5).astype(np.float32)
    x = rng.uniform(-1, 1, 8 * F).astype(np.float32)
    model = MatrixModel(1, 1)
    model.set_routes([(0, 0, h)])
    got = np.concatenate([model.process(x[None, a:a + 2 * F]) for a in range(0, x.size, 2 * F)], axis=1)[0]
    want = direct_convolve(x, h, x.size)
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    ref = CpuConvolver("oracle")
    assert ref.init(h, rank)
    cpu = ref.run(x, F)
    assert np.max(np.abs(got - cpu)) <= 1e-5 * np.max(np.abs(want))
