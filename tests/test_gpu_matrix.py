"""The matrix convolver (b200conv_mx_*, MatrixConvolver) on the GPU against the float64 model of
tests/matrix_model.py.  Bar: max |gpu - model| <= 1e-5 of the model's peak, the engine's."""
import ctypes

import numpy as np
import pytest

from matrix_model import MatrixModel
import synth

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


def _ir(seed, n):
    return synth.decaying_ir(seed, n) if n > 1 else np.array([0.75], dtype=np.float32)


def _inputs(seed, inputs, n, nyquist=()):
    """White noise rows; the rows in `nyquist` also carry a (-1)^n component, whose energy sits in
    the Nyquist half of packed bin 0."""
    x = np.stack([synth.noise(seed + i, n) for i in range(inputs)])
    for i in nyquist:
        x[i] = 0.5 * x[i] + 0.5 * np.where(np.arange(n) % 2 == 0, 1.0, -1.0).astype(np.float32)
    return x


def _feed(mx, x, frames_per_call):
    """Runs x through mx in calls of the given frame counts (cycled); returns the concatenated output."""
    F = mx.frame_size()
    out, at, k = [], 0, 0
    while at < x.shape[1]:
        n = min(frames_per_call[k % len(frames_per_call)] * F, x.shape[1] - at)
        out.append(mx.process(x[:, at:at + n]))
        at += n
        k += 1
    return np.concatenate(out, axis=1)


def _err(got, want):
    return float(np.max(np.abs(got - want)) / max(np.max(np.abs(want)), 1e-30))


@pytest.mark.parametrize("rank", [8, 9, 11, 13, 14, 16])
def test_true_stereo_ring_wraps(pkg, rank):
    F = 1 << (rank - 1)
    mx = pkg.MatrixConvolver(2, 2, rank, device=0)
    # lengths 1, F - 1, F + 1, several partitions; then F and others after a second set_routes
    routes = [(0, 0, _ir(1, 3 * F + 7)), (0, 1, _ir(2, F - 1)), (1, 0, _ir(3, F + 1)), (1, 1, _ir(4, 1))]
    frames = 48                         # > ring slots (longest route's partitions + one launch group)
    x = _inputs(10 * rank, 2, frames * F, nyquist=(1,))
    mx.set_routes(routes)
    model = MatrixModel(2, 2)
    model.set_routes(routes)
    want = model.process(x)
    got = _feed(mx, x, [1, 3, 2])
    assert _err(got, want) <= TOL, rank

    routes = [(0, 0, _ir(5, F)), (1, 0, _ir(6, 2 * F + 3)), (0, 1, _ir(7, 5)), (1, 1, _ir(8, 4 * F))]
    mx.set_routes(routes)
    model.set_routes(routes)
    x = _inputs(10 * rank + 5, 2, 16 * F, nyquist=(0,))
    assert _err(_feed(mx, x, [2, 1]), model.process(x)) <= TOL, rank
    mx.close()


def _check_shape(pkg, inputs, outputs, routes, rank=9, frames=24):
    F = 1 << (rank - 1)
    mx = pkg.MatrixConvolver(inputs, outputs, rank, device=0)
    mx.set_routes(routes)
    model = MatrixModel(inputs, outputs)
    model.set_routes(routes)
    x = _inputs(77 + inputs, inputs, frames * F, nyquist=(0,))
    got = _feed(mx, x, [1, 3])
    want = model.process(x)
    assert _err(got, want) <= TOL
    mx.close()
    return got


def test_fan_out_one_by_eight(pkg):
    _check_shape(pkg, 1, 8, [(0, o, _ir(20 + o, 300 + 200 * o)) for o in range(8)])


def test_fan_in_eight_by_one(pkg):
    _check_shape(pkg, 8, 1, [(i, 0, _ir(40 + i, 1 + 250 * i)) for i in range(8)])


def test_sparse_with_unrouted_input_and_output(pkg):
    routes = [(0, 0, _ir(60, 700)), (1, 0, _ir(61, 90)), (1, 1, _ir(62, 1500)), (3, 1, _ir(63, 256)),
              (2, 0, _ir(64, 511))]          # input 4 and output 2 have no route
    got = _check_shape(pkg, 5, 3, routes)
    assert not np.any(got[2])


def test_block_diagonal_sixteen_true_stereo(pkg):
    routes = []
    for b in range(16):
        for i in range(2):
            for o in range(2):
                routes.append((2 * b + i, 2 * b + o, _ir(100 + 4 * b + 2 * i + o, 400 + 37 * b + 11 * i + 5 * o)))
    _check_shape(pkg, 32, 32, routes)


def test_in_place_device(pkg):
    torch = pytest.importorskip("torch")
    rank, n_io = 10, 3
    F = 1 << (rank - 1)
    routes = [(i, o, _ir(200 + 3 * i + o, 700 + 100 * (i + o))) for i in range(n_io) for o in range(n_io) if i != o or i == 0]
    mx = pkg.MatrixConvolver(n_io, n_io, rank, device=0)
    mx.set_routes(routes)
    model = MatrixModel(n_io, n_io)
    model.set_routes(routes)
    x = _inputs(300, n_io, 20 * F)
    buf = torch.from_numpy(x.copy()).cuda()
    stride = buf.stride(0)
    for at in range(0, x.shape[1], 2 * F):
        mx.process_device(buf.data_ptr() + 4 * at, stride, buf.data_ptr() + 4 * at, stride, 2 * F)
    mx.sync()
    assert _err(buf.cpu().numpy(), model.process(x)) <= TOL
    mx.close()


def test_set_routes_twice_zero_routes_and_clear(pkg):
    rank = 9
    F = 1 << (rank - 1)
    mx = pkg.MatrixConvolver(2, 2, rank, device=0)
    x = _inputs(400, 2, 12 * F, nyquist=(1,))
    # before any routing: zeros
    assert not np.any(mx.process(x[:, :2 * F]))
    short = [(0, 0, _ir(401, 100)), (1, 1, _ir(402, 200))]
    mx.set_routes(short)
    first = _feed(mx, x, [1])
    # a longer IR grows the ring; history is discarded: the output equals a fresh object's
    longer = [(0, 1, _ir(403, 9 * F + 3)), (1, 0, _ir(404, 50)), (1, 1, _ir(405, 3 * F))]
    mx.set_routes(longer)
    model = MatrixModel(2, 2)
    model.set_routes(longer)
    assert _err(_feed(mx, x, [2]), model.process(x)) <= TOL
    # zero routes: zeros
    mx.set_routes([])
    assert mx.routes() == 0
    assert not np.any(_feed(mx, x, [3]))
    # clear() after some history equals a fresh object
    mx.set_routes(short)
    _feed(mx, x[:, :5 * F], [1])
    mx.clear()
    assert np.array_equal(_feed(mx, x, [1]), first)
    mx.close()


def test_failed_calls_change_nothing(pkg):
    rank = 9
    F = 1 << (rank - 1)
    lib = pkg.lib()
    routes = [(0, 0, _ir(500, 700)), (1, 0, _ir(501, 300)), (1, 1, _ir(502, 1000))]
    mx = pkg.MatrixConvolver(2, 2, rank, device=0)
    mx.set_routes(routes)
    model = MatrixModel(2, 2)
    model.set_routes(routes)
    x = _inputs(510, 2, 16 * F, nyquist=(0,))
    want = model.process(x)
    got = [mx.process(x[:, :3 * F])]

    out = np.zeros((2, F + 1), dtype=np.float32)
    src = np.ascontiguousarray(x[:, :F + 1])
    assert lib.b200conv_mx_process_planar(mx._h, out.ctypes.data, F + 1, src.ctypes.data, F + 1, F + 1) == pkg.ERR_ARG
    assert not np.any(out)

    h = _ir(503, 64)
    SZ, FP = ctypes.c_size_t, ctypes.POINTER(ctypes.c_float)

    def bad_routes(ins, outs, lens, irs):
        n = len(ins)
        return lib.b200conv_mx_set_routes(mx._h, n, (SZ * n)(*ins), (SZ * n)(*outs), (FP * n)(*irs), (SZ * n)(*lens))

    hp = h.ctypes.data_as(FP)
    assert bad_routes([0, 0], [1, 1], [64, 64], [hp, hp]) == pkg.ERR_ARG           # duplicate pair
    assert bad_routes([2], [0], [64], [hp]) == pkg.ERR_ARG                           # input out of range
    assert bad_routes([0], [2], [64], [hp]) == pkg.ERR_ARG                           # output out of range
    assert bad_routes([0], [0], [0], [hp]) == pkg.ERR_ARG                            # length 0
    assert bad_routes([0], [0], [64], [FP()]) == pkg.ERR_ARG                         # NULL impulse response
    assert mx.routes() == len(routes)

    got.append(_feed(mx, x[:, 3 * F:], [1, 2]))
    assert _err(np.concatenate(got, axis=1), want) <= TOL
    mx.close()


def test_caller_stream_order(pkg):
    torch = pytest.importorskip("torch")
    rank, frames = 11, 12
    F = 1 << (rank - 1)
    routes = [(0, 0, _ir(600, 5000)), (0, 1, _ir(601, 3000)), (1, 1, _ir(602, 7000))]
    mx = pkg.MatrixConvolver(2, 2, rank, device=0)
    mx.set_routes(routes)
    model = MatrixModel(2, 2)
    model.set_routes(routes)
    x = _inputs(610, 2, frames * F)
    host = torch.from_numpy(x)
    s = torch.cuda.Stream()
    res = []
    with torch.cuda.stream(s):
        for k in range(frames):
            src = torch.empty((2, F), device="cuda")
            src.copy_(host[:, k * F:(k + 1) * F].to("cuda", non_blocking=False) * 2.0)      # a kernel writes the input
            dst = torch.empty((2, F), device="cuda")
            mx.process_device(dst.data_ptr(), F, src.data_ptr(), F, F, stream=s.cuda_stream)
            res.append(dst * 0.5)                                                          # a kernel reads the output
    s.synchronize()
    got = torch.cat(res, dim=1).cpu().numpy()
    assert _err(got, model.process(x)) <= TOL
    mx.close()


def test_planar_and_device_paths_are_bit_identical(pkg):
    torch = pytest.importorskip("torch")
    rank = 10
    F = 1 << (rank - 1)
    routes = [(i, o, _ir(700 + 4 * i + o, 900 + 300 * i + 70 * o)) for i in range(3) for o in range(4)]
    a = pkg.MatrixConvolver(3, 4, rank, device=0)
    b = pkg.MatrixConvolver(3, 4, rank, device=0)
    a.set_routes(routes)
    b.set_routes(routes)
    x = _inputs(710, 3, 10 * F, nyquist=(2,))
    host = _feed(a, x, [2])
    src = torch.from_numpy(x).cuda()
    dst = torch.empty((4, x.shape[1]), device="cuda")
    for at in range(0, x.shape[1], 2 * F):
        b.process_device(dst.data_ptr() + 4 * at, dst.stride(0), src.data_ptr() + 4 * at, src.stride(0), 2 * F)
    b.sync()
    assert np.array_equal(host, dst.cpu().numpy())
    a.close()
    b.close()


def test_diagonal_matches_convolver_batch(pkg):
    rank, n = 10, 4
    F = 1 << (rank - 1)
    irs = [_ir(800 + i, 2000 + 900 * i) for i in range(n)]
    mx = pkg.MatrixConvolver(n, n, rank, device=0)
    mx.set_routes([(i, i, irs[i]) for i in range(n)])
    batch = pkg.ConvolverBatch(n, device=0)
    for i in range(n):
        assert batch.init(i, irs[i], rank)
    x = _inputs(810, n, 30 * F, nyquist=(3,))
    got = _feed(mx, x, [1, 2])
    want = np.concatenate([batch.process(x[:, at:at + F]) for at in range(0, x.shape[1], F)], axis=1)
    assert _err(got, want) <= TOL
    mx.close()
    batch.close()


def test_full_size_true_stereo_bank(pkg):
    """Config A of tools/bench_mx.py: 16 true-stereo reverbs (32 x 32, block-diagonal 2 x 2) with
    480 000-tap IRs at rank 11, 640 one-frame calls: the ring (470 partitions + 32) wraps."""
    torch = pytest.importorskip("torch")
    rank, taps, blocks = 11, 480000, 640
    F = 1 << (rank - 1)
    routes = [(2 * b + i, 2 * b + o, synth.decaying_ir(1000 + 4 * b + 2 * i + o, taps))
              for b in range(16) for i in range(2) for o in range(2)]
    mx = pkg.MatrixConvolver(32, 32, rank, device=0)
    mx.set_routes(routes)
    x = _inputs(1100, 32, blocks * F, nyquist=(5,))
    src = torch.from_numpy(x).cuda()
    dst = torch.empty_like(src)
    for k in range(blocks):
        at = k * F
        mx.process_device(dst.data_ptr() + 4 * at, dst.stride(0), src.data_ptr() + 4 * at, src.stride(0), F)
    mx.sync()
    got = dst.cpu().numpy()
    mx.close()
    for o in (4, 27):                                   # 4 <- inputs 4, 5 (5 carries (-1)^n); 27 <- 26, 27
        want = MatrixModel(32, 32)
        want.set_routes([r for r in routes if r[1] == o])
        y = want.process(x)[o]
        assert _err(got[o], y) <= TOL, o
