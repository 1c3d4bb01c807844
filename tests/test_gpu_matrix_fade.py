"""b200conv_mx_set_irs / MatrixConvolver.set_irs on the GPU: new impulse responses for running routes,
keeping the input history and crossfading old to new, against the float64 model of
tests/matrix_fade_model.py.  Bar: max |gpu - model| <= 1e-5 of the model's peak, as for the matrix."""
import ctypes

import numpy as np
import pytest

from matrix_fade_model import MatrixFadeModel
import synth

pytestmark = pytest.mark.gpu

TOL = 1e-5
SZ, FP = ctypes.c_size_t, ctypes.POINTER(ctypes.c_float)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


def _ir(seed, n):
    return synth.decaying_ir(seed, n) if n > 1 else np.array([0.75], dtype=np.float32)


def _inputs(seed, inputs, n):
    return np.stack([synth.noise(seed + i, n) for i in range(inputs)])


def _err(got, want):
    return float(np.max(np.abs(got - want)) / max(np.max(np.abs(want)), 1e-30))


class _Feeder:
    """Feeds consecutive frames of x to any number of objects (GPU or model) in the same calls."""

    def __init__(self, x, F):
        self.x, self.F, self.at = x, F, 0

    def run(self, objs, frames, sizes=(1,)):
        outs = [[] for _ in objs]
        left, k = frames, 0
        while left > 0:
            n = min(sizes[k % len(sizes)], left)
            blk = self.x[:, self.at:self.at + n * self.F]
            for o, obj in zip(outs, objs):
                o.append(obj.process(blk))
            self.at += n * self.F
            left -= n
            k += 1
        return [np.concatenate(o, axis=1) for o in outs]


# 3 inputs x 2 outputs; output 0 has fan-in 3, output 1 fan-in 2.  Route 0 is the longest (7 rows).
def _routes(F, seed):
    return [(0, 0, _ir(seed, 6 * F + 5)), (1, 0, _ir(seed + 1, 2 * F)), (2, 0, _ir(seed + 2, F // 2)),
            (0, 1, _ir(seed + 3, 3 * F + 1)), (2, 1, _ir(seed + 4, F + 3))]


@pytest.mark.parametrize("rank", [8, 11, 13, 16])
def test_chain_of_fades_against_model(pkg, rank):
    """A chain of set_irs calls, each after the previous fade has ended: fades of 0, 1, F/3, F,
    5F + 17 samples and one longer than a launch group (32 frames), in calls of 1, 3 and 8 frames so
    that fades end inside calls and launch groups.  Replacements are shorter than, equal to and longer
    than the old IRs (up to the ring's reach, 7F taps); some stages change part of an output's routes,
    some every route into an output."""
    F = 1 << (rank - 1)
    routes = _routes(F, 40 * rank)
    mx = pkg.MatrixConvolver(3, 2, rank, device=0)
    mx.set_routes(routes)
    model = MatrixFadeModel(3, 2)
    model.set_routes(routes)
    fades = [0, 1, F // 3, F, 5 * F + 17, 40 * F + 3]
    stages = [
        [(0, 4 * F)],                                       # part of output 0, shorter
        [(3, 5 * F), (4, F + 3)],                           # every route into output 1: longer, equal
        [(1, 7 * F), (2, 1)],                               # longer up to the reach; one tap
        [(0, 6 * F + 5), (1, F // 2), (2, 2 * F), (3, 3)],  # routes of both outputs
        [(2, 5 * F), (4, 7 * F)],
        [(0, 1), (1, 2 * F), (2, 3 * F), (3, F), (4, 6 * F)],
    ]
    total = 10 + sum(-(-f // F) + 5 for f in fades)
    x = _inputs(50 * rank, 3, total * F)
    feed = _Feeder(x, F)
    got, want = feed.run([mx, model], 10, (3, 1))
    gots, wants = [got], [want]
    for s, (fade, stage) in enumerate(zip(fades, stages)):
        changes = [(r, _ir(1000 * rank + 10 * s + r, n)) for r, n in stage]
        mx.set_irs(changes, fade=fade)
        model.set_irs(changes, fade=fade)
        assert mx.fade_remaining() == model.fade_remaining() == fade
        got, want = feed.run([mx, model], -(-fade // F) + 5, (1, 3, 8))
        assert mx.fade_remaining() == 0
        gots.append(got)
        wants.append(want)
        assert _err(got, want) <= TOL, (rank, fade)
    assert _err(np.concatenate(gots, axis=1), np.concatenate(wants, axis=1)) <= TOL
    mx.close()


def _pair(pkg, rank, routes, n=2):
    objs = [pkg.MatrixConvolver(3, 2, rank, device=0) for _ in range(n)]
    for o in objs:
        o.set_routes(routes)
    return objs


# rank 13 runs the half-frame inverse (k_inv_half with park and tickets) with and without the delta jobs
@pytest.mark.parametrize("rank", [11, 13])
def test_replacing_an_ir_with_itself_is_bit_identical(pkg, rank):
    F = 1 << (rank - 1)
    routes = _routes(F, 300)
    a, b = _pair(pkg, rank, routes)
    feed = _Feeder(_inputs(310, 3, 40 * F), F)
    ga, gb = feed.run([a, b], 5)
    assert np.array_equal(ga, gb)
    a.set_irs([(0, routes[0][2]), (4, routes[4][2])], fade=3 * F + 5)
    ga, gb = feed.run([a, b], 12)
    assert np.array_equal(ga, gb)
    a.set_irs([(1, routes[1][2]), (2, routes[2][2]), (3, routes[3][2])], fade=0)
    ga, gb = feed.run([a, b], 6)
    assert np.array_equal(ga, gb)
    a.close()
    b.close()


@pytest.mark.parametrize("rank", [11, 13])
def test_equal_length_replacement_bit_identity(pkg, rank):
    """Outputs with no changed route match an untouched object during and after the fade; once the
    fade is over every output matches a fresh object routed with the new IRs from the start."""
    F = 1 << (rank - 1)
    routes = _routes(F, 400)
    new = {0: _ir(410, 6 * F + 5), 1: _ir(411, 2 * F)}       # routes into output 0 only, same lengths
    routed_new = [(i, o, new.get(r, h)) for r, (i, o, h) in enumerate(routes)]
    a, b = _pair(pkg, rank, routes)
    c = _pair(pkg, rank, routed_new, 1)[0]
    feed = _Feeder(_inputs(420, 3, 40 * F), F)
    feed.run([a, b, c], 5)
    a.set_irs(list(new.items()), fade=3 * F + 5)
    during_a, during_b, _ = feed.run([a, b, c], 4)
    assert a.fade_remaining() == 0
    after_a, after_b, after_c = feed.run([a, b, c], 10)
    assert np.array_equal(during_a[1], during_b[1])
    assert np.array_equal(after_a[1], after_b[1])
    assert np.array_equal(after_a, after_c)
    for o in (a, b, c):
        o.close()


def test_failed_calls_change_nothing(pkg):
    rank = 9
    F = 1 << (rank - 1)
    lib = pkg.lib()
    routes = _routes(F, 500)
    a, b = _pair(pkg, rank, routes)
    feed = _Feeder(_inputs(510, 3, 40 * F), F)
    feed.run([a, b], 4)
    h = _ir(520, 64)
    long = _ir(521, 7 * F + 1)                              # 9 rows: beyond the ring's reach (8)

    def bad(idx, irs, lens, fade=F):
        n = len(idx)
        return lib.b200conv_mx_set_irs(a._h, n, (SZ * n)(*idx), (FP * n)(*irs), (SZ * n)(*lens), fade, None)

    hp, lp = h.ctypes.data_as(FP), long.ctypes.data_as(FP)
    assert bad([5], [hp], [64]) == pkg.ERR_ARG                              # route out of range
    assert bad([1, 1], [hp, hp], [64, 64]) == pkg.ERR_ARG                   # route twice
    assert bad([0], [FP()], [64]) == pkg.ERR_ARG                            # NULL impulse response
    assert bad([0], [hp], [0]) == pkg.ERR_ARG                               # empty impulse response
    assert bad([0, 2], [hp, lp], [64, long.size]) == pkg.ERR_ARG            # longer than the ring reaches
    assert bad([0], [hp], [2 ** 64 - 1]) == pkg.ERR_ARG                     # a length whose partition count would wrap
    assert bad([], [], []) == pkg.OK                                        # no-op
    assert a.fade_remaining() == 0
    ga, gb = feed.run([a, b], 6, (1, 3))
    assert np.array_equal(ga, gb)

    change = [(2, _ir(530, 3 * F))]
    a.set_irs(change, fade=6 * F)
    b.set_irs(change, fade=6 * F)
    ga, gb = feed.run([a, b], 2)
    assert a.fade_remaining() == 4 * F
    assert bad([0], [hp], [64]) == pkg.ERR_STATE                            # a fade is in progress
    assert a.fade_remaining() == 4 * F
    ga, gb = feed.run([a, b], 8, (1, 3))
    assert np.array_equal(ga, gb)
    a.close()
    b.close()


def test_widest_matrix_with_delta_outputs(pkg):
    """4096 x 4096, the largest object: a launch group of one frame during a fade has 4096 + 4096 + 1
    transform jobs, more than a group of the same object without a fade."""
    rank, n_io = 8, 4096
    F = 1 << (rank - 1)
    routes = [(0, 0, _ir(1100, 3 * F + 7)), (4095, 4095, _ir(1101, 2 * F)), (7, 4095, _ir(1102, F + 1))]
    mx = pkg.MatrixConvolver(n_io, n_io, rank, device=0)
    mx.set_routes(routes)
    model = MatrixFadeModel(n_io, n_io)
    model.set_routes(routes)
    x = np.zeros((n_io, 12 * F), dtype=np.float32)
    for i in (0, 7, 4095):
        x[i] = synth.noise(1110 + i, 12 * F)
    feed = _Feeder(x, F)
    got, want = feed.run([mx, model], 3)
    change = [(2, _ir(1103, 3 * F))]
    mx.set_irs(change, fade=2 * F + 5)
    model.set_irs(change, fade=2 * F + 5)
    g2, w2 = feed.run([mx, model], 9, (1, 3))
    assert mx.fade_remaining() == 0
    got, want = np.concatenate([got, g2], axis=1), np.concatenate([want, w2], axis=1)
    assert _err(got[[0, 4095]], want[[0, 4095]]) <= TOL
    rest = np.ones(n_io, dtype=bool)
    rest[[0, 4095]] = False
    assert not np.any(got[rest])
    mx.close()


def test_fade_remaining_counts_down(pkg):
    rank = 10
    F = 1 << (rank - 1)
    mx = pkg.MatrixConvolver(3, 2, rank, device=0)
    mx.set_routes(_routes(F, 600))
    feed = _Feeder(_inputs(610, 3, 20 * F), F)
    assert mx.fade_remaining() == 0
    mx.set_irs([(3, _ir(620, 2 * F))], fade=5 * F + 17)
    assert mx.fade_remaining() == 5 * F + 17
    for frames, left in ((1, 4 * F + 17), (3, F + 17), (1, 17), (1, 0)):
        feed.run([mx], frames, (frames,))
        assert mx.fade_remaining() == left
    mx.set_irs([(3, _ir(621, 2 * F))], fade=0)
    assert mx.fade_remaining() == 0
    mx.close()


def test_clear_and_set_routes_during_a_fade(pkg):
    rank = 10
    F = 1 << (rank - 1)
    routes = _routes(F, 700)
    mx = pkg.MatrixConvolver(3, 2, rank, device=0)
    mx.set_routes(routes)
    model = MatrixFadeModel(3, 2)
    model.set_routes(routes)
    feed = _Feeder(_inputs(710, 3, 60 * F), F)
    feed.run([mx, model], 4)
    change = [(0, _ir(720, 5 * F)), (3, _ir(721, F))]
    mx.set_irs(change, fade=10 * F)
    model.set_irs(change, fade=10 * F)
    feed.run([mx, model], 2)
    # clear: the fade ends with the new IRs in place, the history goes
    mx.clear()
    model.clear()
    assert mx.fade_remaining() == 0
    got, want = feed.run([mx, model], 8, (1, 3))
    assert _err(got, want) <= TOL
    # set_routes: replaces everything, the fade included
    mx.set_irs(change[:1], fade=10 * F)
    feed.run([mx], 1)
    other = [(1, 1, _ir(730, 4 * F)), (2, 0, _ir(731, 3 * F))]
    mx.set_routes(other)
    model.set_routes(other)
    assert mx.fade_remaining() == 0
    mx.set_irs([(1, _ir(732, 2 * F))], fade=F // 2)
    model.set_irs([(1, _ir(732, 2 * F))], fade=F // 2)
    got, want = feed.run([mx, model], 8, (3, 1))
    assert _err(got, want) <= TOL
    mx.close()


def test_caller_stream_order_without_host_sync(pkg):
    """process_device, set_irs, process_device on a torch stream with no host sync in between gives
    the same bits as the synchronous planar path."""
    torch = pytest.importorskip("torch")
    rank, frames = 11, 14
    F = 1 << (rank - 1)
    routes = _routes(F, 800)
    a, b = _pair(pkg, rank, routes)
    x = _inputs(810, 3, frames * F)
    change = [(1, _ir(820, 5 * F)), (4, _ir(821, 2))]
    host = []
    for k in range(frames):
        if k == 4:
            a.set_irs(change, fade=3 * F + 100)
        host.append(a.process(x[:, k * F:(k + 1) * F]))
    src = torch.from_numpy(x).cuda()
    dst = torch.empty((2, frames * F), device="cuda")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for k in range(frames):
            if k == 4:
                b.set_irs(change, fade=3 * F + 100, stream=s.cuda_stream)
            b.process_device(dst.data_ptr() + 4 * k * F, dst.stride(0), src.data_ptr() + 4 * k * F, src.stride(0),
                             F, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(np.concatenate(host, axis=1), dst.cpu().numpy())
    a.close()
    b.close()


def test_set_irs_does_not_wait_for_the_device(pkg):
    torch = pytest.importorskip("torch")
    rank = 11
    F = 1 << (rank - 1)
    mx = pkg.MatrixConvolver(3, 2, rank, device=0)
    mx.set_routes(_routes(F, 900))
    src = torch.from_numpy(_inputs(910, 3, 4 * F)).cuda()
    dst = torch.empty((2, 4 * F), device="cuda")
    s = torch.cuda.Stream()
    torch.cuda.synchronize()

    def run(frames):
        for k in range(frames):
            mx.process_device(dst.data_ptr() + 4 * k * F, dst.stride(0), src.data_ptr() + 4 * k * F, src.stride(0),
                              F, stream=s.cuda_stream)

    change = [(0, _ir(920, 3 * F)), (3, _ir(921, 2 * F))]
    mx.set_irs(change, fade=F, stream=s.cuda_stream)          # warm-up: staging, pool
    run(2)
    s.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                          # about 100 ms
    mx.set_irs(change, fade=F, stream=s.cuda_stream)
    busy = not s.query()
    s.synchronize()
    assert busy
    run(2)
    s.synchronize()
    mx.close()


def test_device_memory_stays_bounded(pkg):
    torch = pytest.importorskip("torch")
    rank = 11
    F = 1 << (rank - 1)
    taps = 200 * F
    routes = [(i, o, _ir(1000 + 2 * i + o, taps)) for i in range(2) for o in range(2)]
    ir_set = len(routes) * (taps // F + 1) * F * 8              # G rows of every route
    mx = pkg.MatrixConvolver(2, 2, rank, device=0)
    mx.set_routes(routes)
    x = _inputs(1010, 2, 2 * F)
    bank = [[(r, _ir(2000 + 10 * c + r, taps)) for r in range(4)] for c in range(3)]

    def cycle(c):
        mx.set_irs(bank[c % 3], fade=F + 1)
        mx.process(x)
        assert mx.fade_remaining() == 0

    cycle(0)
    mx.sync()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for c in range(1, 101):
        cycle(c)
    mx.sync()
    free1 = torch.cuda.mem_get_info()[0]
    assert free0 - free1 <= ir_set, (free0, free1, ir_set)
    mx.close()
