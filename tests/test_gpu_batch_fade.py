"""b200conv_set_irs / ConvolverBatch.set_irs on the GPU: new impulse responses for running instances,
keeping their input history and crossfading old to new, against the float64 model of
tests/batch_fade_model.py.  Bar: max |gpu - model| <= 1e-5 of the model's peak, per instance."""
import ctypes

import numpy as np
import pytest

from batch_fade_model import BatchFadeModel
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


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _ir(seed, n):
    return synth.decaying_ir(seed, n)


def _err(got, want):
    peak = np.max(np.abs(want))
    return float(np.max(np.abs(np.asarray(got, np.float64) - want)) / peak) if peak > 0 else float(np.max(np.abs(got)))


class Rig:
    """One input matrix fed to GPU batches and to one model per instance in the same calls, through
    one entry point: "device" (process_device on the batch's stream, or on `stream`), "inplace"
    (process_device with dst == src), "host" (b200conv_process: pointer table), "planar"
    (process_planar, pageable) or "pinned" (process_planar on page-locked matrices)."""

    def __init__(self, torch, x, F, entry="device", stream=None):
        self.torch, self.x, self.F, self.entry, self.stream = torch, x, F, entry, stream
        self.at, self.n, self.total = 0, x.shape[0], x.shape[1]
        self.want = np.zeros(x.shape)
        if entry in ("device", "inplace"):
            self.src = torch.from_numpy(x).cuda()
            self.dst = self.src.clone() if entry == "inplace" else torch.zeros_like(self.src)
            if entry == "inplace":
                self.src = self.dst
            torch.cuda.synchronize()
        elif entry == "pinned":
            self.pinned = (torch.from_numpy(x).pin_memory(), torch.zeros(x.shape, dtype=torch.float32).pin_memory())
            self.hsrc, self.hdst = self.pinned[0].numpy(), self.pinned[1].numpy()
        else:
            self.hsrc, self.hdst = np.ascontiguousarray(x), np.zeros(x.shape, dtype=np.float32)

    def call(self, b, at, n):
        if self.entry in ("device", "inplace"):
            st = None if self.stream is None else self.stream.cuda_stream
            b.process_device(self.dst.data_ptr() + 4 * at, self.src.data_ptr() + 4 * at, self.total, n, st)
        elif self.entry == "host":
            b.process_pointers([self.hdst[i, at:at + n] for i in range(self.n)],
                               [self.hsrc[i, at:at + n] for i in range(self.n)], n)
        else:
            b.process(self.hsrc[:, at:at + n], out=self.hdst[:, at:at + n])

    def run(self, b, models, samples, sizes, check=None):
        """`check(b, models)` after every call"""
        end, k = self.at + samples, 0
        while self.at < end:
            n = min(sizes[k % len(sizes)], end - self.at)
            self.call(b, self.at, n)
            for i, m in enumerate(models):
                self.want[i, self.at:self.at + n] = m.process(self.x[i, self.at:self.at + n])
            self.at += n
            k += 1
            if check is not None:
                check(b, models)

    def out(self):
        if self.entry in ("device", "inplace"):
            self.torch.cuda.synchronize()
            return self.dst.cpu().numpy()
        return np.array(self.hdst)

    def check(self, got=None):
        got = self.out() if got is None else got
        for i in range(self.n):
            assert _err(got[i, :self.at], self.want[i, :self.at]) <= TOL, i


def _batch(pkg, rank, irs, phases=None):
    b = pkg.ConvolverBatch(len(irs), 0)
    models = []
    for c, ir in enumerate(irs):
        assert b.init(c, ir, rank, 0.0 if phases is None else phases[c])
        models.append(BatchFadeModel(1 << (rank - 1)))
        models[-1].init(ir)
    return b, models


def _set_irs(b, models, changes, fade):
    b.set_irs([i for i, _ in changes], [h for _, h in changes], fade=fade)
    for i, h in changes:
        models[i].set_irs(h, fade=fade)


def _remaining_matches(b, models):
    for i, m in enumerate(models):
        assert b.fade_remaining(i) == m.fade_remaining(), i


SHAPES = {
    # name: (call sizes in units of F / 12, phases, lookahead option)
    "frame": ((12,), None, None),
    "frame_la2": ((12,), None, 2),
    "frame_la0": ((12,), None, 0),
    "multi": ((36, 96, 12), None, None),
    "sub": ((3,), (0.5, 0.25, 0.0), None),
    "mixed": ((4, 12, 29, 1), (0.5, 0.0, 0.25), None),
}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("rank", [8, 10, 11, 13, 14, 16])
def test_fades_against_model(pkg, torch, rank, shape):
    """Three instances (6F + 5, 3F + 1 and 2F taps).  Instance 0 swaps to a shorter IR right after its
    ring (40 slots) wrapped, with a fade of 4F + 7 samples; 2F later, while 0 still fades, instance 1
    starts a fade of 5F + 17 samples (equal length), so set_irs rebuilds the twin around the running
    fade.  0 hands over first and 1 keeps fading in a twin with a free slot, which the next set_irs
    (instance 2, F + 5 samples) leaves behind; 1's fade ends inside a call.  Then 0 fades out to a
    one-tap zero IR and 2 swaps to a slightly shorter IR in one set_irs.  With the "sub" and "mixed"
    shapes the swaps fall inside frames (phases), so the pending blocks are recomputed."""
    F = 1 << (rank - 1)
    unit, phases, la = SHAPES[shape]
    sizes = tuple(max(1, u * F // 12) for u in unit)
    irs = [_ir(10 * rank, 6 * F + 5), _ir(10 * rank + 1, 3 * F + 1), _ir(10 * rank + 2, 2 * F)]
    b, models = _batch(pkg, rank, irs, phases)
    if la is not None and rank <= 13:
        b.set_option("lookahead", la)
    x = np.stack([synth.noise(100 * rank + c, 60 * F) for c in range(3)])
    rig = Rig(torch, x, F)
    rig.run(b, models, 41 * F, sizes)
    _set_irs(b, models, [(0, _ir(1000 + rank, 4 * F))], 4 * F + 7)
    rig.run(b, models, 2 * F, sizes, _remaining_matches)
    assert b.fade_remaining(0) == 2 * F + 7                 # still fading: set_irs moves it into a new twin
    _set_irs(b, models, [(1, _ir(2000 + rank, 3 * F + 1))], 5 * F + 17)
    assert b.fade_remaining(1) == 5 * F + 17 and b.fade_remaining(0) == 2 * F + 7
    rig.run(b, models, 3 * F, sizes, _remaining_matches)
    assert b.fade_remaining(0) == 0 and b.fade_remaining(1) > 0     # 0 handed over, 1 runs on
    _set_irs(b, models, [(2, _ir(2500 + rank, 2 * F - 3))], F + 5)  # the twin had a free slot
    rig.run(b, models, 4 * F, sizes, _remaining_matches)
    assert b.fade_remaining(2) == 0
    assert b.fade_remaining(1) == 0
    assert b.state(0)["conv_size"] == 4 * F and b.state(0)["partitions"] == 5
    _set_irs(b, models, [(0, np.zeros(1, np.float32)), (2, _ir(3000 + rank, 2 * F - 3))], 2 * F)
    rig.run(b, models, 10 * F, sizes, _remaining_matches)
    rig.check()
    got = rig.out()
    assert not np.any(got[0, 57 * F:])                  # faded out
    b.close()


@pytest.mark.parametrize("fade", [0, 3])
@pytest.mark.parametrize("rank", [11, 14])
def test_swap_inside_a_frame_recomputes_the_pending_block(pkg, torch, rank, fade):
    """Half a frame in, the pending block (what the complete frames add to the frame in progress)
    was made with the old IR; after the swap the rest of that frame must come from the new one."""
    F = 1 << (rank - 1)
    b, models = _batch(pkg, rank, [_ir(7, 3 * F + 1)])
    rig = Rig(torch, synth.noise(8, 12 * F)[None, :], F)
    rig.run(b, models, 3 * F + F // 2, (F, F, F, F // 2))
    _set_irs(b, models, [(0, _ir(9, 2 * F + 7))], fade)
    rig.run(b, models, 4 * F, (F // 4, F // 2, F))
    rig.check()
    b.close()


def _bit_rig(pkg, torch, rank, irs, x):
    b = pkg.ConvolverBatch(len(irs), 0)
    b.set_option("lookahead", 0)
    for c, ir in enumerate(irs):
        assert b.init(c, ir, rank, 0.0)
    return b, Rig(torch, x, 1 << (rank - 1))


@pytest.mark.parametrize("rank", [11, 14])
def test_bit_identity(pkg, torch, rank):
    """One-frame process_device calls, equal-length IRs, lookahead off.  While instance 1 fades, the
    other instances are bit-identical to the same batch without set_irs; once the fade is over,
    instance 1 is bit-identical to a batch that had the new IR from the start."""
    F = 1 << (rank - 1)
    irs = [_ir(40 + c, 5 * F - 3) for c in range(3)]
    h_new = _ir(50, 5 * F - 3)
    x = np.stack([synth.noise(60 + c, 40 * F) for c in range(3)])
    fad, rf = _bit_rig(pkg, torch, rank, irs, x)
    ref, rr = _bit_rig(pkg, torch, rank, irs, x)
    fresh, rn = _bit_rig(pkg, torch, rank, [irs[0], h_new, irs[2]], x)
    for b, r in ((fad, rf), (ref, rr), (fresh, rn)):
        r.run(b, [], 9 * F, (F,))
    fad.set_irs([1], [h_new], fade=3 * F + 5)
    for b, r in ((fad, rf), (ref, rr), (fresh, rn)):
        r.run(b, [], 31 * F, (F,))
    a, o, n = rf.out(), rr.out(), rn.out()
    assert fad.fade_remaining(1) == 0
    assert np.array_equal(a[0], o[0]) and np.array_equal(a[2], o[2])
    assert np.array_equal(a[1, :9 * F], o[1, :9 * F])
    assert np.array_equal(a[1, 13 * F:], n[1, 13 * F:])
    assert not np.array_equal(a[1, 9 * F:12 * F], o[1, 9 * F:12 * F])
    for b in (fad, ref, fresh):
        b.close()


@pytest.mark.parametrize("entry", ["device", "stream", "inplace", "host", "planar", "pinned"])
def test_every_entry_point(pkg, torch, entry):
    """The same fade through every process entry point, with call sizes that are and are not whole
    frames; on a caller's stream nothing synchronises the host between calls."""
    rank = 11
    F = 1 << (rank - 1)
    irs = [_ir(70, 4 * F + 9), _ir(71, 2 * F), _ir(72, 3 * F)]
    b, models = _batch(pkg, rank, irs, (0.0, 0.5, 0.0))
    x = np.stack([synth.noise(80 + c, 30 * F) for c in range(3)])
    stream = torch.cuda.Stream() if entry == "stream" else None
    rig = Rig(torch, x, F, "device" if entry == "stream" else entry, stream)
    rig.run(b, models, 6 * F, (F, 2 * F, 300))
    _set_irs(b, models, [(0, _ir(73, 3 * F)), (1, _ir(74, F + 1))], 4 * F + 11)
    rig.run(b, models, 12 * F, (F, 300, 2 * F))
    _set_irs(b, models, [(2, _ir(75, 3 * F))], F // 2)
    rig.run(b, models, 12 * F - 300, (F, 77))
    if stream is not None:
        stream.synchronize()
    rig.check()
    assert all(b.fade_remaining(i) == 0 for i in range(3))
    b.close()


@pytest.mark.parametrize("rank", [11, 14])
def test_cascade_with_the_first_batch_fading(pkg, torch, rank):
    """Two batches on one caller stream, the second reading what the first writes, while the first
    one's instance fades."""
    F = 1 << (rank - 1)
    n, frames = 2, 24
    irs_a = [_ir(90 + c, 3 * F + 2) for c in range(n)]
    irs_b = [_ir(95 + c, 2 * F + 5) for c in range(n)]
    a, ma = _batch(pkg, rank, irs_a)
    bb, mb = _batch(pkg, rank, irs_b)
    x = np.stack([synth.noise(99 + c, frames * F) for c in range(n)])
    src = torch.from_numpy(x).cuda()
    mid, out = torch.zeros_like(src), torch.zeros_like(src)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    want = np.zeros(x.shape)
    for f in range(frames):
        if f == 5:
            _set_irs(a, ma, [(1, _ir(98, 2 * F))], 4 * F + 3)
        o = 4 * f * F
        a.process_device(mid.data_ptr() + o, src.data_ptr() + o, frames * F, F, st.cuda_stream)
        bb.process_device(out.data_ptr() + o, mid.data_ptr() + o, frames * F, F, st.cuda_stream)
        for c in range(n):
            want[c, f * F:(f + 1) * F] = mb[c].process(ma[c].process(x[c, f * F:(f + 1) * F]))
    st.synchronize()
    got = out.cpu().numpy()
    for c in range(n):
        assert _err(got[c], want[c]) <= TOL, c
    a.close()
    bb.close()


def test_errors_leave_no_trace(pkg, torch):
    """Every refused set_irs leaves the batch's output bit-identical to a batch that never saw it."""
    rank = 11
    F = 1 << (rank - 1)
    irs = [_ir(110 + c, 3 * F) for c in range(3)]
    x = np.stack([synth.noise(120 + c, 20 * F) for c in range(4)])
    objs = []
    for _ in range(2):
        b = pkg.ConvolverBatch(4, 0)
        for c, ir in enumerate(irs):
            assert b.init(c, ir, rank, 0.0)
        objs.append((b, Rig(torch, x, F)))
    for b, r in objs:
        r.run(b, [], 4 * F, (F,))
        b.set_irs([2], [_ir(130, 2 * F)], fade=6 * F)       # both: a fade in progress
    (b, r), lib = objs[0], pkg.lib()
    h = _ir(131, 2 * F)
    cases = [
        (pkg.ERR_ARG, [4], [h]),                            # out of range
        (pkg.ERR_ARG, [0, 0], [h, h]),                      # twice
        (pkg.ERR_ARG, [0], [np.zeros(0, np.float32)]),      # empty
        (pkg.ERR_ARG, [0], [_ir(132, 3 * F + 1)]),          # more partitions than the ring reaches
        (pkg.ERR_STATE, [3], [h]),                          # not initialised
        (pkg.ERR_STATE, [2], [h]),                          # already fading
        (pkg.ERR_STATE, [0, 2], [h, h]),                    # one of them already fading
    ]
    for code, idx, hs in cases:
        with pytest.raises(pkg.B200ConvError) as e:
            b.set_irs(idx, hs, fade=F)
        assert "error %d:" % code in str(e.value), (idx, str(e.value))
    rc = lib.b200conv_set_irs(b._h, 1, (SZ * 1)(0), None, (SZ * 1)(F), 0)
    assert rc == pkg.ERR_ARG
    rc = lib.b200conv_set_irs(b._h, 1, (SZ * 1)(0), (FP * 1)(), (SZ * 1)(F), 0)
    assert rc == pkg.ERR_ARG
    assert lib.b200conv_set_irs(b._h, 0, None, None, None, 5) == pkg.OK
    assert b.init_shared(3, 0)
    objs[1][0].init_shared(3, 0)
    with pytest.raises(pkg.B200ConvError) as e:
        b.set_irs([0], [h], fade=F)                         # lends its spectra
    assert "error %d:" % pkg.ERR_STATE in str(e.value)
    with pytest.raises(pkg.B200ConvError):
        b.init_shared(1, 2)                                 # borrowing from a fading instance
    for b, r in objs:
        r.run(b, [], 16 * F, (F, 300))
    a, o = objs[0][1].out(), objs[1][1].out()
    assert np.array_equal(a, o)
    for b, _ in objs:
        b.close()


def test_init_and_destroy_end_a_fade_and_a_borrower_fades(pkg, torch):
    rank = 10
    F = 1 << (rank - 1)
    irs = [_ir(140 + c, 4 * F) for c in range(4)]
    b, models = _batch(pkg, rank, irs[:3] + [irs[0]])
    assert b.init_shared(3, 0)                             # 3 borrows 0's spectra
    x = np.stack([synth.noise(150 + c, 40 * F) for c in range(4)])
    rig = Rig(torch, x, F)
    rig.run(b, models, 5 * F, (F, 100))
    _set_irs(b, models, [(1, _ir(160, 2 * F)), (2, _ir(161, 3 * F)), (3, _ir(162, 4 * F))], 8 * F)
    rig.run(b, models, 2 * F, (F, 100))
    assert b.fade_remaining(1) > 0
    b.init(1, irs[1], rank, 0.0)                            # ends the fade: a fresh instance
    models[1].init(irs[1])
    b.destroy(2)
    models[2].destroy()
    assert b.fade_remaining(1) == b.fade_remaining(2) == 0 and b.fade_remaining(3) > 0
    with pytest.raises(pkg.B200ConvError):
        b.destroy(0)                                        # still lends to 3 until its fade is over
    rig.run(b, models, 10 * F, (F, 100))
    assert b.fade_remaining(3) == 0
    rig.check()
    b.destroy(0)                                            # 3 owns its spectra now
    models[0].destroy()
    rig.run(b, models, 5 * F, (F,))
    rig.check()
    b.close()


def test_device_memory_returns_after_the_handover(pkg, torch):
    """Fades of instances whose IRs are alone in their allocations: once the new IRs have taken over,
    device memory is back at its level before the first set_irs on the batch (new and old IRs are the
    same length).  A batch of its own runs one fade first, so that loading the fade kernels is not
    counted; during a fade the twin's memory is visible."""
    rank = 11
    F = 1 << (rank - 1)
    taps = 200000
    x = torch.rand((4, 64 * F), device="cuda") * 2 - 1
    y = torch.zeros_like(x)

    def batch(seed):
        b = pkg.ConvolverBatch(4, 0)
        for c in range(4):
            assert b.init(c, _ir(seed + c, taps), rank, 0.0)
        for f in range(4):
            b.process_device(y.data_ptr() + 4 * f * F, x.data_ptr() + 4 * f * F, 64 * F, F)
        b.sync()
        return b

    def cycle(b, k, mid=None):
        b.set_irs([k % 4], [_ir(180 + k, taps)], fade=3 * F)
        for f in range(5):
            b.process_device(y.data_ptr() + 4 * f * F, x.data_ptr() + 4 * f * F, 64 * F, F)
            if f == 0 and mid is not None:
                b.sync()
                mid.append(torch.cuda.mem_get_info()[0])
        b.sync()
        assert b.fade_remaining(k % 4) == 0

    warm = batch(160)
    cycle(warm, 0)
    warm.close()
    b = batch(170)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    mid = []
    cycle(b, 0, mid)
    for k in range(1, 9):
        cycle(b, k)
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    assert free0 - mid[0] > (2 << 20), (free0, mid[0])
    assert abs(free0 - free1) <= (2 << 20), (free0, free1)
    b.close()
