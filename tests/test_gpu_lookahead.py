"""k_frame lookahead for streams of one-frame calls (kernels.cuh, LA_BUFS; DESIGN 4.1c).

The launches of a group of K blocks sum, each over one bin slice, the partitions q >= 2K of the
next group's blocks.  Only the order of the partition sum changes, so results are checked against
float64 truth at 1e-5 of peak, and every way of running a stream (programmatic launch on or off,
profiling, interruptions) must give the same bits."""
import numpy as np
import pytest
from scipy.signal import fftconvolve

import synth

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    p = ge.load()
    p.lib()
    return p


def truth(src, ir, n):
    return fftconvolve(np.asarray(src, np.float64), np.asarray(ir, np.float64))[:n]


def rel_err(got, want):
    peak = np.max(np.abs(want))
    return float(np.max(np.abs(np.asarray(got, np.float64) - want)) / peak) if peak > 0 else float(np.max(np.abs(got)))


def one_frame_calls(b, dst, src, F, first, count, stride, stream=None):
    for i in range(first, first + count):
        b.process_device(dst.data_ptr() + 4 * i * F, src.data_ptr() + 4 * i * F, stride, F, stream)


@pytest.mark.parametrize("rank", [8, 9, 10, 11, 12, 13])
@pytest.mark.parametrize("K", [2, 4, 8])
def test_lookahead_ragged_batches_every_rank_and_group_size(pkg, rank, K):
    """IRs shorter than the head (bins + 1 < 2K), exactly the head (= 2K), one partition of tail
    (2K + 1), a single tap, a long one and an uninitialised instance in one batch."""
    torch = pytest.importorskip("torch")
    F = 1 << (rank - 1)
    lens = [(2 * K - 2) * F, (2 * K - 1) * F, 2 * K * F, 1, 23 * F + 5, 0, (2 * K - 1) * F - 3]
    n, frames = len(lens), 5 * K + 30
    irs = [synth.decaying_ir(c, L) if L else None for c, L in enumerate(lens)]
    g = torch.Generator(device="cuda").manual_seed(100 + rank * 10 + K)
    src = torch.rand((n, frames * F), generator=g, device="cuda") * 2 - 1
    b = pkg.ConvolverBatch(n, 0)
    b.set_option("lookahead", K)
    for c, ir in enumerate(irs):
        if ir is not None:
            assert b.init(c, ir, rank, 0.0)
    dst = torch.zeros_like(src)
    b.reset_stats()
    one_frame_calls(b, dst, src, F, 0, frames, frames * F)
    b.sync()
    st = b.stats()
    assert st["launches"] == frames and st["mac_launches"] == frames
    out, x = dst.cpu().numpy(), src.cpu().numpy()
    for c, ir in enumerate(irs):
        if ir is None:
            assert not out[c].any()
        else:
            assert rel_err(out[c], truth(x[c], ir, frames * F)) <= TOL, (c, lens[c])
    b.close()


def test_lookahead_full_size_cfg3_ring_wraps_twice(pkg):
    """64 x 480 000 taps at rank 11 (the automatic choice), 1100 blocks: the input-spectrum ring
    (502 slots) wraps twice."""
    torch = pytest.importorskip("torch")
    n, taps, rank, frames = 64, 480000, 11, 1100
    F = 1 << (rank - 1)
    irs = [synth.decaying_ir(c, taps) for c in range(4)]
    g = torch.Generator(device="cuda").manual_seed(11)
    src = torch.rand((n, frames * F), generator=g, device="cuda") * 2 - 1
    b = pkg.ConvolverBatch(n, 0)
    assert b.init_many(list(range(n)), [irs[c % 4] for c in range(n)], rank)
    dst = torch.zeros_like(src)
    b.reset_stats()
    one_frame_calls(b, dst, src, F, 0, frames, frames * F)
    b.sync()
    st = b.stats()
    assert st["launches"] == frames and st["mac_launches"] == frames
    # steady state streams far fewer bytes than the one-pass schedule
    assert st["mac_stream_bytes"] * 3 < st["mac_algo_bytes"]
    for c in (0, 1, 38, 63):
        want = truth(src[c].cpu().numpy(), irs[c % 4], frames * F)
        assert rel_err(dst[c].cpu().numpy(), want) <= TOL, c
    b.close()


def run_interrupted(pkg, torch, pdl, lookahead, n=6, taps=70000, rank=10):
    """A stream of one-frame device calls interrupted in the middle of groups by every kind of
    call that ends a lookahead schedule.  Returns (outputs, inputs, irs, re-init frame)."""
    F = 1 << (rank - 1)
    frames = 120
    irs = [synth.decaying_ir(c, taps) for c in range(n)]
    new_ir = synth.decaying_ir(99, taps // 3)
    g = torch.Generator(device="cuda").manual_seed(5)
    src = torch.rand((n, frames * F), generator=g, device="cuda") * 2 - 1
    b = pkg.ConvolverBatch(n, 0)
    b.set_option("pdl", pdl)
    b.set_option("lookahead", lookahead)
    for c in range(n):
        assert b.init(c, irs[c], rank, 0.0)
    dst = torch.zeros_like(src)
    stride = frames * F
    f = 0

    def frames_(k):
        nonlocal f
        one_frame_calls(b, dst, src, F, f, k, stride)
        f += k

    frames_(11)                                                     # group of 4: stops at c = 3 of group 2
    # a partial call, then the rest of the frame (the general path)
    b.process_device(dst.data_ptr() + 4 * f * F, src.data_ptr() + 4 * f * F, stride, 300)
    b.process_device(dst.data_ptr() + 4 * (f * F + 300), src.data_ptr() + 4 * (f * F + 300), stride, F - 300)
    f += 1
    frames_(6)
    # a multi-frame call
    b.process_device(dst.data_ptr() + 4 * f * F, src.data_ptr() + 4 * f * F, stride, 3 * F)
    f += 3
    frames_(9)
    # re-init of one instance
    reinit_at = f
    assert b.init(2, new_ir, rank, 0.0)
    frames_(10)
    # profiling on, then off
    b.set_profiling(True)
    frames_(7)
    b.sync()
    b.profile()
    b.set_profiling(False)
    frames_(5)
    # synchronous host calls (the eager pending-MAC path)
    b.sync()
    for _ in range(3):
        blk = src[:, f * F:(f + 1) * F].cpu().numpy()
        dst[:, f * F:(f + 1) * F] = torch.from_numpy(b.process(blk)).cuda()
        f += 1
    frames_(frames - f)
    b.sync()
    out = dst.cpu().numpy()
    b.close()
    return out, src.cpu().numpy(), irs, new_ir, reinit_at, F


@pytest.mark.parametrize("lookahead", [4, 8])
def test_lookahead_interruptions_pdl_bit_identity_and_truth(pkg, lookahead):
    torch = pytest.importorskip("torch")
    o1, x, irs, new_ir, at, F = run_interrupted(pkg, torch, 1, lookahead)
    o0, _, _, _, _, _ = run_interrupted(pkg, torch, 0, lookahead)
    assert np.array_equal(o1, o0)
    n = x.shape[1]
    for c in range(len(irs)):
        if c == 2:
            cut = at * F
            assert rel_err(o1[c][:cut], truth(x[c][:cut], irs[c], cut)) <= TOL
            assert rel_err(o1[c][cut:], truth(x[c][cut:], new_ir, n - cut)) <= TOL
        else:
            assert rel_err(o1[c], truth(x[c], irs[c], n)) <= TOL, c
    # lookahead off: the same results up to the order of the partition sum
    off, _, _, _, _, _ = run_interrupted(pkg, torch, 1, 0)
    assert float(np.max(np.abs(off - o1)) / np.max(np.abs(off))) <= TOL


def test_lookahead_automatic_vs_off_at_cfg3(pkg):
    """The automatic choice at the headline shape, against lookahead off: within 1e-5 of peak,
    and one launch per block either way."""
    torch = pytest.importorskip("torch")
    n, taps, rank, frames = 64, 480000, 11, 200
    F = 1 << (rank - 1)
    irs = [synth.decaying_ir(c, taps) for c in range(4)]
    g = torch.Generator(device="cuda").manual_seed(12)
    src = torch.rand((n, frames * F), generator=g, device="cuda") * 2 - 1
    outs, streamed = [], []
    for la in (-1, 0):
        b = pkg.ConvolverBatch(n, 0)
        b.set_option("lookahead", la)
        assert b.init_many(list(range(n)), [irs[c % 4] for c in range(n)], rank)
        dst = torch.zeros_like(src)
        b.reset_stats()
        one_frame_calls(b, dst, src, F, 0, frames, frames * F)
        b.sync()
        st = b.stats()
        assert st["launches"] == frames
        streamed.append(st["mac_stream_bytes"])
        outs.append(dst.cpu().numpy())
        b.close()
    assert streamed[0] < streamed[1]
    assert float(np.max(np.abs(outs[0] - outs[1])) / np.max(np.abs(outs[1]))) <= TOL
