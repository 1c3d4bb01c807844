"""The k_frame lookahead tail's stage geometry (kernels.cuh frame_body), restated in Python: QT
partitions per stage, NS buffers of G slices and one circular window of ring slices per CTA, each
ring slice copied once.  For ranks 8..13, K = 2, 4, 8, ragged splits and the split-0 bias the model
replays the copies and the reads of every thread in the kernel's order and checks that every
(partition, segment, column) product is formed exactly once from the right G and ring slices, that
no window slot is overwritten while a later stage still reads it, and that the bytes copied equal
the engine's la_stream_bytes (engine.cu).  A GPU test holds the engine's mac_stream_bytes counter
to the same count."""
import pytest

NS_DEFAULT = 2
EARLY_MAX_BYTES = 450000000


def chunk_range(nq, split, splits, bias):
    even = nq // splits
    if nq < splits:
        return min(split, nq), min(split + 1, nq)
    if splits <= 1 or bias == 0 or even <= bias + 1:
        return nq * split // splits, nq * (split + 1) // splits
    len0 = even - bias
    rest = nq - len0
    if split == 0:
        return 0, len0
    return len0 + rest * (split - 1) // (splits - 1), len0 + rest * split // (splits - 1)


def tile_geometry(rank, K, tile, NS):
    M = 1 << (rank - 1)
    TB = min(M, 1024)
    stage_elems = (1024 // TB) * TB
    W = M // K
    Wg = min(W, TB)
    nj = max(1, TB // W)
    QT = ((2 * NS * stage_elems) // Wg - (nj - 1)) // (2 * NS)
    return dict(M=M, TB=TB, T=TB // 4, stage_elems=stage_elems, W=W, Wg=Wg, Wc4=Wg // 2, nj=nj,
                j0=tile * TB // W, p0=tile * TB % W, QT=QT, NW=NS * QT + nj - 1)


def replay_cta(rank, K, tile, NS, tq0, tq1, t0):
    """Copies and reads of one CTA's tail, in the kernel's order.  Returns the slices it copies and
    the products {(q, j, column): (G partition, frame)} its threads form."""
    g = tile_geometry(rank, K, tile, NS)
    QT, NW, nj, Wc4, T = g["QT"], g["NW"], g["nj"], g["Wc4"], g["T"]
    assert QT >= 1
    # shared memory, in slices of Wg bins: NS x QT G slices, then the window
    assert NS * QT + NW <= (2 * NS * g["stage_elems"]) // g["Wg"]
    n_titer = (tq1 - tq0 + QT - 1) // QT
    gbuf = [[None] * QT for _ in range(NS)]
    window = [None] * NW
    fmax = t0 + K + g["j0"] + nj - 1 - tq0
    copied = 0

    def issue(k):
        nonlocal copied
        q = tq0 + k * QT
        rows = min(QT, tq1 - q)
        for r in range(rows):
            gbuf[k % NS][r] = q + r
        s0 = 0 if k == 0 else k * QT + nj - 1
        nx = rows + (nj - 1 if k == 0 else 0)
        for s in range(s0, s0 + nx):
            window[s % NW] = fmax - s
        copied += rows + nx

    products = {}
    run = nj > 1
    threads = []
    for tid in range(T):
        if run:
            col, jv = tid % Wc4, 2 * (tid // Wc4)
            threads.append(((col, jv), (col, jv + 1)))
        else:
            threads.append(((tid, 0), (tid + T, 0)))
    for k in range(min(NS, n_titer)):
        issue(k)
    xs = {tid: nj - 1 - threads[tid][0][1] for tid in range(T)}
    xp = {}
    for k in range(n_titer):
        rows = min(QT, tq1 - (tq0 + k * QT))
        for tid, ((c0, j_0), (c1, j_1)) in enumerate(threads):
            if run and k == 0:
                xp[tid] = window[(xs[tid] - 1) % NW]
            for r in range(rows):
                q = tq0 + k * QT + r
                gq = gbuf[k % NS][r]
                x0 = window[xs[tid]]
                if run:
                    x1, xp[tid] = xp[tid], x0
                else:
                    x1 = window[xs[tid]]
                for (col, j), x in (((c0, j_0), x0), ((c1, j_1), x1)):
                    key = (q, j, col)
                    assert key not in products, "product formed twice"
                    products[key] = (gq, x)
                xs[tid] = (xs[tid] + 1) % NW
        # __syncthreads(): then stage k + NS may overwrite what stage k read
        if k + NS < n_titer:
            issue(k + NS)
    return g, products, copied


def la_stream_bytes(F, q_lo, nq, K, use, splits, bias, TB):
    """engine.cu la_stream_bytes"""
    q_hi = q_lo + nq
    qs = max(q_lo, min(q_hi, 2 * K))
    nh = (qs - q_lo) if use else nq
    nt = q_hi - qs
    W = F // K
    Wg, nj = min(W, TB), max(1, TB // W)
    slices = 0
    for s in range(splits):
        e0, e1 = chunk_range(nt, s, splits, bias)
        if e1 > e0:
            slices += 2 * (e1 - e0) + nj - 1
    return 16 * F * nh + (F // TB) * slices * 8 * Wg + 8 * F * splits * (2 if use else 1) + 8 * F


def la_stream_bytes_one_pass(F, q_lo, nq, K, use, splits):
    """the figure la_stream_bytes gave before: one pass over the window, (2 nt + K - 1) slices"""
    q_hi = q_lo + nq
    qs = max(q_lo, min(q_hi, 2 * K))
    nh = (qs - q_lo) if use else nq
    nt = q_hi - qs
    tail = (8 * F // K) * (2 * nt + K - 1) if nt > 0 else 0
    return 16 * F * nh + tail + 8 * F * splits * (2 if use else 1) + 8 * F


CASES = [(rank, K, nq, splits, bias)
         for rank in range(8, 14) for K in (2, 4, 8)
         for nq, splits, bias in ((6 * K + 1, 1, 0), (8 * K + 5, 3, 0), (469, 8, 6), (8 * K + 13, 5, 2), (2 * K + 3, 4, 6))]


@pytest.mark.parametrize("NS", [2, 3])
@pytest.mark.parametrize("rank,K,nq,splits,bias", CASES)
def test_tail_products_once_window_safe_bytes_exact(rank, K, nq, splits, bias, NS):
    t0 = 1000
    q_lo, qs = 0, min(nq, 2 * K)
    nt = nq - qs
    M = 1 << (rank - 1)
    tiles = M // min(M, 1024)
    copied = 0
    for tile in range(tiles):
        seen = {}
        for split in range(splits):
            e0, e1 = chunk_range(nt, split, splits, bias)
            g, products, n = replay_cta(rank, K, tile, NS, qs + e0, qs + e1, t0)
            copied += n * 8 * g["Wg"]
            for key, (gq, frame) in products.items():
                q, j, col = key
                assert gq == q, "G slice of the wrong partition"
                assert frame == t0 + K + g["j0"] + j - q, "ring slice of the wrong frame"
                assert key not in seen
                seen[key] = split
        g = tile_geometry(rank, K, tile, NS)
        assert set(seen) == {(q, j, c) for q in range(qs, nq) for j in range(g["nj"]) for c in range(g["Wc4"])}
    fixed = 16 * M * qs + 8 * M * splits * 2 + 8 * M
    assert copied + fixed == la_stream_bytes(M, q_lo, nq, K, True, splits, bias, min(M, 1024))


def test_rank11_k8_stage_holds_six_partitions_and_copies_each_slice_once():
    g = tile_geometry(11, 8, 0, NS_DEFAULT)
    assert (g["QT"], g["NW"], g["nj"]) == (6, 19, 8)
    _, _, n = replay_cta(11, 8, 0, NS_DEFAULT, 16, 73, 1000)
    assert n == 2 * (73 - 16) + 7


def plan_splits(n, rank, max_nq, sm_count=148):
    M = 1 << (rank - 1)
    TB = min(M, 1024)
    tiles, QB = M // TB, 1024 // TB
    splits = (7 * sm_count // 2) // (n * tiles)
    return max(1, min(splits, max_nq // (2 * QB), 32))


@pytest.mark.parametrize("n,taps,rank,K", [
    (64, 480000, 11, 8), (32, 480000, 11, 8), (16, 480000, 11, 8),     # config 3 on 1, 2, 4 GPUs
    (4096, 48000, 11, 4),                                              # config 4, one frame per call
    (64, 480000, 9, 2)])                                               # 64 x 10 s at rank 9
def test_early_transform_gate_decides_as_before(n, taps, rank, K):
    F = 1 << (rank - 1)
    nq = (taps + F - 1) // F + 1
    splits = plan_splits(n, rank, nq)
    for use in (False, True):
        new = n * la_stream_bytes(F, 0, nq, K, use, splits, 6, min(F, 1024))
        old = n * la_stream_bytes_one_pass(F, 0, nq, K, use, splits)
        assert new >= old
        assert (new <= EARLY_MAX_BYTES) == (old <= EARLY_MAX_BYTES)


@pytest.mark.gpu
@pytest.mark.parametrize("rank,K,splits", [(11, 8, 8), (12, 4, 3), (9, 2, 5)])
def test_engine_counts_the_bytes_the_tail_copies(rank, K, splits):
    torch = pytest.importorskip("torch")
    import __graft_entry__ as ge
    import synth
    pkg = ge.load()
    n, taps = 3, 90000
    F = 1 << (rank - 1)
    b = pkg.ConvolverBatch(n, 0)
    b.set_option("lookahead", K)
    b.set_option("mac_splits", splits)
    for c in range(n):
        assert b.init(c, synth.decaying_ir(c, taps), rank, 0.0)
    src = torch.rand((n, 64 * F), device="cuda") * 2 - 1
    dst = torch.empty_like(src)
    for i in range(2 * K):
        b.process_device(dst.data_ptr() + 4 * i * F, src.data_ptr() + 4 * i * F, 64 * F, F)
    b.sync()
    b.reset_stats()
    calls = 3 * K
    for i in range(2 * K, 2 * K + calls):
        b.process_device(dst.data_ptr() + 4 * i * F, src.data_ptr() + 4 * i * F, 64 * F, F)
    b.sync()
    st = b.stats()
    b.close()
    nq = (taps + F - 1) // F + 1
    want = n * la_stream_bytes(F, 0, nq, K, True, splits, 6, min(F, 1024))
    assert st["mac_launches"] == calls
    assert st["mac_stream_bytes"] == calls * want
