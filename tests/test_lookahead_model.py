"""The k_frame lookahead schedule (float64 model, tests/engine_model.py LookaheadModel) against the
direct partition sum and against direct convolution, for K = 2, 4, 8 and IRs whose partition count
bins + 1 is below, equal to and one above the head of 2K rows, with interruptions inside groups."""
import numpy as np
import pytest

import engine_model as em
import lookahead_model as la
import synth


def spectra(ir, rank):
    F = 1 << (rank - 1)
    tw = em.twiddle_table(1 << rank)
    bins = (ir.size + F - 1) // F
    padded = np.zeros(bins * F, np.float32)
    padded[:ir.size] = ir
    H = np.stack([em.fwd_half_spectrum(padded[p * F:(p + 1) * F], rank, tw) for p in range(bins)])
    return em.fold_partitions(H), tw


@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("extra", [-1, 0, 1, 9])
def test_lookahead_schedule_matches_direct_sum_and_convolution(K, extra):
    rank = 8
    F = 1 << (rank - 1)
    nq = 2 * K + extra                        # bins + 1
    ir = synth.decaying_ir(K * 10 + extra + 1, (nq - 1) * F - 5)
    G, tw = spectra(ir, rank)
    assert G.shape[0] == nq
    frames = 6 * K + nq + 5
    src = synth.noise(3 + K, frames * F)
    X = [em.fwd_half_spectrum(src[t * F:(t + 1) * F], rank, tw) for t in range(frames)]
    model = la.LookaheadModel(G, K, splits=3)
    # interruptions in the middle of groups: a block without lookahead, and a bare interruption
    plain_at = {K + 1, 3 * K + 2}
    out = np.zeros(frames * F, np.float32)
    for t in range(frames):
        if t == 4 * K + 1:
            model.interrupt()
        Y = model.block(X[t].astype(np.complex128), lookahead=t not in plain_at)
        direct = sum(la.pmul(G[q].astype(np.complex128), X[t - q].astype(np.complex128))
                     for q in range(nq) if t - q >= 0)
        assert np.max(np.abs(Y - direct)) <= 1e-9 * max(1.0, np.max(np.abs(direct)))
        out[t * F:(t + 1) * F] = em.inv_first_half(Y.astype(np.complex64), rank, tw)
    # priming groups: the first one, and one after each interruption
    assert model.primed >= 3 * K
    want = np.convolve(src.astype(np.float64), ir.astype(np.float64))[:frames * F]
    assert np.max(np.abs(out - want)) <= 1e-5 * np.max(np.abs(want))
