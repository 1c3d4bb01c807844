"""Float64 model of the k_frame lookahead schedule (kernels.cuh, LA_BUFS; engine.cu,
process_uniform; DESIGN 4.1c), on the packed spectra of tests/engine_model.py."""
import numpy as np


LA_BUFS = 3     # group buffers of tail sums (kernels.cuh, LA_BUFS)


def pmul(g, x):
    """Packed spectrum product: bins 1.. complex, bin 0 = (DC * DC, Nyquist * Nyquist)."""
    y = g * x
    y[..., 0] = g[..., 0].real * x[..., 0].real + 1j * (g[..., 0].imag * x[..., 0].imag)
    return y


def chunk(n, split, splits):
    return (n * split) // splits, (n * (split + 1)) // splits


class LookaheadModel:
    """The k_frame lookahead schedule for one instance in float64 (kernels.cuh, LA_BUFS; engine.cu,
    process_uniform), index for index: block t of group g (first block t0, t = t0 + c) sums its head
    q < 2K (or every partition when the tails of its group are incomplete: the priming group after
    a (re)start) plus the split rows of T_t, and writes bin slice c of the tails
    T_{t0+K+j} = sum_{q >= 2K} G_q X_{t0+K+j-q}, j < K, into group buffer (g + 1) mod LA_BUFS.
    Every ring row it reads is asserted to hold the frame it wants."""

    def __init__(self, G, K, splits=3, spare=32):
        self.G = np.asarray(G, np.complex128)
        self.nq, self.M = self.G.shape
        self.K, self.splits = K, splits
        self.S = self.nq + spare
        self.ring = np.zeros((self.S, self.M), np.complex128)
        self.frame_of = np.full(self.S, -1, np.int64)       # which frame each ring slot holds
        self.T = np.zeros((LA_BUFS, K, splits, self.M), np.complex128)
        self.t = 0
        self.live = False
        self.origin = 0
        self.next_t = 0
        self.primed = 0                                      # blocks that ran a full sum with lookahead

    def x(self, f, newest):
        s = (-f) % self.S
        assert 0 <= f <= newest and self.frame_of[s] == f, (f, newest)
        return self.ring[s]

    def interrupt(self):
        """any call that is not a lookahead launch: a partial or multi-frame call, a synchronous call,
        a re-init or a table change"""
        self.live = False

    def block(self, X, lookahead=True):
        t = self.t
        s = (-t) % self.S
        self.ring[s] = X
        self.frame_of[s] = t
        K, M, nq = self.K, self.M, self.nq
        qs = min(nq, 2 * K)
        if not lookahead:
            self.live = False
            Y = sum(pmul(self.G[q], self.x(t - q, t)) for q in range(nq) if t - q >= 0)
            self.t += 1
            return Y if not np.isscalar(Y) else np.zeros(M, np.complex128)
        if (not self.live) or (self.next_t != t):
            self.origin = t
        rel = t - self.origin
        c, g = rel % K, (rel // K) % LA_BUFS
        use = rel >= K
        put, get = (g + 1) % LA_BUFS, g
        t0 = t - c
        W = M // K
        sl = slice(c * W, (c + 1) * W)
        for split in range(self.splits):
            a, b = chunk(nq - qs, split, self.splits)
            for j in range(K):
                acc = np.zeros(W, np.complex128)
                for q in range(qs + a, qs + b):
                    f = t0 + K + j - q
                    if f >= 0:
                        assert f <= t0 - 1
                        acc += pmul(self.G[q], self.x(f, t0 - 1))[sl]      # bin 0 sits in slice 0 only
                self.T[put, j, split, sl] = acc
        hq = qs if use else nq
        Y = np.zeros(M, np.complex128)
        for split in range(self.splits):
            a, b = chunk(hq, split, self.splits)
            for q in range(a, b):
                if t - q >= 0:
                    Y += pmul(self.G[q], self.x(t - q, t))
        if use:
            for split in range(self.splits):
                Y += self.T[get, c, split]
        else:
            self.primed += 1
        self.live = True
        self.next_t = t + 1
        self.t += 1
        return Y
