"""Float64 models of the batched Equalizer, SpectralProcessor and SpectralSplitter that step every
instance of a batch at once, numpy on an instance axis (axis 0).  The per-instance models
(equalizer_model.ModelEqualizer, spectral_model.ModelSpectralProcessor,
splitter_model.ModelSpectralSplitter) are Python loops per instance; these check thousands of rows.
tests/test_batch_models.py holds them to the per-instance models.

Instances whose phases differ have different frame schedules: the spectral models group the rows
by their current offset and step each group vectorised.  For a real input and any table H of N
bins, Re(IFFT(X H)) = IRFFT(X[k] (H[k] + conj(H[N - k])) / 2) over the N / 2 + 1 unique bins, so
the table paths transform with rfft / irfft (half the work of the full complex transforms)."""
import numpy as np


def fold(H):
    """[..., N] full tables -> [..., N / 2 + 1] Hermitian parts (H[k] + conj(H[N - k])) / 2."""
    H = np.asarray(H, dtype=np.complex128)
    N = H.shape[-1]
    k = np.arange(N // 2 + 1)
    return 0.5 * (H[..., k] + np.conj(H[..., (N - k) % N]))


class BatchEqualizer:
    """ModelEqualizer (Equalizer.cpp:474-518) for `n` instances fed the same call sizes."""

    def __init__(self, n, fir_rank):
        self.n, self.F = n, 1 << fir_rank
        F = self.F
        self.inb = np.zeros((n, F))
        self.outb = np.zeros((n, 2 * F))
        self.conv = np.zeros((n, F))
        self.new = np.zeros((n, F))
        self.xfade = np.zeros(n, dtype=bool)
        self.nbuf = 0

    def set_kernel(self, rows, irs, smooth=False):     # Equalizer.cpp:336-345, on the rows `rows`
        rows = np.asarray(rows, dtype=np.int64)
        irs = np.asarray(irs, dtype=np.float64).reshape(rows.size, self.F)
        if smooth:
            self.new[rows] = irs
            self.xfade[rows] = True
        else:
            self.conv[rows] = irs

    def clear(self):                                    # Equalizer.cpp:273-278
        self.inb[:] = 0.0
        self.outb[:] = 0.0
        self.nbuf = 0

    def _convolve(self, X, kern):
        """Linear convolution of the blocks (spectra X, length 2F) with `kern`: [rows, 2F - 1] + a 0."""
        F = self.F
        y = np.fft.irfft(X * np.fft.rfft(kern, 2 * F, axis=1), 2 * F, axis=1)
        y[:, 2 * F - 1] = 0.0
        return y

    def _block(self):
        F, half = self.F, self.F // 2
        X = np.fft.rfft(self.inb, 2 * F, axis=1)
        self.outb[:, :F] = self.outb[:, F:]
        self.outb[:, F:] = 0.0
        self.outb += self._convolve(X, self.conv)
        rows = np.flatnonzero(self.xfade)
        if rows.size:                                   # :486-501
            self.conv[rows] = self.new[rows]
            fft = self._convolve(X[rows], self.conv[rows])
            ramp = np.arange(F) / F
            ob = self.outb[rows]
            ob[:, half:half + F] = ob[:, half:half + F] * (1.0 - ramp) + fft[:, half:half + F] * ramp
            ob[:, F + half:] = fft[:, F + half:]
            self.outb[rows] = ob
            self.xfade[rows] = False
        self.nbuf = 0

    def process(self, x):
        """x: [n, count] -> [n, count] float64."""
        F = self.F
        x = np.asarray(x, dtype=np.float64)
        y = np.empty_like(x)
        pos = 0
        while pos < x.shape[1]:
            if self.nbuf >= F:
                self._block()
            m = min(x.shape[1] - pos, F - self.nbuf)
            self.inb[:, self.nbuf:self.nbuf + m] = x[:, pos:pos + m]
            y[:, pos:pos + m] = self.outb[:, self.nbuf:self.nbuf + m]
            self.nbuf += m
            pos += m
        return y


class BatchSpectralProcessor:
    """ModelSpectralProcessor (SpectralProcessor.cpp:114-199) for `len(phases)` instances.

    kind[i]: 0 no operation, 1 table (tables[i]: N complex bins; a real gain curve is a table with
    a zero imaginary part), 2 function: fn(X, rows) gets the full N-bin spectra X [k, N] of the
    frames of instances `rows` and returns the new spectra."""

    def __init__(self, rank, phases, kind, tables=None, fn=None):
        self.N = 1 << rank
        self.F = self.N // 2
        n = len(phases)
        self.w = np.sin(np.pi * np.arange(self.N) / self.N)
        self.inb = np.zeros((n, self.N))
        self.outb = np.zeros((n, self.N))
        ph = np.asarray(phases, dtype=np.float32)
        self.off = (np.float32(self.N) * (ph * np.float32(0.5))).astype(np.int64)     # :123, fp32
        self.kind = np.asarray(kind, dtype=np.int64)
        self.Hf = None
        if np.any(self.kind == 1):
            self.Hf = np.zeros((n, self.F + 1), dtype=np.complex128)
            t = np.flatnonzero(self.kind == 1)
            self.Hf[t] = fold(np.asarray(tables)[t])
        self.fn = fn

    def _frame(self, r):
        fr = self.inb[r] * self.w
        for k, apply in ((1, self._table), (2, self._function)):
            s = self.kind[r] == k
            if np.any(s):
                fr[s] = apply(fr[s], r[s])
        ob = np.zeros((r.size, self.N))
        ob[:, :self.F] = self.outb[r, self.F:]
        self.outb[r] = ob + fr * self.w
        self.inb[r, :self.F] = self.inb[r, self.F:]

    def _table(self, fr, rows):
        return np.fft.irfft(np.fft.rfft(fr, axis=1) * self.Hf[rows], self.N, axis=1)

    def _function(self, fr, rows):
        return np.real(np.fft.ifft(self.fn(np.fft.fft(fr, axis=1), rows), axis=1))

    def process(self, x):
        """x: [n, count] -> [n, count] float64."""
        x = np.asarray(x, dtype=np.float64)
        out = np.empty_like(x)
        count = x.shape[1]
        start = self.off.copy()
        for o0 in np.unique(start):
            r = np.flatnonzero(start == o0)
            o, pos = int(o0), 0
            while pos < count:
                if o >= self.F:
                    self._frame(r)
                    o = 0
                m = min(self.F - o, count - pos)
                self.inb[r, self.F + o:self.F + o + m] = x[r, pos:pos + m]
                out[r, pos:pos + m] = self.outb[r, o:o + m]
                o += m
                pos += m
            self.off[r] = o
        return out

    def remaining(self):
        """[n] samples until the next transform (:241-245)."""
        return self.F - self.off


class BatchSpectralSplitter:
    """ModelSpectralSplitter (SpectralSplitter.cpp:227-383) for `len(phases)` instances.

    kinds[i][h]: 0 unbound, 1 table (tables[i, h]: N complex bins, real gains with a zero imaginary
    part), 2 sink only.  An instance with nothing bound produces nothing and keeps its state."""

    def __init__(self, rank, kinds, tables, phases, chunk_rank=0):
        self.N = 1 << rank
        cr = min(max(chunk_rank, 5), rank) if chunk_rank > 0 else rank
        self.F = 1 << (cr - 1)
        F = self.F
        self.kinds = np.asarray(kinds, dtype=np.int64)
        n, self.H = self.kinds.shape
        self.w = np.sin(np.pi * np.arange(2 * F) / (2 * F)) ** 2
        ph = np.asarray(phases, dtype=np.float32)
        self.fill = (np.float32(F) * (ph * np.float32(0.5))).astype(np.int64)           # :241, fp32
        self.hist = np.zeros((n, self.N))               # the last N input samples, newest last
        self.cur = np.zeros((n, self.H, F))             # what the sink sees during the current hop
        self.tail = np.zeros((n, self.H, F))            # W_{j-1}[F:]
        self.Hf = np.zeros((n, self.H, self.N // 2 + 1), dtype=np.complex128)
        t = self.kinds == 1
        if np.any(t):
            self.Hf[t] = fold(np.asarray(tables)[t])
        self.live = np.any(self.kinds != 0, axis=1)

    def latency(self):
        return 2 * self.F

    def _frame(self, r):
        F, N = self.F, self.N
        win = self.hist[r]
        kr = self.kinds[r]
        fx = np.any(kr == 1, axis=1)
        X = np.zeros((r.size, N // 2 + 1), dtype=np.complex128)
        if np.any(fx):
            X[fx] = np.fft.rfft(win[fx], axis=1)
        for h in range(self.H):
            frame = np.zeros((r.size, 2 * F))
            t = kr[:, h] == 1
            if np.any(t):
                frame[t] = np.fft.irfft(X[t] * self.Hf[r[t], h], N, axis=1)[:, N - 2 * F:]
            s = kr[:, h] == 2
            frame[s] = win[s, :2 * F]
            W = frame * self.w
            b = kr[:, h] != 0
            self.cur[r[b], h] = W[b, :F] + self.tail[r[b], h]
            self.tail[r[b], h] = W[b, F:]

    def process(self, x):
        """x: [n, count] -> [H, n, count] float64 (zero where nothing is bound)."""
        x = np.asarray(x, dtype=np.float64)
        n, count = x.shape
        out = np.zeros((self.H, n, count))
        F = self.F
        start = self.fill.copy()
        for f0 in np.unique(start[self.live]):
            r = np.flatnonzero(self.live & (start == f0))
            bound = (self.kinds[r] != 0).T[:, :, None]  # [H, k, 1]
            f, pos = int(f0), 0
            while pos < count:
                if f >= F:
                    self._frame(r)
                    f = 0
                m = min(F - f, count - pos)
                self.hist[r] = np.concatenate([self.hist[r, m:], x[r, pos:pos + m]], axis=1)
                out[:, r, pos:pos + m] = np.where(bound, self.cur[r, :, f:f + m].transpose(1, 0, 2), 0.0)
                f += m
                pos += m
            self.fill[r] = f
        return out
