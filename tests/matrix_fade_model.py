"""Float64 model of b200conv_mx_set_irs: the matrix convolver of tests/matrix_model.py whose routes can
take new impulse responses while it runs, keeping the input history.  With k counting samples from the
first sample of the first call after set_irs and w(k) = min(1, (k + 1) / fade) (w = 1 when fade == 0),
a changed route contributes

    (1 - w) * (h_old (*) x) + w * (h_new (*) x)

with both convolutions over the whole history since set_routes / clear.  Once w reaches 1 the new IR
replaces the old one for good.  Each call computes only its own samples, from the input window the
longest IR reaches, so long runs stay cheap."""
import numpy as np
from scipy.signal import fftconvolve

from matrix_model import MatrixModel


class FadeInProgress(RuntimeError):
    pass


class MatrixFadeModel(MatrixModel):
    def set_routes(self, routes):
        self.fade = None                    # (start sample, fade length, {route: old ir})
        super().set_routes(routes)

    def clear(self):
        self._end_fade()
        super().clear()

    def _end_fade(self):
        self.fade = None

    def fade_remaining(self):
        if self.fade is None:
            return 0
        start, length, _ = self.fade
        return max(0, start + length - self.x.shape[1])

    def set_irs(self, changes, fade=0):
        """changes: [(route, ir), ...] -- the model checks what the engine returns B200CONV_ERR_* for."""
        changes = [(int(r), np.asarray(h, dtype=np.float64)) for r, h in changes]
        if not changes:
            return
        if self.fade_remaining() > 0:
            raise FadeInProgress()
        old = {}
        for r, h in changes:
            i, o, h_old = self.routes[r]
            old[r] = h_old
            self.routes[r] = (i, o, h)
        self.fade = (self.x.shape[1], int(fade), old) if fade > 0 else None

    def _conv(self, x, h, n0, n):
        """(h (*) x)[n0 : n0 + n] from the window of x that h reaches"""
        a = max(0, n0 - h.size + 1)
        return fftconvolve(x[a:n0 + n], h)[n0 - a:n0 - a + n]

    def process(self, src):
        src = np.asarray(src, dtype=np.float64)
        n0, n = self.x.shape[1], src.shape[1]
        self.x = np.concatenate([self.x, src], axis=1)
        y = np.zeros((self.outputs, n))
        w = None
        if self.fade is not None:
            start, length, old = self.fade
            k = np.arange(n0, n0 + n) - start
            w = np.minimum(1.0, (k + 1) / length)
        for r, (i, o, h) in enumerate(self.routes):
            new = self._conv(self.x[i], h, n0, n)
            if w is not None and r in self.fade[2]:
                y[o] += (1.0 - w) * self._conv(self.x[i], self.fade[2][r], n0, n) + w * new
            else:
                y[o] += new
        if self.fade is not None and self.fade_remaining() == 0:
            self._end_fade()
        return y
