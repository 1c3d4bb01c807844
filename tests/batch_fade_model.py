"""Float64 model of one convolver-batch instance with b200conv_set_irs: its impulse response can be
replaced while it runs, keeping the input history.  With k counting samples from the first sample of
the first call after set_irs and w(k) = min(1, (k + 1) / fade) (w = 1 when fade == 0), the instance
outputs

    (1 - w) * (h_old (*) x) + w * (h_new (*) x)

with both convolutions over the whole history since init.  Once w reaches 1 the new IR replaces the
old one for good, and with it the instance's reported size (conv_size, bins, partitions), which is
also what the next set_irs is checked against.  Each call computes only its own samples, from the
input window the IRs reach, so long runs stay cheap.  The model raises for the cases the engine
returns B200CONV_ERR_ARG / B200CONV_ERR_STATE for, and then changes nothing."""
import numpy as np
from scipy.signal import fftconvolve


class ArgError(ValueError):
    pass


class StateError(RuntimeError):
    pass


class BatchFadeModel:
    def __init__(self, F):
        self.F = F
        self.destroy()

    def destroy(self):
        self.h = None
        self.x = np.zeros(0)
        self.fade = None                    # (start sample, fade length, old ir)

    def init(self, ir):
        self.destroy()
        self.h = np.asarray(ir, dtype=np.float64)

    def state(self):
        if self.h is None:
            return {"conv_size": 0, "bins": 0, "partitions": 0}
        bins = -(-self.h.size // self.F)
        return {"conv_size": self.h.size, "bins": bins, "partitions": bins + 1}

    def fade_remaining(self):
        if self.fade is None:
            return 0
        start, length, _ = self.fade
        return max(0, start + length - self.x.size)

    def set_irs(self, ir, fade=0, lends=False):
        ir = np.asarray(ir, dtype=np.float64)
        if ir.size == 0:
            raise ArgError("empty impulse response")
        if self.h is None:
            raise StateError("not initialised")
        if self.fade is not None:
            raise StateError("already fading")
        if lends:
            raise StateError("lends its IR spectra")
        if -(-ir.size // self.F) + 1 > self.state()["partitions"]:
            raise ArgError("more partitions than the ring reaches")
        old, self.h = self.h, ir
        self.fade = (self.x.size, int(fade), old) if fade > 1 else None

    def _conv(self, h, n0, n):
        """(h (*) x)[n0 : n0 + n] from the window of x that h reaches"""
        a = max(0, n0 - h.size + 1)
        return fftconvolve(self.x[a:n0 + n], h)[n0 - a:n0 - a + n]

    def process(self, src):
        src = np.asarray(src, dtype=np.float64)
        n0, n = self.x.size, src.size
        self.x = np.concatenate([self.x, src])
        if self.h is None:
            return np.zeros(n)
        y = self._conv(self.h, n0, n)
        if self.fade is not None:
            start, length, old = self.fade
            w = np.minimum(1.0, (np.arange(n0, n0 + n) - start + 1) / length)
            y = (1.0 - w) * self._conv(old, n0, n) + w * y
            if self.fade_remaining() == 0:
                self.fade = None
        return y
