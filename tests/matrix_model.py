"""Float64 model of the matrix convolver (b200conv_mx_*): output o is the sum, over the routes
(i, o, h), of input i convolved with h.  State across calls is kept the simple way: the model holds
every input sample since the last set_routes / clear and recomputes the outputs of each call."""
import numpy as np
from scipy.signal import fftconvolve


class MatrixModel:
    def __init__(self, inputs, outputs):
        self.inputs = inputs
        self.outputs = outputs
        self.routes = []
        self.clear()

    def set_routes(self, routes):
        self.routes = [(int(i), int(o), np.asarray(h, dtype=np.float64)) for i, o, h in routes]
        self.clear()

    def clear(self):
        self.x = np.zeros((self.inputs, 0))

    def process(self, src):
        src = np.asarray(src, dtype=np.float64)
        n0, n = self.x.shape[1], src.shape[1]
        self.x = np.concatenate([self.x, src], axis=1)
        y = np.zeros((self.outputs, n0 + n))
        for i, o, h in self.routes:
            y[o] += fftconvolve(self.x[i], h)[:n0 + n]
        return y[:, n0:]
