"""Float64 model of lsp::dspu::SpectralSplitter::process(src, count) (reference
src/main/util/SpectralSplitter.cpp:227-383), independent of any FFT restatement (numpy.fft) and of
the reference's sliding buffers: written from what the code computes, as a function of the input
STREAM.

    N = 2^rank transform size, F = 2^(chunk_rank - 1) hop (chunk_rank = rank unless set: :233),
    a transform before input sample s_j = (F - f0) + j F, f0 = floor(F * (phase / 2)) in fp32 (:241),
    over the N samples x[s_j - N, s_j) (zeros before the start), no window before the transform;
    handler with a function:    y = Re(IFFT(func(FFT(window)))), the LAST 2 F samples of it (:324);
    handler without a function: the FIRST 2 F samples of the window (:327);
    times w[i] = sin(pi i / (2 F))^2 (misc/windows.cpp:249-260), overlap-added with hop F, and
    the sink sees the sum one hop later: out[s_j + i] = W_j[i] + W_{j-1}[F + i], i < F (:331-340,365-371).
Latency 2 F = 2^chunk_rank (:289)."""
import numpy as np


class ModelSpectralSplitter:
    def __init__(self, rank, handlers, chunk_rank=0, phase=0.0):
        self.rank = rank
        self.N = 1 << rank
        cr = min(max(chunk_rank, 5), rank) if chunk_rank > 0 else rank
        self.F = 1 << (cr - 1)
        self.w = np.sin(np.pi * np.arange(2 * self.F) / (2 * self.F)) ** 2
        self.f0 = int(np.float32(self.F) * (np.float32(phase) * np.float32(0.5)))
        self.hooks = [None] * handlers      # None = unbound; "copy" = sink only; else function of the N-bin spectrum
        self.x = np.zeros(0)
        self.tail = [np.zeros(self.F) for _ in range(handlers)]     # W_{j-1}[F:]
        self.cur = [np.zeros(self.F) for _ in range(handlers)]      # what the sink sees during the current hop
        self.fill = self.f0                 # nFrameSize

    def latency(self):
        return 2 * self.F

    def bind(self, handler, hook):
        self.hooks[handler] = hook
        self.tail[handler] = np.zeros(self.F)
        self.cur[handler] = np.zeros(self.F)

    def process(self, src):
        src = np.asarray(src, np.float64)
        out = np.zeros((len(self.hooks), src.size))
        if all(h is None for h in self.hooks):
            return out
        pos = 0
        while pos < src.size:
            if self.fill >= self.F:
                win = np.zeros(self.N)
                have = min(self.N, self.x.size)
                if have:
                    win[self.N - have:] = self.x[self.x.size - have:]
                X = None
                for h, hook in enumerate(self.hooks):
                    if hook is None:
                        continue
                    if isinstance(hook, str):
                        frame = win[:2 * self.F]
                    else:
                        if X is None:
                            X = np.fft.fft(win)
                        frame = np.real(np.fft.ifft(hook(X)))[self.N - 2 * self.F:]
                    W = frame * self.w
                    self.cur[h] = W[:self.F] + self.tail[h]
                    self.tail[h] = W[self.F:].copy()
                self.fill = 0
            n = min(self.F - self.fill, src.size - pos)
            self.x = np.concatenate([self.x, src[pos:pos + n]])[-(self.N + self.F):]
            for h, hook in enumerate(self.hooks):
                if hook is not None:
                    out[h, pos:pos + n] = self.cur[h][self.fill:self.fill + n]
            self.fill += n
            pos += n
        return out
