"""Float64 model of lsp::dspu::SpectralProcessor::process(dst, src, count) (reference
src/main/util/SpectralProcessor.cpp:114-199), independent of any FFT restatement (numpy.fft):
sine ("cosine" in the reference's naming, misc/windows.cpp:238-246) window w[i] = sin(pi i / N)
before and after the spectral hook, frames of N = 2^rank samples every N/2, latency N,
first transform after N/2 - floor(N * (phase / 2)) samples."""
import numpy as np


class ModelSpectralProcessor:
    def __init__(self, rank, phase=0.0, hook=None):
        self.N = 1 << rank
        self.F = self.N // 2
        self.w = np.sin(np.pi * np.arange(self.N) / self.N)
        self.inb = np.zeros(self.N)
        self.outb = np.zeros(self.N)
        # nOffset = buf_size * (fPhase * 0.5f), in fp32 like the reference (:123)
        self.off = int(np.float32(self.N) * (np.float32(phase) * np.float32(0.5)))
        self.hook = hook            # None, or a function of the complex spectrum (N bins) -> spectrum

    def process(self, src):
        src = np.asarray(src, np.float64)
        out = np.empty_like(src)
        pos = 0
        while pos < src.size:
            if self.off >= self.F:
                frame = self.inb * self.w
                if self.hook is not None:
                    frame = np.real(np.fft.ifft(self.hook(np.fft.fft(frame))))
                self.outb[:self.F] = self.outb[self.F:]
                self.outb[self.F:] = 0.0
                self.outb += frame * self.w
                self.inb[:self.F] = self.inb[self.F:]
                self.off = 0
            n = min(self.F - self.off, src.size - pos)
            self.inb[self.F + self.off:self.F + self.off + n] = src[pos:pos + n]
            out[pos:pos + n] = self.outb[self.off:self.off + n]
            self.off += n
            pos += n
        return out

    def remaining(self):
        """Samples until the next transform (SpectralProcessor::remaining, :241-245)."""
        return self.F - self.off

    def reset(self):
        """SpectralProcessor::reset (:247-257): buffers cleared, offset kept."""
        self.inb[:] = 0.0
        self.outb[:] = 0.0
