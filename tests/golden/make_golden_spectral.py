"""Generates tests/golden/spectral_golden.npz from the reference's own SpectralProcessor.cpp and
SpectralSplitter.cpp (scope-table row f4).

Run in the build container (needs /root/reference to build oracle/_ref):

    python tests/golden/make_golden_spectral.py

Each case stores the settings, the tables bound, the input, the call pattern and the output produced
by oracle/_ref/libref_convolver.so (the reference classes compiled verbatim over the restated
lsp::dsp:: kernels, host callbacks in oracle/ref_wrap_spectral.cpp / ref_wrap_splitter.cpp).  The
reference ships no golden vectors for these classes (its only test of them is
utest/util/spectral_proc.cpp, reproduced in tests/test_oracle_spectral.py); the fixtures freeze their
behaviour as observed here so that it stays checkable where /root/reference does not exist.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))

from oracle import bindings  # noqa: E402
import synth  # noqa: E402
from spectral_cases import GOLDEN, SP_CASES, SS_CASES, tables  # noqa: E402


def main():
    bindings.build()
    out = {}
    for k, (name, rank, phase, step, n, kind) in enumerate(SP_CASES):
        src = synth.noise(300 + k, n)
        gain, H = tables(rank, 300 + k)
        sp = bindings.CpuSpectralProcessor(14)
        sp.set_rank(rank)
        sp.set_phase(phase)
        if kind == 1:
            sp.bind_complex(H)
        elif kind == 2:
            sp.bind_gain(gain)
        # input and tables are regenerated from their seeds by the tests (synth.noise, tables())
        out[name + ".dst"] = sp.run(src, step)
        out[name + ".meta"] = np.array([rank, phase, step, kind, sp.latency(), 300 + k, n], dtype=np.float64)
    for k, (name, rank, chunk, phase, step, n, kinds) in enumerate(SS_CASES):
        src = synth.noise(400 + k, n)
        ss = bindings.CpuSpectralSplitter(13, len(kinds))
        ss.set_rank(rank)
        if chunk:
            ss.set_chunk_rank(chunk)
        ss.set_phase(phase)
        for h, kind in enumerate(kinds):
            gain, H = tables(rank, 10 * (400 + k) + h)
            if kind == 1:
                ss.bind_complex(h, H)
            elif kind == 2:
                ss.bind_gain(h, gain)
            elif kind == 3:
                ss.bind_sink(h)
        dst = ss.run(src, step)
        out[name + ".dst"] = dst[[h for h, kind in enumerate(kinds) if kind != 0]]     # rows of unbound handlers are zero
        out[name + ".kinds"] = np.array(kinds, dtype=np.int64)
        out[name + ".meta"] = np.array([rank, chunk, phase, step, ss.latency(), 400 + k, n], dtype=np.float64)
    np.savez_compressed(GOLDEN, **out)
    print("wrote", len(SP_CASES) + len(SS_CASES), "cases")


if __name__ == "__main__":
    main()
