"""Scope-table row f4: outputs of the reference's own SpectralProcessor / SpectralSplitter frozen in
tests/golden/spectral_golden.npz (tests/golden/make_golden_spectral.py; the cases are listed in
tests/spectral_cases.py).  The verbatim build must reproduce them bit for bit (it does not depend on
the machine: scalar restated kernels, no FMA contraction in the schedulers), and the independent
float64 models must agree with them.  CPU only."""
import numpy as np
import pytest

import spectral_cases as cases
import spectral_model
import splitter_model
import synth
from oracle.bindings import CpuSpectralProcessor, CpuSpectralSplitter


@pytest.fixture(scope="module")
def golden():
    return np.load(cases.GOLDEN)


def _hook(kind, gain, H):
    if kind == 1:
        return lambda X: X * H.astype(np.complex128)
    if kind == 2:
        return lambda X: X * gain.astype(np.float64)
    return None


def test_spectral_processor_cases(golden):
    for name, *_ in cases.SP_CASES:
        rank, phase, step, kind, latency, seed, n = golden[name + ".meta"]
        rank, step, kind, seed, n = int(rank), int(step), int(kind), int(seed), int(n)
        src = synth.noise(seed, n)
        gain, H = cases.tables(rank, seed)
        want = golden[name + ".dst"]
        model = spectral_model.ModelSpectralProcessor(rank, float(phase), _hook(kind, gain, H)).process(src)
        assert np.max(np.abs(model - want)) <= 2e-5 * max(1.0, np.max(np.abs(want))), name
        if CpuSpectralProcessor.available():
            sp = CpuSpectralProcessor(14)
            sp.set_rank(rank)
            sp.set_phase(float(phase))
            if kind == 1:
                sp.bind_complex(H)
            elif kind == 2:
                sp.bind_gain(gain)
            assert np.array_equal(sp.run(src, step), want), name
            assert sp.latency() == int(latency)


def test_spectral_splitter_cases(golden):
    for name, *_ in cases.SS_CASES:
        rank, chunk, phase, step, latency, seed, n = golden[name + ".meta"]
        rank, chunk, step, seed, n = int(rank), int(chunk), int(step), int(seed), int(n)
        kinds = [int(k) for k in golden[name + ".kinds"]]
        src = synth.noise(seed, n)
        want = golden[name + ".dst"]
        bound = [h for h, kind in enumerate(kinds) if kind != 0]
        m = splitter_model.ModelSpectralSplitter(rank, len(kinds), chunk, float(phase))
        ref = CpuSpectralSplitter(13, len(kinds)) if CpuSpectralSplitter.available() else None
        if ref is not None:
            ref.set_rank(rank)
            if chunk:
                ref.set_chunk_rank(chunk)
            ref.set_phase(float(phase))
        for h, kind in enumerate(kinds):
            gain, H = cases.tables(rank, 10 * seed + h)
            if kind == 3:
                m.bind(h, "copy")
            elif kind != 0:
                m.bind(h, _hook(kind, gain, H))
            if ref is not None:
                if kind == 1:
                    ref.bind_complex(h, H)
                elif kind == 2:
                    ref.bind_gain(h, gain)
                elif kind == 3:
                    ref.bind_sink(h)
        model = m.process(src)[bound]
        assert np.max(np.abs(model - want)) <= 2e-5 * max(1.0, np.max(np.abs(want))), name
        if ref is not None:
            assert np.array_equal(ref.run(src, step)[bound], want), name
            assert ref.latency() == int(latency)
