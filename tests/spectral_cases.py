"""The SpectralProcessor / SpectralSplitter cases frozen in tests/golden/spectral_golden.npz, and the
seeded spectral tables every spectral test binds.  Shared by tests/golden/make_golden_spectral.py,
which wrote the fixtures, and the tests that read them."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "spectral_golden.npz")


def tables(rank, seed):
    """A real gain curve and a complex table of 2**rank bins, neither of them symmetric on purpose."""
    N = 1 << rank
    rng = np.random.Generator(np.random.PCG64(seed))
    gain = rng.uniform(0.2, 1.5, N).astype(np.float32)
    H = (rng.uniform(-1, 1, N) + 1j * rng.uniform(-1, 1, N)).astype(np.complex64)
    return gain, H


#            name        rank  phase  step  samples  kind (0 none, 1 complex, 2 gain)
SP_CASES = [("sp_r8_gain",    8,  0.0,  31,   3000,  2),
            ("sp_r9_cplx",    9,  0.37, 256,  4000,  1),
            ("sp_r10_none",   10, 0.5,  1000, 6000,  0),
            ("sp_r12_gain",   12, 1.0,  4096, 12000, 2)]
#            name        rank  chunk phase  step  samples  kinds per handler (0 unbound, 1 complex, 2 gain, 3 sink only)
SS_CASES = [("ss_r8",         8,  0,   0.0,  31,   3000,  (2, 1, 0, 3)),
            ("ss_r10_c8",     10, 8,   0.37, 1000, 6000,  (1, 2, 3, 0)),
            ("ss_r12_c10",    12, 10,  1.0,  4096, 9000,  (2, 2, 2, 0)),
            ("ss_r9_c3",      9,  3,   0.5,  77,   4000,  (3, 0, 1, 0))]
