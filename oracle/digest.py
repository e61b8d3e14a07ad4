"""Digests of float arrays for the golden checks that demand bit identity (TEST INFRASTRUCTURE ONLY).

The digests in tests/golden/reference_checks.npz were taken from the reference's outputs on the
machine that ran oracle/make_golden.py; the tests compare them with the oracle run wherever the
tests run.  Some of those values pass through transcendental ufuncs (the Hann window's cos, the
weighting tables' log10, ...), whose last bit numpy may compute differently on another CPU (its
SIMD dispatch, e.g. SVML on AVX-512).  A digest mismatch of such a value on a new host therefore
first calls for rerunning oracle/make_golden.py there against the reference, before it is read as
a change of the oracle.
"""
import hashlib

import numpy as np


def digest(*arrays):
    """SHA-256 over the shapes and float64 bytes of `arrays` (a list of arrays counts as its
    elements in order).  For NaN-free arrays two digests agree exactly when np.array_equal holds
    element by element, so bit-identity checks need not store the arrays themselves."""
    h = hashlib.sha256()
    for a in arrays:
        for v in (a if isinstance(a, (list, tuple)) else [a]):
            v = np.ascontiguousarray(v, dtype="<f8") + 0.0          # -0.0 == 0.0, as in array_equal
            h.update(repr(v.shape).encode())
            h.update(v.tobytes())
    return h.hexdigest()
