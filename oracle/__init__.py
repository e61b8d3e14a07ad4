"""CPU oracle for the Friture spectral hot path -- TEST INFRASTRUCTURE ONLY.

Nothing under ``oracle/`` is part of the product.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it, and only as the checker / the timed CPU baseline -- never on the
product path (``friture_b200`` fails loudly when its CUDA library is missing and has
no CPU fallback).

Parity status: PINNED.  The restatement in :mod:`oracle.friture_oracle` is validated
against golden vectors that ``oracle/make_golden.py`` generates from the unmodified
reference (imported in place by ``oracle/ref_import.py``) and that are committed under
``tests/golden/``; ``tests/test_oracle_vs_reference.py`` and ``tests/test_oracle_golden.py``
check them without the reference tree.
"""
