"""CPU: the oracle restatement against the UNMODIFIED reference, through what oracle/make_golden.py
recorded of the reference's outputs (tests/golden/reference_checks.npz): digests where the oracle
must be bit-identical to the reference (see oracle/digest.py), values where it may differ by
rounding.  The seeded inputs are regenerated here; their digests are stored with the outputs."""
import os

import numpy as np
import pytest

from oracle import friture_oracle as fo
from oracle.digest import digest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref():
    with np.load(os.path.join(GOLD, "reference_checks.npz")) as d:
        return {k: d[k] for k in d.files}


def same(g, key, *arrays):
    return digest(*arrays) == str(g[key])


def seeded(g, key, *arrays):
    """The regenerated inputs are the ones the reference was run on."""
    assert same(g, key, *arrays), "%s: numpy's seeded stream changed; rerun oracle/make_golden.py" % key


def coeffs(bpo):
    with np.load(os.path.join(GOLD, "coefficients.npz")) as c:
        return c["bdec"], c["adec"], list(c["b%d" % bpo]), list(c["a%d" % bpo])


def test_analyzelive_all_sizes(ref):
    for k in range(10):
        n = 32 * 2 ** k                                   # spectrum_settings.py:61-70
        rng = np.random.default_rng(n)
        x = rng.standard_normal(n)
        seeded(ref, "analyzelive_x_%d" % n, x)
        assert same(ref, "analyzelive_%d" % n, fo.analyzelive(x)), n
        assert same(ref, "window_%d" % n, fo.hann_window(n)), n


def test_lfilter_bit_identical(ref):
    from oracle import iir_c
    bdec, adec, boct, aoct = coeffs(3)
    rng = np.random.default_rng(0)
    x = rng.standard_normal(700)
    seeded(ref, "lfilter_x", x)
    for name, b, a in [("dec", bdec, adec), ("band", boct[1], aoct[1])]:
        zi = rng.standard_normal(len(b) - 1) * 0.01
        seeded(ref, "lfilter_%s_zi" % name, zi)
        for fn in (fo.lfilter_df2t, fo.lfilter_df2t_loop, iir_c.lfilter):
            y, z = fn(b, a, x, zi.copy())
            assert same(ref, "lfilter_%s" % name, y, z), fn


def test_bank_and_smoothing(ref):
    for bpo in (1, 3, 24):
        bdec, adec, boct, aoct = coeffs(bpo)
        rng = np.random.default_rng(bpo)
        zo = fo.bank_filtic(bdec, adec, boct, aoct)
        for step in range(3):
            x = rng.standard_normal(512)
            seeded(ref, "bank_bpo%d_x%d" % (bpo, step), x)
            yo, do, zo = fo.octave_filter_bank_decimation(bdec, adec, boct, aoct, x, zo)
            assert np.array_equal(do, ref["bank_bpo%d_dec%d" % (bpo, step)])
            assert same(ref, "bank_bpo%d_y%d" % (bpo, step), yo), (bpo, step)
            assert same(ref, "bank_bpo%d_z%d" % (bpo, step), zo), (bpo, step)
    k = fo.smoothing_kernel(0.01, 64)
    d = np.random.default_rng(1).random(40)
    seeded(ref, "smoothing_data", d)
    assert ref["smoothing_value"] == fo.exp_smoothed_value(k, 0.01, d, 0.3)


def test_octave_filters_attributes_and_gcc(ref):
    fi, fl, fh = fo.octave_frequencies(27, 3)
    assert same(ref, "of3_fi", fi) and same(ref, "of3_flow", fl) and same(ref, "of3_fhigh", fh)
    assert fo.get_decs(3) == list(ref["of3_decs"])
    A, B, C = fo.weighting_tables(fi, eps=0.0)
    assert same(ref, "of3_A", A) and same(ref, "of3_B", B) and same(ref, "of3_C", C)
    rng = np.random.default_rng(3)
    d0, d1 = rng.standard_normal(24000), rng.standard_normal(24000)
    seeded(ref, "gcc_x", d0, d1)
    assert same(ref, "gcc", fo.generalized_cross_correlation(d0, d1))


def test_filter_data_matches_reference():
    """friture_b200/data/filters.npz carries exactly the reference's coefficients
    (tests/golden/coefficients.npz holds them as the reference's generated_filters.PARAMS)."""
    from friture_b200 import filter_data
    bdec_r, adec_r, _, _ = coeffs(3)
    bdec, adec, sos = filter_data.decimator()
    assert np.array_equal(bdec, bdec_r) and np.array_equal(adec, adec_r)
    for bpo in (1, 3, 6, 12, 24):
        _, _, b_r, a_r = coeffs(bpo)
        b, a, s = filter_data.bands(bpo)
        assert np.array_equal(b, np.array(b_r)) and np.array_equal(a, np.array(a_r))


def test_shim_labels_and_attributes_match_reference(ref):
    """Octave_Filters host-side attributes (no GPU needed)."""
    from friture_b200.octavefilters import Octave_Filters
    for bpo in (1, 3, 6, 12, 24):
        m = Octave_Filters(bpo)
        assert m.f_nominal == list(ref["of%d_f_nominal" % bpo])
        for name in ("fi", "flow", "fhigh", "A", "B", "C", "bdec", "adec", "boct", "aoct"):
            assert same(ref, "of%d_%s" % (bpo, name), getattr(m, name)), (bpo, name)
        assert m.get_decs() == list(ref["of%d_decs" % bpo]) and m.nbands == int(ref["of%d_nbands" % bpo])
    from friture_b200 import audioproc
    pm = audioproc()
    for n in (1024, 2048):
        pm.set_fftsize(n)
        for name in ("window", "freq", "A", "B", "C", "size_sq", "fft_size"):
            assert same(ref, "audioproc%d_%s" % (n, name), getattr(pm, name)), (n, name)


def test_live_fft_bank_restatement_and_fir_data(ref):
    """oracle.octave_filter_bank_decimation_fft == the unmodified reference's Octave_Filters.filter
    (live FFT overlap-add path, friture/filter.py:136-247) to 1e-15; the direct FIR form the GPU
    kernel computes equals it to rounding; data/fir.npz holds the reference's taps.  The reference's
    band outputs are stored whole at 1 and 3 bands per octave, as 16 fixed positions of every band
    at 24, with every band's L2 norm and peak; the per-element bounds imply the norm bounds
    (triangle inequality) and bound the direct form against the restatement everywhere."""
    from friture_b200 import filter_data
    assert fo.fft_bank_sizes() == [1536, 1024, 768, 640, 576, 576, 540, 540, 540]
    rng = np.random.default_rng(1)
    for bpo in (1, 3, 24):
        boct_fir, bdec_fir = filter_data.fir_taps(bpo)
        assert same(ref, "fft%d_taps" % bpo, boct_fir, bdec_fir)
        oo, od = fo.fft_bank_state(bpo)
        hist = [np.zeros(511) for _ in range(9)]
        for blk in range(5):
            x = rng.standard_normal(512 if blk % 2 else 1024) * 0.1
            seeded(ref, "fft%d_x%d" % (bpo, blk), x)
            y, dec, oo, od = fo.octave_filter_bank_decimation_fft(boct_fir, bdec_fir, x, oo, od)
            y2, hist = fo.fir_bank_direct(boct_fir, bdec_fir, x, hist)
            assert np.array_equal(dec, ref["fft%d_dec%d" % (bpo, blk)])
            val = ref["fft%d_val%d" % (bpo, blk)]
            sel = ref.get("fft%d_idx%d" % (bpo, blk), slice(None))
            lens, norm, peak = (ref["fft%d_%s%d" % (bpo, k, blk)] for k in ("len", "norm", "peak"))
            assert [len(v) for v in y] == list(lens) == [len(v) for v in y2]
            tol2 = np.repeat(1e-12 * np.maximum(peak, 1.0), lens)
            yc, y2c = np.concatenate(y), np.concatenate(y2)
            assert np.max(np.abs(yc[sel] - val)) < 1e-14
            assert np.all(np.abs(y2c[sel] - val) < tol2[sel])
            assert np.all(np.abs(y2c - yc) < tol2 + 1e-14)
            assert np.all(np.abs([np.linalg.norm(v) for v in y] - norm) <= 1e-14 * np.sqrt(lens))
