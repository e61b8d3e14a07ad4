"""CPU: the oracle restatement (oracle/friture_oracle.py, oracle/iir_df2t.c) against golden vectors
generated from the unmodified reference by oracle/make_golden.py.  Runs anywhere (no GPU, no
reference tree)."""
import os

import numpy as np
import pytest

from oracle import friture_oracle as fo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with np.load(os.path.join(GOLD, name)) as d:
        return {k: d[k] for k in d.files}


def test_analyzelive_and_window():
    g = load("analyzelive.npz")
    for n in (1024, 2048, 8192):
        x = g["x_%d" % n].astype(np.float64)
        assert np.array_equal(fo.hann_window(n), g["window_%d" % n])
        got = fo.analyzelive(x)
        assert np.allclose(got, g["power_%d" % n], rtol=1e-13, atol=0)
        f = np.linspace(0, 48000 // 2, n // 2 + 1)
        assert np.array_equal(f, g["freq_%d" % n])
        A, B, C = fo.weighting_tables(f)
        assert np.allclose(A, g["A_%d" % n], rtol=1e-14) and np.allclose(C, g["C_%d" % n], rtol=1e-14)
        assert np.allclose(B, g["B_%d" % n], rtol=1e-14)


def test_spectrogram_framing():
    """End-index framing of the ring buffer (ringbuffer.py:87-99) == frame f starts at f*hop."""
    g = load("spectrogram.npz")
    n_fft, hop = int(g["n_fft"]), int(g["hop"])
    p = fo.stft_power_batch(g["x"], n_fft, hop)
    assert p.shape == g["power"].shape
    assert np.allclose(p, g["power"], rtol=1e-12, atol=1e-300)
    logpower = 10. * np.log10(g["power"] + 1e-30)          # the reference's log_spectrogram
    assert np.allclose(fo.log_spectrogram(p), logpower, rtol=0, atol=1e-10)
    p1 = np.stack([fo.stft_power(g["x"][c], n_fft, hop) for c in range(g["x"].shape[0])])
    assert np.allclose(p1, g["power"], rtol=1e-13, atol=0)


def coeffs(bpo):
    c = load("coefficients.npz")
    return c["bdec"], c["adec"], list(c["b%d" % bpo]), list(c["a%d" % bpo])


@pytest.mark.parametrize("bpo,block", [(3, 256), (3, 512), (3, 1024), (12, 512)])
def test_iir_bank_energies(bpo, block):
    g = load("octave_bank.npz")
    bdec, adec, boct, aoct = coeffs(bpo)
    orc = fo.OctaveSpectrumOracle(bdec, adec, boct, aoct)
    x = g["x"].astype(np.float64)
    E = np.array([orc.push(x[b * block:(b + 1) * block])[0] for b in range(len(x) // block)])
    ref = g["energies_bpo%d_block%d" % (bpo, block)]
    assert np.allclose(E, ref, rtol=1e-12, atol=0)
    if block == 512:
        assert np.array_equal(np.array(orc.decs), g["dec_bpo%d" % bpo])
        assert np.allclose(np.concatenate(orc.zis), g["zis_bpo%d" % bpo], rtol=1e-12, atol=1e-300)


def test_iir_bank_outputs_and_block_invariance():
    g = load("octave_bank.npz")
    bdec, adec, boct, aoct = coeffs(3)
    x = g["x"].astype(np.float64)
    outs = {}
    for block in (512, 2048):
        zis = fo.bank_filtic(bdec, adec, boct, aoct)
        ys = [[] for _ in range(27)]
        for b in range(len(x) // block):
            y, dec, zis = fo.octave_filter_bank_decimation(bdec, adec, boct, aoct,
                                                           x[b * block:(b + 1) * block], zis)
            for k in range(27):
                ys[k].append(y[k])
        outs[block] = [np.concatenate(v) for v in ys]
    for k in (0, 13, 26):
        assert np.allclose(outs[512][k], g["y_bpo3_band%d" % k], rtol=1e-12, atol=1e-18)
        assert np.allclose(outs[512][k], outs[2048][k], rtol=1e-10, atol=1e-15)   # blocking-invariant
    # energies at common instants do not depend on the blocking (reference golden)
    e256, e512, e1024 = (g["energies_bpo3_block%d" % b] for b in (256, 512, 1024))
    assert np.allclose(e256[3::4], e1024, rtol=1e-10) and np.allclose(e512[1::2], e1024, rtol=1e-10)


def test_c_restatement_matches():
    from oracle import iir_c
    g = load("octave_bank.npz")
    bdec, adec, boct, aoct = coeffs(3)
    x = g["x"]
    orc = fo.OctaveSpectrumOracle(bdec, adec, boct, aoct)
    bank = iir_c.BankC(bdec, adec, boct, aoct, orc.alphas, n_channels=2)
    E = bank.process(np.stack([x, x]), 512)
    ref = g["energies_bpo3_block512"]
    assert np.allclose(E[0], ref, rtol=1e-11) and np.array_equal(E[0], E[1])
    y, z = iir_c.lfilter(bdec, adec, x[:300].astype(np.float64), np.zeros(12))
    y2, z2 = fo.lfilter_df2t_loop(bdec, adec, x[:300].astype(np.float64), np.zeros(12))
    assert np.array_equal(y, y2) and np.array_equal(z, z2)            # same rounding, no FMA
    y3, z3 = fo.lfilter_df2t(bdec, adec, x[:300].astype(np.float64), np.zeros(12))
    assert np.array_equal(y, y3) and np.array_equal(z, z3)


def test_live_fft_bank_distance():
    """The reference's live FFT-OLA path differs from its IIR path by ~5e-4 on band energies
    (its own tolerance is 5 %, test_octave_filters.py:58-59); report that distance."""
    g = load("octave_bank.npz")
    bdec, adec, boct, aoct = coeffs(3)
    zis = fo.bank_filtic(bdec, adec, boct, aoct)
    acc = np.zeros(27)
    x = g["x"].astype(np.float64)
    for b in range(16):
        y, _, zis = fo.octave_filter_bank_decimation(bdec, adec, boct, aoct, x[b * 512:(b + 1) * 512], zis)
        acc += np.array([np.sum(v ** 2) for v in y])
    d = np.max(np.abs(g["fft_bank_energy_sum_bpo3"] / acc - 1.0))
    assert 1e-6 < d < 5e-2


def test_gcc_phat_and_decimate():
    g = load("gcc_phat.npz")
    xc = fo.generalized_cross_correlation(g["d0"], g["d1"])
    assert np.allclose(xc, g["xcorr"], rtol=0, atol=1e-12)
    i, v, sm = fo.delay_peak(xc)
    assert i == int(g["argmax"]) == 137
    xcb = fo.generalized_cross_correlation(g["d0b"], g["d1b"])
    i2, v2, sm2 = fo.delay_peak(xcb, sm)
    assert i2 == int(g["argmax_b"]) and np.allclose(sm2, g["smoothed_b"], atol=1e-12)
    c = load("coefficients.npz")
    zis = [np.zeros(12), np.zeros(12)]
    o1, zis = fo.decimate_multiple(2, c["bdec"], c["adec"], g["dec_in"][:1024], zis)
    o2, zis = fo.decimate_multiple(2, c["bdec"], c["adec"], g["dec_in"][1024:], zis)
    assert np.allclose(np.concatenate([o1, o2]), g["dec_out"], rtol=1e-12, atol=1e-18)


def test_exp_smoothing_2d():
    g = load("exp_smoothing.npz")
    alpha = float(g["alpha"])
    kernel = fo.smoothing_kernel(alpha, 8192)
    out = fo.exp_smoothed_value_2d(kernel, alpha, g["data"], g["prev"])
    assert np.allclose(out, g["out"], rtol=1e-13)
    assert np.isclose(alpha, fo.smoothing_alpha(0.125, 48000 / 1024.))
    # recursive form == block form
    s = g["prev"].copy()
    for t in range(g["data"].shape[1]):
        s = alpha * g["data"][:, t] + (1 - alpha) * s
    assert np.allclose(s, g["out"], rtol=1e-12)
