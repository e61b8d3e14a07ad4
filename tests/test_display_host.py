"""CPU: the spectrogram display chain -- oracle restatement and host-side logic against golden
vectors produced by the reference's Frequency_Resampler / Online_Linear_2D_resampler classes."""
import os
from fractions import Fraction

import numpy as np

from oracle import friture_oracle as fo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load():
    with np.load(os.path.join(GOLD, "display.npz")) as d:
        return {k: d[k] for k in d.files}


def ratio_LM():
    return Fraction(48000, 2048) / (Fraction(1) - Fraction(3, 4)) / 1000, Fraction(700, 10000)


def test_oracle_display_chain_matches_reference():
    g = load()
    freq = np.linspace(0, 24000, 1025)
    L, M = ratio_LM()
    tr = fo.OnlineLinear2DResamplerOracle(L, M, 96)
    for tick in range(3):
        norm = (g["db_%d" % tick].astype(np.float64) + 140.0) / 140.0
        res = tr.push(fo.frequency_resample(norm, freq, g["xscaled"]))
        assert res.shape == g["resampled_%d" % tick].shape
        assert np.array_equal(res, g["resampled_%d" % tick])
        assert np.array_equal(fo.color_transform(g["lut"], res), g["pixels_%d" % tick])


def test_host_tables_and_index_bookkeeping():
    from friture_b200.display import Mel, OnlineResamplerIndex, load_lut, screen_rows, SCALES
    g = load()
    freq = np.linspace(0, 24000, 1025)
    xs, i0, t = screen_rows(freq, Mel, 20., 24000., 96)
    assert np.array_equal(xs, g["xscaled"])
    col = np.random.default_rng(0).random(1025)
    assert np.allclose(col[i0] + t * (col[i0 + 1] - col[i0]), np.interp(xs, freq, col), rtol=1e-13)
    assert np.array_equal(load_lut(), g["lut"])
    L, M = ratio_LM()
    idx = OnlineResamplerIndex()
    idx.set_ratio(L, M)
    assert abs(idx.resampling_ratio - float(g["ratio"])) < 1e-15
    for tick, ncols in enumerate((5, 1, 9)):
        cols, a = idx.push(ncols)
        assert len(cols) == g["resampled_%d" % tick].shape[1]
        assert np.all((a >= -1e-12) & (a <= 1 + 1e-12)) and np.all(np.diff(cols) >= 0)
    for s in SCALES.values():       # transform / inverse are inverse pairs
        f = np.array([20., 440., 1000., 20000.])
        assert np.allclose(s.inverse(s.transform(f)), f, rtol=1e-12)
    # every scale: the (i0, t) table reproduces np.interp on the screen rows, from below the first
    # bin above 0 Hz up to a clamped last row at exactly 24 kHz, for 1 / 96 / 600 rows
    rng = np.random.default_rng(1)
    for s in SCALES.values():
        for nb, minfreq in ((17, 20.), (1025, 20.), (8193, 1.5)):
            fq = np.linspace(0, 24000, nb)
            col = rng.standard_normal(nb) * 30 - 60
            for h in (1, 96, 600):
                xs, i0, t = screen_rows(fq, s, minfreq, 24000., h)
                ref_xs = np.atleast_1d(s.inverse(np.linspace(s.transform(minfreq), s.transform(24000.), h)))
                assert np.array_equal(xs, ref_xs) and xs.shape == (h, )
                assert np.all((i0 >= 0) & (i0 <= nb - 2) & (t >= 0) & (t <= 1))
                assert np.allclose(col[i0] + t * (col[i0 + 1] - col[i0]), np.interp(xs, fq, col),
                                   rtol=0, atol=1e-11)
    # the index bookkeeping == the oracle resampler, column for column, over a long irregular tick
    # sequence: downsampling (several ticks emit nothing) and upsampling (several columns per input)
    for L, M in ((Fraction(48000, 32) / (Fraction(1) - Fraction(3, 4)) / 1000, Fraction(8219, 10000)),
                 (Fraction(48000, 2048) / (Fraction(1) - Fraction(3, 4)) / 1000, Fraction(2534, 10000))):
        idx = OnlineResamplerIndex()
        idx.set_ratio(L, M)
        tr = fo.OnlineLinear2DResamplerOracle(L, M, 2)
        old = np.zeros(2)
        n_out = []
        for F in rng.integers(0, 13, 400):
            data = rng.standard_normal((2, F))
            cols, a = idx.push(int(F))
            ref = tr.push(data)
            prev = np.concatenate([old[:, None], data[:, :-1]], axis=1)
            got = data[:, cols] * (1 - a) + prev[:, cols] * a if len(cols) else np.zeros((2, 0))
            assert got.shape == ref.shape and np.allclose(got, ref, rtol=0, atol=1e-12)
            if F:
                old = data[:, -1]
            n_out.append(len(cols))
        n_out = np.array(n_out)
        assert (n_out == 0).sum() > 50 if L > M else (n_out > 13).sum() > 50
