"""GPU parity against the golden vectors generated from the UNMODIFIED reference
(oracle/make_golden.py -> tests/golden/).  These are the reference-derived anchors that travel to
the GPU box."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import TOL, rel_err, assert_logpower_parity  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with np.load(os.path.join(GOLD, name)) as d:
        return {k: d[k] for k in d.files}


@pytest.mark.parametrize("n_fft", [1024, 2048, 8192])
def test_analyzelive_golden(n_fft):
    from friture_b200 import audioproc
    g = load("analyzelive.npz")
    p = audioproc()
    p.set_fftsize(n_fft)
    sp = p.analyzelive(g["x_%d" % n_fft])
    assert sp.shape == (n_fft // 2 + 1,) and sp.dtype == np.float64
    assert rel_err(sp, g["power_%d" % n_fft]) < TOL
    assert_logpower_parity(10 * np.log10(sp + 1e-30), 10 * np.log10(g["power_%d" % n_fft] + 1e-30))


def test_spectrogram_golden():
    import torch
    from friture_b200 import audioproc
    g = load("spectrogram.npz")
    p = audioproc()
    p.set_fftsize(int(g["n_fft"]))
    logpower = 10. * np.log10(g["power"] + 1e-30)          # the reference's log_spectrogram
    got = p.stft(torch.from_numpy(g["x"]).cuda(), hop=int(g["hop"]), log=True).cpu().numpy()
    assert got.shape == logpower.shape
    e = assert_logpower_parity(got, logpower)
    print("spectrogram golden:", e)
    pw = p.stft(torch.from_numpy(g["x"]).cuda(), hop=int(g["hop"]), log=False).cpu().numpy()
    assert rel_err(pw, g["power"]) < TOL


@pytest.mark.parametrize("bpo,block", [(3, 256), (3, 512), (3, 1024), (12, 512)])
def test_bank_energies_golden(bpo, block):
    import torch
    from friture_b200.octavefilters import Octave_Filters
    g = load("octave_bank.npz")
    bank = Octave_Filters(bpo)
    e = bank.energies_batch(torch.from_numpy(g["x"]).cuda()[None, :], block=block)[0].cpu().numpy()
    ref = g["energies_bpo%d_block%d" % (bpo, block)]
    assert e.shape == ref.shape
    assert np.max(np.abs(e - ref) / np.max(ref, axis=-1, keepdims=True)) < TOL
    db = 10 * np.log10(e.astype(np.float64) + 1e-30)
    assert rel_err(db, 10 * np.log10(ref + 1e-30)) < TOL


def test_bank_outputs_golden():
    from friture_b200.octavefilters import Octave_Filters
    g = load("octave_bank.npz")
    bank = Octave_Filters(3)
    ys = [[] for _ in range(27)]
    for b in range(16):
        y, dec = bank.filter(g["x"][b * 512:(b + 1) * 512])
        for k in range(27):
            ys[k].append(y[k])
    assert dec == list(g["dec_bpo3"])
    for k in (0, 13, 26):
        got = np.concatenate(ys[k])
        ref = g["y_bpo3_band%d" % k]
        assert np.max(np.abs(got - ref)) / np.max(np.abs(ref)) < 5e-5
    # distance to the reference's live FFT-OLA path (secondary; its own tolerance is 5 %)
    acc = np.array([np.sum(np.concatenate(v) ** 2) for v in ys])
    d = np.max(np.abs(acc / g["fft_bank_energy_sum_bpo3"] - 1.0))
    print("distance to the live FFT-OLA path on band energy:", d)
    assert d < 0.05
