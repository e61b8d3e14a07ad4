"""CPU: the spectrum widget's per-tick reduction (friture_b200/csrc/reduce.cu,
spectrum_reduce_kernel) -- a float32 NumPy replica of the kernel's smoothing recurrence against the
float64 block smoothing of the reference, and the batched oracle restatement the GPU tests use
(tests/test_spectrum_gpu.py) against the per-tick ``SpectrumWidgetOracle``.

At small FFT sizes and long response times alpha is tiny (3.5e-5 at N = 32, 5 s).  The direct form
s <- fma(alpha, p, (1 - alpha) s) rounds 1 - alpha to float32, which moves the effective time
constant by up to ~1e-3 of itself and biases the steady state beyond the 1e-5 criterion; the
complement form s <- fma(alpha, p - s, s) keeps alpha as it is."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import TOL, rel_err  # noqa: E402

F32 = np.float32


# ---------------------------------------------------------------------------- recurrence replica
def fmaf(a, b, c):
    """float32 fma: a*b of two float32 is exact in float64, so the sum rounds once to 53 bits and
    then to 24 (a double rounding that differs from a true fma only on exact ties)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


def smooth_direct(alpha, s, frames):
    """The recurrence as reduce.cu first ran it: om = 1.0f - alpha; s = fmaf(alpha, p, om * s)."""
    a = F32(alpha)
    om = F32(1.0) - a
    a = np.full_like(s, a)
    for p in frames:
        s = fmaf(a, p, om * s)
    return s


def smooth_complement(alpha, s, frames):
    """The recurrence reduce.cu runs: s = fmaf(alpha, p - s, s)."""
    a = np.full_like(s, F32(alpha))
    for p in frames:
        s = fmaf(a, p - s, s)
    return s


def _steady_state_errors(fft_size, response_time, level_db, nbins=17, seed=0):
    from oracle import friture_oracle as fo
    hop = fft_size // 4
    alpha = fo.smoothing_alpha(response_time, 48000 / hop)
    kernel = fo.smoothing_kernel(alpha, 2 * 4096)
    n = int(np.ceil(5 / alpha))
    rng = np.random.default_rng(seed)
    # exponential-distributed per-bin powers (|X|^2 of broadband noise), mean level_db per bin
    p = (rng.exponential(size=(n, nbins)) * 10 ** (level_db / 10)).astype(F32)
    ref = np.zeros(nbins)
    got = {"direct": np.zeros(nbins, F32), "complement": np.zeros(nbins, F32)}
    step = 4096
    for f0 in range(0, n, step):
        blk = p[f0:f0 + step]
        ref = fo.exp_smoothed_value_2d(kernel, alpha, blk.T.astype(np.float64), ref)
        got["direct"] = smooth_direct(alpha, got["direct"], blk)
        got["complement"] = smooth_complement(alpha, got["complement"], blk)
    rdb = fo.log_spectrogram(ref)
    return {k: rel_err(fo.log_spectrogram(v.astype(np.float64)), rdb) for k, v in got.items()}


@pytest.mark.parametrize("fft_size,response_time", [(32, 5.0), (64, 5.0), (32, 1.0)])
def test_smoothing_recurrence_complement_form(fft_size, response_time):
    """After 5/alpha frames of -20 dB/bin broadband power the complement form stays well inside
    the criterion and the direct form does not."""
    e = _steady_state_errors(fft_size, response_time, -20.0)
    assert e["complement"] < 0.2 * TOL, e
    assert e["direct"] > (3 * TOL if (fft_size, response_time) == (32, 5.0) else TOL), e


# ---------------------------------------------------------------------------- widget restatement
def tick_frame_counts(chunk_sizes, hop):
    """Frames each tick realizes when the stream arrives in these chunks: the widget's
    floor((offset - old_index) / hop), old_index advancing by one hop per frame
    (friture/spectrum.py:125-155)."""
    counts, offset, old = [], 0, 0
    for n in chunk_sizes:
        offset += int(n)
        r = (offset - old) // hop if offset > old else 0
        old += r * hop
        counts.append(int(r))
    return counts


def widget_ticks(x, fft_size, frame_counts, response_time, weight=None):
    """Batched float64 restatement of SpectrumWidgetOracle.tick for C channels at once.
    x: [C, T] stream; frame f ends at sample f*hop of the zero-prefixed stream (the widget's
    zero-initialised ring buffer).  Yields per tick (smoothed power [C, bins], dB [C, bins],
    HPS [C, bins//3])."""
    from oracle import friture_oracle as fo
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    C = x.shape[0]
    hop = fft_size // 4
    nb = fft_size // 2 + 1
    total = int(sum(frame_counts))
    xz = np.concatenate([np.zeros((C, fft_size)), x], axis=1)[:, :fft_size + max(total - 1, 0) * hop]
    P = fo.stft_power_batch(xz, fft_size, hop) if total else np.zeros((C, 0, nb))
    assert P.shape[1] == total
    alpha = fo.smoothing_alpha(response_time, 48000 / hop)
    kernel = fo.smoothing_kernel(alpha, 2 * 4096)
    w = np.zeros(nb) if weight is None else np.asarray(weight, dtype=np.float64)
    s = np.zeros(C * nb)
    f0 = 0
    for n in frame_counts:
        data = P[:, f0:f0 + n, :].transpose(0, 2, 1).reshape(C * nb, n)
        s = fo.exp_smoothed_value_2d(kernel, alpha, data, s)
        f0 += n
        sp = s.reshape(C, nb)
        yield sp, fo.log_spectrogram(sp) + w, np.stack([fo.harmonic_product_spectrum(v) for v in sp])


@pytest.mark.parametrize("fft_size,response_time,weighting", [(64, 0.125, 0), (1024, 1.0, 1)])
def test_widget_restatement_matches_oracle_tick(fft_size, response_time, weighting):
    """widget_ticks == SpectrumWidgetOracle.tick fed the samples of each tick's frames."""
    from oracle import friture_oracle as fo
    C, hop = 2, fft_size // 4
    rng = np.random.default_rng(fft_size)
    chunks = list(rng.integers(1, 3 * fft_size, 12)) + [0, hop - 1, 1]
    x = rng.standard_normal((C, int(sum(chunks)))) * 0.3
    counts = tick_frame_counts(chunks, hop)
    assert 0 in counts and sum(counts) > 20
    w = None if not weighting else fo.weighting_tables(np.linspace(0, 24000, fft_size // 2 + 1))[weighting - 1]
    orcs = [fo.SpectrumWidgetOracle(fft_size, response_time=response_time, weight=w) for _ in range(C)]
    xz = np.concatenate([np.zeros((C, fft_size)), x], axis=1)
    old = 0
    for n, (sp, db, hps) in zip(counts, widget_ticks(x, fft_size, counts, response_time, w)):
        seg = xz[:, old * hop: old * hop + fft_size + (n - 1) * hop] if n else xz[:, :0]
        old += n
        for c in range(C):
            rdb, _, _, ri, rp = orcs[c].tick(seg[c])
            assert np.allclose(orcs[c].disp, sp[c], rtol=1e-12, atol=0)
            assert np.allclose(rdb, db[c], rtol=1e-12, atol=0)
            assert ri == int(np.argmax(db[c])) and rp == int(np.argmax(hps[c]))
