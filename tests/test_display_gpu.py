"""GPU parity: the fused spectrogram display chain vs the reference-derived golden pixels."""
import os
from fractions import Fraction

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_display_pixels_golden():
    import torch
    from friture_b200.display import Mel, SpectrogramDisplay
    with np.load(os.path.join(GOLD, "display.npz")) as d:
        g = {k: d[k] for k in d.files}
    C = 3
    disp = SpectrogramDisplay(C, fft_size=2048, freqscale=Mel, minfreq=20., maxfreq=24000.,
                              spec_min=-140., spec_max=0., height=96, width=700, timerange_s=10.)
    lut = g["lut"]
    inv = {int(v): i for i, v in enumerate(lut)}          # colour word -> LUT index (first wins)
    for tick in range(3):
        db = g["db_%d" % tick].T.copy()                                    # [F, bins]
        x = torch.from_numpy(np.tile(db[None], (C, 1, 1))).cuda().contiguous()
        px = disp.push(x).cpu().numpy().view(np.uint32)
        ref = g["pixels_%d" % tick]
        assert px.shape == (C, ) + ref.shape
        for c in range(C):
            same = px[c] == ref
            # float32 vs float64 upstream: a value within 1e-6 of a LUT step may land one entry off
            assert same.mean() > 0.995
            bad = np.argwhere(~same)
            for r, o in bad[:200]:
                v = g["resampled_%d" % tick][r, o]
                assert abs(v * 255 - round(v * 255)) < 1e-3, (r, o, v)
        assert np.array_equal(px[0], px[1]) and np.array_equal(px[0], px[2])


def test_display_after_stft_runs():
    import torch
    from friture_b200 import audioproc
    from friture_b200.display import SpectrogramDisplay
    p = audioproc()
    p.set_fftsize(4096)
    x = (torch.randn(2, 4096 + 20 * 1024) * 0.1).cuda()
    db = p.stft(x, hop=1024, log=True)
    disp = SpectrogramDisplay(2, fft_size=4096, height=300, width=1200, weighting=1)
    px = disp.push(db)
    assert px.shape[0] == 2 and px.shape[1] == 300 and px.shape[2] >= 1
    assert bool(((px.cpu().numpy().view(np.uint32) >> 24) == 0xFF).all())     # opaque RGB32 words


# ------------------------------------------------------------------ the chain vs the oracle
class OracleChain:
    """fo.frequency_resample -> fo.OnlineLinear2DResamplerOracle -> fo.color_transform per channel,
    fed the same float32 dB columns as the kernel (cast to float64).  A second chain carries the
    magnitudes the float32 arithmetic rounds, (|dB + w| + |spec_min|) / range, through the same
    non-negative interpolation weights: it bounds each pixel value's rounding error."""

    def __init__(self, C, fft_size, scale, minfreq, weighting, spec_min, spec_max, height, L, M):
        from oracle import friture_oracle as fo
        self.C = C
        self.freq = np.linspace(0, 24000, fft_size // 2 + 1)
        A, B, Cw = fo.weighting_tables(self.freq)
        self.w = [np.zeros_like(self.freq), A, B, Cw][weighting]
        self.scale, self.minfreq = scale, minfreq
        self.spec_min, self.range = spec_min, spec_max - spec_min
        self.restart(height, L, M)

    def restart(self, height, L, M):
        from oracle import friture_oracle as fo
        s = self.scale
        self.xs = np.atleast_1d(s.inverse(np.linspace(s.transform(self.minfreq), s.transform(24000.), height)))
        self.tr = [fo.OnlineLinear2DResamplerOracle(L, M, height) for _ in range(2 * self.C)]

    def set_ratio(self, L, M):
        """Online_Linear_2D_resampler.set_ratio: new ratio, indices restart, carried column kept."""
        for tr in self.tr:
            tr.ratio = float(L) / M
            tr.orig_index = tr.resampled_index = 0.

    def push(self, db32):
        from oracle import friture_oracle as fo
        res, mag = [], []
        for c in range(self.C):
            lin = db32[c].T.astype(np.float64) + self.w[:, None]
            norm = (lin - self.spec_min) / self.range
            bound = (np.abs(lin) + abs(self.spec_min)) / abs(self.range)
            res.append(self.tr[c].push(fo.frequency_resample(norm, self.freq, self.xs)))
            mag.append(self.tr[self.C + c].push(fo.frequency_resample(bound, self.freq, self.xs)))
        return np.stack(res), np.stack(mag)


def assert_pixels(px, res, mag, lut):
    """Equal to lut[int(clip(v)*255)] of the oracle's value v, except where v lies within the
    float32 rounding bound of a LUT step; there the pixel is one of the two neighbouring entries."""
    from oracle import friture_oracle as fo
    assert px.shape == res.shape
    bad = px != fo.color_transform(lut, res)
    if not bad.any():
        return
    v, tol = res[bad], 1e-6 * (1.0 + mag[bad])
    lo = (np.clip(v - tol, 0., 1.) * 255).astype(np.intp)
    hi = (np.clip(v + tol, 0., 1.) * 255).astype(np.intp)
    got = px[bad]
    ok = (hi == lo + 1) & ((got == lut[lo]) | (got == lut[np.minimum(hi, 255)]))
    assert ok.all(), (np.argwhere(bad)[~ok][:5], v[~ok][:5], tol[~ok][:5])
    assert bad.mean() < 0.01


def _db_ticks(rng, C, nb, frames):
    """Distinct float32 dB columns per channel (means -70, -60, -50 ... dB, 20 dB spread)."""
    for F in frames:
        mean = -70.0 + 10.0 * np.arange(C)[:, None, None]
        yield (rng.standard_normal((C, F, nb)) * 20.0 + mean).astype(np.float32)


def _input_rate(fft_size):
    return Fraction(48000, fft_size) / (Fraction(1) - Fraction(3, 4)) / 1000     # columns per ms


@pytest.mark.parametrize("weighting", [0, 1, 2, 3])
@pytest.mark.parametrize("scale_id", [0, 1, 2, 3, 4])
def test_display_chain_vs_oracle(scale_id, weighting):
    """Every frequency scale x weighting at N = 32, 2048, 16384, heights 1 / 96 / 600 (three CTAs
    per channel in the carry launch), screen/input column ratios of 1/7.3 (most ticks emit no
    column) and 1/0.37 (one input column feeds several screen columns), ticks of 0 frames, a narrow
    dB range that clips at both ends, minfreq below the first bin above 0 Hz and maxfreq at 24 kHz."""
    import torch
    from friture_b200.display import SCALES, SpectrogramDisplay, load_lut
    C = 3
    scale = SCALES[scale_id]
    lut = load_lut()
    for k, fft_size in enumerate((32, 2048, 16384)):
        nb = fft_size // 2 + 1
        minfreq = 1.5 if fft_size == 16384 else 20.0          # first bin above 0 Hz: 2.9 / 23 / 1500 Hz
        for ri, target in enumerate((7.3, 0.37)):
            height = (1, 96, 600)[(k + ri + scale_id + weighting) % 3]
            spec_min, spec_max = (-75.0, -55.0) if (k + ri + weighting) % 2 else (-140.0, 0.0)
            width = max(1, int(round(float(_input_rate(fft_size)) * 10000 / target)))
            rng = np.random.default_rng([scale_id, weighting, fft_size, ri])
            frames = [int(f) for f in rng.integers(0, 9, 14)]
            frames[1] = frames[6] = 0
            disp = SpectrogramDisplay(C, fft_size=fft_size, freqscale=scale, minfreq=minfreq,
                                      maxfreq=24000.0, spec_min=spec_min, spec_max=spec_max,
                                      weighting=weighting, height=height, width=width, timerange_s=10.)
            orc = OracleChain(C, fft_size, scale, minfreq, weighting, spec_min, spec_max, height,
                              _input_rate(fft_size), Fraction(width, 10000))
            silent = multi = 0
            for F, db in zip(frames, _db_ticks(rng, C, nb, frames)):
                px = disp.push(torch.from_numpy(db).cuda()).cpu().numpy().view(np.uint32)
                res, mag = orc.push(db)
                assert_pixels(px, res, mag, lut)
                silent += F > 0 and px.shape[2] == 0
                multi += px.shape[2] > F
            assert (silent if target > 1 else multi) > 0, (fft_size, target)


def test_display_set_screen_restart():
    """A new height restarts the time resampler with a zero carried column (display.py set_screen);
    a new width only changes the ratio (indices restart, the carried column stays)."""
    import torch
    from friture_b200.display import Mel, SpectrogramDisplay, load_lut
    C, fft_size, weighting = 3, 2048, 2
    nb = fft_size // 2 + 1
    lut = load_lut()
    rng = np.random.default_rng(11)
    disp = SpectrogramDisplay(C, fft_size=fft_size, freqscale=Mel, minfreq=20., maxfreq=24000.,
                              weighting=weighting, height=96, width=300, timerange_s=10.)
    L = _input_rate(fft_size)
    orc = OracleChain(C, fft_size, Mel, 20., weighting, -140., 0., 96, L, Fraction(300, 10000))
    for phase in range(3):
        if phase == 1:
            disp.set_screen(600, 300)
            orc.restart(600, L, Fraction(300, 10000))
        elif phase == 2:
            disp.set_screen(600, 2000)
            orc.set_ratio(L, Fraction(2000, 10000))
        frames = [5, 0, 3, 1, 7]
        for db in _db_ticks(rng, C, nb, frames):
            px = disp.push(torch.from_numpy(db).cuda()).cpu().numpy().view(np.uint32)
            res, mag = orc.push(db)
            assert_pixels(px, res, mag, lut)
