"""GPU parity: the spectrum widget's per-tick reductions (smoothing across frames, weighting, dB,
peak, harmonic product spectrum) vs the CPU oracle (friture/spectrum.py:125-222)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import TOL, assert_logpower_parity, rel_err  # noqa: E402
from test_spectrum_host import tick_frame_counts, widget_ticks  # noqa: E402

pytestmark = pytest.mark.gpu

FFT_SIZES = [32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384]   # spectrum_settings.py:59-70
RESPONSE_TIMES = [0.025, 0.125, 0.3, 1.0, 5.0]                        # spectrum_settings.py:119-125


def bin_index(f_hz, fft_size):
    """Bin of a frequency returned by SpectrumAnalyzer.process (freq = linspace(0, 24000, bins));
    the 1e-20 Hz of a zero pitch maps to bin 0."""
    return np.rint(np.asarray(f_hz) * (fft_size // 2) / 24000.0).astype(int)


def assert_argmax(got_i, ref_vals, tol, what):
    """got_i must be the oracle's arg-max, except on a genuine near-tie: the oracle's own values at
    the two indices within `tol` (float32 cannot order them)."""
    ref_i = int(np.argmax(ref_vals))
    if got_i != ref_i:
        assert 0 <= got_i < len(ref_vals) and ref_vals[ref_i] - ref_vals[got_i] <= tol, \
            (what, int(got_i), ref_i, float(ref_vals[got_i]), float(ref_vals[ref_i]), tol)


def check_indices(fmax, fpitch, rdb, hps, fft_size, lo=0):
    """Peak over the dB vector (near-tie: TOL of the vector's scale, the dB criterion), pitch over
    the HPS product (near-tie: 1e-5 relative).  `lo` = 1 leaves bin 0 out of the dB scale (its
    weighting offset is -998 dB)."""
    for c in range(rdb.shape[0]):
        tol_db = TOL * max(np.max(np.abs(rdb[c, lo:])), 1.0)
        assert_argmax(bin_index(fmax[c], fft_size), rdb[c], tol_db, ("peak", c))
        assert_argmax(bin_index(fpitch[c], fft_size), hps[c], 1e-5 * np.max(hps[c]), ("pitch", c))


def weight_table(fft_size, weighting):
    from oracle import friture_oracle as fo
    if not weighting:
        return None
    return fo.weighting_tables(np.linspace(0, 24000, fft_size // 2 + 1))[weighting - 1]


# ------------------------------------------------------------------ few ticks, tonal input
def _tick_case(fft_size, weighting, level_db=None):
    tag = "%d-%d" % (fft_size, weighting) + ("" if level_db is None else "-quiet%d" % -level_db)
    return pytest.param(fft_size, weighting, level_db, id=tag)


@pytest.mark.parametrize("fft_size,weighting,level_db", [
    _tick_case(2048, 0), _tick_case(8192, 1), _tick_case(1024, 3),
    _tick_case(32, 1), _tick_case(32, 2), _tick_case(32, 3),
    _tick_case(2048, 1), _tick_case(2048, 2), _tick_case(2048, 3),
    _tick_case(16384, 1), _tick_case(16384, 2), _tick_case(16384, 3),
    # quiet inputs: the HPS product of three float32 powers reaches the denormal range near -115 dBFS
    _tick_case(8192, 0, -60), _tick_case(8192, 0, -100), _tick_case(8192, 0, -120),
    _tick_case(1024, 0, -120), _tick_case(2048, 1, -100),
])
def test_spectrum_ticks(fft_size, weighting, level_db):
    import torch
    from friture_b200.spectrum import SpectrumAnalyzer
    from oracle import friture_oracle as fo
    C = 3
    rng = np.random.default_rng(fft_size)
    hop = fft_size // 4
    t = np.arange(fft_size + 9 * hop) / 48000.0
    gain = 1.0 if level_db is None else 10 ** (level_db / 20) / 0.3    # fundamental at level_db dBFS
    ticks = []
    for k in range(3):
        x = rng.standard_normal((C, len(t))) * 0.05
        for c in range(C):
            f0 = 220.0 * (c + 1)
            x[c] += sum(0.3 / h * np.sin(2 * np.pi * f0 * h * t + k) for h in (1, 2, 3))
        ticks.append((x * gain).astype(np.float32))
    an = SpectrumAnalyzer(C, fft_size=fft_size, response_time=0.125, weighting=weighting)
    w = weight_table(fft_size, weighting)
    orcs = [fo.SpectrumWidgetOracle(fft_size, response_time=0.125, weight=w) for _ in range(C)]
    for x in ticks:
        db, fmax, fpitch = an.process(torch.from_numpy(x).cuda())
        db = db.cpu().numpy().astype(np.float64)
        rdb = np.empty_like(db)
        for c in range(C):
            rdb[c], rfmax, rfpitch, ri, rp = orcs[c].tick(x[c])
            if weighting == 0:
                assert_logpower_parity(db[c], rdb[c], min_frac=0.0, strict=False, floor_db=40.0)
            else:   # bin 0 carries A/B/C(0 Hz) = -998 dB (eps = 1e-50): the criterion on bins 1..
                assert rel_err(db[c, 1:], rdb[c, 1:]) < TOL, (c, rel_err(db[c, 1:], rdb[c, 1:]))
        hps = np.stack([fo.harmonic_product_spectrum(o.disp) for o in orcs])
        check_indices(fmax, fpitch, rdb, hps, fft_size, lo=1 if weighting else 0)
        if level_db is not None:    # a clear tone: no near-tie excuse for the pitch
            for c in range(C):
                assert bin_index(fpitch[c], fft_size) == int(np.argmax(hps[c])), (c, level_db)
    assert abs(an.alpha - orcs[0].alpha) < 1e-15


# ------------------------------------------------------------------ widget settings at steady state
def _broadband(rng, C, T):
    """C distinct broadband channels: white at sigma 0.5 and 0.005, then tilted (one-pole) noise."""
    from scipy.signal import lfilter
    sig = [0.5, 0.005] + [0.05] * (C - 2)
    x = rng.standard_normal((C, T)) * np.asarray(sig)[:, None]
    for c in range(2, C):
        x[c] = lfilter([1.0], [1.0, -0.5], x[c])
    return x.astype(np.float32)


def _chunks(rng, total):
    """Irregular pushes summing to >= total: mostly 441..4096 samples, some of 1..15 samples and
    some empty ones (a timer tick with no new audio realizes no frame; the second tick is one)."""
    out, n = [4096, 0], 4096
    while n < total:
        u = rng.random()
        k = 0 if u < 0.08 else int(rng.integers(1, 16)) if u < 0.2 else int(rng.integers(441, 4097))
        out.append(k)
        n += k
    return out


def drive_widget(an, x, chunks):
    """Push x [C, T] (CUDA) through a StreamFramer in these chunks and process every take(),
    including the ones that realize no frame.  Yields (n_frames, dB [C, bins], fmax, fpitch)."""
    import torch
    from friture_b200.stream import StreamFramer
    C = x.shape[0]
    fr = StreamFramer(C, an.fft_size, an.hop, x.device)
    empty = torch.empty((C, 0), dtype=torch.float32, device=x.device)
    p = 0
    for n in chunks:
        fr.push(x[:, p:p + n])
        p += n
        view, nf = fr.take()
        db, fmax, fpitch = an.process(view if nf else empty)
        yield nf, db.cpu().numpy().astype(np.float64), fmax, fpitch


@pytest.mark.parametrize("response_time", RESPONSE_TIMES)
@pytest.mark.parametrize("fft_size", FFT_SIZES)
def test_spectrum_widget_settings_steady_state(fft_size, response_time):
    """Every FFT size x response time of the widget, driven tick by tick as the widget is, for at
    least 5/alpha frames.  Once smoothing averages >= 8 frames and the stream is past 5/alpha
    frames, every bin of every tick meets the strict criterion (smoothed broadband power has no
    deep nulls); before that, and for short memories, the floor-aware one."""
    import torch
    from friture_b200.spectrum import SpectrumAnalyzer
    C = 3
    hop = fft_size // 4
    rng = np.random.default_rng([fft_size, int(response_time * 1000)])
    an = SpectrumAnalyzer(C, fft_size=fft_size, response_time=response_time)
    settle = 5.0 / an.alpha
    chunks = _chunks(rng, int(np.ceil(settle)) * hop + 3 * 4096 + fft_size)
    counts = tick_frame_counts(chunks, hop)
    x = _broadband(rng, C, sum(chunks))
    ref = widget_ticks(x, fft_size, counts, response_time)
    done, strict_ticks = 0, 0
    gpu = drive_widget(an, torch.from_numpy(x).cuda(), chunks)
    for tick, ((nf, db, fmax, fpitch), (_, rdb, hps), n) in enumerate(zip(gpu, ref, counts)):
        assert nf == n
        done += n
        if 1.0 / an.alpha >= 8 and done >= settle:
            strict_ticks += 1
            for c in range(C):
                e = rel_err(db[c], rdb[c])
                assert e < TOL, (tick, c, done, e)
        else:
            for c in range(C):
                assert_logpower_parity(db[c], rdb[c], min_frac=0.999, strict=False)
        check_indices(fmax, fpitch, rdb, hps, fft_size)
    assert done >= settle and 0 in counts
    assert strict_ticks >= 3 or 1.0 / an.alpha < 8


# ------------------------------------------------------------------ edges
@pytest.mark.parametrize("fft_size", [32, 2048])
@pytest.mark.parametrize("weighting", [0, 1, 2, 3])
def test_spectrum_edges(fft_size, weighting):
    import torch
    from friture_b200.spectrum import SpectrumAnalyzer
    C, hop = 2, fft_size // 4
    w = weight_table(fft_size, weighting)
    w = np.zeros(fft_size // 2 + 1) if w is None else w
    an = SpectrumAnalyzer(C, fft_size=fft_size, response_time=0.3, weighting=weighting)
    # all-zero input: dB = 10 log10(1e-30) + w on every bin, pitch 1e-20 Hz
    db, fmax, fpitch = an.process(torch.zeros((C, fft_size + 5 * hop), device="cuda"))
    db = db.cpu().numpy().astype(np.float64)
    for c in range(C):
        assert rel_err(db[c], -300.0 + w) < TOL
        if weighting:
            assert_argmax(bin_index(fmax[c], fft_size), w, TOL * np.max(np.abs(-300 + w[1:])), "peak")
        else:
            assert fmax[c] == 0.0
        assert fpitch[c] == 1e-20
    # a tick with no frame leaves the state as it was
    x = (torch.randn(C, fft_size + 7 * hop) * 0.1).cuda()
    db1, fmax1, fpitch1 = an.process(x)
    state = an._disp.clone()
    for short in (x[:, :0], x[:, :fft_size - 1]):
        db2, fmax2, fpitch2 = an.process(short)
        assert torch.equal(an._disp, state) and torch.equal(db2, db1)
        assert np.array_equal(fmax2, fmax1) and np.array_equal(fpitch2, fpitch1)
    # 8192 frames in one call is the reference's kernel length; more is rejected, state untouched
    with pytest.raises(ValueError):
        an.process(torch.zeros((C, fft_size + 8192 * hop), device="cuda"))
    assert torch.equal(an._disp, state)


def test_spectrum_tick_of_8192_frames():
    """The longest accepted tick (the reference's 8192-tap smoothing kernel), at N = 32, 5 s."""
    import torch
    from friture_b200.spectrum import SpectrumAnalyzer
    fft_size, hop, rt = 32, 8, 5.0
    x = _broadband(np.random.default_rng(7), 3, fft_size + 2 * 8192 * hop)
    counts = [1, 8192, 8191]        # ticks of 1 (the zero frame), 8192 and 8191 frames
    an = SpectrumAnalyzer(3, fft_size=fft_size, response_time=rt)
    xd = torch.from_numpy(x).cuda()
    xz = torch.cat([torch.zeros((3, fft_size), device="cuda"), xd], dim=1)
    f0 = 0
    for n, (sp, rdb, hps) in zip(counts, widget_ticks(x, fft_size, counts, rt)):
        db, fmax, fpitch = an.process(xz[:, f0 * hop: f0 * hop + fft_size + (n - 1) * hop].contiguous())
        f0 += n
        db = db.cpu().numpy().astype(np.float64)
        for c in range(3):
            assert_logpower_parity(db[c], rdb[c], min_frac=0.999, strict=False)
        check_indices(fmax, fpitch, rdb, hps, fft_size)


def test_smoothing_state_carries_and_resets():
    import torch
    from friture_b200.spectrum import SpectrumAnalyzer
    x = (torch.randn(2, 2048 + 3 * 512) * 0.1).cuda()
    an = SpectrumAnalyzer(2, fft_size=2048, response_time=1.0)
    a1, _, _ = an.process(x)
    a2, _, _ = an.process(x)
    assert not torch.equal(a1, a2)            # history matters
    an.setfftsize(2048)                       # settings change restarts the buffers (spectrum.py:224-226)
    a3, _, _ = an.process(x)
    assert torch.equal(a1, a3)
