"""CPU: StreamFramer host logic against the reference ring buffer's framing
(friture/ringbuffer.py:87-99 + the widgets' loops), restated with plain NumPy."""
import os

import numpy as np
import pytest


def reference_frames(stream, frame_len, hop, chunk, pre_increment):
    """Frames a widget would see when `stream` arrives in `chunk`-sized pushes."""
    hist = np.concatenate([np.zeros(frame_len), stream])     # zero-initialised ring buffer
    frames, old_index, offset = [], 0, 0
    for p in range(0, len(stream), chunk):
        offset += min(chunk, len(stream) - p)
        r = int(np.floor((offset - old_index) / hop)) if offset > old_index else 0
        for _ in range(r):
            if pre_increment:
                old_index += hop
            frames.append(hist[old_index:old_index + frame_len].copy())   # samples ending at old_index
            if not pre_increment:
                old_index += hop
    return frames


@pytest.mark.parametrize("frame_len,hop,chunk,pre", [(2048, 512, 512, False), (2048, 1024, 512, False),
                                                     (24000, 12000, 128, True), (64, 16, 40, False),
                                                     (100, 30, 7, True)])
def test_framer_matches_reference_framing(frame_len, hop, chunk, pre):
    import torch
    from friture_b200.stream import StreamFramer
    rng = np.random.default_rng(frame_len + hop)
    total = 3 * frame_len + 11 * hop + 5
    x = rng.standard_normal((2, total)).astype(np.float32)
    fr = StreamFramer(2, frame_len, hop, "cpu", capacity=frame_len + 3 * hop + chunk, pre_increment=pre)
    got = [[], []]
    for p in range(0, total, chunk):
        fr.push(torch.from_numpy(x[:, p:p + chunk]))
        view, r = fr.take()
        for f in range(r):
            for c in range(2):
                got[c].append(view[c, f * hop:f * hop + frame_len].numpy().copy())
    for c in range(2):
        ref = reference_frames(x[c].astype(np.float64), frame_len, hop, chunk, pre)
        assert len(ref) == len(got[c]) and len(ref) > 3
        assert all(np.array_equal(a.astype(np.float32), b) for a, b in zip(ref, got[c]))


def test_framer_vs_reference_ringbuffer():
    """Against the unmodified RingBuffer, through the frame counts and frame digests
    oracle/make_golden.py recorded from it (tests/golden/reference_checks.npz)."""
    import torch
    from friture_b200.stream import StreamFramer
    from oracle.digest import digest
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                              "reference_checks.npz")) as g:
        x_digest, counts, frames = str(g["ring_x"]), list(g["ring_counts"]), list(g["ring_frames"])
    rng = np.random.default_rng(1)
    x = rng.standard_normal(20000)
    assert digest(x) == x_digest, "numpy's seeded stream changed; rerun oracle/make_golden.py"
    fr = StreamFramer(1, 2048, 512, "cpu")
    got = []
    for p, realizable in zip(range(0, len(x), 512), counts):
        fr.push(torch.from_numpy(x[None, p:p + 512].astype(np.float32)))
        view, r = fr.take()
        assert r == realizable
        for f in range(r):
            got.append(digest(view[0, f * 512:f * 512 + 2048].numpy()))
    assert len(counts) == len(range(0, len(x), 512)) and got == frames
