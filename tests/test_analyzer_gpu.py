"""GPU: the combined per-hop analysis (friture_b200.analyzer.ChannelAnalyzer) -- BASELINE configs[4]'s
unit: one log-power column + one 30-band dB vector per channel and hop -- device path, host path
and the 2-rank NCCL gather, against the oracle."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import TOL, assert_logpower_parity, rel_err  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_units(x, n_oct=10, weighting=None):
    from oracle import friture_oracle as fo
    from friture_b200 import filter_data
    bdec, adec, _ = filter_data.decimator()
    boct, aoct, _ = filter_data.bands(3)
    C, T = x.shape
    spec = fo.log_spectrogram(fo.stft_power_batch(x, 2048, 1024))
    bands = np.zeros((C, T // 1024, 3 * n_oct))
    for c in range(C):
        orc = fo.OctaveSpectrumOracle(bdec, adec, list(boct), list(aoct), noctave=n_oct)
        for b in range(T // 1024):
            bands[c, b] = orc.push(x[c, b * 1024:(b + 1) * 1024].astype(np.float64))[1]
    if weighting is not None:
        bands = bands + weighting
    return spec, bands


def test_combined_device_and_host_paths_match_oracle():
    import torch
    from friture_b200.analyzer import ChannelAnalyzer
    x = (np.random.default_rng(3).standard_normal((7, 17 * 1024)) * 0.1).astype(np.float32)
    ref_spec, ref_bands = oracle_units(x)
    an = ChannelAnalyzer(7)
    spec, bands = an.process(torch.from_numpy(x).cuda())
    assert tuple(spec.shape) == (7, 16, 1025) and tuple(bands.shape) == (7, 17, 30)
    assert_logpower_parity(spec.cpu().numpy(), ref_spec)
    assert rel_err(bands.cpu().numpy(), ref_bands) < TOL
    # sequential (one stream) == overlapped (two streams)
    an2 = ChannelAnalyzer(7)
    spec2, bands2 = an2.process(torch.from_numpy(x).cuda(), overlap=False)
    assert torch.equal(spec, spec2) and torch.equal(bands, bands2)
    # host path: pinned buffers, pipelined over time segments inside the C call
    an3 = ChannelAnalyzer(7)
    xh = torch.from_numpy(x).pin_memory()
    sh, bh = an3.process_host(xh)
    assert torch.equal(sh, spec.cpu())
    assert rel_err(bh.numpy(), ref_bands) < TOL        # cut into launches at other instants: same state, same result
    # a stream fed in two pieces gives the same band vectors (state carried in the handle)
    an4 = ChannelAnalyzer(7)
    xd = torch.from_numpy(x).cuda()
    _, b_a = an4.process(xd[:, :8 * 1024].contiguous())
    _, b_b = an4.process(xd[:, 8 * 1024:].contiguous())
    assert rel_err(torch.cat([b_a, b_b], 1).cpu().numpy(), ref_bands) < TOL


def test_combined_long_host_stream_and_weighting():
    import torch
    from friture_b200.analyzer import ChannelAnalyzer
    x = (np.random.default_rng(4).standard_normal((3, 65 * 1024)) * 0.1).astype(np.float32)
    an = ChannelAnalyzer(3, weighting="A")
    ref_spec, ref_bands = oracle_units(x, weighting=an.bank.A)
    sh, bh = an.process_host(torch.from_numpy(x).pin_memory())      # 8 time segments
    assert_logpower_parity(sh.numpy(), ref_spec)
    assert rel_err(bh.numpy(), ref_bands) < TOL


_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
from friture_b200.analyzer import ChannelAnalyzer
from oracle import friture_oracle as fo
C, F = 6, 16
xs = [(np.random.default_rng(100 + r).standard_normal((C, (F + 1) * 1024)) * 0.1).astype(np.float32) for r in range(world)]
ref = np.concatenate([fo.log_spectrogram(fo.stft_power_batch(x, 2048, 1024)) for x in xs], axis=0)
for transport, engine in (("nccl", "auto"), ("peer", "ce"), ("peer", "kernel")):
    an = ChannelAnalyzer(C)
    gathered = torch.empty((4, world * C, F // 4, 1025), dtype=torch.float32, device="cuda") if transport == "nccl" else None
    chunks, bands, gathered = an.process_sharded(torch.from_numpy(xs[rank]).cuda(), gathered, n_chunks=4,
                                                 transport=transport, engine=engine)
    if transport == "peer":
        an.peer_gather.wait_all()           # every rank's pushes have landed
    torch.cuda.synchronize()
    # every rank must hold every rank's columns, in global channel order, equal to the oracle's
    g = gathered.reshape(4, world * C, F // 4, 1025)
    full = g.permute(1, 0, 2, 3).reshape(world * C, F, 1025).cpu().numpy()
    err = float(np.max(np.abs(full - ref)) / max(np.max(np.abs(ref)), 1.0))
    own = chunks.permute(1, 0, 2, 3).reshape(C, F, 1025)
    same = bool(torch.equal(own, g.permute(1, 0, 2, 3).reshape(world * C, F, 1025)[rank * C:(rank + 1) * C]))
    print("RESULT %%s-%%s rank %%d err %%.3g own_block_identical %%s" %% (transport, engine, rank, err, same), flush=True)
    assert err < 1e-5 and same
    if transport == "peer":
        an.peer_gather.close()
dist.destroy_process_group()
'''


def test_gather_of_columns_two_ranks(tmp_path):
    """north_star's collective on two real GPUs, both transports: NCCL all-gather per frame chunk on
    a side stream, and copy-engine pushes into the peers' IPC-opened buffers over NVLink;
    gathered == the oracle's columns of all channels on every rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT})
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("RESULT nccl-auto rank") == 2
    assert out.stdout.count("RESULT peer-ce rank") == 2 and out.stdout.count("RESULT peer-kernel rank") == 2


def test_peer_push_kernel_single_gpu():
    """frt_peer_push with local buffers standing in for the peers': every destination receives the
    block, bytes outside it stay untouched, odd sizes that are not a multiple of the grid stride work."""
    import ctypes
    from ctypes import c_size_t, c_void_p
    import torch
    from friture_b200 import _lib
    h = _lib.default_handle()
    n = 3 * 1000 * 1025 + 4                      # floats; 16-byte multiple, not a multiple of anything else
    src = torch.randn(n, device="cuda")
    dsts = [torch.full((n + 8,), -7.0, device="cuda") for _ in range(3)]
    table = (c_void_p * 3)(*[d.data_ptr() + 16 for d in dsts])      # offset by 4 floats, still 16-byte aligned
    st = torch.cuda.current_stream()
    h.call("frt_peer_push", c_void_p(src.data_ptr()), table, 3, c_size_t(n * 4), 0, c_void_p(st.cuda_stream))
    torch.cuda.synchronize()
    for d in dsts:
        assert torch.equal(d[4:4 + n], src)
        assert float(d[:4].max()) == -7.0 and float(d[4 + n:].min()) == -7.0
    with pytest.raises(_lib.FrtError):
        h.call("frt_peer_push", c_void_p(src.data_ptr() + 4), table, 3, c_size_t(n * 4), 0, c_void_p(st.cuda_stream))
