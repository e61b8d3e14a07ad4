#!/usr/bin/env python
"""bench.py -- throughput of the Friture spectral hot path on B200 (one JSON line on stdout).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload combined|stft|bank|gcc]
                    [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic 48 kHz float32 audio.  The default
workload is the one BASELINE.json's metric is quoted on ("2048-pt STFT + 30-band 1/3-octave"),
configs[4]'s unit on one GPU's share of the channels: 1024 channels per GPU, and per channel and
hop of 1024 new samples ONE unit = one 2048-point log-power spectrogram column (50 % overlap; what
`audioproc.analyzelive` + `log_spectrogram` give Spectrogram_Widget per column) + one vector of
30 smoothed 1/3-octave band levels in dB (what OctaveSpectrum_Widget computes per chunk:
`Octave_Filters.filter`, y**2, `exp_smoothed_value`, 10*log10).  `metric` is spectra/sec, counted
in these units.

  value      whole-job units/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e        same through the public API with HOST buffers (pinned): H2D + kernels + D2H in the
             timed region
  roofline   the step's dominant kernel (the filterbank): algorithmic bytes per launch / its
             CUDA-event duration against the measured HBM peak, plus its FP32 issue-slot fraction
             (the recursion is issue/latency-bound, not HBM-bound)
  cpu_baseline / --impl reference   the CPU oracle (a validated restatement of the reference's
             NumPy path; the reference is pure Python and cannot travel to the GPU box) on the
             host's usable cores

Multi-GPU (torchrun, one process per GPU): channels are independent streams, sharded over the
ranks with no collective while computing; at N > 1 the north-star's final all-gather of the
spectrogram columns over NVLink IS inside the timed region, issued per frame chunk on a side
stream so that it overlaps the filterbank kernel.  `other_workloads` holds the named extras
(configs[1], [2], [3], the channel sweep, the gather variants), each with its own roofline.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_FFT = 2048
HOP = 1024
NBINS = N_FFT // 2 + 1
N_OCT = 10          # "30-band": 10 octaves x 3 bands (SURVEY M3)
NBANDS = 3 * N_OCT
STFT_BYTES_PER_SPECTRUM = HOP * 4 + NBINS * 4      # 8196 B: each sample read once, each bin written once
SM_COUNT, SM_MHZ = 148, 1965.0


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bank_state_bytes(n_oct, bpo=3):
    return (n_oct * (2 * bpo + 6) * 2 + n_oct * bpo) * 4


def bank_bytes_per_launch(C, block, n_blocks, n_oct, bpo=3):
    """input samples + band vectors + filter/smoothing state read and written once per launch"""
    return C * (block * n_blocks * 4 + n_blocks * n_oct * bpo * 4 + 2 * bank_state_bytes(n_oct, bpo))


def bank_fp32_ops_per_sample(n_oct, bpo=3):
    """lane-operations per input sample: 4 per normalised biquad step, 2 for y^2 + smoothing"""
    return sum(((2 * bpo + 6) * 4 + bpo * 2) / 2 ** j for j in range(n_oct))


def traffic_for(kernel_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture -- only if it
    was taken from the very source that is being run (keyed by the .cu file's hash)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            t = json.load(f).get(kernel_key)
        src = os.path.join(ROOT, "friture_b200", "csrc", t["source"])
        with open(src, "rb") as f:
            sha = hashlib.sha256(f.read()).hexdigest()[:16]
        if sha == t["source_sha16"]:
            return t
    except Exception:
        pass
    return None


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            try:
                self.proc.kill()
            except Exception:
                pass

    def summary(self, t0, t1):
        sm, mx, reasons, power = [], [], set(), []
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            p = [q.strip() for q in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
                power.append(float(p[6]))
            except ValueError:
                continue
            for name, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": float(max(power)) if power else None}


# ----------------------------------------------------------------------------- host placement
def bind_to_gpu_numa(local_rank):
    """Pin this process to the CPUs of the GPU's NUMA node BEFORE any pinned allocation, so that
    the staging buffers of the host path live next to the GPU's PCIe root (SCALE_r01: unbound
    ranks lost two thirds of the PCIe rate at 8 GPUs)."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:].lower(), rest.lower())
        node = int(open(path).read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["bound"] = True
            info["cpus"] = len(allowed)
    except Exception as e:      # placement is an optimisation, never a failure
        info["error"] = repr(e)[:120]
    return info


def usable_cpus():
    """CPUs this process may actually use: min(affinity, cgroup cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(np.ceil(int(quota) / int(period)))))
    except Exception:
        pass
    return max(1, n)


# ----------------------------------------------------------------------------- CPU reference (oracle port)
_W = {}


def _cpu_init(workload, seed_base, ch_per_worker, hops):
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    _W["cfg"] = (workload, seed_base, ch_per_worker, hops)
    _W["data"] = {}


def _cpu_data(idx, shape):
    if idx not in _W["data"]:
        rng = np.random.default_rng(_W["cfg"][1] + idx)
        _W["data"][idx] = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    return _W["data"][idx]


def _cpu_step(idx):
    """One worker's share of a step, the way the reference does it: per channel the spectrogram
    loop (per frame `analyzelive`, friture/spectrogram.py:149-159, then log_spectrogram :161) and
    the octave-spectrum chain per 1024-sample chunk (friture/octavespectrum.py:101-121; the IIR
    recursion runs through the plain-C restatement oracle/iir_df2t.c, bit-identical to the
    reference's pure-Python loop and ~1000x faster -- the literal loop is timed separately)."""
    from oracle import friture_oracle as fo
    workload, _, nch, hops = _W["cfg"]
    acc = 0.0
    units = 0
    if workload in ("combined", "stft"):
        x = _cpu_data(idx, (nch, (hops + 1) * HOP))
        for c in range(nch):
            sp = fo.stft_power(x[c].astype(np.float64), N_FFT, HOP)
            acc += float(fo.log_spectrogram(sp)[0, 0])
            units += sp.shape[0]
    if workload in ("combined", "bank"):
        from friture_b200 import filter_data
        from oracle import iir_c
        n_oct = N_OCT if workload == "combined" else 9
        block = HOP if workload == "combined" else 512
        nblk = hops + 1 if workload == "combined" else hops
        x = _cpu_data(idx, (nch, nblk * block))
        if "bank" not in _W:
            bdec, adec, _ = filter_data.decimator()
            boct, aoct, _ = filter_data.bands(3)
            orc = fo.OctaveSpectrumOracle(bdec, adec, list(boct), list(aoct), noctave=n_oct)
            _W["bank"] = iir_c.BankC(bdec, adec, list(boct), list(aoct), orc.alphas, n_channels=nch,
                                     noctave=n_oct)
        e = _W["bank"].process(x, block)
        acc += float(np.sum(10 * np.log10(e[:, -1] + 1e-30)))
        if workload == "bank":
            units += nch * nblk
    if workload == "gcc":
        rng = np.random.default_rng(idx)
        d0 = rng.standard_normal((nch, 24000))
        d1 = np.roll(d0, 137, axis=1) + 0.1 * rng.standard_normal((nch, 24000))
        for p in range(nch):
            fo.delay_peak(fo.generalized_cross_correlation(d0[p], d1[p]))
        units += nch
    return units, acc


class CpuReference:
    """The CPU path on `workers` processes; one step = every worker's fixed share."""

    SHARE = {"combined": (32, 64), "stft": (32, 128), "bank": (16, 256), "gcc": (8, 0)}

    def __init__(self, workload, workers):
        import multiprocessing as mp
        self.workload, self.workers = workload, workers
        nch, hops = self.SHARE[workload]
        self.pool = mp.get_context("fork").Pool(workers, initializer=_cpu_init,
                                                initargs=(workload, 4321, nch, hops))
        what = {"combined": "%d hops of 1024: per-frame analyzelive + log10, and the 30-band IIR bank "
                            "(C restatement of the reference recursion) + smoothing + dB" % hops,
                "stft": "%d frames (N=2048, hop=1024): per-frame analyzelive loop + log10" % hops,
                "bank": "%d blocks of 512: 27-band IIR bank (C restatement) + smoothing + dB" % hops,
                "gcc": "L=24000 GCC-PHAT + peak pick (numpy.fft, as the reference)"}[workload]
        self.sample = "%d worker processes x %d channels x %s" % (workers, nch, what)

    def step(self):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_step, range(self.workers), chunksize=1)
        return sum(r[0] for r in res), time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def best_cpu_reference(workload):
    """The worker count (one or two per usable CPU) that gives the CPU path its best throughput."""
    ncpu = usable_cpus()
    best = None
    for workers in sorted({ncpu, min(2 * ncpu, os.cpu_count() or ncpu)}):
        ref = CpuReference(workload, workers)
        ref.step()
        n, dt = ref.step()
        if best is None or n / dt > best[1]:
            if best is not None:
                best[0].close()
            best = (ref, n / dt)
        else:
            ref.close()
    best[0].cores = ncpu
    return best[0]


def literal_python_bank_rate():
    """The true cost of the reference's own pure-Python recursion (friture/signal/lfilter.py:131-139),
    one 1024-sample chunk of the 30-band bank on one core."""
    from oracle import friture_oracle as fo
    from friture_b200 import filter_data
    bdec, adec, _ = filter_data.decimator()
    boct, aoct, _ = filter_data.bands(3)
    zis = fo.bank_filtic(bdec, adec, list(boct), list(aoct), noctave=N_OCT)
    y = np.random.default_rng(0).standard_normal(HOP) * 0.1
    t0 = time.perf_counter()
    zi = 0
    for j in range(N_OCT):
        for i in (2, 1, 0):
            fo.lfilter_df2t_loop(boct[i], aoct[i], y, zis[zi]); zi += 1
        yd, _ = fo.lfilter_df2t_loop(bdec, adec, y, zis[zi]); zi += 1
        y = yd[::2]
    return 1.0 / (time.perf_counter() - t0)


WORKLOAD_TEXT = {
    "combined": "configs[4] unit on one GPU: %d ch/GPU x %d hops, 48 kHz: per channel-hop (1024 new samples) one "
                "2048-pt log-power column (50%% overlap) + one 30-band 1/3-octave dB vector (10 octaves, "
                "IIR bank + exponential RMS)",
    "stft": "configs[1]: %d ch/GPU x %d frames, 48 kHz, 2048-pt STFT hop 1024 (50%% overlap) + log-power spectrogram",
    "bank": "configs[2]: %d ch/GPU x %d blocks of 512, 27-band 1/3-octave filterbank (SOS decimator + biquads + RMS, dB)",
    "gcc": "configs[3]: %d channel-pairs/GPU, GCC-PHAT L=24000 (rFFT -> phase -> irFFT -> argmax)%.0s",
}


def workload_config(args, world):
    return {"workload": WORKLOAD_TEXT[args.workload] % (args.channels, args.frames),
            "n_fft": N_FFT, "hop": HOP, "channels_per_gpu": args.channels,
            "hops_per_channel": args.frames, "global_channels": args.channels * world,
            "parallelism": ("channel-sharded x%d" % world) +
                           (", final all-gather of the spectrogram columns over NVLink inside the timed region, "
                            "overlapped with the filterbank" if world > 1 and args.workload == "combined"
                            else ", no data-path collective"),
            "l2_policy": "inputs and outputs of a step (%.2f GB/GPU) are larger than L2; no flush needed"
                         % (args.channels * (args.frames + 1) * HOP * 4 * 2 / 1e9)}


def run_reference_arm(args, rank, world):
    """--impl reference: the CPU path alone.  Under torchrun only rank 0 works."""
    if rank != 0:
        return
    ref = best_cpu_reference(args.workload)
    for _ in range(max(args.warmup, 1)):
        ref.step()
    tot_n, tot_t = 0, 0.0
    for _ in range(args.steps):
        n, dt = ref.step()
        tot_n += n
        tot_t += dt
    ref.close()
    value = tot_n / tot_t
    line = {
        "impl": "reference", "metric": "spectra/sec", "value": value, "unit": "spectra/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "spectra/s", "cores": ref.cores,
                         "workers": ref.workers, "kind": "port", "sample": ref.sample},
        "e2e": {"value": value, "unit": "spectra/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "note": "reference is pure Python/NumPy and cannot travel to the GPU box; this is oracle/, its "
                "validated restatement (same numpy.fft calls and per-frame loop; the IIR recursion through "
                "the bit-identical plain-C port), on all usable host cores",
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU workloads
PROBE_ROWS, PROBE_SEED = 2, 1234


def synth(C, T, dev, seed):
    """Synthetic broadband audio (sigma 0.1), generated in chunks to bound host memory.  The first
    PROBE_ROWS channels are the same on every rank (fixed seed): the parity gate checks them, inside
    the very buffer that is timed, with the strict every-bin criterion -- which a float32 transform
    can only meet on a sample without deep spectral nulls (tests/parity.py), so the sample must not
    change from rank to rank or run to run."""
    import torch
    x = torch.empty((C, T), dtype=torch.float32, device=dev)
    p = min(PROBE_ROWS, C)
    gen = torch.Generator(device="cpu").manual_seed(PROBE_SEED)
    x[:p] = (torch.randn((p, T), generator=gen, dtype=torch.float32) * 0.1).to(dev)
    gen = torch.Generator(device="cpu").manual_seed(seed)
    step = max(1, (32 << 20) // max(T, 1))
    for c0 in range(p, C, step):
        c1 = min(C, c0 + step)
        x[c0:c1] = (torch.randn((c1 - c0, T), generator=gen, dtype=torch.float32) * 0.1).to(dev)
    return x


def strict_rel(got, ref):
    """north_star's criterion: max|got-ref| / max(max|ref|, 1) on the log-power / band-dB vector."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(got - ref)) / max(float(np.max(np.abs(ref))), 1.0))


def event_pair():
    import torch
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


class Combined:
    """configs[4]'s unit: STFT column + 30-band vector per channel-hop; at world > 1 the columns are
    all-gathered inside the step (chunked, overlapped)."""
    name = "combined"
    kernel = "bank_pipe_kernel (filterbank) -- ~90% of the step; stft2048_kernel runs behind it"

    def __init__(self, C, F, dev, rank, world, gather=True, n_oct=N_OCT, transport="peer"):
        import torch
        from friture_b200.analyzer import ChannelAnalyzer
        self.C, self.F, self.dev, self.world = C, F, dev, world
        self.n_oct = n_oct
        self.T = (F + 1) * HOP
        self.an = ChannelAnalyzer(C, N_FFT, HOP, 3, n_oct, device=dev.index)
        self.x = synth(C, self.T, dev, 1234 + rank)
        self.bands = torch.empty((C, F + 1, 3 * n_oct), dtype=torch.float32, device=dev)
        self.gather = gather and world > 1
        self.n_chunks = 8 if F % 8 == 0 else 1
        self.transport, self.engine = (transport.split("-") + ["auto"])[:2]
        if self.gather:
            fc = F // self.n_chunks
            self.spec_chunks = self.gathered = None
            if self.transport == "nccl":
                self.spec_chunks = torch.empty((self.n_chunks, C, fc, NBINS), dtype=torch.float32, device=dev)
                self.gathered = torch.empty((self.n_chunks, world * C, fc, NBINS), dtype=torch.float32, device=dev)
            self.spec = None
        else:
            self.spec = torch.empty((C, F, NBINS), dtype=torch.float32, device=dev)
        self.units = C * F
        # our kernels per step (copy-engine pushes / NCCL kernels are not ours, the push kernel is)
        self.launches_per_step = (1 + self.n_chunks) if self.gather else 2
        if self.gather and self.transport == "peer" and (self.engine == "kernel" or
                                                         (self.engine == "auto" and world > 4)):
            self.launches_per_step += self.n_chunks
        self.bank_events = []

    def step(self, timed=False):
        import torch
        if self.gather:
            self.spec_chunks, _, self.gathered = self.an.process_sharded(
                self.x, self.gathered, self.spec_chunks, self.bands, self.n_chunks, transport=self.transport,
                engine=self.engine)
            return
        if timed:     # the dominant kernel's own duration, on the stream it runs on
            e0, e1 = event_pair()
            self.an.proc.stft(self.x, hop=HOP, log=True, out=self.spec)
            e0.record()
            self.an._bank(self.x, self.bands)
            e1.record()
            self.bank_events.append((e0, e1))
        else:
            self.an.process(self.x, self.spec, self.bands)

    def parity(self):
        """Oracle as checker on a slice of the very buffers being timed (strict criterion)."""
        import torch
        from oracle import friture_oracle as fo
        from friture_b200 import filter_data
        self.an.bank.reset() if self.an.bank._plan_key is not None else None
        self.step()
        torch.cuda.synchronize()
        cs, fs = min(self.C, 2), min(self.F, 16)
        xs = self.x[:cs, :(fs + 1) * HOP].cpu().numpy()
        if self.gather:
            fc = self.F // self.n_chunks
            got_spec = self.spec_chunks[0, :cs, :min(fs, fc)].cpu().numpy()
            fs_spec = min(fs, fc)
        else:
            got_spec = self.spec[:cs, :fs].cpu().numpy()
            fs_spec = fs
        ref_spec = fo.log_spectrogram(fo.stft_power_batch(xs[:, :(fs_spec + 1) * HOP], N_FFT, HOP))
        bdec, adec, _ = filter_data.decimator()
        boct, aoct, _ = filter_data.bands(3)
        ref_b = np.zeros((cs, fs + 1, 3 * self.n_oct))
        for c in range(cs):
            orc = fo.OctaveSpectrumOracle(bdec, adec, list(boct), list(aoct), noctave=self.n_oct)
            for b in range(fs + 1):
                ref_b[c, b] = orc.push(xs[c, b * HOP:(b + 1) * HOP].astype(np.float64))[1]
        got_b = self.bands[:cs, :fs + 1].cpu().numpy()
        res = {"logpower_rel": strict_rel(got_spec, ref_spec), "band_db_rel": strict_rel(got_b, ref_b),
               "criterion": "max|got-ref| / max(max|ref|, 1) < 1e-5 on %d ch x %d hops" % (cs, fs)}
        res["ok"] = res["logpower_rel"] < 1e-5 and res["band_db_rel"] < 1e-5
        if self.gather:
            # the collective: every rank's block of the gathered array equals what that rank computed
            import torch.distributed as dist
            if self.transport == "peer":
                self.an.peer_gather.wait_all()
            g = self.gathered.reshape(self.n_chunks, self.world, self.C, -1)
            mine = float(g[0, dist.get_rank(), 0].double().sum().item())
            sums = [None] * self.world
            dist.all_gather_object(sums, mine)
            got = [float(g[0, r, 0].double().sum().item()) for r in range(self.world)]
            res["gathered_blocks_match"] = bool(all(a == b for a, b in zip(got, sums)))
            res["ok"] = res["ok"] and res["gathered_blocks_match"]
        self.an.bank.reset()
        return res

    def outputs(self):
        """What a caller of the step receives: log-power columns (gathered over the ranks at N > 1)
        and band-level vectors in dB."""
        if self.gather:
            if self.transport == "peer":
                self.an.peer_gather.wait_all()
            return {"spectrogram_logpower_gathered": self.gathered, "bands_db": self.bands}
        return {"spectrogram_logpower": self.spec, "bands_db": self.bands}

    def roofline(self, peak, peak_src):
        ms = [a.elapsed_time(b) for a, b in self.bank_events]
        if not ms:
            return None
        kern_ms = float(np.mean(ms))
        byts = bank_bytes_per_launch(self.C, HOP, self.F + 1, self.n_oct)
        achieved = byts / (kern_ms * 1e-3) / 1e9
        ops = bank_fp32_ops_per_sample(self.n_oct) * self.C * (self.F + 1) * HOP
        issue_peak = SM_COUNT * 128 * SM_MHZ * 1e6
        r = {"bound": "hbm", "kernel": "bank_pipe_kernel<6,1,3,2> (30-band filterbank, the step's dominant kernel)",
             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
             "peak_source": peak_src, "algorithmic_bytes_per_launch": byts,
             "bytes_per_unit": byts / (self.C * (self.F + 1)), "kernel_ms": kern_ms,
             "fp32_lane_ops_per_launch": ops, "fp32_issue_frac": ops / (kern_ms * 1e-3) / issue_peak,
             "note": "the recursion is FP32-issue / dependency-latency bound (SURVEY 8d #3): at 100% FP32 issue "
                     "rate it would sit near 36% of the HBM peak; both fractions are reported"}
        t = traffic_for("bank_pipe_kernel")
        if t and t.get("channels") == self.C and t.get("blocks") == self.F + 1:
            r["traffic"] = t.get("dram_bytes_per_launch")
        return r

    def e2e(self, steps, barrier):
        import torch
        xh = torch.empty((self.C, self.T), dtype=torch.float32, pin_memory=True)
        xh.copy_(self.x)
        sh = torch.empty((self.C, self.F, NBINS), dtype=torch.float32, pin_memory=True)
        bh = torch.empty((self.C, self.F + 1, 3 * self.n_oct), dtype=torch.float32, pin_memory=True)
        self.an.bank.reset()
        self.an.process_host(xh, sh, bh)       # warm-up (allocates the device staging)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.an.process_host(xh, sh, bh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out = {"h2d_bytes_per_step": int(xh.numel() * 4), "d2h_bytes_per_step": int((sh.numel() + bh.numel()) * 4),
               "steps": steps, "api": "ChannelAnalyzer.process_host -> frt_combined_process_host (pinned host in/out)"}
        if self.spec is not None:
            self.an.bank.reset()
            self.an.process_host(xh, sh, bh)
            self.an.bank.reset()
            self.an.process(self.x, self.spec, self.bands)
            torch.cuda.synchronize()
            out["matches_device_path"] = bool(torch.equal(sh[:2, :8], self.spec[:2, :8].cpu()) and
                                              torch.allclose(bh[:2, :8], self.bands[:2, :8].cpu(), rtol=0, atol=2e-4))
        del xh, sh, bh
        return dt, out


class StftOnly:
    """configs[1]: 2048-pt STFT, hop 1024, log-power."""
    name = "stft"

    def __init__(self, C, F, dev, rank, world, **_):
        import torch
        from friture_b200 import audioproc
        from friture_b200._lib import Handle
        self.C, self.F, self.dev = C, F, dev
        self.T = N_FFT + (F - 1) * HOP
        self.proc = audioproc(Handle(dev.index))
        self.proc.set_fftsize(N_FFT)
        self.x = synth(C, self.T, dev, 1234 + rank)
        self.out = torch.empty((C, F, NBINS), dtype=torch.float32, device=dev)
        self.units = C * F
        self.launches_per_step = 1
        self.events = []

    def step(self, timed=False):
        if timed:
            e0, e1 = event_pair()
            e0.record()
            self.proc.stft(self.x, hop=HOP, log=True, out=self.out)
            e1.record()
            self.events.append((e0, e1))
        else:
            self.proc.stft(self.x, hop=HOP, log=True, out=self.out)

    def parity(self):
        import torch
        from oracle import friture_oracle as fo
        self.step()
        torch.cuda.synchronize()
        cs, fs = min(self.C, 4), min(self.F, 32)
        ref = fo.log_spectrogram(fo.stft_power_batch(self.x[:cs, :N_FFT + (fs - 1) * HOP].cpu().numpy(), N_FFT, HOP))
        rel = strict_rel(self.out[:cs, :fs].cpu().numpy(), ref)
        return {"logpower_rel": rel, "ok": rel < 1e-5,
                "criterion": "max|got-ref| / max(max|ref|, 1) < 1e-5 on %d ch x %d frames" % (cs, fs)}

    def outputs(self):
        return {"spectrogram_logpower": self.out}

    def roofline(self, peak, peak_src):
        if not self.events:
            return None
        kern_ms = float(np.mean([a.elapsed_time(b) for a, b in self.events]))
        byts = self.C * self.F * STFT_BYTES_PER_SPECTRUM
        achieved = byts / (kern_ms * 1e-3) / 1e9
        r = {"bound": "hbm", "kernel": "stft2048_kernel<LOGPOWER,VEC>", "achieved": achieved, "peak": peak,
             "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
             "algorithmic_bytes_per_launch": byts, "bytes_per_unit": STFT_BYTES_PER_SPECTRUM, "kernel_ms": kern_ms}
        t = traffic_for("stft2048_kernel")
        if t and t.get("channels") == self.C and t.get("frames") == self.F:
            r["traffic"] = t.get("dram_bytes_per_launch")
        return r

    def e2e(self, steps, barrier):
        import torch
        xh = torch.empty((self.C, self.T), dtype=torch.float32, pin_memory=True)
        xh.copy_(self.x)
        oh = torch.empty((self.C, self.F, NBINS), dtype=torch.float32, pin_memory=True)
        self.proc.stft_host(xh, hop=HOP, log=True, out=oh)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.proc.stft_host(xh, hop=HOP, log=True, out=oh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out = {"h2d_bytes_per_step": int(xh.numel() * 4), "d2h_bytes_per_step": int(oh.numel() * 4), "steps": steps,
               "api": "audioproc.stft_host -> frt_stft_process_host (pinned host in/out)",
               "matches_device_path": bool(torch.equal(oh[:2, :8], self.out[:2, :8].cpu()))}
        del xh, oh
        return dt, out


class BankOnly:
    """configs[2]: 27-band 1/3-octave filterbank + RMS, blocks of 512."""
    name = "bank"

    def __init__(self, C, F, dev, rank, world, n_oct=9, block=512, **_):
        import torch
        from friture_b200.octavefilters import Octave_Filters
        self.C, self.F, self.dev, self.n_oct, self.block = C, F, dev, n_oct, block
        self.bank = Octave_Filters(3, device=dev.index, n_octaves=n_oct)
        self.x = synth(C, F * block, dev, 99 + rank)
        self.units = C * F
        self.launches_per_step = 1
        self.events = []
        self.e = None

    def step(self, timed=False):
        if timed:
            e0, e1 = event_pair()
            e0.record()
            self.e = self.bank.energies_batch(self.x, block=self.block, db=True)
            e1.record()
            self.events.append((e0, e1))
        else:
            self.e = self.bank.energies_batch(self.x, block=self.block, db=True)

    def parity(self):
        import torch
        from oracle import friture_oracle as fo
        self.bank.reset()
        self.step()
        torch.cuda.synchronize()
        cs, fs = min(self.C, 2), min(self.F, 32)
        ref = np.zeros((cs, fs, 3 * self.n_oct))
        xs = self.x[:cs, :fs * self.block].cpu().numpy()
        for c in range(cs):
            orc = fo.OctaveSpectrumOracle(self.bank.bdec, self.bank.adec, self.bank.boct, self.bank.aoct,
                                          noctave=self.n_oct)
            for b in range(fs):
                ref[c, b] = orc.push(xs[c, b * self.block:(b + 1) * self.block].astype(np.float64))[1]
        rel = strict_rel(self.e[:cs, :fs].cpu().numpy(), ref)
        self.bank.reset()
        return {"band_db_rel": rel, "ok": rel < 1e-5,
                "criterion": "max|got-ref| / max(max|ref|, 1) < 1e-5 on %d ch x %d blocks" % (cs, fs)}

    def outputs(self):
        return {"bands_db": self.e}

    def roofline(self, peak, peak_src):
        if not self.events:
            return None
        kern_ms = float(np.mean([a.elapsed_time(b) for a, b in self.events]))
        byts = bank_bytes_per_launch(self.C, self.block, self.F, self.n_oct)
        achieved = byts / (kern_ms * 1e-3) / 1e9
        ops = bank_fp32_ops_per_sample(self.n_oct) * self.C * self.F * self.block
        return {"bound": "hbm", "kernel": "bank_pipe_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": byts, "bytes_per_unit": byts / (self.C * self.F), "kernel_ms": kern_ms,
                "fp32_issue_frac": ops / (kern_ms * 1e-3) / (SM_COUNT * 128 * SM_MHZ * 1e6),
                "note": "FP32-issue / dependency-latency bound recursion, not HBM-bound"}

    def e2e(self, steps, barrier):
        return None, None


class GccOnly:
    """configs[3]: GCC-PHAT delay estimation, L = 24000."""
    name = "gcc"

    def __init__(self, C, F, dev, rank, world, **_):
        import torch
        from friture_b200.correlation import GccPhat
        self.C, self.dev = C, dev
        g = torch.Generator(device="cpu").manual_seed(7 + rank)
        L = 24000
        self.d0 = torch.randn((C, L), generator=g, dtype=torch.float32).to(dev)
        self.d1 = torch.roll(self.d0, 137, 1) + 0.1 * torch.randn((C, L), generator=g, dtype=torch.float32).to(dev)
        self.est = GccPhat(L)
        self.units = C
        self.launches_per_step = 1
        self.events = []

    def step(self, timed=False):
        if timed:
            e0, e1 = event_pair()
            e0.record()
            self.res = self.est.estimate(self.d0, self.d1, smooth=False)
            e1.record()
            self.events.append((e0, e1))
        else:
            self.res = self.est.estimate(self.d0, self.d1, smooth=False)

    def parity(self):
        import torch
        from oracle import friture_oracle as fo
        self.step()
        torch.cuda.synchronize()
        idx = self.res[0]
        ok = bool((idx == 137).all().item())
        xc = fo.generalized_cross_correlation(self.d0[0].cpu().numpy().astype(np.float64),
                                              self.d1[0].cpu().numpy().astype(np.float64))
        i_ref = fo.delay_peak(xc)[0]
        return {"delays_recovered": ok, "argmax_matches_oracle": bool(int(idx[0].item()) == int(i_ref)),
                "ok": ok and int(idx[0].item()) == int(i_ref), "criterion": "identical arg-max (known delay 137)"}

    def outputs(self):
        idx, val, _ = self.res
        return {"delay_index": idx.double(), "peak_value": val}

    def roofline(self, peak, peak_src):
        if not self.events:
            return None
        kern_ms = float(np.mean([a.elapsed_time(b) for a, b in self.events]))
        byts = self.C * 2 * 24000 * 4
        achieved = byts / (kern_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "gcc_phat_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": byts, "bytes_per_unit": 192000, "kernel_ms": kern_ms}

    def e2e(self, steps, barrier):
        return None, None


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(outputs, out_dir):
    """Write each output as <out_dir>/<name>.npy (float32 / float64), DUMP_BYTES in all.  An output
    larger than its share is viewed as rows of its last dimension (of single elements when one such
    row alone exceeds the share) and keeps a fixed, seeded sample of those rows in ascending order,
    written as [rows, width]; two builds run with the same arguments write the same rows."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(outputs) - 4096          # room for the .npy headers
    for name, t in outputs.items():
        if t.numel() * t.element_size() > share:
            width = t.shape[-1] if t.shape[-1] * t.element_size() <= share else 1
            flat = t.reshape(-1, width)
            keep = share // (width * t.element_size())
            rows = np.sort(np.random.default_rng(0).choice(flat.shape[0], keep, replace=False))
            t = flat[torch.from_numpy(rows).to(t.device)]
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


WORKLOADS = {"combined": Combined, "stft": StftOnly, "bank": BankOnly, "gcc": GccOnly}
DEFAULTS = {"combined": (1024, 128), "stft": (256, 4096), "bank": (1024, 256), "gcc": (4096, 0)}


def time_workload(wl, steps, warmup, barrier, world, dev):
    """W warm-up steps, then K steps bracketed by barrier + synchronize; CUDA events; max over ranks."""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        wl.step()
    barrier()
    e0, e1 = event_pair()
    e0.record()
    for _ in range(steps):
        wl.step(timed=True)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps


def quick(cls, C, F, dev, rank, world, barrier, peak, peak_src, reps=5, **kw):
    """A named extra: short timed run of another workload with its own roofline."""
    import torch
    wl = cls(C, F, dev, rank, world, **kw)
    ms = time_workload(wl, reps, 2, barrier, world, dev)
    r = wl.roofline(peak, peak_src) or {}
    out = {"channels_per_gpu": C, "hops_or_frames": F, "ms_per_step": ms, "units_per_s": wl.units * world / (ms * 1e-3),
           "roofline": {k: r.get(k) for k in ("kernel", "achieved", "peak", "frac", "kernel_ms", "fp32_issue_frac",
                                              "bytes_per_unit") if k in r}}
    del wl
    torch.cuda.empty_cache()
    return out


def other_workloads(args, dev, rank, world, barrier, peak, peak_src):
    import torch
    res = {}
    if world == 1:
        res["stft_config1_256ch"] = quick(StftOnly, 256, 4096, dev, rank, world, barrier, peak, peak_src)
        res["bank_config2_27band_block512"] = quick(BankOnly, 1024, 256, dev, rank, world, barrier, peak, peak_src)
        res["gcc_phat_config3_4096pairs"] = quick(GccOnly, 4096, 0, dev, rank, world, barrier, peak, peak_src, reps=3)
        # north_star's channel sweep, combined unit
        sweep = {}
        for C, F in ((1, 128), (256, 128), (1024, 128), (8192, 32)):
            sweep[str(C)] = quick(Combined, C, F, dev, rank, world, barrier, peak, peak_src, reps=3)
        res["combined_channel_sweep"] = sweep
        # the widgets' default FFT sizes (spectrogram 4096, spectrum 8192), 75 % overlap as the widgets use
        from friture_b200 import audioproc
        x = synth(256, 256 * 1024, dev, 5)
        for n_fft in (256, 1024, 4096, 8192):
            pw = audioproc()
            pw.set_fftsize(n_fft)
            hopw = n_fft // 4
            nfr = (x.shape[1] - n_fft) // hopw + 1
            outw = torch.empty((256, nfr, n_fft // 2 + 1), dtype=torch.float32, device=dev)
            pw.stft(x, hop=hopw, log=True, out=outw)
            barrier()
            e0, e1 = event_pair()
            e0.record()
            for _ in range(3):
                pw.stft(x, hop=hopw, log=True, out=outw)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1) / 3
            gbs = 256 * nfr * (hopw + n_fft // 2 + 1) * 4 / (ms * 1e-3) / 1e9
            res["stft_%d_overlap75" % n_fft] = {"channels_per_gpu": 256, "frames_per_channel": nfr, "ms": ms,
                                               "spectra_per_s": 256 * nfr / (ms * 1e-3),
                                               "roofline": {"achieved": gbs, "peak": peak, "frac": gbs / peak}}
            del outw, pw
        res["dropin_1ch"] = dropin_single_channel(dev)
    else:
        # the same step without the collective, and the gather after the spectrum widget's per-tick
        # reduction (one smoothed column per channel and tick instead of one per frame)
        res["combined_no_gather"] = quick(Combined, args.channels, args.frames, dev, rank, world, barrier, peak,
                                          peak_src, reps=5, gather=False)
        auto = "peer-ce" if world <= 4 else "peer-kernel"
        for other in ("nccl", "peer-ce", "peer-kernel"):
            if other != args.transport and not (args.transport == "peer" and other == auto):
                res["combined_gather_via_%s" % other] = quick(Combined, args.channels, args.frames, dev, rank, world,
                                                              barrier, peak, peak_src, reps=5, transport=other)
        from friture_b200.spectrum import SpectrumAnalyzer
        from friture_b200.sharded import allgather_channels
        C, F = args.channels, args.frames
        x = synth(C, N_FFT + (F - 1) * HOP, dev, 77 + rank)
        an = SpectrumAnalyzer(C, fft_size=N_FFT, overlap=0.5, response_time=0.125)
        full_tick = torch.empty((C * world, NBINS), dtype=torch.float32, device=dev)

        def tick():
            db, _, _ = an.process(x)
            allgather_channels(db, C * world, out=full_tick)
        tick()
        barrier()
        e0, e1 = event_pair()
        e0.record()
        for _ in range(5):
            tick()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / 5
        res["spectrum_tick_with_allgather"] = {"channels_per_gpu": C, "frames_per_tick": F, "ms": ms,
                                               "spectra_per_s": C * F * world / (ms * 1e-3),
                                               "note": "gathered payload = one smoothed column per channel per tick"}
    return res


def dropin_single_channel(dev):
    """The literal drop-in calls (one frame / one chunk of one channel, NumPy in and out)."""
    from friture_b200 import audioproc
    from friture_b200.octavefilters import Octave_Filters
    p = audioproc()
    p.set_fftsize(N_FFT)
    x = np.random.default_rng(0).standard_normal(N_FFT)
    for _ in range(20):
        p.analyzelive(x)
    t0 = time.perf_counter()
    for _ in range(200):
        p.analyzelive(x)
    t_an = (time.perf_counter() - t0) / 200
    bank = Octave_Filters(3)
    xb = np.random.default_rng(1).standard_normal(512)
    for _ in range(5):
        bank.filter(xb)
    t0 = time.perf_counter()
    for _ in range(50):
        bank.filter(xb)
    t_f = (time.perf_counter() - t0) / 50
    return {"analyzelive_us_per_call": 1e6 * t_an, "octave_filter_us_per_512_chunk": 1e6 * t_f,
            "note": "one channel, one frame/chunk per call: launch + copy latency dominates; the reference's NumPy "
                    "analyzelive takes ~16 us, its FFT-OLA filter() ~390 us (SURVEY 6) -- the GPU path pays off on "
                    "the batched entry points"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="combined", choices=sorted(WORKLOADS))
    ap.add_argument("--channels", type=int, default=None, help="channels (pairs for gcc) per GPU")
    ap.add_argument("--frames", type=int, default=None, help="hops / frames / blocks per channel per step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-gather", action="store_true", help="N > 1: leave the all-gather out of the step")
    ap.add_argument("--transport", default="peer", choices=["peer", "peer-ce", "peer-kernel", "nccl"],
                    help="N > 1: one-hop pushes over NVLink peer memory (default; copy engines at 2 GPUs, a copy "
                         "kernel above 4) or NCCL all-gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")
    dC, dF = DEFAULTS[args.workload]
    args.channels = args.channels or dC
    args.frames = dF if args.frames is None else args.frames

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    placement = bind_to_gpu_numa(local_rank)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; friture_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from friture_b200 import _lib
    wl = WORKLOADS[args.workload](args.channels, args.frames, dev, rank, world, gather=not args.no_gather,
                                  transport=args.transport)
    perr = wl.parity()
    if not perr.get("ok"):
        raise SystemExit("bench.py: parity gate failed: %r" % (perr,))

    # ---- device-resident timing
    for _ in range(args.warmup):
        wl.step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    e0, e1 = event_pair()
    t_wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        wl.step(timed=True)
    e1.record()
    barrier()
    t_wall1 = time.time()
    total_ms = e0.elapsed_time(e1)
    time.sleep(0.2)
    sampler.stop()
    clocks = sampler.summary(t_wall0, t_wall1)
    if args.dump_outputs:       # before the e2e and extra runs reuse the buffers
        outs = wl.outputs()
        if rank == 0:
            dump_outputs(outs, args.dump_outputs)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = wl.units * world / (ms_per_step * 1e-3)
    peak, peak_src = load_peaks()
    roofline = wl.roofline(peak, peak_src)
    if world > 1 and args.workload == "combined" and not args.no_gather:
        recv = wl.units * NBINS * 4 * (world - 1)
        roofline = {"bound": "hbm", "kernel": "all-gather of the spectrogram columns over NVLink (%s), link-bound step"
                              % ("one-hop pushes into peer memory" if args.transport.startswith("peer") else "NCCL"),
                    "achieved": recv / (ms_per_step * 1e-3) / 1e9, "peak": 770.0, "unit": "GB/s",
                    "frac": recv / (ms_per_step * 1e-3) / 1e9 / 770.0, "traffic": None,
                    "peak_source": "measured NVLink peer copy, GB/s per direction per GPU (B200_PROFILING.md)",
                    "note": "at N > 1 the step is bounded by NVLink ingress: every GPU receives (N-1)/N of all columns; "
                            "achieved = bytes received per GPU per step / step time"}

    # ---- end to end through the public API with pinned host buffers
    e2e = None
    if not args.no_e2e:
        dt, e2e = wl.e2e(args.e2e_steps, barrier)
        if e2e is not None:
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
            e2e = dict({"value": wl.units * world * args.e2e_steps / dt, "unit": "spectra/s",
                        "ms_per_step": 1e3 * dt / args.e2e_steps, "host_placement": placement}, **e2e)
            e2e["pcie_note"] = ("PCIe-bound: %.2f GB in + %.2f GB out per step and GPU at ~50 GB/s each way"
                                % (e2e["h2d_bytes_per_step"] / 1e9, e2e["d2h_bytes_per_step"] / 1e9))

    launches = wl.launches_per_step * args.steps
    others = {}
    if not args.no_others:
        others = other_workloads(args, dev, rank, world, barrier, peak, peak_src)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = best_cpu_reference(args.workload)
        n, dt = ref.step()
        n2, dt2 = ref.step()
        ref.close()
        cpu_baseline = {"value": (n + n2) / (dt + dt2), "unit": "spectra/s", "cores": ref.cores,
                        "workers": ref.workers, "kind": "port", "sample": ref.sample}
        if args.workload in ("combined", "bank") and not args.no_others:
            cpu_baseline["literal_python_recursion_30band_chunks_per_s_1core"] = literal_python_bank_rate()

    if rank == 0:
        line = {
            "metric": "spectra/sec", "value": value, "unit": "spectra/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, world),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches), "parity": perr, "other_workloads": others,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
