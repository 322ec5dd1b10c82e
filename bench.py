#!/usr/bin/env python
"""bench.py — headline benchmark of the librosa FFT time-frequency hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg3|cfg4|cfg5|stats|speech400]
                    [--dump-outputs DIR]

Metric (BASELINE.json): mel-spectrogram frames/sec, n_fft=2048, hop=512, n_mels=128, float32, on
BASELINE.json configs[1] — batch = 1024 clips x 10 s mono @ 22050 Hz per GPU.  One "step" is one pass of
the fused stft -> |.|^2 -> mel kernel over that batch.  Weak scaling: every rank owns a 1024-clip shard,
no collective on the data path; `value` = frames of all ranks / max-over-ranks device time.

One JSON line on stdout (rank 0).  Extra keys beyond the base contract:
  roofline      dominant kernel vs the measured HBM peak (MEASURED_PEAKS.json), algorithmic bytes
  cpu_baseline  the oracle port (oracle/ref_np.py == the reference's algorithm, bit-exact here) timed on
                this box's host cores on a bounded sample: the three ways SURVEY 8d lists (batched call /
                one-process loop / forked workers), best reported, all listed under `variants`
  e2e           same metric through the public drop-in call with HOST (pinned) buffers, H2D + D2H inside;
                `pageable` = the same call on an ordinary ndarray; `h2d_ceiling_gbs_per_gpu` = plain upload
                bandwidth with every rank transferring at once (the floor of the end-to-end step)
  secondary     device-resident ms / frames/s / roofline of BASELINE.json configs 3, 4, 5 (per-GPU shards) and of the
                n_fft = 400 speech front end (`speech400`, mixed-radix kernel; not a BASELINE.json config)
  clocks        NVML samples taken during the timed region

--dump-outputs DIR writes what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float32: whole
clips picked by a fixed seed, as many as fit in 64 MB; complex spectra get a trailing (real, imag) axis.  The
inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (clips per GPU, channels, samples, sr, op, kwargs, algorithmic bytes per frame (SURVEY §8d))
    "cfg2": dict(clips=1024, n=220500, sr=22050, op="mel", kw=dict(n_fft=2048, hop_length=512, n_mels=128, power=2.0),
                 desc="batch=1024 clips x10s mono sr=22050 -> melspectrogram n_fft=2048 hop=512 n_mels=128 power=2.0"),
    "cfg3": dict(clips=2048, n=441000, sr=44100, op="stft", kw=dict(n_fft=4096, hop_length=1024),
                 desc="2048 channel-clips (1024 stereo, 1/8 of batch=8192) x10s sr=44100 -> stft n_fft=4096 hop=1024 per GPU"),
    "cfg4": dict(clips=512, n=480000, sr=16000, op="mfcc", kw=dict(n_mfcc=40, n_mels=128, n_fft=1024, hop_length=256),
                 desc="512 clips x30s mono sr=16000 -> mfcc n_mfcc=40 n_mels=128 n_fft=1024 hop=256 per GPU"),
    # SURVEY 8f rank 2: frame-wise statistics fused with the stft (cfg-2 shapes); one launch yields all six rows
    "stats": dict(clips=1024, n=220500, sr=22050, op="centroid", kw=dict(n_fft=2048, hop_length=512),
                  desc="batch=1024 clips x10s mono sr=22050 -> spectral_centroid n_fft=2048 hop=512 (fused statistics kernel)"),
    "cfg5": dict(clips=256, n=220500, sr=22050, op="roundtrip", kw=dict(n_fft=2048, hop_length=512),
                 desc="256 clips x10s -> stft -> istft n_fft=2048 hop=512 per GPU"),
    # not a BASELINE.json config: the 25 ms / 10 ms / 80-band log-mel front end of speech models (n_fft is not a power
    # of two: mixed-radix kernel, csrc/mr_kernel.cuh)
    "speech400": dict(clips=1024, n=160000, sr=16000, op="mel", kw=dict(n_fft=400, hop_length=160, n_mels=80, power=2.0),
                      desc="1024 clips x10s mono sr=16000 -> melspectrogram n_fft=400 hop=160 n_mels=80 per GPU"),
}
METRIC = "mel-spectrogram frames/sec (n_fft=2048,hop=512,n_mels=128)"
OUTPUT_NAMES = {"mel": "melspectrogram", "stft": "stft", "mfcc": "mfcc", "centroid": "spectral_centroid",
                "roundtrip": "istft"}
DUMP_BYTES = 60 * 10**6         # under 64 MB however MB is counted, .npy header included


def n_frames(n, n_fft, hop):
    return 1 + n // hop   # center=True, even n_fft (SURVEY Appendix A.1)


def algorithmic_bytes_per_step(w):
    """Compulsory HBM traffic of one step: every input sample read once + every output element written once."""
    T = n_frames(w["n"], w["kw"]["n_fft"], w["kw"]["hop_length"])
    F = 1 + w["kw"]["n_fft"] // 2
    clips, n = w["clips"], w["n"]
    if w["op"] == "mel":
        return clips * (4 * n + 4 * w["kw"]["n_mels"] * T)
    if w["op"] == "stft":
        return clips * (4 * n + 8 * F * T)
    if w["op"] == "mfcc":
        return clips * (4 * n + 4 * w["kw"]["n_mfcc"] * T)
    if w["op"] == "roundtrip":
        return clips * (4 * n + 8 * F * T) + clips * (8 * F * T + 4 * n)
    if w["op"] == "centroid":
        return clips * (4 * n + 4 * 6 * T)      # six statistics rows per frame
    raise ValueError(w["op"])


def make_batch(w, rank):
    import signals

    base = signals.make("A", (64, w["n"]), seed=1000 * rank)       # mix A: 0.1 * N(0,1), SURVEY §8d
    reps = -(-w["clips"] // 64)
    scale = (1.0 + 0.01 * np.arange(reps, dtype=np.float32))[:, None, None]
    return np.ascontiguousarray((base[None] * scale).reshape(-1, w["n"])[: w["clips"]])


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profiled_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture, if any."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    try:
        with open(path) as fh:
            return json.load(fh).get(workload)
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 5 ms from a background thread while the
    timed region runs (nvidia-smi -lms cannot sample a region that lasts tens of milliseconds)."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, device):
        import threading

        self.samples, self.bits, self.max_mhz, self.power = [], 0, None, []
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            self._stop.wait(0.005)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._thread is None:
            return out
        self._stop.set()
        self._thread.join(timeout=2)
        if self.samples:
            out.update(sm_mhz=statistics.median(self.samples), samples=len(self.samples),
                       reasons=sorted(k for k, bit in self.REASONS.items() if self.bits & bit),
                       power_w_max=max(self.power) if self.power else None)
        return out


# ------------------------------------------------------------------------------------------- CPU port
_CPU_BATCH = None      # the sample batch; forked workers inherit it (no per-step pickling of audio)


def _cpu_one(op, kw, sr, y):
    from oracle import ref_np as O

    if op == "mel":
        return O.melspectrogram(y=y, sr=sr, **kw).shape[-1]
    if op == "stft":
        return O.stft(y, **kw).shape[-1]
    if op == "mfcc":
        return O.mfcc(y=y, sr=sr, **kw).shape[-1]
    if op == "centroid":
        return O.spectral_centroid(y=y, sr=sr, **kw).shape[-1]
    D = O.stft(y, **kw)
    O.istft(D, hop_length=kw["hop_length"], length=y.shape[-1])
    return D.shape[-1]


def _cpu_range_job(args):
    """A worker's share of one pass: the clips [lo, hi) of the inherited batch, one reference call per clip."""
    op, kw, sr, lo, hi = args
    return sum(_cpu_one(op, kw, sr, _CPU_BATCH[i]) for i in range(lo, hi))


def _cpu_worker_init():
    # one BLAS / OpenMP thread per worker process: the pool already uses every core
    global _BLAS_LIMIT
    try:
        import threadpoolctl

        _BLAS_LIMIT = threadpoolctl.threadpool_limits(limits=1)
    except Exception:
        _BLAS_LIMIT = None


def cpu_quota():
    """CPU time this container may use, in cores (cgroup v2 cpu.max / v1 cfs quota), or None if unlimited."""
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()[:2]
        if quota != "max":
            return float(quota) / float(period)
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as fh:
            quota = float(fh.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fh:
            period = float(fh.read())
        if quota > 0:
            return quota / period
    except Exception:
        pass
    return None


class CpuPort:
    """The reference's algorithm (oracle port, bit-exact with librosa here) on the host cores, the three ways
    SURVEY 8d lists: (i) one batched call, BLAS threads = all cores; (ii) per-clip loop in one process;
    (iii) per-clip loop over persistent forked workers reading the clips of a batch they inherited at fork
    (>= 4 clips per core and pass, jobs are clip indices, one BLAS thread each)."""

    def __init__(self, w, clips_per_core=4, min_clips=64):
        import multiprocessing as mp

        global _CPU_BATCH
        self.w = w
        self.visible = len(os.sched_getaffinity(0)) or (os.cpu_count() or 1)
        self.quota = cpu_quota()
        # a container may show every core of the box and still be throttled to a few cores' worth of time
        # (cgroup cpu.max): more workers than that only adds context switches
        self.cores = self.visible if self.quota is None else max(1, min(self.visible, int(round(self.quota))))
        if os.environ.get("B2L_CPU_WORKERS"):
            self.cores = max(1, int(os.environ["B2L_CPU_WORKERS"]))
        self.clips = max(min_clips, clips_per_core * self.cores)
        _CPU_BATCH = make_batch(dict(w, clips=self.clips), rank=0)
        self.T = n_frames(w["n"], w["kw"]["n_fft"], w["kw"]["hop_length"])
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_worker_init)
        # one clip per job, >= 4 jobs per core and pass: idle workers pull the next clip index (a few bytes)
        self.jobs = [(w["op"], w["kw"], w["sr"], i, i + 1) for i in range(self.clips)]
        self.pool.map(_cpu_range_job, [(w["op"], w["kw"], w["sr"], 0, 1)] * self.cores, chunksize=1)   # imports, FFT plans

    def step_pool(self):
        t0 = time.perf_counter()
        frames = sum(self.pool.map(_cpu_range_job, self.jobs, chunksize=1))
        return frames, time.perf_counter() - t0

    def step_loop(self, k):
        w = self.w
        t0 = time.perf_counter()
        frames = sum(_cpu_one(w["op"], w["kw"], w["sr"], _CPU_BATCH[i]) for i in range(k))
        return frames, time.perf_counter() - t0

    def step_batched(self, k):
        w = self.w
        t0 = time.perf_counter()
        frames = k * _cpu_one(w["op"], w["kw"], w["sr"], _CPU_BATCH[:k])
        return frames, time.perf_counter() - t0

    def variants(self, small=32):
        """frames/s of the three ways on this box (a warm-up of each first; (i) and (ii) on `small` clips)."""
        out = {}
        k = min(small, self.clips)
        self.step_batched(min(4, k))
        f, s = self.step_batched(k)
        out["batched_call_all_blas_threads"] = f / s
        self.step_loop(2)
        f, s = self.step_loop(min(16, k))
        out["per_clip_loop_1_process"] = f / s
        self.step_pool()
        f, s = self.step_pool()
        out[f"per_clip_loop_{self.cores}_forked_workers"] = f / s
        return out

    def describe(self, variants):
        return (f"{self.clips} clips of the workload per pass ({self.clips // self.cores} per worker), {self.cores} persistent "
                f"forked workers ({self.visible} CPUs visible, cgroup quota "
                f"{'none' if self.quota is None else '%.1f cores' % self.quota}) read a fork-inherited batch; variants frames/s: "
                + ", ".join(f"{k}={v:.0f}" for k, v in variants.items()))

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_measure(w, seconds):
    """Best of the three SURVEY 8d variants, the pool variant re-timed for `seconds`."""
    port = CpuPort(w)
    var = port.variants()
    f = s = 0.0
    t_end = time.perf_counter() + seconds
    while True:
        fi, si = port.step_pool()
        f += fi
        s += si
        if time.perf_counter() > t_end:
            break
    pool_key = [k for k in var if k.endswith("forked_workers")][0]
    var[pool_key] = f / s
    best = max(var, key=var.get)
    out = {"value": var[best], "unit": "frames/s", "cores": port.cores, "cpus_visible": port.visible,
           "cgroup_cpu_quota": port.quota, "kind": "port", "best_variant": best,
           "variants": var, "sample": port.describe(var)}
    port.close()
    return out


def run_reference(args, w, rank, world):
    if rank != 0:
        return
    port = CpuPort(w)
    var = port.variants()
    best = max(var, key=var.get)
    if best.startswith("batched"):
        step = lambda: port.step_batched(min(64, port.clips))
    elif best.startswith("per_clip_loop_1_"):
        step = lambda: port.step_loop(min(32, port.clips))
    else:
        step = port.step_pool
    for _ in range(max(1, args.warmup)):
        step()
    frames = secs = 0.0
    for _ in range(args.steps):
        f, s = step()
        frames += f
        secs += s
    value = frames / secs
    var[best] = value
    line = {
        "impl": "reference", "metric": METRIC if w["op"] == "mel" else f"{w['op']} frames/sec", "value": value,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 in / f64 FFT (reference numerics)", "data": "synthetic",
        "config": {"workload": w["desc"], "name": args.workload},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": port.cores, "cpus_visible": port.visible,
                         "cgroup_cpu_quota": port.quota, "kind": "port",
                         "best_variant": best, "variants": var, "sample": port.describe(var)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    port.close()
    emit(line)


# ------------------------------------------------------------------------------------------- GPU arm
def make_steps(lb, w, dev, host):
    kw, op, sr = w["kw"], w["op"], w["sr"]

    def step_resident():
        """One step on the device-resident batch; returns the result (a DeviceArray the caller frees)."""
        if op == "mel":
            return lb.feature.melspectrogram(y=dev, sr=sr, **kw)
        if op == "stft":
            return lb.stft(dev, **kw)
        if op == "mfcc":
            return lb.feature.mfcc(y=dev, sr=sr, **kw)
        if op == "centroid":
            return lb.feature.spectral_centroid(y=dev, sr=sr, **kw)
        D = lb.stft(dev, **kw)
        y = lb.istft(D, hop_length=kw["hop_length"], length=w["n"])
        D.free()
        return y

    def step_e2e(src=None):
        y = host if src is None else src
        if op == "mel":
            return lb.feature.melspectrogram(y=y, sr=sr, **kw)
        if op == "stft":
            return lb.stft(y, **kw)
        if op == "mfcc":
            return lb.feature.mfcc(y=y, sr=sr, **kw)
        if op == "centroid":
            return lb.feature.spectral_centroid(y=y, sr=sr, **kw)
        return lb.istft(lb.stft(y, **kw), hop_length=kw["hop_length"], length=w["n"])

    return step_resident, step_e2e


def dump_outputs(out, name, directory):
    """Copy a seeded sample of whole clips of the device result ``out`` (clips leading) to DIR/<name>.npy."""
    from librosa_b200 import _native as nat

    n_clips = out.shape[0]
    clip_bytes = out.nbytes // n_clips
    clips = np.sort(np.random.default_rng(0).choice(n_clips, min(n_clips, DUMP_BYTES // clip_bytes), replace=False))
    rows = []
    for c in clips:
        view = nat.DeviceArray(out.ctx, out.ptr + int(c) * clip_bytes, out.shape[1:], out.dtype, layout=out.layout,
                               owner=False)
        host = view.get(out=np.empty(view._mem_shape(), out.dtype))
        rows.append(np.stack([host.real, host.imag], axis=-1) if host.dtype.kind == "c" else host)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, f"{name}.npy"), np.stack(rows).astype(np.float32))


KERNEL_NAMES = {"mel": "fwd_kernel<10,32,16,MODE_MEL>", "stft": "fwd_kernel<.,.,.,MODE_STFT>",
                "mfcc": "fwd_kernel<.,.,.,MODE_MEL>+dct_clamp_kernel", "roundtrip": "fwd_kernel+inv_kernel",
                "centroid": "fwd_kernel<10,32,16,MODE_STATS>"}


def run_ours(args, w, rank, world, local_rank):
    import librosa_b200 as lb

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    # one process per GPU: keep this process (and the pinned buffers it allocates) on the CPUs local to its GPU,
    # as `numactl --cpunodebind` would; released again before the CPU baseline uses every core
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = None if os.environ.get("B2L_BENCH_NO_NUMA_BIND") else lb.bind_host_to_device(local_rank)
    ctx = lb.default_context(local_rank)

    def barrier():
        ctx.synchronize()
        if dist is not None:
            dist.barrier()
            import torch

            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch

        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peak, peak_src = measured_peak()

    def resident(wl, steps, warmup, sample_clocks):
        """Device-resident timing of one workload: (ms per step max over ranks, launches, clocks, frames per GPU,
        result of the last timed step)."""
        T = n_frames(wl["n"], wl["kw"]["n_fft"], wl["kw"]["hop_length"])
        host = lb.pinned_empty((wl["clips"], wl["n"]), np.float32)
        host[...] = make_batch(wl, rank)
        dev = ctx.to_device(host)
        step_resident, step_e2e = make_steps(lb, wl, dev, host)
        for _ in range(max(3, warmup)):
            step_resident().free()
        barrier()
        sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks) else None
        launches0 = ctx.launch_count
        e0, e1 = ctx.event(), ctx.event()
        out = None
        e0.record()
        for _ in range(steps):
            if out is not None:
                out.free()
            out = step_resident()
        e1.record()
        ms = e0.elapsed_ms(e1)
        barrier()
        launches = ctx.launch_count - launches0
        clocks = sampler.stop() if sampler else None
        ms_per_step = max_over_ranks(ms) / steps
        return dict(ms_per_step=ms_per_step, launches=launches, clocks=clocks, frames=wl["clips"] * T, host=host,
                    dev=dev, step_e2e=step_e2e, out=out)

    def roofline_of(wl, ms_per_step, name):
        alg_bytes = algorithmic_bytes_per_step(wl)
        achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": profiled_traffic(name), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel": "mr_kernel<2> (mixed radix 5,5,8)" if name == "speech400" else KERNEL_NAMES[wl["op"]],
                "note": "kernel time == step time (CUDA events on the launching stream); bytes = inputs read once + outputs written once"}

    # ---- device-resident: warm-up, then K steps between events (inputs 0.9 GB >> 126 MB L2: no flush needed)
    r = resident(w, args.steps, args.warmup, True)
    ms_per_step, launches, clocks, frames_per_step = r["ms_per_step"], r["launches"], r["clocks"], r["frames"]
    host, dev, step_e2e = r["host"], r["dev"], r["step_e2e"]
    value = world * frames_per_step / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(r["out"], OUTPUT_NAMES[w["op"]], args.dump_outputs)
    r["out"].free()

    # ---- end to end through the public call with host buffers (H2D + D2H inside the timed region)
    def time_e2e(src, steps):
        out = step_e2e(src)                   # warm-up: second stream, plans, device and pinned pools
        nbytes = int(out.nbytes)
        out2 = step_e2e(src)                  # a second result while the first is alive: both pinned buffers exist
        del out, out2
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = step_e2e(src)
        ctx.synchronize()
        sec = (time.perf_counter() - t0) / steps
        del out
        return max_over_ranks(sec), nbytes

    e2e_steps = max(3, min(args.steps, 10))
    e2e_s, d2h = time_e2e(host, e2e_steps)
    e2e_value = world * frames_per_step / e2e_s
    # the same call on a PAGEABLE ndarray (what a drop-in user passes): the library stages it through pinned
    # buffers with several host threads (b2l_h2d -> staged_h2d)
    pageable = np.array(host)               # ordinary malloc'ed copy
    e2e_pg_s, _ = time_e2e(pageable, max(3, e2e_steps // 2))
    del pageable
    # PCIe upload ceiling with every rank transferring at once: explains the end-to-end scaling
    import ctypes as C

    from librosa_b200 import _native as nat

    probe = ctx.empty(host.shape, np.float32)
    nat.check(nat.lib().b2l_h2d(ctx.handle, C.c_void_p(probe.ptr), host.ctypes.data_as(C.c_void_p), host.nbytes))
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        nat.check(nat.lib().b2l_h2d(ctx.handle, C.c_void_p(probe.ptr), host.ctypes.data_as(C.c_void_p), host.nbytes))
    ctx.synchronize()
    h2d_gbs = 3 * host.nbytes / max_over_ranks(time.perf_counter() - t0) / 1e9
    probe.free()
    h2d_bytes = int(host.nbytes)
    dev.free()
    del host

    # ---- split / join over NVLink through the product's own NCCL path (b2l_comm_*, rendezvous over TCP, no
    # torch): rank 0 holds the whole device-resident batch, scatters the shards, every rank runs its shard,
    # rank 0 gathers the mel spectrograms.  Timed with CUDA events on rank 0's stream, max over ranks.
    join = None
    if world > 1 and not args.no_join and w["op"] == "mel":
        from librosa_b200 import distributed as D

        comm = D.init_from_env(ctx)
        T = n_frames(w["n"], w["kw"]["n_fft"], w["kw"]["hop_length"])
        shard = ctx.empty((w["clips"], w["n"]), np.float32)
        full_in = full_out = None
        if rank == 0:
            full_in = ctx.empty((world * w["clips"], w["n"]), np.float32)
            one = ctx.to_device(make_batch(w, 0))
            for r_ in range(world):
                lb.device_copy(ctx, full_in, r_ * one.nbytes, one)
            one.free()
            full_out = ctx.empty((world * w["clips"], w["kw"]["n_mels"], T), np.float32)

        def join_step():
            comm.scatter(full_in, shard)
            M = lb.feature.melspectrogram(y=shard, sr=w["sr"], **w["kw"])
            comm.gather(M, full_out)
            M.free()

        for _ in range(3):
            join_step()
        barrier()
        js = max(3, min(args.steps, 10))
        e0, e1 = ctx.event(), ctx.event()
        e0.record()
        for _ in range(js):
            join_step()
        e1.record()
        jms = max_over_ranks(e0.elapsed_ms(e1)) / js
        barrier()
        comm.close()
        shard.free()
        if rank == 0:
            full_in.free()
            full_out.free()
        moved = (world - 1) * (w["clips"] * w["n"] * 4 + w["clips"] * w["kw"]["n_mels"] * T * 4)
        join = {"mode": "nccl scatter -> mel -> nccl gather (b2l_comm_*, root = rank 0)", "ms_per_step": jms,
                "value": world * frames_per_step / (jms * 1e-3), "unit": "frames/s",
                "nvlink_bytes_per_step": moved, "nvlink_gbs_at_root": moved / (jms * 1e-3) / 1e9}

    # ---- the other BASELINE.json configs, device-resident (driver-recorded secondary numbers)
    secondary = []
    if not args.no_secondary and args.workload == "cfg2":
        for name in ("cfg3", "cfg4", "cfg5", "speech400"):
            wl = WORKLOADS[name]
            try:
                rr = resident(wl, max(5, args.steps // 2), 3, False)
            except Exception as exc:                      # e.g. not enough free HBM next to another job
                secondary.append({"name": name, "error": repr(exc)[:200]})
                continue
            rr["dev"].free()
            rr["out"].free()
            ms2 = rr["ms_per_step"]
            secondary.append({"name": name, "workload": wl["desc"], "metric": f"{wl['op']} frames/sec",
                              "value": world * rr["frames"] / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2,
                              "per_gpu_clips": wl["clips"], "gpu_launches": rr["launches"],
                              "roofline": roofline_of(wl, ms2, name)})
            del rr
        ctx.empty_cache()

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    roofline = roofline_of(w, ms_per_step, args.workload)

    # ---- CPU baseline on this box (bounded sample)
    cpu = None
    if numa_cpus:
        os.sched_setaffinity(0, all_cpus)
    if world == 1 and not args.no_cpu:
        cpu = cpu_measure(w, 10.0)

    op = w["op"]
    line = {
        "metric": METRIC if op == "mel" else f"{op} frames/sec", "value": value, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "name": args.workload, "per_gpu_clips": w["clips"],
                   "frames_per_step_per_gpu": frames_per_step, "parallelism": f"clips sharded x{world}, no collective",
                   "host_cpus_bound_to_gpu": len(numa_cpus) if numa_cpus else None,
                   "l2": "inputs (%.0f MB per step) exceed the 126 MB L2; no flush" % (w["clips"] * w["n"] * 4 / 1e6)},
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s * 1e3,
                "path": "librosa_b200 public call on a pinned host ndarray -> ndarray",
                "pageable": {"value": world * frames_per_step / e2e_pg_s, "ms_per_step": e2e_pg_s * 1e3,
                             "path": "same call on an ordinary (pageable) ndarray; staged upload inside the library"},
                "h2d_ceiling_gbs_per_gpu": h2d_gbs,
                "h2d_floor_ms": h2d_bytes / (h2d_gbs * 1e9) * 1e3},
        "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary, "join": join,
    }
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else that libraries print on file
    descriptor 1 while the benchmark runs (NCCL's version banner, torchrun notices) was redirected to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg3 / cfg4 / cfg5 / speech400 secondary numbers")
    ap.add_argument("--no-join", action="store_true", help="skip the NCCL scatter -> mel -> gather leg (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's result to "
                                                           "DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w, rank, world)
    else:
        run_ours(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
