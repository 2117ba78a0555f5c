#!/usr/bin/env python
"""Benchmark of the phase-retrieval hot path on B200: headline = batched fast Griffin-Lim (BASELINE.json configs[1]),
plus every other named config and the communicating (frame-sharded) path in a `configs` object of the same line.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (torchrun launches N ranks)
    python bench.py --impl reference --gpus N --steps K ...  # the unmodified reference on the host CPUs
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's output (see dump_outputs)

Headline: a *step* is one whole griffin_lim job over one batch of synthetic magnitudes,
    griffin_lim(mag, max_iter=64, alpha=0.99, tol=0, eva_iter=10, hop_length=256, window=hann(1024))
with mag = |STFT| of B=512 unit-variance noise signals of 10 s @ 24 kHz (spec 512 x 513 x 938): the real-magnitude
entry of the public API (one-shot phase_init, 64 fused iterations, 6 metric evaluations).
metric = audio-seconds x iterations / second, whole job over all N GPUs (batch-sharded, weak scaling: every rank runs
its own B=512 batch; the path needs no collective).

  value        : inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          : the same call with HOST (pinned) input and output, copies inside the timed region; value from the MEAN
                 step, median / p95 / max beside it
  roofline     : fused GL-iteration kernel, algorithmic bytes 20*B*F*T + 8*B*L per launch / event-timed average
                 launch duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline : the unmodified reference (baseline/_ref) on the host CPUs on a bounded sample of the workload (the
                 oracle port beside it, or alone when the reference is not installed); `parity` compares the final
                 spectral convergence of the GPU run, the reference and the CPU port on that same sample
  reference_cuda : the unmodified reference (baseline/_ref) with device='cuda' on the same inputs (cuFFT + cuDNN)
  configs      : cfg1 / cfg3 / cfg4 / cfg5 of BASELINE.json (ms per job, per iteration, audio-s*it/s, roofline
                 fraction); for N > 1: cfg2 STRONG-scaled (B = 512 / N per rank), cfg3 / cfg4 batch-sharded, and cfg5
                 FRAME-SHARDED over the N ranks through the NVLink peer-memory halo exchange (ms / iteration, speed-up
                 over one GPU, exchange time, boundary checks); `generic400`: the generic (mixed-radix) path at
                 torchaudio's default transform, with the reference's CUDA path on the same inputs beside it
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "audio_seconds_x_iterations_per_second"
UNIT = "audio-s*it/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

WORKLOADS = {
    # BASELINE.json configs[0..4]; sizes as in SURVEY.md section 8 (T = 1 + N // hop)
    "cfg1": dict(algo="gl", B=1, N=661500, sr=22050, n_fft=2048, hop=512, iters=100, coef=0.3,
                 desc="griffin_lim one 30 s @ 22.05 kHz signal, n_fft=2048 hop=512 hann, 100 iters, alpha=0.3"),
    "cfg2": dict(algo="gl", B=512, N=240000, sr=24000, n_fft=1024, hop=256, iters=64, coef=0.99,
                 desc="batched griffin_lim B=512 x 10 s @ 24 kHz, n_fft=1024 hop=256 hann, 64 iters, alpha=0.99, "
                      "tol=0, eva_iter=10 (the metric sums are computed on every 10th iteration as in the reference; at "
                      "tol=0 with verbose off nothing can observe them, so the host does not wait for them), "
                      "real-magnitude input (phase_init inside)"),
    "cfg3": dict(algo="rtisi", B=256, N=240000, sr=24000, n_fft=1024, hop=256, iters=25, coef=0.99, look_ahead=3,
                 desc="RTISI_LA B=256 x 10 s @ 24 kHz, n_fft=1024 hop=256 hann, look_ahead=3, max_iter=25, alpha=0.99"),
    "cfg4": dict(algo="admm", B=128, N=882000, sr=44100, n_fft=2048, hop=512, iters=100, coef=0.1,
                 desc="ADMM B=128 x 20 s @ 44.1 kHz, n_fft=2048 hop=512 hann, 100 iters, rho=0.1"),
    "cfg5": dict(algo="gl", B=1, N=172800000, sr=48000, n_fft=4096, hop=1024, iters=100, coef=0.99,
                 desc="griffin_lim one 1 h @ 48 kHz signal, n_fft=4096 hop=1024 hann, 100 iters, alpha=0.99"),
    # not a BASELINE config: the GENERIC path (mixed-radix team kernels, csrc/specinv_generic_mr.cu) at torchaudio's
    # default transform (n_fft=400, hop=200), reported beside the reference's own CUDA path on the same inputs
    "generic400": dict(algo="gl", B=64, N=160000, sr=16000, n_fft=400, hop=200, iters=32, coef=0.99,
                       desc="GENERIC path: griffin_lim B=64 x 10 s @ 16 kHz, n_fft=400 hop=200 hann (torchaudio's "
                            "default transform), 32 iters, alpha=0.99"),
}


def hann(n):
    return (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(n) / n)).astype(np.float32)


def dims(w):
    F, T = w["n_fft"] // 2 + 1, 1 + w["N"] // w["hop"]
    return F, T, (T - 1) * w["hop"]


def workload_config(w, n_gpus):
    F, T, _ = dims(w)
    return {"workload": w["desc"], "batch_per_gpu": w["B"], "spec_shape": [w["B"], F, T],
            "parallelism": f"batch-sharded x{n_gpus}, no collective",
            "l2": "inputs larger than L2 (each iteration streams %.2f GB)" % (iter_bytes(w) / 1e9)}


def iter_bytes(w, B=None, T=None):
    """Algorithmic HBM bytes of one fused iteration, fp32 (SURVEY.md section 8d): GL reads q (8) + writes q (8) +
    reads mag (4) per bin, ADMM reads and writes X and U + reads mag (36), both read x (4) + write x (4) per sample.
    RTISI-LA: the whole call reads the magnitudes once and writes the signal once."""
    B = w["B"] if B is None else B
    F, T0, _ = dims(w)
    T = T0 if T is None else T
    L = (T - 1) * w["hop"]
    if w["algo"] == "rtisi":
        return 4 * B * F * T + 4 * B * L
    per_bin = 36 if w["algo"] == "admm" else (20 if w["coef"] > 0 else 4)
    return per_bin * B * F * T + 8 * B * L


def frame_flops(n_fft):
    """SURVEY.md section 8d count convention per frame and iteration: real FFT of n via an n/2-point complex FFT
    5 (n/2) log2(n/2) + 8 (n/2), x 2 (forward + inverse), + 12 F point-wise, + 4 n_fft window / overlap-add."""
    h = n_fft // 2
    return 2 * (5 * h * math.log2(h) + 8 * h) + 12 * (h + 1) + 4 * n_fft


def units(w, B=None):
    return (w["B"] if B is None else B) * w["N"] / w["sr"] * w["iters"]


# ----------------------------------------------------------------------------- CPU legs
def cpu_inputs(w, B, threads, seed=0):
    from oracle import specinv_oracle as O
    rs = np.random.RandomState(seed)
    win = hann(w["n_fft"])
    a = O.args_helper(w["n_fft"] // 2 + 1, np.float32, window=win, hop_length=w["hop"])
    x = rs.randn(B, w["N"]).astype(np.float32)
    mag = O.run_batched(lambda s: np.abs(O.stft(s, a)), x, threads)
    return win, a, mag


def cpu_job(w, B, threads, seed=0):
    """The oracle's griffin_lim on B signals of the workload, batch split over `threads` host threads."""
    from oracle import specinv_oracle as O
    win, a, mag = cpu_inputs(w, B, threads, seed)

    def run():
        t = time.perf_counter()
        y = O.run_batched(lambda s: O.griffin_lim(s, max_iter=w["iters"], tol=0, alpha=w["coef"], eva_iter=10,
                                                  window=win, hop_length=w["hop"]), mag, threads)
        return time.perf_counter() - t, y
    return run, (win, a, mag)


def cpu_sample_size(w):
    cores = os.cpu_count() or 1
    threads = min(cores, 64)
    B = max(1, min(w["B"], 2 * threads))
    return B, threads


def reference_available():
    return os.path.exists(os.path.join(REF_DIR, "torch_specinv", "methods.py"))


def import_reference():
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import torch_specinv
    return torch_specinv


def run_reference(args, w):
    """Reference arm: the UNMODIFIED reference (baseline/_ref, installed by baseline/install_ref.py) through its own
    public API on the host CPUs with all the threads torch uses (kind "reference"); the oracle port (kind "port") only
    when the reference is not installed.  Each step is a bounded sample of the workload (B' of the B signals, full
    length and iteration count), sized after one probe so that the K + W steps end within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget_s = 150.0
    B0, threads = cpu_sample_size(w)
    n_jobs = args.steps + args.warmup
    if reference_available():
        import torch
        ref = import_reference()
        kind = "reference"
        threads = torch.get_num_threads()
        torch.manual_seed(0)
        win = torch.hann_window(w["n_fft"])
        x = torch.randn(B0, w["N"])
        mag_all = torch.stft(x, w["n_fft"], w["hop"], window=win, return_complex=True).abs()

        def make(B):
            mag = mag_all[:B]

            def run():
                t = time.perf_counter()
                with torch.no_grad():
                    ref.griffin_lim(mag, max_iter=w["iters"], tol=0, alpha=w["coef"], verbose=False, eva_iter=10,
                                    hop_length=w["hop"], window=win)
                return time.perf_counter() - t
            return run
    else:
        kind = "port"

        def make(B):
            run, _ = cpu_job(w, B, threads)
            return lambda: run()[0]
    Bp = max(1, min(B0, 4))
    t_probe = make(Bp)()                                           # untimed probe (also pages everything in)
    per_signal = t_probe / Bp
    B = int(max(1, min(B0, budget_s / (n_jobs * per_signal))))
    run = make(B)
    for _ in range(args.warmup):
        run()
    times = [run() for _ in range(args.steps)]
    total = sum(times)
    value = units(w, B) * args.steps / total
    sample = (f"B={B} of {w['B']} signals, full length and iteration count, {threads} threads"
              + ("" if kind == "reference" else " (baseline/_ref not installed: oracle port)"))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU leg
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_to_gpu_numa(torch, index):
    """Pin this process (and the pinned host buffers it allocates afterwards: first touch) to the CPUs NVML reports as
    local to its GPU.  Under torchrun eight ranks otherwise float over both sockets and the e2e leg's host <-> device
    copies (1.48 GB per step and rank) cross the socket interconnect.  SPECINV_BENCH_NUMA_BIND=0 switches it off.
    Returns a short description for the JSON line."""
    if os.environ.get("SPECINV_BENCH_NUMA_BIND", "1") == "0":
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cpus local to the GPU"
    except Exception as ex:      # no NVML / not permitted: run unbound
        return f"unbound ({type(ex).__name__})"


class Ctx:
    """torch / distributed plumbing shared by the measurement functions."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa(torch, self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def ev(self):
        return self.torch.cuda.Event(enable_timing=True)

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def min_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return t.tolist()


def synth_mag(cx, w, B, seed, length=None):
    """mag = |STFT(randn)| of B signals through the library's own STFT kernel, (B, F, T) with frame-major strides
    (what torch.stft returns); outside every timed region."""
    torch = cx.torch
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    F, T, L = dims(w)
    win = torch.from_numpy(hann(w["n_fft"])).to(cx.dev)
    g = torch.Generator(device=cx.dev).manual_seed(seed)
    plan0 = StftPlan(args_helper(torch.empty(B, F, T, device="meta"), hop_length=w["hop"], window=win), T, B,
                     torch.float32, cx.dev)
    # the plan's L is (T-1)*hop: feed exactly that many samples, like the reference's round trip does
    x = torch.randn(B, plan0.length, device=cx.dev, generator=g)
    mag = plan0.unpack(plan0.stft(x)).abs()
    del x, plan0
    return win, mag


DUMP_BYTES = 32 << 20


def dump_outputs(directory, signal):
    """--dump-outputs: the signal the last timed step returned, as DIR/signal.npy (float32, one row per signal).  The
    inputs are seeded, so two builds of the library run with the same arguments can be compared output for output.
    A batch larger than DUMP_BYTES is sampled: whole rows, drawn with a fixed seed, in ascending order."""
    os.makedirs(directory, exist_ok=True)
    y = signal.reshape(-1, signal.shape[-1])
    B, L = y.shape
    n = max(1, min(B, DUMP_BYTES // (L * y.element_size())))
    rows = np.sort(np.random.RandomState(0).choice(B, n, replace=False))
    np.save(os.path.join(directory, "signal.npy"), y[rows.tolist()].cpu().numpy())


def make_job(cx, w, mag, win, loop_ms=None):
    """One whole public call on device-resident input, step by step like methods.griffin_lim / ADMM so that events
    can bracket the iteration loop (-> ms per fused launch)."""
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200 import methods
    from spectrogram_inversion_b200.engine import ADMMSolver, GriffinLimSolver, training_loop
    kw = dict(hop_length=w["hop"], window=win)
    if w["algo"] == "rtisi":
        return lambda: S.RTISI_LA(mag, look_ahead=w["look_ahead"], max_iter=w["iters"], alpha=w["coef"], verbose=0, **kw)
    Solver = GriffinLimSolver if w["algo"] == "gl" else ADMMSolver

    def job():
        plan, C, m = methods._setup(mag, dict(kw))
        solver = Solver(plan, C, m, w["coef"])
        e0, e1 = cx.ev(), cx.ev()
        e0.record()
        training_loop(solver, w["iters"], 0.0, False, 10, "sc")
        e1.record()
        if loop_ms is not None:
            loop_ms.append((e0, e1))
        return methods._finish(solver.signal, mag)
    return job


def final_sc_db(cx, w, mag, win, y):
    """Spectral convergence (metrics.py:4-14) of a result: sc(|STFT(y)|, mag) through the library's own kernels."""
    import spectrogram_inversion_b200 as S
    torch = cx.torch
    from spectrogram_inversion_b200.engine import StftPlan
    from spectrogram_inversion_b200.stft_args import args_helper
    B, F, T = mag.shape
    plan = StftPlan(args_helper(mag, hop_length=w["hop"], window=win), T, B, torch.float32, cx.dev)
    est = plan.unpack(plan.stft(y.contiguous())).abs()
    return float(S.sc(est, mag))


def measure_config(cx, name, w, B, n_jobs, n_warm, seed, with_reference_cuda=False):
    """Device-resident timing of one BASELINE config at B signals per rank: n_warm untimed + n_jobs timed whole
    public calls, barrier + synchronize on both sides, max over ranks."""
    torch = cx.torch
    win, mag = synth_mag(cx, w, B, seed)
    loop_ms = []
    job = make_job(cx, w, mag, win, loop_ms)
    y = None
    for _ in range(n_warm):
        y = job()
    loop_ms.clear()
    cx.barrier()
    s, e = cx.ev(), cx.ev()
    s.record()
    for _ in range(n_jobs):
        y = job()
    e.record()
    cx.barrier()
    job_ms = s.elapsed_time(e) / n_jobs
    it_ms = (sum(a.elapsed_time(b) for a, b in loop_ms) / (len(loop_ms) * w["iters"])) if loop_ms else 0.0
    job_ms, it_ms = cx.max_over_ranks([job_ms, it_ms])
    F, T, L = dims(w)
    out = {"workload": w["desc"], "batch_per_gpu": B, "n_gpus": cx.world, "ms_per_job": job_ms,
           "value": cx.world * units(w, B) / (job_ms / 1e3), "unit": UNIT, "jobs_timed": n_jobs}
    if w["algo"] == "rtisi":
        steps = (T + w["look_ahead"]) * w["iters"]
        flops = B * steps * (w["look_ahead"] + 1) * frame_flops(w["n_fft"])
        fp32_peak, fp32_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "fp32_peak.json")) as f:
                pk = json.load(f)
            fp32_peak, fp32_src = float(pk["fp32_fma_tflops"]), pk["source"]
        except Exception:
            pass
        tfl = flops / (job_ms / 1e3) / 1e12
        out.update({"us_per_inner_iteration": 1e3 * job_ms / steps, "bound": "latency / fp32 (HBM traffic negligible)",
                    "tflops_achieved": tfl, "fp32_peak_tflops": fp32_peak,
                    "fp32_frac": (tfl / fp32_peak) if fp32_peak else None,      # per GPU: B signals of this rank
                    "fp32_peak_source": fp32_src,
                    "flops_convention": "SURVEY.md 8d: B x (T+LA) x max_iter x (LA+1) frames x frame_flops(n_fft)",
                    "hbm_bytes_per_job": iter_bytes(w, B)})
    else:
        bytes_it = iter_bytes(w, B)
        gbs = bytes_it / (it_ms / 1e3) / 1e9
        out.update({"ms_per_iteration": it_ms, "algorithmic_bytes_per_launch": bytes_it, "achieved_gbs": gbs,
                    "frac": gbs / cx.peak, "iteration_value": cx.world * units(w, B) / w["iters"] / (it_ms / 1e3)})
    if y is not None:
        try:
            out["final_sc_db"] = final_sc_db(cx, w, mag, win, y)
        except Exception as ex:   # never let a diagnostic kill the line
            out["final_sc_db"] = f"unavailable: {ex}"
    if with_reference_cuda:
        out["reference_cuda"] = measure_reference_cuda(cx, w, mag, win)
    del mag, y
    torch.cuda.empty_cache()
    return out


def measure_cfg5_sharded(cx, w, n_iter=100, n_check=3):
    """cfg5 with the FRAMES of the one signal sharded over the ranks (rank order = time order): per iteration every
    rank runs the fused kernel on its range and exchanges the partial overlap-add sums of the n_fft - hop boundary
    samples with its neighbours through NVLink peer memory (sharding.PeerHalo, csrc/specinv_p2p.cu)."""
    torch, dist = cx.torch, cx.dist
    from spectrogram_inversion_b200.engine import GriffinLimSolver, SplitSpec, StftPlan
    from spectrogram_inversion_b200.sharding import CudaRangeEngine, FrameShardedGriffinLim, shard_bounds
    from spectrogram_inversion_b200.stft_args import StftArgs
    F, T, L = dims(w)
    n_fft, hop = w["n_fft"], w["hop"]
    win = torch.from_numpy(hann(n_fft)).to(cx.dev)
    args = StftArgs(n_fft, hop, n_fft, win, True, "reflect", False, True)
    # every rank synthesises the SAME global problem (same seed) and keeps its frame range
    g = torch.Generator(device=cx.dev).manual_seed(55)
    plan = StftPlan(args, T, 1, torch.float32, cx.dev)
    x = torch.randn(1, plan.length, device=cx.dev, generator=g)
    S = plan.stft(x)
    mag = plan.spec_abs(S)
    C = SplitSpec(mag.main * torch.exp(2j * math.pi * torch.rand(mag.main.shape, device=cx.dev, generator=g)),
                  mag.nyq.to(S.nyq.dtype))
    del x, S
    lo, hi = shard_bounds(T, cx.world, cx.rank)
    Tg = hi - lo

    def local(s):
        # clone: the solver owns (and ping-pongs into) what it is given; a prefix slice is already contiguous
        return SplitSpec(s.main[:, lo:hi].clone(), s.nyq[:, lo:hi].clone())

    engine = CudaRangeEngine(args, Tg, 1, torch.float32, cx.dev, lo, T)
    solver = FrameShardedGriffinLim(engine, local(C), local(mag), w["coef"])
    peer = solver.peer is not None
    # ---- parity with the single-GPU run after n_check iterations (rank 0 runs the whole signal as well)
    for _ in range(n_check):
        solver.step()
    ov = n_fft - hop
    xl = solver.signal_local
    checks = {}
    # (1) neighbours hold bit-identical samples in the region they share
    if cx.rank + 1 < cx.world:
        dist.send(xl[:, xl.shape[1] - ov:].contiguous(), cx.rank + 1)
    same = 1.0
    if cx.rank > 0:
        got = torch.empty(1, ov, device=cx.dev)
        dist.recv(got, cx.rank - 1)
        same = float(torch.equal(got, xl[:, :ov]))
    checks["boundary_bit_identical_between_neighbours"] = bool(cx.min_over_ranks([same])[0] == 1.0)
    # (2) against the un-sharded solver on rank 0: its right boundary block and its whole owned piece
    diff_b = diff_all = 0.0
    single_ms = 0.0
    if cx.rank == 0:
        ref = GriffinLimSolver(plan, SplitSpec(C.main.clone(), C.nyq.clone()), mag, w["coef"])
        for _ in range(n_check):
            ref.step()
        start, piece = solver.owned_piece()
        diff_all = float((piece - ref.signal[:, start:start + piece.shape[1]]).abs().max())
        # the block rank 0 shares with rank 1 (the last n_fft - hop samples of its local buffer, owned by rank 1)
        g0 = engine.padded_offset + xl.shape[1] - ov - engine.pad
        diff_b = float((xl[:, xl.shape[1] - ov:] - ref.signal[:, g0:g0 + ov]).abs().max())
        # single-GPU iteration time on the same box for the speed-up
        for _ in range(5):
            ref.step()
        torch.cuda.synchronize()
        e0, e1 = cx.ev(), cx.ev()
        e0.record()
        for _ in range(n_iter):
            ref.step()
        e1.record()
        torch.cuda.synchronize()
        single_ms = e0.elapsed_time(e1) / n_iter
        del ref
    del C, mag, plan
    torch.cuda.empty_cache()
    checks["rank0_boundary_block_max_abs_diff_vs_1gpu"] = diff_b
    checks["rank0_owned_piece_max_abs_diff_vs_1gpu"] = diff_all
    checks["after_iterations"] = n_check
    # ---- timing: n_iter iterations (fused kernel + exchange + padding refresh each)
    for _ in range(5):
        solver.step()
    cx.barrier()
    e0, e1 = cx.ev(), cx.ev()
    e0.record()
    for _ in range(n_iter):
        solver.step()
    e1.record()
    cx.barrier()
    it_ms = e0.elapsed_time(e1) / n_iter
    # the exchange alone (peer stores + flags + add, then the padding refresh), on a scratch copy of the signal
    scratch = solver.signal_local.clone()
    for _ in range(3):
        solver._exchange(scratch)
    cx.barrier()
    e0, e1 = cx.ev(), cx.ev()
    e0.record()
    for _ in range(50):
        solver._exchange(scratch)
    e1.record()
    cx.barrier()
    ex_us = 1e3 * e0.elapsed_time(e1) / 50
    it_ms, ex_us, single_ms = cx.max_over_ranks([it_ms, ex_us, single_ms])
    bytes_it = iter_bytes(w, 1)
    gbs = bytes_it / (it_ms / 1e3) / 1e9
    if solver.peer is not None:
        solver.peer.close()
    return {"workload": w["desc"] + f"; frames sharded over {cx.world} ranks ({Tg} frames on rank {cx.rank}), "
            "per-iteration halo exchange of n_fft - hop = 3072 samples with each neighbour",
            "n_gpus": cx.world, "exchange": "NVLink peer-memory kernel (PeerHalo)" if peer else "NCCL send/recv",
            "ms_per_iteration": it_ms, "ms_per_iteration_1gpu_same_box": single_ms,
            "speedup_vs_1gpu": (single_ms / it_ms) if it_ms > 0 else None, "exchange_us": ex_us,
            "value": units(w, 1) / w["iters"] / (it_ms / 1e3), "unit": UNIT + " (per-iteration rate)",
            "algorithmic_bytes_per_iteration": bytes_it, "achieved_gbs_aggregate": gbs,
            "frac_of_n_gpu_peak": gbs / (cx.peak * cx.world), "checks": checks}


def measure_reference_cuda(cx, w, mag, win, n_jobs=2):
    """The unmodified reference with device='cuda' on the same inputs: torch.stft (cuFFT) + conv_transpose1d (cuDNN) +
    ~12 element-wise kernels per iteration (methods.py:237-250, :127-128) -- 'the existing GPU path'."""
    torch = cx.torch
    if not reference_available():
        return {"unavailable": "baseline/_ref not installed (python baseline/install_ref.py)"}
    try:
        ref = import_reference()
        kw = dict(max_iter=w["iters"], tol=0, alpha=w["coef"], verbose=False, eva_iter=10, hop_length=w["hop"], window=win)
        B = mag.shape[0]
        while True:
            try:
                with torch.no_grad():
                    y = ref.griffin_lim(mag[:B], **kw)
                break
            except torch.cuda.OutOfMemoryError:
                torch.cuda.empty_cache()
                if B == 1:
                    raise
                B //= 2
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad():
            y = ref.griffin_lim(mag[:B], **kw)          # second warm-up, also sizes the timed run
        torch.cuda.synchronize()
        if time.perf_counter() - t0 > 8.0:
            n_jobs = 1
        e0, e1 = cx.ev(), cx.ev()
        e0.record()
        with torch.no_grad():
            for _ in range(n_jobs):
                y = ref.griffin_lim(mag[:B], **kw)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_jobs
        sc = final_sc_db(cx, w, mag[:B].contiguous() if B != mag.shape[0] else mag, win, y)
        del y
        torch.cuda.empty_cache()
        return {"value": units(w, B) / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "batch": B, "jobs_timed": n_jobs,
                "final_sc_db": sc, "what": "torch_specinv 0.2.1 (baseline/_ref) griffin_lim on device='cuda', same "
                "magnitudes, device-resident input (torch " + torch.__version__ + ": cuFFT + cuDNN)"}
    except Exception as ex:
        torch.cuda.empty_cache()
        return {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}


def run_ours(args, w):
    cx = Ctx()
    torch, dist = cx.torch, cx.dist
    import spectrogram_inversion_b200 as S
    from spectrogram_inversion_b200 import _ops, methods
    from spectrogram_inversion_b200.engine import GriffinLimSolver

    world, rank, dev = cx.world, cx.rank, cx.dev
    B = args.batch or w["B"]
    iters = w["iters"]
    win, mag = synth_mag(cx, w, B, 1234 + rank)
    kw = dict(hop_length=w["hop"], window=win)
    mag_host = torch.empty(mag.shape, dtype=mag.dtype, pin_memory=True)
    mag_host.copy_(mag)
    torch.cuda.synchronize()

    loop_ms = []
    job_device = make_job(cx, w, mag, win, loop_ms)

    def job_e2e():
        return S.griffin_lim(mag_host, max_iter=iters, tol=0, alpha=w["coef"], verbose=False, eva_iter=10, **kw)

    # ---- the fused iteration kernel timed alone (burst): a few back-to-back launches on the still idle board, so
    # that the figure is free of the power capping a 64-iteration job runs into (roofline.burst_*; `achieved` is
    # the sustained figure measured inside the timed steps below)
    burst_ms = None
    try:
        plan_b, C_b, m_b = methods._setup(mag, dict(kw))
        solver_b = GriffinLimSolver(plan_b, C_b, m_b, w["coef"])
        for _ in range(3):
            solver_b.step()
        torch.cuda.synchronize()
        b0, b1 = cx.ev(), cx.ev()
        b0.record()
        for _ in range(8):
            solver_b.step()
        b1.record()
        torch.cuda.synchronize()
        burst_ms = b0.elapsed_time(b1) / 8
        del plan_b, C_b, m_b, solver_b
    except Exception:
        burst_ms = None

    for _ in range(args.warmup):
        job_device()
    loop_ms.clear()
    cx.barrier()
    sampler = ClockSampler(cx.local) if rank == 0 else None
    launches0 = _ops.LAUNCHES[0]
    s, e = cx.ev(), cx.ev()
    s.record()
    for _ in range(args.steps):
        y = job_device()
    e.record()
    cx.barrier()
    launches = _ops.LAUNCHES[0] - launches0
    total_ms = s.elapsed_time(e)
    it_ms = sum(a.elapsed_time(b) for a, b in loop_ms) / (len(loop_ms) * iters)
    sc_gpu = final_sc_db(cx, w, mag, win, y)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y)
    del y

    # ---- e2e through the public API with host buffers: every step timed on its own (host buffers in, host buffers
    # out, blocking call).  The reported value comes from the MEAN step; median / p95 / max are listed beside it.
    yh = None
    for _ in range(max(3, min(args.warmup, 5))):
        yh = job_e2e()      # keep the result alive like the timed loop does (pinned-buffer cache warm)
    cx.barrier()
    n_e2e = args.steps
    marks = [cx.ev() for _ in range(n_e2e + 1)]
    marks[0].record()
    for k in range(n_e2e):
        yh = job_e2e()
        marks[k + 1].record()
    cx.barrier()
    e2e_steps = [marks[k].elapsed_time(marks[k + 1]) for k in range(n_e2e)]
    e2e_mean = float(np.mean(e2e_steps))
    clocks = sampler.stop() if sampler else None

    total_ms, e2e_mean, it_ms, burst_ms = cx.max_over_ranks([total_ms, e2e_mean, it_ms, burst_ms or 0.0])

    units_per_step = world * units(w, B)
    value = units_per_step * args.steps / (total_ms / 1e3)
    e2e_value = units_per_step / (e2e_mean / 1e3)
    achieved = iter_bytes(w, B) / (it_ms / 1e3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get("gl_iter_dram_bytes_per_launch")
    except Exception:
        pass
    h2d, d2h = mag_host.numel() * 4, yh.numel() * 4

    # ---- reference_cuda, cpu_baseline + parity on its sample (rank 0 of a single-GPU run only)
    ref_cuda = cpu = parity = None
    if world == 1 and not args.no_cpu:
        ref_cuda = measure_reference_cuda(cx, w, mag, win)
        Bc, threads = cpu_sample_size(w)
        run_cpu, (win_c, a_c, mag_c) = cpu_job(w, Bc, threads)
        mag_s = torch.from_numpy(mag_c).to(dev)
        y_ref = None
        if reference_available():
            # the UNMODIFIED reference on the host CPUs, on the sample's very magnitudes
            try:
                ref = import_reference()
                mag_cpu, win_cpu = torch.from_numpy(mag_c), torch.from_numpy(hann(w["n_fft"]))
                t0 = time.perf_counter()
                with torch.no_grad():
                    y_ref = ref.griffin_lim(mag_cpu, max_iter=iters, tol=0, alpha=w["coef"], verbose=False, eva_iter=10,
                                            hop_length=w["hop"], window=win_cpu)
                tcpu = time.perf_counter() - t0
                cpu = {"value": units(w, Bc) / tcpu, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "reference",
                       "sample": f"B={Bc} of {w['B']} signals, full length and iteration count, one run of {tcpu:.1f} s of "
                                 "torch_specinv 0.2.1 (baseline/_ref) on the host CPUs"}
            except Exception as ex:
                y_ref, cpu = None, {"reference_failed": f"{type(ex).__name__}: {ex}"[:200]}
        tcpu, y_cpu = run_cpu()
        port = {"value": units(w, Bc) / tcpu, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"B={Bc} of {w['B']} signals, full length and iteration count, one run of {tcpu:.1f} s"}
        if y_ref is None:
            cpu = dict(port, **(cpu or {}))
        else:
            cpu["oracle_port"] = port
        # the GPU path on the CPU sample's very magnitudes: final spectral convergence of all results, judged by the
        # same (GPU) STFT.  north_star: within 1 % (0.0864 dB) of the reference.
        y_gpu = S.griffin_lim(mag_s, max_iter=iters, tol=0, alpha=w["coef"], verbose=False, eva_iter=10, **kw)
        sc_g = final_sc_db(cx, w, mag_s, win, y_gpu)
        sc_c = final_sc_db(cx, w, mag_s, win, torch.from_numpy(np.ascontiguousarray(y_cpu)).to(dev))
        one_pct = 20 * math.log10(1.01)
        parity = {"sample": f"the cpu_baseline sample (B={Bc}, seed 0)", "final_sc_db_gpu": sc_g,
                  "final_sc_db_cpu_port": sc_c, "diff_db": sc_g - sc_c, "one_percent_db": one_pct,
                  "within_1pct": abs(sc_g - sc_c) <= one_pct}
        if y_ref is not None:
            sc_r = final_sc_db(cx, w, mag_s, win, y_ref.to(dev).contiguous())
            parity.update({"final_sc_db_reference": sc_r, "diff_db_vs_reference": sc_g - sc_r,
                           "within_1pct_of_reference": abs(sc_g - sc_r) <= one_pct,
                           "max_abs_diff_vs_reference": float((y_gpu - y_ref.to(dev)).abs().max())})
        del mag_s, y_gpu
    del mag, yh, mag_host
    torch.cuda.empty_cache()

    # ---- the other configs (device-resident, bounded: 2 warm-up + 3 timed whole calls each)
    configs = {}
    if args.configs != "none":
        want = ["cfg1", "cfg3", "cfg4", "cfg5", "generic400"] if args.configs == "all" else \
            [c for c in args.configs.split(",") if c in WORKLOADS]
        for name in want:
            wc = WORKLOADS[name]
            try:
                if name == "cfg5" and world > 1:
                    configs["cfg5_frame_sharded"] = measure_cfg5_sharded(cx, wc)
                    continue
                Bc = wc["B"] if wc["B"] == 1 else max(1, wc["B"] // world)      # batch configs: strong scaling
                r = measure_config(cx, name, wc, Bc, 3, 2, 77 + rank,
                                   with_reference_cuda=(name == "generic400" and world == 1 and not args.no_cpu))
                if wc["B"] == 1 and world > 1:
                    r["note"] = "a single signal does not shard by batch: every rank ran its own replica"
                elif world > 1:
                    r["scaling"] = f"strong: B={wc['B']} split into {Bc} per rank"
                configs[name] = r
            except Exception as ex:
                configs[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
                torch.cuda.empty_cache()
        if world > 1 and args.configs == "all":
            try:
                r = measure_config(cx, "cfg2", w, max(1, w["B"] // world), 3, 2, 1234 + rank)
                r["scaling"] = f"strong: B={w['B']} split into {max(1, w['B'] // world)} per rank"
                configs["cfg2_strong"] = r
            except Exception as ex:
                configs["cfg2_strong"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    if rank == 0:
        cfg = workload_config(w, world)
        cfg["batch_per_gpu"] = B
        srt = sorted(e2e_steps)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "final_sc_db": sc_gpu,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s",
                             "frac": achieved / cx.peak, "traffic": traffic,
                             "traffic_source": "ncu --set full capture of this kernel at this shape, committed under "
                                               "profiles/ (a constant, not measured in this run)",
                             "kernel": "fused GL iteration",
                             "ms_per_launch": it_ms, "algorithmic_bytes_per_launch": iter_bytes(w, B),
                             "peak_source": cx.peak_src, "timing": "sustained: averaged over the timed 64-iteration jobs "
                             "(includes the 6 evaluating launches per job and any power capping)",
                             "burst_ms_per_launch": burst_ms or None,
                             "burst_frac": (iter_bytes(w, B) / (burst_ms / 1e3) / 1e9 / cx.peak) if burst_ms else None},
                "cpu_baseline": cpu, "parity": parity, "reference_cuda": ref_cuda,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_mean, "ms_per_step_median": srt[len(srt) // 2],
                        "ms_per_step_p95": srt[min(len(srt) - 1, int(math.ceil(0.95 * len(srt))) - 1)],
                        "ms_per_step_max": srt[-1], "ms_per_step_all": e2e_steps,
                        "timing": f"value from the MEAN of {len(e2e_steps)} steps (rank 0's steps listed in call order; "
                                  "the mean is the max over ranks)"},
                "gpu_launches": launches, "clocks": clocks, "host_binding": cx.numa,
                "configs": configs}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2"],
                    help="headline workload (cfg2 = the configuration BASELINE.json's metric is quoted on)")
    ap.add_argument("--configs", default="all", help="extra configs reported in `configs`: all | none | cfg1,cfg3,...")
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (debugging only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity / reference_cuda legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the signal the last one returned (a seeded sample of its rows "
                         "when larger than 32 MiB) to DIR/signal.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this library's path computed (--impl ours)")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
