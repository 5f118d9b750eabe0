#!/usr/bin/env python
"""Benchmark of the nnaudio-b200 hot path (contract: task brief §④ / base contract).

  python bench.py --gpus N --steps K --warmup W [--workload cfg2] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic white noise:
by default ``cfg2`` of BASELINE.json (MelSpectrogram n_fft=2048 hop=512
n_mels=128 on 64 x 10 s @ 22 050 Hz per GPU; the configuration the headline
metric is quoted on).  ``value`` is whole-job frames/s with inputs resident in
HBM; ``e2e`` is the same metric through the public nn.Module call with pinned
HOST buffers (H2D of the input and D2H of the spectrogram inside the timed
region).  Under torchrun (N > 1) every rank processes its own batch shard
(weak scaling) and the shards' outputs are all-gathered over NCCL/NVLink.

``--impl reference`` times the CPU arm instead: the NumPy oracle port of the
reference's conv1d path (oracle/nnaudio_oracle.py) on the host cores — the
reference itself is Python and cannot travel to the GPU box.

``--dump-outputs DIR`` writes the spectrograms the last timed step of the headline workload returned as
``DIR/<workload>.npy`` (float32; a seeded sample of whole clips when they exceed 64 MB).  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ from the modules imported here

# torchrun exports OMP_NUM_THREADS=1 to its workers.  The CPU arm is meant to use the host cores
# ("all the host threads it can use"), and BLAS sizes its pool when it is first loaded, so put the
# count back before numpy / torch are imported.  Only for --impl reference: the GPU arm does no
# host compute worth threading.
if "--impl" in sys.argv and "reference" in sys.argv and os.environ.get("OMP_NUM_THREADS") == "1" \
        and int(os.environ.get("WORLD_SIZE", "1")) > 1:
    try:
        os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    except AttributeError:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

# ----------------------------------------------------------------------------
# workloads (BASELINE.json configs; shapes from SURVEY.md §8 config table)
# ----------------------------------------------------------------------------
WORKLOADS = {
    "cfg2": dict(cls="MelSpectrogram", ctor=dict(sr=22050, n_fft=2048, hop_length=512, n_mels=128),
                 B=64, L=220500, fwd={}, desc="MelSpectrogram n_fft=2048 hop=512 n_mels=128, 64x10s@22050Hz"),
    "stft2048": dict(cls="STFT", ctor=dict(n_fft=2048, hop_length=512, sr=22050, output_format="Magnitude"),
                     B=64, L=220500, fwd={}, desc="STFT n_fft=2048 hop=512 Magnitude, 64x10s@22050Hz"),
    "cfg3": dict(cls="CQT1992v2", ctor=dict(sr=44100, n_bins=84, bins_per_octave=12, fmin=32.7),
                 B=128, L=441000, fwd={}, desc="CQT1992v2 84 bins fmin=32.7, 128x10s@44100Hz"),
    "cfg4": dict(cls="CQT2010v2", ctor=dict(sr=22050, n_bins=88), B=256, L=661500, fwd={},
                 desc="CQT2010v2 88 bins, 256x30s@22050Hz"),
    "cfg5": dict(cls="MFCC", ctor=dict(sr=16000), B=1024, L=80000, fwd={},
                 desc="MFCC (STFT->Mel->dB->DCT) n_fft=2048 hop=512, 1024x5s@16kHz"),
    # not a BASELINE config: the dense-bank member of the STFT family at the cfg2 shape (VERDICT r1: "never
    # benchmarked").  Two framed launches per step (STFT -> operand planes, planes x bank): roofline per STEP.
    "gammatone": dict(cls="Gammatonegram", ctor=dict(sr=22050, n_fft=2048, hop_length=512, n_bins=64),
                      B=64, L=220500, fwd={}, framed_per_step=True,
                      desc="Gammatonegram n_fft=2048 hop=512 64 bins, 64x10s@22050Hz"),
}


# which roof bounds a workload (SURVEY.md 8(d)): the fused pyramid is HBM-bound, the rest tensor-bound
WORKLOAD_BOUND = {"cfg2": "tensor", "stft2048": "tensor", "cfg3": "tensor", "cfg5": "tensor", "cfg4": "hbm",
                  "gammatone": "tensor"}
# the other configurations BASELINE.json's metric names, reported inside the same JSON line
SECONDARY = ["stft2048", "cfg3", "cfg4", "cfg5", "gammatone"]

GATHER_DESC = {"peer": "kernels write into symmetric memory, copy-engine pushes over NVLink, stream-memop "
                       "handshakes: no SMs, no kernels, no NCCL on the data path",
               "symm": "copy-engine pushes into symmetric memory over NVLink, torch barrier kernels",
               "nccl": "ncclAllGather on reserved SMs", "none": "-", "auto": "-"}

# SMs left to the NCCL gather while the persistent kernels run, and the matching NCCL CTA cap
# (the gather of (N-1) x 14 MB must hide under one ~0.47 ms transform; measured ~14.5 GB/s per
# NCCL CTA next to the kernels: 8 CTAs suffice at N=4, not at N=8 — profiles/README.md)
DEFAULT_RESERVE = {1: 0, 2: 8, 4: 8, 8: 16}


def frames_per_clip(w):
    hop = w["ctor"].get("hop_length", 512)
    return w["L"] // hop + 1


def framed_algorithmic_flops(mod, cls, B, T):
    """Algorithmic FLOPs of ONE launch of the dominant kernel (the framed
    contraction) — SURVEY.md §8(d) per-frame figures times B*T frames."""
    if cls in ("MelSpectrogram", "Gammatonegram", "MFCC", "STFT"):
        st = mod.melspec_layer.stft if cls == "MFCC" else (mod if cls == "STFT" else mod.stft)
        F, K = st.wsin.shape[0], st.wsin.shape[-1]
        return B * T * (2.0 * K * 2 * F + 3.0 * F)
    if cls == "CQT1992v2":
        return B * T * 4.0 * float(mod.lenghts.sum().item())
    if cls == "CQT2010v2":
        nf, w = mod.cqt_kernels_real.shape[0], mod.cqt_kernels_real.shape[-1]
        return B * T * 2.0 * w * 2 * nf  # per octave launch
    return float("nan")


# ----------------------------------------------------------------------------
# clocks sampling (nvidia-smi recipe of B200_PROFILING.md, through NVML)
# ----------------------------------------------------------------------------
class ClockSampler:
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, device_index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.nv = pynvml
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # older binding name
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.001)  # short timed regions still get samples

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's conv1d path
# ----------------------------------------------------------------------------
def cpu_arm(workload, steps, warmup, budget_s):
    """Times the NumPy oracle (fp32, BLAS-threaded) on a bounded sample of the workload: as many
    clips per step as fit ``budget_s`` overall.  The BLAS thread count is the best of
    {all cores, /2, /4, ...} on a calibration batch (128 OpenBLAS threads are slower than 32 on
    these GEMM shapes), and ``cores`` in the result is the count actually used."""
    import numpy as np

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import build as build_module, run_oracle

    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits
    except Exception:  # noqa: BLE001  (no threadpoolctl: whatever the environment set)
        threadpool_limits = None

    w = WORKLOADS[workload]
    mod = build_module(w["cls"], w["ctor"])
    T = frames_per_clip(w)
    rng = np.random.RandomState(1234)

    def timed(x, n):
        t0 = time.perf_counter()
        for _ in range(n):
            run_oracle(w["cls"], mod, x, w["fwd"], dtype=np.float32)
        return time.perf_counter() - t0

    # calibration batch (one clip alone under-uses the BLAS threads)
    n_cal = int(min(8, w["B"]))
    xc = rng.standard_normal((n_cal, w["L"])).astype(np.float32)
    def best_of(n):  # single runs are noisy on a shared host: minimum of n
        return min(timed(xc, 1) for _ in range(n))

    timed(xc, 1)  # warm BLAS threads
    threads, best = avail, best_of(3)
    if threadpool_limits is not None:
        cand = avail // 2
        while cand >= 4:
            with threadpool_limits(limits=cand):
                timed(xc, 1)
                t = best_of(3)
            if t < 0.9 * best:  # switch only for a clear win
                threads, best = cand, t
            cand //= 2
    per_clip = max(best / n_cal, 1e-4)
    clips = int(max(1, min(w["B"], budget_s / ((steps + warmup) * per_clip))))
    x = rng.standard_normal((clips, w["L"])).astype(np.float32)
    import contextlib
    limiter = threadpool_limits(limits=threads) if threadpool_limits is not None else contextlib.nullcontext()
    with limiter:
        timed(x, warmup)
        dt = timed(x, steps)
    return {
        "value": clips * T * steps / dt, "unit": "frames/s", "cores": threads, "kind": "port",
        "sample": f"{clips} clip(s) x {w['L']} samples of {workload} per step, {steps} steps, "
                  f"NumPy fp32 oracle (oracle/nnaudio_oracle.py), {threads} BLAS threads of {avail} "
                  f"cores, {dt:.1f}s",
        "ms_per_step": 1e3 * dt / steps,
    }


def static_traffic(workload):
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            return json.load(f).get(workload, {}).get("framed_dram_bytes_per_launch")
    except Exception:  # noqa: BLE001
        return None


REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "nnAudio"))


def _reference_module(workload):
    """The UNMODIFIED reference module of a workload, imported from oracle/_ref
    (copied there by oracle/install_ref.sh during build())."""
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import importlib

    feats = importlib.import_module("nnAudio.features")
    assert os.path.realpath(feats.__file__).startswith(os.path.realpath(REF_DIR)), feats.__file__
    w = WORKLOADS[workload]
    return getattr(feats, w["cls"])(verbose=False, **w["ctor"])


def reference_cpu_arm(workload, steps, warmup, budget_s):
    """The reference's own CPU path (torch conv1d -> oneDNN, every host thread): a bounded sample
    of the workload per step, sized from a calibration run so the whole arm fits ``budget_s``."""
    import torch

    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    torch.set_num_threads(avail)
    w = WORKLOADS[workload]
    T = frames_per_clip(w)
    mod = _reference_module(workload)
    gen = torch.Generator().manual_seed(1234)

    def timed(x, n):
        t0 = time.perf_counter()
        with torch.no_grad():
            for _ in range(n):
                mod(x, **w["fwd"])
        return time.perf_counter() - t0

    # oneDNN's conv1d does not always scale to every core of a big host: give the reference the
    # thread count that is fastest on a calibration batch ({all, /2, /4, /8}; ``cores`` reports it)
    n_cal = int(min(8, w["B"]))
    xc = torch.randn(n_cal, w["L"], generator=gen)
    timed(xc, 1)
    best_t, threads = min(timed(xc, 1) for _ in range(2)), avail
    cand = avail // 2
    while cand >= 8:
        torch.set_num_threads(cand)
        timed(xc, 1)
        t = min(timed(xc, 1) for _ in range(2))
        if t < 0.9 * best_t:
            best_t, threads = t, cand
        cand //= 2
    torch.set_num_threads(threads)
    per_clip = max(best_t / n_cal, 1e-4)
    clips = int(max(1, min(w["B"], budget_s / ((steps + warmup) * per_clip))))
    x = torch.randn(clips, w["L"], generator=gen)
    timed(x, warmup)
    dt = timed(x, steps)
    return {
        "value": clips * T * steps / dt, "unit": "frames/s", "cores": threads, "kind": "reference",
        "sample": f"{clips} clip(s) x {w['L']} samples of {workload} per step, {steps} steps, unmodified "
                  f"nnAudio 0.3.3 {w['cls']} (oracle/_ref) on CPU, torch {torch.__version__} conv1d, "
                  f"{threads} threads (fastest of all / 2 / 4 / 8 of {avail} cores), {dt:.1f}s",
        "ms_per_step": 1e3 * dt / steps,
    }


def reference_gpu_leg(workload, dev, budget_s=20.0):
    """SURVEY.md §2.1 / §8(d): the reference's own modules (cuDNN conv1d) on the SAME B200, inputs
    resident, CUDA events.  The batch is halved until the reference fits in memory / its time
    budget; frames/s is reported for the batch that ran."""
    import torch

    w = WORKLOADS[workload]
    T = frames_per_clip(w)
    mod = _reference_module(workload).to(dev)
    B = w["B"]
    gen = torch.Generator(device=dev).manual_seed(99)
    last_err = None
    while B >= 1:
        try:
            x = torch.randn(B, w["L"], generator=gen, device=dev)
            with torch.no_grad():
                t0 = time.perf_counter()
                mod(x, **w["fwd"])
                torch.cuda.synchronize(dev)
                first = time.perf_counter() - t0
                mod(x, **w["fwd"])
                torch.cuda.synchronize(dev)
                t0 = time.perf_counter()
                mod(x, **w["fwd"])
                torch.cuda.synchronize(dev)
                one = time.perf_counter() - t0
                n = int(max(3, min(20, budget_s / max(one, 1e-4) / 2)))
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    y = mod(x, **w["fwd"])
                e1.record()
                torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / n
            del x, y
            torch.cuda.empty_cache()
            return {"value": B * T / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "batch": B,
                    "steps": n, "first_call_s": round(first, 3),
                    "what": f"unmodified nnAudio 0.3.3 {w['cls']} on cuda (cuDNN conv1d, torch "
                            f"{torch.__version__}), inputs resident, {B} of {w['B']} clips"}
        except Exception as e:  # noqa: BLE001  (OOM / cuDNN workspace: smaller batch)
            last_err = f"{type(e).__name__}: {str(e)[:120]}"
            torch.cuda.empty_cache()
            B //= 2
    return {"value": None, "unavailable": last_err}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, name, y):
    """``out_dir/<name>.npy``: ``y`` (a CPU tensor, clips first) as float32, or, above DUMP_LIMIT_BYTES, the
    clips of a fixed seeded sample in ascending order."""
    import numpy as np

    a = y.float().numpy()
    per_clip = a[0].nbytes
    if a.nbytes > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // per_clip)
        a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


# ----------------------------------------------------------------------------
def main():
    # stdout carries exactly ONE line (the JSON); libraries that print there (NCCL's version
    # banner) are routed to stderr for the duration of the run.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = _run()
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
    if line is not None:
        os.write(1, (json.dumps(line) + "\n").encode())


def _run():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--path", default=None, choices=[None, "auto", "simt", "tcgen05"])
    ap.add_argument("--batch", type=int, default=None, help="override per-GPU batch (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=8)
    ap.add_argument("--no-workloads", action="store_true", help="skip the secondary configs (stft2048, cfg3, cfg4, cfg5)")
    ap.add_argument("--workload-steps", type=int, default=None,
                    help="timed steps of each secondary config (default: --steps)")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference's cuDNN leg")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--watchdog", type=int, default=900, help="seconds after which a stuck run is aborted")
    ap.add_argument("--e2e-copy-streams", type=int, default=1)
    ap.add_argument("--gather", default="auto", choices=["auto", "nccl", "symm", "peer"],
                    help="peer = kernels write into symmetric memory, copy-engine pushes, stream-memop "
                         "handshakes (no SMs, no kernels); symm = same pushes with torch's barrier kernels; "
                         "nccl = all_gather_into_tensor with an SM reserve; auto = peer when it works here")
    ap.add_argument("--gather-to", default="root", choices=["all", "root"],
                    help="rank 0 receives the whole batch's spectrograms (the north star's gather), or every rank")
    ap.add_argument("--reserve-sms", type=int, default=None,
                    help="SMs kept free for the concurrent NCCL gather (default: by world size)")
    ap.add_argument("--nccl-max-ctas", type=int, default=-1,
                    help="-1 = same as the SM reserve (default), 0 = NCCL's own default")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the headline workload's output of the last timed step to DIR/<workload>.npy")
    args = ap.parse_args()
    if args.workload_steps is None:
        args.workload_steps = args.steps
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "ours":
        # a wedged device-side handshake must end the run, not sit on the box until the driver's limit
        import faulthandler

        faulthandler.dump_traceback_later(args.watchdog, exit=True)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["B"] = args.batch
    T = frames_per_clip(w)
    metric = "spectrogram frames/sec"

    # ------------------------------------------------------------ CPU arm --
    if args.impl == "reference":
        if rank != 0:
            return None
        if reference_available():
            res = reference_cpu_arm(args.workload, args.steps, args.warmup, budget_s=120.0)
            arm = "the UNMODIFIED reference (oracle/_ref, nnAudio 0.3.3) on the host cores: torch conv1d (oneDNN)"
        else:
            res = cpu_arm(args.workload, args.steps, args.warmup, budget_s=120.0)
            arm = "CPU oracle port of the reference conv1d path (oracle/_ref not installed)"
        line = {
            "impl": "reference", "metric": metric, "value": res["value"], "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {w['desc']}", "arm": arm},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "frames/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        return line

    # ------------------------------------------------------------ GPU arm --
    import torch
    import torch.distributed as dist

    import nnaudio_b200 as nb
    from nnaudio_b200 import _C
    from nnaudio_b200.host import HostPipeline, alloc_pinned, gpu_local_cpus
    from nnaudio_b200.parallel import BatchShardedTransform

    if args.path:
        os.environ["NNAUDIO_B200_PATH"] = args.path
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # host threads of this rank on the GPU's NUMA node: pinned buffers are first-touched there and
    # the launch thread does not cross sockets (the e2e copies are PCIe-bound)
    local_cpus = gpu_local_cpus(local_rank)
    if local_cpus and not args.no_numa_bind:
        try:
            os.sched_setaffinity(0, local_cpus)
        except OSError:
            local_cpus = None
    gather_impl = "none"
    if world > 1:
        # NCCL path: few CTAs for the output gather -- it overlaps the next batch's kernels (which
        # leave SMs free for it, nnaudio_b200.parallel) and 99 MB per step does not need more
        reserve_plan = args.reserve_sms if args.reserve_sms is not None else DEFAULT_RESERVE.get(world, 16)
        max_ctas = args.nccl_max_ctas if args.nccl_max_ctas >= 0 else reserve_plan
        if max_ctas > 0 and args.gather not in ("symm", "peer"):
            os.environ["NCCL_MAX_CTAS"] = str(max_ctas)
        dist.init_process_group("nccl", device_id=dev)
        gather_impl = args.gather
        if args.gather in ("auto", "symm", "peer"):
            # does the copy-engine gather work here?  (symmetric memory needs P2P / fabric handles,
            # the handshakes need stream memory operations); every rank must agree: reduce the outcome
            want_impl = "symm" if args.gather == "symm" else "peer"
            ok = 1
            try:
                probe = BatchShardedTransform(lambda t: t * 1.0, gather=True, reserve_sms=0)
                want = torch.arange(world, device=dev, dtype=torch.float32).repeat_interleave(2)[:, None].expand(-1, 8)
                for it in range(3):  # slot reuse included
                    xp = torch.full((2, 8), float(rank), device=dev)
                    if want_impl == "peer":
                        wk, got = probe.forward_async_peer(xp, slot=it & 1, gather_to="all")
                    else:
                        wk, got = probe.forward_async_symm(xp, slot=it & 1, gather_to="all")
                    wk.wait()
                    torch.cuda.synchronize(dev)
                    ok &= int(torch.equal(got, want))
                    if want_impl == "peer":
                        probe.release_peer(it & 1)
                    else:
                        probe.release(it & 1)
                torch.cuda.synchronize(dev)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] rank {rank}: {want_impl} gather unavailable: {type(e).__name__}: {e}\n")
                ok = 0
            flag = torch.tensor([ok], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 1:
                gather_impl = want_impl
            elif args.gather != "auto":
                raise RuntimeError(f"--gather {args.gather} requested but it failed its probe")
            else:
                gather_impl = "nccl"

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:  # noqa: BLE001
        pass
    tensor_peak = float(peaks.get("bf16_tflops", 1590.0))
    hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
    peak_src = ("measured (MEASURED_PEAKS.json: bf16_tflops burst, hbm_gbs)" if peaks
                else "fallback (B200_PROFILING.md): 1590 TFLOP/s bf16, 6500 GB/s")

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    reserve = args.reserve_sms if args.reserve_sms is not None else DEFAULT_RESERVE.get(world, 16)
    if gather_impl in ("symm", "peer") and args.reserve_sms is None:
        reserve = 0  # the copy engines do the gather: the kernels keep every SM

    def measure(name, steps, warmup, gather, keep_output=False):
        """One workload, inputs resident in HBM: ``steps`` timed steps between two CUDA events on the
        launching stream (max over ranks), the framed contraction timed per launch with in-stream
        events (nnab_profile_*), clocks sampled through NVML during the timed region."""
        w = dict(WORKLOADS[name])
        if args.batch and name == args.workload:
            w["B"] = args.batch
        B, T = w["B"], frames_per_clip(w)
        mod = getattr(nb.features, w["cls"])(verbose=False, **w["ctor"]).to(dev)
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        batch_bytes = B * w["L"] * 4
        # rotating input batches, > 126 MB of L2 in total: no step re-reads a cached input
        n_rot = 1 if batch_bytes > 160e6 else max(3, int(-(-160e6 // batch_bytes)))
        xs = [torch.randn(B, w["L"], generator=gen, device=dev, dtype=torch.float32) for _ in range(n_rot)]
        sharded = BatchShardedTransform(lambda inp: mod(inp, **w["fwd"]), gather=(gather and world > 1),
                                        reserve_sms=reserve if gather else 0)

        def run_steps(n):
            """n steps; the gather of step i overlaps the transform of step i+1 (two gather buffers);
            every gather completes inside the timed region."""
            prev, y = None, None
            for i in range(n):
                if gather_impl == "peer" and gather and world > 1:
                    work, y = sharded.forward_async_peer(xs[i % n_rot], slot=i & 1, gather_to=args.gather_to)
                elif gather_impl == "symm" and gather and world > 1:
                    work, y = sharded.forward_async_symm(xs[i % n_rot], slot=i & 1, gather_to=args.gather_to)
                else:
                    work, y = sharded.forward_async(xs[i % n_rot], slot=i & 1)
                if prev is not None:
                    prev.wait()
                    if gather and world > 1:
                        if gather_impl == "peer":
                            sharded.release_peer((i - 1) & 1, None if args.gather_to == "all" else [0])
                        elif gather_impl == "symm":
                            sharded.release((i - 1) & 1)
                prev = work
            if prev is not None:
                prev.wait()
                # the last step's slot must be handed back too: the next run_steps() reuses it
                if gather and world > 1:
                    if gather_impl == "peer":
                        sharded.release_peer((n - 1) & 1, None if args.gather_to == "all" else [0])
                    elif gather_impl == "symm":
                        sharded.release((n - 1) & 1)
            return y

        with torch.no_grad():
            y = run_steps(warmup)
            sync_all()
            out_shape = (B,) + tuple(y.shape[1:])  # this rank's own spectrograms
            out_bytes = int(torch.tensor(out_shape).prod().item()) * 4
            del y  # else the timed loop holds one more live output than the warm-up did (cudaMalloc)
            run_steps(2)
            sync_all()
            sampler = ClockSampler(local_rank)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            _C.profile_read()
            _C.profile_read_exec_flops()
            _C.profile_enable(True)
            launches0 = _C.launch_count()
            sampler.start()
            sync_all()
            e0.record()
            y = run_steps(steps)
            e1.record()
            sync_all()
            clocks = sampler.stop()
            y = y.cpu() if keep_output else None
            _C.profile_enable(False)
            launches = _C.launch_count() - launches0
            framed_ms, framed_n = _C.profile_read()
            exec_flops = _C.profile_read_exec_flops()
            dev_ms = e0.elapsed_time(e1)
        dev_ms, framed_ms = reduce_max([dev_ms, framed_ms])
        frames_total = world * B * T * steps
        flops_launch = framed_algorithmic_flops(mod, w["cls"], B, T)
        avg_launch_ms = framed_ms / max(framed_n, 1)
        if w.get("framed_per_step"):  # several framed launches make up one transform: time them together
            avg_launch_ms = framed_ms / max(steps, 1)
        tensor_alg = flops_launch / (avg_launch_ms * 1e-3) / 1e12 if framed_n else None
        tensor_exec = exec_flops / (framed_ms * 1e-3) / 1e12 if framed_ms > 0 else None
        alg_bytes = batch_bytes + out_bytes  # per step and rank: waveform in + spectrogram out
        hbm_ach = alg_bytes / (dev_ms / steps * 1e-3) / 1e9
        bound = WORKLOAD_BOUND.get(name, "tensor")
        roof = {
            "kernel": "framed contraction (frames x basis), pad/split pre-pass included",
            "bound": bound,
            "achieved": tensor_alg if bound == "tensor" else hbm_ach,
            "peak": tensor_peak if bound == "tensor" else hbm_peak,
            "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
            "frac": ((tensor_alg / tensor_peak) if tensor_alg else None) if bound == "tensor" else hbm_ach / hbm_peak,
            "traffic": static_traffic(name),
            "traffic_note": "dram__bytes_read + write of the dominant kernel per launch from the committed ncu --set "
                            "full capture (profiles/ncu_summary.json): static, not re-measured in this run",
            "peak_source": peak_src,
            "algorithmic_flops_per_launch": flops_launch, "avg_launch_ms": avg_launch_ms,
            "launches_timed": framed_n, "share_of_step": framed_ms / dev_ms if dev_ms else None,
            # SURVEY.md 8(d): both figures -- algorithmic (the reference's dense flops) and executed
            "tensor_algorithmic_tflops": tensor_alg,
            "tensor_algorithmic_frac": (tensor_alg / tensor_peak) if tensor_alg else None,
            "tensor_pipe": {"executed_tflops": tensor_exec,
                            "frac": (tensor_exec / tensor_peak) if tensor_exec else None,
                            "what": "MMA flops issued (3 bf16 split terms, tile padding, structural zeros) / kernel time / peak"},
            "hbm": {"algorithmic_bytes_per_step": alg_bytes, "achieved_gbs": hbm_ach, "frac": hbm_ach / hbm_peak,
                    "what": "(waveform in + spectrogram out) per step / step time / measured copy bandwidth"},
        }
        used_tc = (os.environ.get("NNAUDIO_B200_PATH", "auto") != "simt") and \
            _C.lib().nnab_packed_basis_bytes(8, 2048) > 0
        res = {
            "desc": w["desc"], "value": frames_total / (dev_ms * 1e-3), "unit": "frames/s",
            "ms_per_step": dev_ms / steps, "steps": steps, "warmup": warmup, "per_gpu_batch": B,
            "frames_per_clip": T, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
            "l2": f"{n_rot} rotating input batch(es) of {batch_bytes / 1e6:.0f} MB (> 126 MB L2 in total), no flush",
            "dtype": "bf16x3 split (fp32-equivalent), f32 accumulate" if used_tc else "f32",
        }
        return res, mod, out_shape, w, y

    main, mod, out_shape, w, y_last = measure(args.workload, args.steps, args.warmup, gather=True,
                                              keep_output=bool(args.dump_outputs) and rank == 0)
    if y_last is not None:
        dump_outputs(args.dump_outputs, args.workload, y_last)
    del y_last
    B = w["B"]
    no_gather = None
    if world > 1:  # SURVEY.md 8(e): frames/s with and without the gather
        ng, m_ng, _, _, _ = measure(args.workload, args.steps, args.warmup, gather=False)
        del m_ng
        no_gather = {"value": ng["value"], "ms_per_step": ng["ms_per_step"],
                     "what": "same run, transform only (shards stay on their GPUs)"}

    # ------------------------------------------------------------ e2e --
    e2e, pcie = None, None
    if not args.no_e2e:
        with torch.no_grad():
            # raw link rate of this box, pinned memory, per direction: one big copy, and the same bytes as
            # 8 MB chunks on the copy streams the pipeline uses (on some of this pool's boxes one 256 MB
            # copy reads the host at 35 GB/s while the pipeline's chunk copies reach 52); the better one is
            # the link rate `frac_of_link` is quoted against
            probe_n = 64 << 20  # floats = 256 MB
            hp, place = alloc_pinned((probe_n,), device_index=local_rank, fill="zeros")
            dp = torch.empty(probe_n, dtype=torch.float32, device=dev)
            n_str = max(1, int(args.e2e_copy_streams))
            streams = [torch.cuda.Stream(device=dev) for _ in range(n_str)]
            pieces = 32  # 8 MB each, the size of the pipeline's chunk copies
            step_n = probe_n // pieces

            def one_copy(dst, src):
                dst.copy_(src, non_blocking=True)

            def striped_copy(dst, src):
                cur = torch.cuda.current_stream(dev)
                fork = torch.cuda.Event()
                fork.record(cur)
                for i in range(pieces):
                    st = streams[i % n_str]
                    if i < n_str:
                        st.wait_event(fork)
                    with torch.cuda.stream(st):
                        dst[i * step_n:(i + 1) * step_n].copy_(src[i * step_n:(i + 1) * step_n], non_blocking=True)
                for st in streams:
                    join = torch.cuda.Event()
                    join.record(st)
                    cur.wait_event(join)

            rates, how = {}, {}
            for key, (dst, src) in (("h2d", (dp, hp)), ("d2h", (hp, dp))):
                best, best_how = 0.0, ""
                for name, fn in (("one copy", one_copy), (f"{pieces} chunks on {n_str} streams", striped_copy)):
                    for _ in range(2):  # warm the link (power state) and the page tables
                        fn(dst, src)
                    torch.cuda.synchronize(dev)
                    for _ in range(5):  # best of 5: the link rate, not its jitter
                        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        fn(dst, src)
                        b_.record()
                        torch.cuda.synchronize(dev)
                        r = probe_n * 4 / (a.elapsed_time(b_) * 1e-3) / 1e9
                        if r > best:
                            best, best_how = r, name
                rates[key], how[key] = best, best_how
            del hp, dp, streams
            pcie = {"h2d_gbs": rates["h2d"], "d2h_gbs": rates["d2h"], "pinned": place, "best": how,
                    "what": "cudaMemcpyAsync of a 256 MB pinned buffer per direction, as one copy and as chunks striped "
                            "over the pipeline's copy streams; best of 5 after 2 warm-up copies each, CUDA events"}

            x_hosts = [alloc_pinned((B, w["L"]), device_index=local_rank, fill="randn")[0] for _ in range(2)]
            y_host, _ = alloc_pinned(out_shape, device_index=local_rank)
            pipe = HostPipeline(mod, chunk_clips=max(1, B // args.e2e_chunks),
                                copy_streams=args.e2e_copy_streams, **w["fwd"])
            for i in range(3):
                pipe(x_hosts[i & 1], y_host, device=dev)
            sync_all()
            n_e2e = args.steps
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(n_e2e):
                pipe(x_hosts[i & 1], y_host, device=dev)
            b_.record()
            sync_all()
            (e2e_ms,) = reduce_max([a.elapsed_time(b_)])
            h2d_b, d2h_b = x_hosts[0].numel() * 4, y_host.numel() * 4
            T_ = frames_per_clip(w)
            ms_step = e2e_ms / n_e2e
            # The host side of a pool box is shared (other tenants' copies cross the same root complex), so a
            # probe taken seconds earlier can read BELOW what the pipeline then sustains (35-39 vs 52 GB/s seen).
            # The link rate is therefore the better of the probe and the pipeline's own sustained rate.
            h2d_link = max(rates["h2d"], h2d_b / (ms_step * 1e-3) / 1e9)
            pcie["h2d_gbs_link"] = h2d_link
            pcie["probe_below_pipeline"] = bool(h2d_link > rates["h2d"])
            link_ms = max(h2d_b / (h2d_link * 1e9), d2h_b / (rates["d2h"] * 1e9)) * 1e3
            e2e = {"value": world * B * T_ * n_e2e / (e2e_ms * 1e-3), "unit": "frames/s",
                   "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b, "ms_per_step": ms_step,
                   "steps": n_e2e, "h2d_gbs_achieved": h2d_b / (ms_step * 1e-3) / 1e9,
                   "link_bound_ms_per_step": link_ms, "frac_of_link": link_ms / ms_step,
                   "path": f"nnaudio_b200.host.HostPipeline: pinned host ({place}) -> {args.e2e_chunks} chunks, "
                           "H2D / kernels / D2H on 3 streams, copies of consecutive calls back to back"}
            del x_hosts, y_host, pipe

    # ------------------------------------------- the metric's other configs --
    others = {}
    if not args.no_workloads:
        del mod
        torch.cuda.empty_cache()
        for name in [n for n in SECONDARY if n != args.workload]:
            try:
                res, m2, _, _, _ = measure(name, steps=args.workload_steps, warmup=3, gather=False)
                del m2
                others[name] = res
            except Exception as e:  # noqa: BLE001  (never cost the headline line)
                others[name] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.empty_cache()

    # --------------------------------- the reference's own cuDNN path, same GPU --
    ref_gpu = {}
    if world == 1 and not args.no_reference_gpu and reference_available():
        for name in [args.workload] + [n for n in ("stft2048", "cfg3") if n != args.workload and not args.no_workloads]:
            try:
                ref_gpu[name] = reference_gpu_leg(name, dev)
            except Exception as e:  # noqa: BLE001
                ref_gpu[name] = {"value": None, "unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.empty_cache()

    if rank == 0:
        T = frames_per_clip(w)
        line = {
            "metric": metric, "value": main["value"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": main["dtype"], "data": "synthetic",
            "config": {
                "workload": f"{args.workload}: {w['desc']}", "per_gpu_batch": B,
                "global_batch": world * B, "frames_per_clip": T,
                "parallelism": f"batch-sharded x{world}" + (
                    f" + gather of the output spectrograms to {args.gather_to} ({GATHER_DESC[gather_impl]}; the "
                    "gather of step i overlaps the transform of step i+1)" if world > 1 else ""),
                "gather": gather_impl if world > 1 else None,
                "l2": main["l2"] + "; one CUDA-event pair around all K steps",
                "kernel_path": os.environ.get("NNAUDIO_B200_PATH", "auto"),
                "sms_reserved_for_gather": reserve if world > 1 else 0,
                "host_cpus": f"{len(local_cpus)} cpus of the GPU's NUMA node" if local_cpus else "unbound",
            },
            "gpu_launches": main["gpu_launches"],
            "clocks": main["clocks"],
            "roofline": main["roofline"],
        }
        if no_gather:
            line["without_gather"] = no_gather
        if e2e:
            line["e2e"] = e2e
            line["pcie"] = pcie
        if others:
            line["workloads"] = others
        if ref_gpu:
            line["reference_gpu"] = ref_gpu
        if world == 1 and not args.no_cpu_baseline:
            try:  # a reported baseline must never cost the measured line
                if local_cpus:
                    try:
                        os.sched_setaffinity(0, range(os.cpu_count() or 1))  # the CPU arm uses every core
                    except OSError:
                        pass
                if reference_available():
                    res = reference_cpu_arm(args.workload, steps=4, warmup=1, budget_s=20.0)
                else:
                    res = cpu_arm(args.workload, steps=8, warmup=1, budget_s=20.0)
                line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port",
                                        "sample": f"failed: {type(e).__name__}: {e}"}
    else:
        line = None
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


if __name__ == "__main__":
    main()
