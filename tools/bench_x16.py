"""fp32 vs bf16 vs fp16 waveform input on the bench.py workloads (one GPU).

Method (that of bench.py): per workload and dtype, rotating input batches larger than the 126 MB L2
in total, warm-up steps, then a CUDA-event-timed window; the three dtypes are alternated round by
round inside one process so that they share the same clocks and neighbours.  Per step it reports the
module call (step ms) and the summed time of the framed-contraction launches (kernel ms, the
library's in-stream event pairs).  The e2e leg times HostPipeline on pinned host batches of each
dtype (what bench.py's e2e number measures, with 16-bit host buffers).  The card's name and power
limit are read in the same call.

    python tools/bench_x16.py [--workloads cfg2,stft2048,...] [--steps 20] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from bench import WORKLOADS, frames_per_clip  # noqa: E402
from helpers import build as build_module  # noqa: E402
from nnaudio_b200 import _C  # noqa: E402
from nnaudio_b200.host import HostPipeline, alloc_pinned  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def time_steps(mod, xs, steps, fwd):
    """(step ms, framed-kernel ms) per step over `steps` calls cycling through `xs`."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _C.profile_read()
    _C.profile_enable(True)
    with torch.no_grad():
        a.record()
        for i in range(steps):
            mod(xs[i % len(xs)], **fwd)
        b.record()
    torch.cuda.synchronize()
    _C.profile_enable(False)
    k_ms, _ = _C.profile_read()
    return a.elapsed_time(b) / steps, k_ms / steps


def bench_workload(name, steps, warmup, rounds):
    w = WORKLOADS[name]
    mod = build_module(w["cls"], w["ctor"]).cuda()
    B, L = w["B"], w["L"]
    gen = torch.Generator(device="cuda").manual_seed(1234)
    xs = {}
    for dn, dt in DTYPES.items():
        nbytes = B * L * torch.finfo(dt).bits // 8
        n_rot = max(3, int(-(-160e6 // nbytes)))
        xs[dn] = [torch.randn(B, L, generator=gen, device="cuda").to(dt) for _ in range(n_rot)]
    with torch.no_grad():
        for dn in DTYPES:
            for i in range(warmup):
                mod(xs[dn][i % len(xs[dn])], **w["fwd"])
    torch.cuda.synchronize()
    runs = {dn: [] for dn in DTYPES}
    for _ in range(rounds):  # alternated: fp32, bf16, fp16, fp32, ...
        for dn in DTYPES:
            runs[dn].append(time_steps(mod, xs[dn], steps, w["fwd"]))
    res = {"desc": w["desc"], "B": B, "L": L, "frames_per_step": B * frames_per_clip(w), "steps": steps,
           "rounds": rounds}
    for dn, r in runs.items():
        step = [s for s, _ in r]
        kern = [k for _, k in r]
        res[dn] = {"step_ms": min(step), "step_ms_all": step, "kernel_ms": min(kern), "kernel_ms_all": kern}
    for dn in ("bf16", "fp16"):
        res[dn]["step_vs_fp32"] = res[dn]["step_ms"] / res["fp32"]["step_ms"]
        res[dn]["kernel_vs_fp32"] = res[dn]["kernel_ms"] / res["fp32"]["kernel_ms"] if res["fp32"]["kernel_ms"] else None
    del xs, mod
    torch.cuda.empty_cache()
    return res


def bench_e2e(name, steps, chunks, rounds):
    w = WORKLOADS[name]
    mod = build_module(w["cls"], w["ctor"]).cuda()
    B, L = w["B"], w["L"]
    res = {"workload": name, "chunks": chunks, "steps": steps, "rounds": rounds}
    legs = {}
    for dn, dt in DTYPES.items():
        x_hosts = [alloc_pinned((B, L), dtype=dt, fill="randn")[0] for _ in range(2)]
        with torch.no_grad():
            y = mod(x_hosts[0][:1].cuda(), **w["fwd"])
        y_host, _ = alloc_pinned((B,) + tuple(y.shape[1:]))
        legs[dn] = (x_hosts, y_host, HostPipeline(mod, chunk_clips=max(1, B // chunks), **w["fwd"]))
        for i in range(3):
            legs[dn][2](x_hosts[i & 1], y_host)
    torch.cuda.synchronize()
    times = {dn: [] for dn in DTYPES}
    for _ in range(rounds):  # alternated: the host link is shared, its rate drifts
        for dn, (x_hosts, y_host, pipe) in legs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(steps):
                pipe(x_hosts[i & 1], y_host)
            b.record()
            torch.cuda.synchronize()
            times[dn].append(a.elapsed_time(b) / steps)
    for dn, (x_hosts, y_host, _) in legs.items():
        ms = min(times[dn])
        h2d = x_hosts[0].numel() * x_hosts[0].element_size()
        res[dn] = {"ms_per_step": ms, "ms_per_step_all": times[dn], "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": y_host.numel() * 4, "h2d_gbs": h2d / (ms * 1e-3) / 1e9}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg2,stft2048,cfg3,cfg4,cfg5,gammatone")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--e2e-chunks", type=int, default=8)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_x16.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_x16 needs a CUDA device")
    torch.cuda.set_device(0)
    t0 = time.time()
    out = {"card": card(), "torch": torch.__version__,
           "method": "CUDA events; per dtype rotating batches > 160 MB in total (> L2); dtypes alternated per "
                     "round, best of rounds reported; kernel_ms = summed framed-contraction launches "
                     "(nnab_profile_read); e2e = HostPipeline on pinned host buffers of the dtype, dtypes "
                     "alternated per round, best of rounds",
           "workloads": {}}
    for name in args.workloads.split(","):
        out["workloads"][name] = bench_workload(name, args.steps, args.warmup, args.rounds)
        r = out["workloads"][name]
        print(f"{name}: step fp32 {r['fp32']['step_ms']:.4f} bf16 {r['bf16']['step_ms']:.4f} "
              f"fp16 {r['fp16']['step_ms']:.4f} ms | kernel fp32 {r['fp32']['kernel_ms']:.4f} "
              f"bf16 {r['bf16']['kernel_ms']:.4f} fp16 {r['fp16']['kernel_ms']:.4f} ms", flush=True)
    out["e2e"] = bench_e2e("cfg2", args.e2e_steps, args.e2e_chunks, args.rounds)
    e = out["e2e"]
    print("e2e cfg2 ms/step: " + " ".join(f"{d} {e[d]['ms_per_step']:.4f}" for d in DTYPES), flush=True)
    out["card_after"] = card()
    out["wall_s"] = time.time() - t0
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
