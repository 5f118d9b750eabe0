#!/usr/bin/env python
"""CFP timing on one B200 (not part of bench.py's line): our dense-contraction formulation
(nnaudio_b200.features.CFP) and, when oracle/_ref is present, the unmodified reference module on the same
GPU (torch.stft + torch.fft through cuFFT), same input, CUDA events after warm-up.

    python tools/bench_cfp.py [--batch 16] [--seconds 10] [--steps 10]
"""
import argparse
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def timed(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    warnings.simplefilter("ignore")
    import nnaudio_b200 as nb

    L = int(16000 * args.seconds)
    x = torch.randn(args.batch, L, device="cuda")
    ours = nb.features.CFP().cuda()
    with torch.no_grad():
        y = ours(x)
        ms = timed(lambda: ours(x), args.steps)
    frames = args.batch * y.shape[-1]
    out = {"workload": f"CFP default (fr=2, fs=16000, hop=320), {args.batch} x {args.seconds:g} s", "frames": frames,
           "ours_ms": ms, "ours_frames_per_s": frames / ms * 1e3}
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "nnAudio")):
        import scipy.signal
        import scipy.signal.windows

        if not hasattr(scipy.signal, "blackmanharris"):
            scipy.signal.blackmanharris = scipy.signal.windows.blackmanharris  # removed SciPy alias
        sys.path.insert(0, ref_dir)
        from nnAudio.features.cfp import CFP as RefCFP

        ref = RefCFP().cuda()
        with torch.no_grad():
            z = ref(x)
            out["reference_gpu_ms"] = timed(lambda: ref(x), args.steps)
        d = (y - z).abs().max().item() / z.abs().max().item()
        out["max_rel_vs_reference_gpu"] = d
    print(json.dumps(out))


if __name__ == "__main__":
    main()
