#!/usr/bin/env python
"""Gammatonegram timing on one B200 (cfg2 shape: 64 x 10 s @ 22.05 kHz, n_fft 2048, hop 512, 64 bins):
dense bank on the tensor cores (NNAB_FB_PLANES=1: operand planes + second tcgen05 contraction), the
round-1 path (NNAB_FB_PLANES=0: fp32 power spectrogram + CUDA-core GEMM), the STFT power alone for scale,
and the unmodified reference on the same GPU when oracle/_ref is present.  CUDA events after warm-up.
"""
import json
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def timed(fn, steps=20, warmup=5):
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
    warnings.simplefilter("ignore")
    import nnaudio_b200 as nb

    xs = [torch.randn(64, 220500, device="cuda") for _ in range(3)]  # 169 MB of inputs > L2
    it = [0]

    def nxt():
        it[0] = (it[0] + 1) % 3
        return xs[it[0]]

    mod = nb.features.Gammatonegram(sr=22050, n_fft=2048, n_bins=64, hop_length=512, verbose=False).cuda()
    stft = nb.features.STFT(n_fft=2048, hop_length=512, sr=22050, output_format="Magnitude", verbose=False).cuda()
    out = {"workload": "Gammatonegram 64 bins, n_fft 2048, hop 512, 64 x 10 s @ 22.05 kHz"}
    with torch.no_grad():
        frames = 64 * mod(xs[0]).shape[-1]
        for tag, env in (("planes_ms", "1"), ("old_path_ms", "0")):
            os.environ["NNAB_FB_PLANES"] = env
            out[tag] = timed(lambda: mod(nxt()))
        os.environ.pop("NNAB_FB_PLANES", None)
        out["default_ms"] = timed(lambda: mod(nxt()))
        out["stft_magnitude_ms"] = timed(lambda: stft(nxt()))
    out["frames"] = frames
    out["planes_frames_per_s"] = frames / out["planes_ms"] * 1e3
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "nnAudio")):
        sys.path.insert(0, ref_dir)
        from nnAudio.features.gammatone import Gammatonegram as Ref

        ref = Ref(sr=22050, n_fft=2048, n_bins=64, hop_length=512, verbose=False).cuda()
        with torch.no_grad():
            out["reference_gpu_ms"] = timed(lambda: ref(nxt()), steps=3, warmup=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
