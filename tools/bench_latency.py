#!/usr/bin/env python
"""Small-batch latency (VERDICT r1 "host overhead per forward"): BASELINE cfg1 (STFT n_fft=512 hop=256, one
1 s clip @ 16 kHz) and a single 10 s clip through MelSpectrogram / CQT1992v2, per call: wall-clock of the
Python call (host side: argument checks, ctypes, workspace allocation, tensor-map encoding, launches) and
device time between CUDA events, ours and the unmodified reference on the same GPU.
"""
import json
import os
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def measure(fn, n=200, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    # host: time to ISSUE the call (no sync inside the loop)
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    host_us = (time.perf_counter() - t0) / n * 1e6
    torch.cuda.synchronize()
    # latency: one call at a time, issue -> result complete
    lat = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        lat.append(time.perf_counter() - t0)
    lat.sort()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return {"host_issue_us": round(host_us, 1), "latency_median_us": round(lat[n // 2] * 1e6, 1),
            "device_back_to_back_us": round(a.elapsed_time(b) / n * 1e3, 1)}


def main():
    warnings.simplefilter("ignore")
    import nnaudio_b200 as nb

    ref_features = None
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "nnAudio")):
        sys.path.insert(0, ref_dir)
        from nnAudio import features as ref_features
    cases = [
        ("cfg1 STFT n_fft=512 hop=256, 1 x 1 s @ 16 kHz", "STFT", dict(n_fft=512, hop_length=256, sr=16000), (1, 16000)),
        ("MelSpectrogram n_fft=2048 128 mels, 1 x 10 s @ 22.05 kHz", "MelSpectrogram",
         dict(sr=22050, n_fft=2048, hop_length=512, n_mels=128), (1, 220500)),
        ("CQT1992v2 84 bins, 1 x 10 s @ 44.1 kHz", "CQT1992v2", dict(sr=44100, n_bins=84, fmin=32.7), (1, 441000)),
    ]
    out = {}
    for name, cls, ctor, shape in cases:
        x = torch.randn(*shape, device="cuda")
        mod = getattr(nb.features, cls)(verbose=False, **ctor).cuda()
        entry = {}
        with torch.no_grad():
            entry["ours"] = measure(lambda: mod(x))
            if ref_features is not None:
                ref = getattr(ref_features, cls)(verbose=False, **ctor).cuda()
                entry["reference_gpu"] = measure(lambda: ref(x), n=50, warmup=5)
        out[name] = entry
    print(json.dumps(out))


if __name__ == "__main__":
    main()
