#!/usr/bin/env python
"""Regenerates docs/API.md from the live signatures of nnaudio_b200.features."""
import contextlib
import inspect
import io
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import nnaudio_b200 as nb  # noqa: E402

REF = {"STFT": "stft.py:66-362", "iSTFT": "stft.py:364-546", "MelSpectrogram": "mel.py:9-194",
       "MFCC": "mel.py:197-329", "Gammatonegram": "gammatone.py:9-194", "CQT1992v2": "cqt.py:561-803",
       "CQT": "cqt.py:1142-1145", "CQT2010v2": "cqt.py:805-1139", "VQT": "vqt.py:9-215",
       "CQT1992": "cqt.py:9-256", "CQT2010": "cqt.py:259-558", "Griffin_Lim": "griffin_lim.py:9-148",
       "Combined_Frequency_Periodicity": "cfp.py:9-246", "CFP": "cfp.py:249-484"}

HEADER = """# API — `nnaudio_b200.features` (generated from the signatures by `python docs/make_api.py`)

Same class names, constructor arguments (names, order, defaults), `forward` signatures, buffer names and public
attributes as `nnAudio.features` v0.3.3 — checked against the unmodified reference by the fixtures in `tests/golden/`
(signatures, buffers bit-identical for 49 + 7 configurations, attribute surface, exception types, outputs ≤1e-4). What differs:

* inputs must be **CUDA** tensors on a B200 (sm_100a); anything else raises — there is no CPU fallback;
* waveform inputs (`STFT.forward`, `MelSpectrogram`, `MFCC`, `Gammatonegram`, the CQTs, `VQT`, `CFP`) may be float32,
  **bfloat16 or float16** (the reference's conv1d would reject a 16-bit waveform against its fp32 kernels); the result
  is float32 and equal to that of the fp32 copy of the same samples, and the input gradient has the input's dtype
  (DESIGN.md §3.10).  Spectrogram inputs (`iSTFT`, `STFT.inverse`, `Griffin_Lim`) stay float32; other dtypes raise;
* multi-GPU: one process per GPU (`nnaudio_b200.parallel.BatchShardedTransform`, INTEGRATION.md) is the fast path;
  `torch.nn.DataParallel`, the reference's own mode, also works (per-device launch attributes and caches);
* `Griffin_Lim.forward(S, rand_phase=None)` takes an optional initial phase (reproducible runs); `device` moves the
  module's buffers at construction, as the reference creates its window there;
* trainable inverse kernels / window of `iSTFT` raise `NotImplementedError` under autograd (no dW path yet);
* `CFP` / `Combined_Frequency_Periodicity` are forward-only (the reference has no parameters there; a waveform that
  requires grad raises `NotImplementedError`); their FFT stages run as dense contractions (DESIGN.md §3.9).

Environment switches: `NNAUDIO_B200_PATH=auto|simt|tcgen05` (kernel family), `NNAUDIO_B200_DECIM_BWD=fir|simt|tc|ola`
(adjoint of the pyramid's FIR stages in training), `NNAB_TALL_BALANCE=0|1` (balanced tile schedule of the CQT1992v2 kernel).

"""


def main():
    out = io.StringIO()
    out.write(HEADER)
    for name, where in REF.items():
        cls = getattr(nb.features, name)
        out.write(f"## `{name}`  — reference `{where}`\n\n```python\n")
        out.write(f"{name}{str(inspect.signature(cls.__init__)).replace('(self, ', '(')}\n")
        for meth in ("forward", "inverse"):
            if meth == "inverse" and meth not in cls.__dict__:
                continue
            out.write(f".{meth}{str(inspect.signature(getattr(cls, meth))).replace('(self, ', '(')}\n")
        out.write("```\n\n")
        doc = inspect.getdoc(cls) or ""
        if doc:
            out.write(doc.split("\n\n")[0].replace("\n", " ") + "\n\n")
        kw = {"Griffin_Lim": dict(n_fft=512)}.get(name, {})
        if "verbose" in inspect.signature(cls.__init__).parameters:
            kw["verbose"] = False
        try:
            with contextlib.redirect_stdout(io.StringIO()), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                mod = cls(**kw)
            bufs = ", ".join(f"`{k}` {tuple(v.shape)}" for k, v in mod.state_dict().items())
            out.write(f"state_dict (defaults): {bufs or '—'}\n\n")
        except ValueError as e:  # CQT1992's own defaults exceed Nyquist, in the reference too
            out.write(f"(the default arguments do not construct, as in the reference: {str(e).split(',')[0]})\n\n")
    with open(os.path.join(ROOT, "docs", "API.md"), "w") as f:
        f.write(out.getvalue())


if __name__ == "__main__":
    main()
