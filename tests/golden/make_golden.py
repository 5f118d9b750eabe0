"""Generate the golden fixtures by running the UNMODIFIED reference (nnAudio
v0.3.3, imported read-only from ``$NNAUDIO_REF`` = /root/reference/Installation)
on CPU in the build container.  The GPU box has no /root/reference, so the
outputs are committed:

  ref_outputs.npz        reference forward() outputs for tests/golden/cases.py
  ref_buffers.json       sha256 of every state_dict buffer of the case modules
  ref_ground_truths.npz  the reference's own golden vectors, re-encoded from
                         Installation/tests/ground-truths/*.npy (test fixtures,
                         not source code) — pinned by tests/test_cqt.py:94-262

Both .npz files keep a seeded sample of each array's entries (cases.pack_sampled).

(The Combined_Frequency_Periodicity / CFP fixtures have their own generator, make_golden_cfp.py ->
ref_cfp.npz / ref_cfp.json.)

Run:  PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("NNAUDIO_REF", "/root/reference/Installation")
sys.dont_write_bytecode = True
sys.path.insert(0, REF)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "..", "..", "oracle"))

from cases import (CASES, DESIGN_CASES, ERROR_CASES, GRAD_CASES, SWEEP_FORWARD, sweep_input, ISTFT_CASES, ISTFT_GRAD_CASES, REF_GROUND_TRUTHS,  # noqa: E402
                   SWEEP_CTOR, WGRAD_CASES, attribute_surface, istft_spectrogram, loss_weights, make_input,
                   out_key, pack_sampled)

from nnAudio import features as ref_features  # noqa: E402


def make_module(namespace, cls, ctor):
    """CQT1992 has no ``verbose`` argument (and always prints)."""
    import contextlib
    import inspect
    import io
    klass = getattr(namespace, cls)
    kw = dict(ctor)
    if "verbose" in inspect.signature(klass.__init__).parameters:
        kw["verbose"] = False
    with contextlib.redirect_stdout(io.StringIO()):
        return klass(**kw)


def sha(t: torch.Tensor) -> str:
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(a.tobytes()).hexdigest()


def main():
    torch.manual_seed(0)
    outputs, buffers = {}, {}
    for cid, cls, ctor, inp, fwds in CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mod = make_module(ref_features, cls, ctor)
        buffers[cid] = {k: [list(v.shape), sha(v)] for k, v in mod.state_dict().items()
                        if v is not None}
        x = torch.from_numpy(make_input(inp))
        if cid == "stft_default_hop_1d_input":
            x = x[0]
        for kw in fwds:
            with torch.no_grad(), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                y = mod(x, **kw)
            outputs[out_key(cid, kw)] = y.numpy().astype(np.float32)
            print(f"{out_key(cid, kw):60s} {tuple(y.shape)}")
    for cid, cls, ctor in DESIGN_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mod = make_module(ref_features, cls, ctor)
        buffers[cid] = {k: [list(v.shape), sha(v)] for k, v in mod.state_dict().items()
                        if v is not None}
        print(f"{cid:60s} {len(buffers[cid])} buffers")
    for cid, cls, ctor in SWEEP_FORWARD:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mod = make_module(ref_features, cls, ctor)
            x = torch.from_numpy(make_input(sweep_input(cid, cls)))
            with torch.no_grad():
                y = mod(x)
        outputs["sweep|" + cid] = y.numpy().astype(np.float32)
        print(f"{'sweep|' + cid:60s} {tuple(y.shape)}")
    attributes = {}
    for cid, cls, ctor in [(c[0], c[1], c[2]) for c in CASES] + list(DESIGN_CASES):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            attributes[cid] = attribute_surface(make_module(ref_features, cls, ctor))
    with open(os.path.join(HERE, "ref_attributes.json"), "w") as f:
        json.dump(attributes, f, indent=1, sort_keys=True)
    import inspect
    signatures = {}
    for cls in ("STFT", "iSTFT", "MelSpectrogram", "MFCC", "Gammatonegram", "CQT1992v2", "CQT", "CQT2010v2", "VQT",
                "CQT1992", "CQT2010", "Griffin_Lim"):
        klass = getattr(ref_features, cls)
        entry = {}
        for meth in ("__init__", "forward", "inverse"):
            if hasattr(klass, meth) and (meth != "inverse" or "inverse" in klass.__dict__):
                params = list(inspect.signature(getattr(klass, meth)).parameters.values())[1:]
                entry[meth] = [[q.name, None if q.default is inspect.Parameter.empty else repr(q.default)]
                               for q in params]
        signatures[cls] = entry
    with open(os.path.join(HERE, "ref_signatures.json"), "w") as f:
        json.dump(signatures, f, indent=1, sort_keys=True)
    errors = {}
    for cid, cls, ctor, call in ERROR_CASES:
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                mod = make_module(ref_features, cls, ctor)
                if call[0] == "forward":
                    mod(torch.zeros(call[1]), **call[2])
                elif call[0] == "inverse":
                    mod.inverse(torch.zeros(call[1]), **call[2])
            errors[cid] = "ok"
        except Exception as e:  # noqa: BLE001  (the point is to record the type)
            errors[cid] = type(e).__name__
        print(f"{cid:60s} -> {errors[cid]}")
    with open(os.path.join(HERE, "ref_errors.json"), "w") as f:
        json.dump(errors, f, indent=1, sort_keys=True)
    # inverse STFT: waveform outputs of the reference (the spectrogram inputs are regenerated by the tests)
    for case in ISTFT_CASES:
        cid, n_fft, hop, win, kind, spec = case
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if kind == "roundtrip":
                st = ref_features.STFT(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True, verbose=False)
                X = torch.from_numpy(istft_spectrogram(case, st.wsin.numpy(), st.wcos.numpy()))
                with torch.no_grad():
                    y = st.inverse(X, onesided=True, length=spec["length"])
            else:
                im = ref_features.iSTFT(n_fft=n_fft, hop_length=hop, window=win, verbose=False)
                X = torch.from_numpy(istft_spectrogram(case))
                with torch.no_grad():
                    y = im(X, onesided=False)
        outputs[cid + "|y"] = y.numpy().astype(np.float32)
        print(f"{cid:60s} X{tuple(X.shape)} -> y{tuple(y.shape)}")
    # gradient of the inverse STFT w.r.t. its spectrogram input
    for case in ISTFT_GRAD_CASES:
        cid, n_fft, hop, win, kind, spec = case
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if kind == "roundtrip":
                st = ref_features.STFT(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True, verbose=False)
                X = torch.from_numpy(istft_spectrogram(case, st.wsin.numpy(), st.wcos.numpy()))
                X.requires_grad_(True)
                y = st.inverse(X, onesided=True, length=spec["length"])
            else:
                im = ref_features.iSTFT(n_fft=n_fft, hop_length=hop, window=win, verbose=False)
                X = torch.from_numpy(istft_spectrogram(case))
                X.requires_grad_(True)
                y = im(X, onesided=False)
        w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
        (y * w).sum().backward()
        outputs[cid + "|dX"] = X.grad.numpy().astype(np.float32)
        print(f"{cid:60s} X{tuple(X.shape)} y{tuple(y.shape)} -> dX{tuple(X.grad.shape)}")
    # input gradients through the reference's own autograd path
    for cid, cls, ctor, inp, kw in GRAD_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mod = make_module(ref_features, cls, ctor)
        x = torch.from_numpy(make_input(inp)).requires_grad_(True)
        y = mod(x, **kw)
        w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
        (y * w).sum().backward()
        outputs["grad|" + cid] = x.grad.numpy().astype(np.float32)
        print(f"{'grad|' + cid:60s} out{tuple(y.shape)} -> dx{tuple(x.grad.shape)}")
    # gradients of trainable kernels / filterbanks
    for cid, cls, ctor, inp, kw, names in WGRAD_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            mod = make_module(ref_features, cls, ctor)
        x = torch.from_numpy(make_input(inp))
        y = mod(x, **kw)
        w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
        (y * w).sum().backward()
        params = dict(mod.named_parameters())
        for n in names:
            outputs[f"wgrad|{cid}|{n}"] = params[n].grad.numpy().astype(np.float32)
            print(f"{'wgrad|' + cid + '|' + n:60s} {tuple(params[n].grad.shape)}")
    np.savez_compressed(os.path.join(HERE, "ref_outputs.npz"), **pack_sampled(outputs))
    with open(os.path.join(HERE, "ref_buffers.json"), "w") as f:
        json.dump(buffers, f, indent=1, sort_keys=True)

    # the reference's own golden vectors + a self-check that the reference still
    # reproduces them at its own tolerance (tests/test_cqt.py: rtol=atol=1e-3)
    gt_dir = os.path.join(REF, "tests", "ground-truths")
    gts = {}
    for key, (cls, method, kw, transform) in REF_GROUND_TRUTHS.items():
        gt = np.load(os.path.join(gt_dir, key + "-ground-truth.npy"))
        gts[key] = gt.astype(np.float32)
        mod = make_module(ref_features, cls, SWEEP_CTOR)
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y = mod(torch.from_numpy(make_input(("chirp", method))), **kw)
        if transform == "log1e-5":
            y = torch.log(y + 1e-5)
        elif transform == "log1e-2":
            y = torch.log(y + 1e-2)
        ok = np.allclose(y.numpy(), gt, rtol=1e-3, atol=1e-3)
        print(f"{key:40s} gt{gt.shape} ref reproduces: {ok}  maxabs {np.abs(y.numpy()-gt).max():.3e}")
        assert ok, key
    np.savez_compressed(os.path.join(HERE, "ref_ground_truths.npz"), **pack_sampled(gts))
    print("wrote fixtures to", HERE)


if __name__ == "__main__":
    main()
