"""Test helpers: build a case module, drive the CPU oracle from the module's
buffers, and the parity metrics of SURVEY.md §7 step 0 / BASELINE.md §4."""
from __future__ import annotations

import contextlib
import inspect
import io
import json
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
for p in (ROOT, GOLDEN, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nnaudio_oracle as oracle  # noqa: E402  (test infrastructure only)
from cases import (CASES, REF_GROUND_TRUTHS, SWEEP_CTOR, istft_spectrogram, make_input,  # noqa: E402,F401
                   out_key, sample_index)

import nnaudio_b200 as nb  # noqa: E402

_REF_OUT = None
_REF_GT = None
_REF_BUF = None


class Sampled:
    """A stored reference array: its full ``shape`` and its ``values`` at the flat indices ``idx``
    (tests/golden/cases.py: ``sample_index``; they include the entries of max |a|, max a and min a).
    Compare a full-size result with ``pick(result)`` against ``values``."""

    def __init__(self, key, shape, peaks, values):
        self.shape = tuple(int(s) for s in shape)
        self.idx = sample_index(key, self.shape, peaks)
        self.values = values
        assert values.shape == self.idx.shape, key

    def pick(self, a):
        """The stored entries of ``a``: an array of the full size (unit axes may differ), or a mask whose
        shape lacks the trailing (real, imag) axis of a complex-format output."""
        a = np.asarray(a)
        if a.shape != self.shape and a.shape + (2,) == self.shape:
            a = np.broadcast_to(a[..., None], self.shape)
        assert a.size == int(np.prod(self.shape)), (a.shape, self.shape)
        return a.reshape(-1)[self.idx]


def _load_sampled(name):
    d = np.load(os.path.join(GOLDEN, name))
    return {k: Sampled(k, d[k + "|shape"], d[k + "|peaks"], d[k])
            for k in d.files if not k.endswith(("|shape", "|peaks"))}


def ref_outputs():
    global _REF_OUT
    if _REF_OUT is None:
        _REF_OUT = _load_sampled("ref_outputs.npz")
    return _REF_OUT


def ref_ground_truths():
    global _REF_GT
    if _REF_GT is None:
        _REF_GT = _load_sampled("ref_ground_truths.npz")
    return _REF_GT


def istft_input(case):
    """The spectrogram the reference inverted for an ISTFT case (cases.ISTFT_CASES / ISTFT_GRAD_CASES)."""
    cid, n_fft, hop, win, kind, spec = case
    if kind == "module":
        return istft_spectrogram(case)
    st = build("STFT", dict(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True))
    return istft_spectrogram(case, st.wsin.detach().cpu().numpy(), st.wcos.detach().cpu().numpy())


def ref_buffers():
    global _REF_BUF
    if _REF_BUF is None:
        with open(os.path.join(GOLDEN, "ref_buffers.json")) as f:
            _REF_BUF = json.load(f)
    return _REF_BUF


def build(cls: str, ctor: dict):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        klass = getattr(nb.features, cls)
        kw = dict(ctor)
        if "verbose" in inspect.signature(klass.__init__).parameters:
            kw["verbose"] = False
        with contextlib.redirect_stdout(io.StringIO()):  # CQT1992 always prints, like the reference
            return klass(**kw)


def rel_errors(a: np.ndarray, b: np.ndarray):
    """(max|a-b| / max|b|, ||a-b||_2 / ||b||_2) in float64."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    d = a - b
    return (float(np.abs(d).max() / max(np.abs(b).max(), 1e-30)),
            float(np.linalg.norm(d) / max(np.linalg.norm(b), 1e-30)))


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def run_oracle(cls: str, mod, x: np.ndarray, kw: dict, dtype=np.float64):
    """Evaluate the CPU oracle with the buffers / configuration of ``mod``
    (one of OUR modules, on any device)."""
    fmt = kw.get("output_format")
    norm = kw.get("normalization_type", "librosa")
    if cls == "STFT":
        return oracle.stft(x, _np(mod.wsin), _np(mod.wcos), mod.stride, mod.center, mod.pad_mode,
                           fmt or mod.output_format, mod.trainable, mod.freq_bins, dtype)
    if cls in ("MelSpectrogram", "Gammatonegram"):
        fb = mod.mel_basis if cls == "MelSpectrogram" else mod.gammatone_basis
        st = mod.stft
        return oracle.melspectrogram(x, _np(st.wsin), _np(st.wcos), _np(fb), st.stride, mod.power,
                                     st.center, st.pad_mode, st.trainable, dtype)
    if cls == "MFCC":
        ml = mod.melspec_layer
        st = ml.stft
        return oracle.mfcc(x, _np(st.wsin), _np(st.wcos), _np(ml.mel_basis), st.stride,
                           mod.n_mfcc, ml.power, float(mod.amin[0]), float(mod.ref[0]), mod.top_db,
                           st.center, st.pad_mode, dtype)
    if cls in ("CQT1992v2", "CQT"):
        return oracle.cqt1992v2(x, _np(mod.cqt_kernels_real), _np(mod.cqt_kernels_imag),
                                _np(mod.lenghts), mod.hop_length, mod.center, mod.pad_mode,
                                fmt or mod.output_format, norm, mod.trainable, dtype)
    if cls == "CQT2010v2":
        early = _np(mod.early_downsample_filter) if mod.earlydownsample else None
        return oracle.cqt2010v2(x, _np(mod.cqt_kernels_real), _np(mod.cqt_kernels_imag),
                                _np(mod.lowpass_filter), _np(mod.lenghts), mod.hop_length,
                                mod.n_bins, mod.n_octaves, mod.pad_mode, early,
                                mod.downsample_factor, fmt or mod.output_format, norm,
                                mod.trainable, dtype)
    if cls == "VQT":
        early = _np(mod.early_downsample_filter) if mod.earlydownsample else None
        banks = [(_np(getattr(mod, f"cqt_kernels_real_{i}")), _np(getattr(mod, f"cqt_kernels_imag_{i}")))
                 for i in range(mod.n_octaves)]
        return oracle.vqt(x, banks, _np(mod.lowpass_filter), _np(mod.lenghts), mod.hop_length,
                          mod.n_bins, mod.pad_mode, early, mod.downsample_factor,
                          fmt or mod.output_format, norm, mod.trainable, dtype)
    if cls == "CQT1992":
        return oracle.cqt1992(x, _np(mod.cqt_kernels_real), _np(mod.cqt_kernels_imag), _np(mod.wcos),
                              _np(mod.wsin), _np(mod.lenghts), mod.hop_length, mod.center,
                              mod.pad_mode, fmt or mod.output_format, norm, dtype)
    if cls == "CQT2010":
        early = _np(mod.early_downsample_filter) if mod.earlydownsample else None
        return oracle.cqt2010(x, _np(mod.cqt_kernels_real), _np(mod.cqt_kernels_imag), _np(mod.wcos),
                              _np(mod.wsin), _np(mod.lowpass_filter), _np(mod.lenghts),
                              mod.hop_length, mod.n_bins, mod.n_octaves, mod.pad_mode, early,
                              mod.downsample_factor, fmt or mod.output_format, norm, dtype)
    raise ValueError(cls)


def case_input(cid, inp):
    x = make_input(inp)
    return x[0] if cid == "stft_default_hop_1d_input" else x


def is_phase(kw):
    return kw.get("output_format") == "Phase"


def phase_to_unit(cls, y):
    """Compare phases as unit vectors: STFT 'Phase' is an angle (wraps at +-pi),
    CQT 'Phase' already is (cos, sin)."""
    if cls == "STFT":
        return np.stack((np.cos(y), np.sin(y)), -1)
    return y
