"""The whole Python host layer on the CPU: every golden CASES configuration runs through OUR modules
(inference path, no autograd) with float64 stand-ins in place of the C wrappers
(tests/cpu_kernels.py, semantics of include/nnab.h), and must reproduce the unmodified reference's
outputs.  What this pins without a GPU is the module -> C-call contract: which basis, hop, padding
mode and padding amount, scale tensors / factors, sqrt-eps, power, dB parameters, DCT rows, octave
banks, early-downsample factor and output format each module hands to the library, plus the caches in
between.  The kernels behind those calls are pinned by the `-m gpu` tests against the same fixtures."""
import warnings

import numpy as np
import pytest
import torch

from helpers import (CASES, build, case_input, is_phase, istft_input, out_key, phase_to_unit, ref_outputs,
                     rel_errors)
import cpu_kernels


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_module_to_library_contract_reproduces_reference(case, monkeypatch):
    cpu_kernels.install(monkeypatch)
    cid, cls, ctor, inp, fwds = case
    mod = build(cls, ctor)
    x = torch.from_numpy(np.ascontiguousarray(case_input(cid, inp)))
    for kw in fwds:
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            got = mod(x, **kw).numpy()
        want = ref_outputs()[out_key(cid, kw)]
        assert got.shape == want.shape, (cid, kw)
        if is_phase(kw):
            with torch.no_grad(), warnings.catch_warnings():
                warnings.simplefilter("ignore")
                mag = mod(x, **dict(kw, output_format="Magnitude")).numpy()
            keep = want.pick(mag > 1e-3 * mag.max())
            d = np.abs(phase_to_unit(cls, want.pick(got))[keep] - phase_to_unit(cls, want.values)[keep]).max()
            assert d < 2e-3, (cid, kw, d)
            continue
        tol = 2e-4 if cls == "MFCC" else 2e-5   # dB of near-zero mel powers amplifies the reference's fp32 noise
        emax, el2 = rel_errors(want.pick(got), want.values)
        assert emax < tol and el2 < tol, (cid, kw, emax, el2)


from cases import ISTFT_CASES  # noqa: E402


@pytest.mark.parametrize("case", ISTFT_CASES, ids=[c[0] for c in ISTFT_CASES])
def test_inverse_modules_reproduce_reference(case, monkeypatch):
    """STFT.inverse / iSTFT host layer (kernel selection, one-sided flag, length slicing)."""
    import nnaudio_b200 as nb

    cpu_kernels.install(monkeypatch)
    cid, n_fft, hop, win, kind, spec = case
    X = torch.from_numpy(istft_input(case))
    with torch.no_grad():
        if kind == "roundtrip":
            st = nb.STFT(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True, verbose=False)
            y = st.inverse(X, onesided=True, length=spec["length"])
        else:
            y = nb.iSTFT(n_fft=n_fft, hop_length=hop, window=win, verbose=False)(X, onesided=False)
    want = ref_outputs()[cid + "|y"]
    assert tuple(y.shape) == want.shape
    emax, el2 = rel_errors(want.pick(y.numpy()), want.values)
    assert emax < 2e-5 and el2 < 2e-5, (cid, emax, el2)


from cases import SWEEP_FORWARD, make_input, sweep_input  # noqa: E402
from helpers import run_oracle  # noqa: E402


@pytest.mark.parametrize("case", SWEEP_FORWARD, ids=[c[0] for c in SWEEP_FORWARD])
def test_constructor_sweep_forward_matches_reference(case, monkeypatch):
    """21 further configurations (windows, frequency scales, htk / un-normalised mel, 24 / 36 bins per
    octave, filter_scale, VQT gammas, no early downsampling ...): our host layer (float64 stand-ins
    for the C wrappers) AND the oracle against the unmodified reference's default-format output."""
    cid, cls, ctor = case
    x = make_input(sweep_input(cid, cls))
    want = ref_outputs()["sweep|" + cid]
    mod = build(cls, ctor)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        orc = run_oracle(cls, mod, x, {})
        cpu_kernels.install(monkeypatch)
        with torch.no_grad():
            got = mod(torch.from_numpy(x)).numpy()
    tol = 4e-4 if cls == "MFCC" else 2e-5
    for name, y in (("host layer", got), ("oracle", orc)):
        assert y.shape == want.shape, (cid, name)
        emax, el2 = rel_errors(want.pick(y), want.values)
        assert emax < tol and el2 < tol, (cid, name, emax, el2)
