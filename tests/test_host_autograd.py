"""CPU checks of the differentiable host compositions (SURVEY.md §8f next #1 / #2): the CQT2010v2 /
VQT octave loop and the iSTFT adjoint, with float64 torch stand-ins in place of the C entry points
(tests/cpu_kernels.py).  What is verified here is the wiring — stage order, per-stage padding,
octave concatenation, shared-bank gradient accumulation, one-sided mirror fold, window-sum-square
adjoint — against the gradients the reference's autograd produced (tests/golden/ref_outputs.npz).
The same cases run through the real kernels in tests/test_backward.py / tests/test_istft.py (gpu)."""
import warnings

import numpy as np
import pytest
import torch

from helpers import build, istft_input, ref_outputs, rel_errors  # noqa: E402 (sets sys.path)
import cpu_kernels  # noqa: E402
import nnaudio_b200.features as nb  # noqa: E402
from cases import CASES, GRAD_CASES, ISTFT_GRAD_CASES, WGRAD_CASES, loss_weights, make_input, out_key

HOST_COMPOSED = ("CQT2010v2", "VQT", "CQT1992", "CQT2010")
PYRAMID_GRAD = [c for c in GRAD_CASES if c[1] in HOST_COMPOSED]
PYRAMID_WGRAD = [c for c in WGRAD_CASES if c[1] in HOST_COMPOSED]
V1_FORWARD = [c for c in CASES if c[1] in ("CQT1992", "CQT2010")]


@pytest.mark.parametrize("case", PYRAMID_GRAD, ids=[c[0] for c in PYRAMID_GRAD])
def test_pyramid_input_gradient_wiring(case, monkeypatch):
    cpu_kernels.install(monkeypatch)
    cid, cls, ctor, inp, kw = case
    mod = build(cls, ctor)
    x = torch.from_numpy(make_input(inp)).requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **kw)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
    (y * w).sum().backward()
    want = ref_outputs()["grad|" + cid]
    emax, el2 = rel_errors(want.pick(x.grad.numpy()), want.values)
    assert x.grad.shape == want.shape and emax < 2e-5 and el2 < 2e-5, (cid, emax, el2)


@pytest.mark.parametrize("case", PYRAMID_WGRAD, ids=[c[0] for c in PYRAMID_WGRAD])
def test_pyramid_shared_bank_gradient_wiring(case, monkeypatch):
    cpu_kernels.install(monkeypatch)
    cid, cls, ctor, inp, kw, names = case
    mod = build(cls, ctor)
    x = torch.from_numpy(make_input(inp))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **kw)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
    (y * w).sum().backward()
    params = dict(mod.named_parameters())
    for n in names:
        want = ref_outputs()[f"wgrad|{cid}|{n}"]
        emax, el2 = rel_errors(want.pick(params[n].grad.numpy()), want.values)
        assert params[n].grad.shape == want.shape and emax < 2e-5 and el2 < 2e-5, (cid, n, emax, el2)


@pytest.mark.parametrize("case", ISTFT_GRAD_CASES, ids=[c[0] for c in ISTFT_GRAD_CASES])
def test_istft_spectrogram_gradient_wiring(case, monkeypatch):
    cpu_kernels.install(monkeypatch)
    cid, n_fft, hop, win, kind, spec = case
    X = torch.from_numpy(istft_input(case)).requires_grad_(True)
    if kind == "roundtrip":
        st = build("STFT", dict(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True))
        y = st.inverse(X, onesided=True, length=spec["length"])
    else:
        y = build("iSTFT", dict(n_fft=n_fft, hop_length=hop, window=win))(X, onesided=False)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
    (y * w).sum().backward()
    want = ref_outputs()[cid + "|dX"]
    emax, el2 = rel_errors(want.pick(X.grad.numpy()), want.values)
    assert X.grad.shape == want.shape and emax < 2e-5 and el2 < 2e-5, (cid, emax, el2)


@pytest.mark.parametrize("case", V1_FORWARD, ids=[c[0] for c in V1_FORWARD])
def test_folded_bank_reproduces_two_stage_reference(case, monkeypatch):
    """CQT1992 / CQT2010: the single folded time-domain bank (DFT rows x spectral kernels) gives the
    reference's two-stage result — values, sign conventions of each output format, normalisation."""
    cpu_kernels.install(monkeypatch)
    cid, cls, ctor, inp, fwds = case
    mod = build(cls, ctor)
    x = torch.from_numpy(make_input(inp)).requires_grad_(True)  # routes through the octave loop
    for kw in fwds:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y = mod(x, **kw).detach().numpy()
        want = ref_outputs()[out_key(cid, kw)]
        assert y.shape == want.shape
        if kw.get("output_format") == "Phase":
            mag = np.hypot(*np.moveaxis(mod(x, **dict(kw, output_format="Complex")).detach().numpy(), -1, 0))
            keep = want.pick(mag > 1e-3 * mag.max())
            assert np.abs(want.pick(y)[keep] - want.values[keep]).max() < 2e-3, (cid, kw)
            continue
        emax, el2 = rel_errors(want.pick(y), want.values)
        assert emax < 2e-5 and el2 < 2e-5, (cid, kw, emax, el2)


@pytest.mark.parametrize("taps,n,L", [(256, 2, 1000), (256, 2, 1001), (256, 4, 4099), (255, 3, 777),
                                      (16, 5, 64), (9, 2, 9)])
def test_polyphase_decimation_adjoint_equals_conv1d_autograd(taps, n, L, monkeypatch):
    """The backward of a decimating FIR stage is computed as n interleaved stride-1 FIRs with the
    polyphase components (no overlap-add): identical to autograd through
    conv1d(stride=n, padding=(taps-1)//2) (utils.py:73-100), for even/odd taps and lengths."""
    from nnaudio_b200.features.cqt import _decimate_autograd

    cpu_kernels.install(monkeypatch)
    g = torch.Generator().manual_seed(taps * 131 + n)
    fir = torch.randn(1, 1, taps, generator=g)
    x = torch.randn(3, L, generator=g)
    holder = torch.nn.Module()

    a = x.clone().requires_grad_(True)
    y = _decimate_autograd(holder, "t", a, fir, n)
    b = x.clone().requires_grad_(True)
    y_ref = torch.nn.functional.conv1d(b[:, None, :].double(), fir.double(), stride=n,
                                       padding=(taps - 1) // 2)[:, 0, :]
    assert y.shape == y_ref.shape
    w = torch.randn(y.shape, generator=g)
    (y * w).sum().backward()
    (y_ref * w.double()).sum().backward()
    assert torch.allclose(y.double(), y_ref, rtol=1e-5, atol=1e-5)
    assert torch.allclose(a.grad.double(), b.grad.double(), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("cls,ctor", [
    ("CQT1992", dict(sr=8000, hop_length=64, fmin=200, n_bins=12, trainable_CQT=True)),
    ("CQT2010", dict(sr=8000, hop_length=64, fmin=200, n_bins=24, trainable_CQT=True, earlydownsample=False)),
], ids=["cqt1992", "cqt2010"])
def test_sgd_loop_never_reuses_a_stale_packed_bank(cls, ctor, monkeypatch):
    """ADVICE r1 (high): the folded v1 bank is a recomputed temporary (``_version`` 0 every step);
    after an optimiser step the allocator may give the new fold the old address, and a cache keyed
    on (data_ptr, _version) alone would then hand back the packing of the *previous* parameters.
    Every step's dx must equal that of a fresh module holding the same parameters."""
    import copy

    cpu_kernels.install(monkeypatch)
    torch.manual_seed(0)
    mod = build(cls, ctor)
    opt = torch.optim.SGD(mod.parameters(), lr=5e-2)
    x0 = torch.randn(2, 4096)
    for step in range(5):
        x = x0.clone().requires_grad_(True)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y = mod(x)
        opt.zero_grad()
        y.square().sum().backward()
        fresh = build(cls, ctor)
        fresh.load_state_dict(copy.deepcopy(mod.state_dict()))
        xf = x0.clone().requires_grad_(True)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            yf = fresh(xf)
        yf.square().sum().backward()
        emax, el2 = rel_errors(x.grad.numpy(), xf.grad.numpy())
        assert el2 < 1e-6, (cls, step, emax, el2)
        opt.step()


def test_recomputed_bank_with_recycled_address_is_repacked(monkeypatch):
    """Direct form of the above: different non-leaf banks that land on the SAME address with
    ``_version`` 0 must not share a cached packing.  The collision is forced by making every tensor
    report one address (the float64 stand-ins never look at addresses)."""
    from nnaudio_b200.features.cqt import _framed_complex_autograd

    cpu_kernels.install(monkeypatch)
    monkeypatch.setattr(torch.Tensor, "data_ptr", lambda self: 0x1234)
    mod = torch.nn.Module()
    p = torch.nn.Parameter(torch.randn(6, 64))
    q = torch.nn.Parameter(torch.randn(6, 64))
    x0 = torch.randn(1, 1024)
    grads = []
    for scale in (1.0, 3.0, -2.0, 0.5):
        w_re, w_im = p * scale, q * scale          # fresh temporaries, _version 0
        x = x0.clone().requires_grad_(True)
        c = _framed_complex_autograd(mod, "t", x, w_re, w_im, 32, True, 0)
        c.square().sum().backward()
        grads.append(x.grad.clone() / scale ** 2)   # dx of |c|^2 is quadratic in the bank
    for g in grads[1:]:
        emax, el2 = rel_errors(g.numpy(), grads[0].numpy())
        assert el2 < 1e-6, (emax, el2)


def test_trainable_forward_stft_can_call_inverse_in_training_mode(monkeypatch):
    """ADVICE r1: ``inverse`` only reads kernel_*_inv / window_mask (buffers), so a
    STFT(trainable=True, iSTFT=True) must be able to invert under autograd; a trainable iSTFT
    kernel (no dW path) still refuses."""
    cpu_kernels.install(monkeypatch)
    st = nb.STFT(n_fft=128, hop_length=32, trainable=True, iSTFT=True, verbose=False)
    x = torch.randn(2, 1024)
    X = st(x, output_format="Complex")
    y = st.inverse(X, length=1024)
    assert y.shape == (2, 1024)
    y.square().sum().backward()
    assert st.wsin.grad is not None and torch.isfinite(st.wsin.grad).all()
    inv = nb.iSTFT(n_fft=128, hop_length=32, trainable_kernels=True, verbose=False)
    with pytest.raises(NotImplementedError):
        inv(X.detach(), onesided=True)
