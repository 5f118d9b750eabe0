"""Gradients w.r.t. the input waveform (SURVEY.md §8f next #1, the dX half) against the
reference's autograd (x.grad recorded by tests/golden/make_golden.py on CPU)."""
import warnings

import pytest
import torch

from helpers import build, ref_outputs, rel_errors
from cases import GRAD_CASES, WGRAD_CASES, loss_weights, make_input

pytestmark = pytest.mark.gpu

_ERRORS = {}


@pytest.fixture(scope="module", autouse=True)
def _dump_errors():
    """Leave the measured gradient errors next to the other GPU evidence (gpurun_out/)."""
    yield
    import json
    import os
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        family = os.environ.get("NNAUDIO_B200_PATH", "auto")  # forward kernel family of this run
        with open(os.path.join(out, f"backward_errors_{family}.json"), "w") as f:
            json.dump(_ERRORS, f, indent=1, sort_keys=True)
    except OSError:
        pass


def _tol(cls):
    # MFCC: the dB + top_db clamp amplifies; everything else holds the 1e-4 bar (measured worst
    # case of the pyramid training path: 6.1e-5, profiles/r01_backward_errors_auto.json)
    return 1e-4  # north_star bar for every module, MFCC included (measured: 3e-7 .. 3e-6, profiles/r02_parity_errors.json)


@pytest.mark.parametrize("case", GRAD_CASES, ids=[c[0] for c in GRAD_CASES])
def test_input_gradient_matches_reference_autograd(case):
    cid, cls, ctor, inp, kw = case
    mod = build(cls, ctor).cuda()
    x = torch.from_numpy(make_input(inp)).cuda().requires_grad_(True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **kw)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape))).cuda()
    (y * w).sum().backward()
    torch.cuda.synchronize()
    want = ref_outputs()["grad|" + cid]
    got = x.grad.cpu().numpy()
    assert got.shape == want.shape
    emax, el2 = rel_errors(want.pick(got), want.values)
    _ERRORS[cid] = {"max_rel": emax, "l2_rel": el2}
    tol = _tol(cls)
    assert emax < tol and el2 < tol, (cid, emax, el2)
    # the differentiable path and the fused inference path must agree on the forward value
    with torch.no_grad():
        y0 = mod(x.detach(), **kw)
    e2, _ = rel_errors(y.detach().cpu().numpy(), y0.cpu().numpy())
    assert e2 < 1e-4


def test_gradient_flows_to_upstream_module():
    """A waveform produced by a trainable layer receives gradients through the spectrogram."""
    lin = torch.nn.Linear(64, 4096).cuda()
    spec = build("MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40)).cuda()
    z = torch.randn(3, 64, device="cuda")
    loss = spec(lin(z)).log1p().mean()
    loss.backward()
    assert lin.weight.grad is not None and torch.isfinite(lin.weight.grad).all()
    assert lin.weight.grad.abs().max() > 0


@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c[0] for c in WGRAD_CASES])
def test_trainable_kernel_gradients_match_reference_autograd(case):
    """trainable=True / trainable_mel / trainable_STFT: parameter gradients (dW) against the
    reference's autograd through conv1d + matmul."""
    cid, cls, ctor, inp, kw, names = case
    mod = build(cls, ctor).cuda()
    x = torch.from_numpy(make_input(inp)).cuda()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **kw)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape))).cuda()
    (y * w).sum().backward()
    torch.cuda.synchronize()
    params = dict(mod.named_parameters())
    for n in names:
        want = ref_outputs()[f"wgrad|{cid}|{n}"]
        got = params[n].grad.cpu().numpy()
        assert got.shape == want.shape, n
        emax, el2 = rel_errors(want.pick(got), want.values)
        _ERRORS[f"{cid}|{n}"] = {"max_rel": emax, "l2_rel": el2}
        assert emax < _tol(cls) and el2 < _tol(cls), (cid, n, emax, el2)


def test_training_step_reduces_loss_with_trainable_stft():
    """A few SGD steps on the Fourier kernels themselves (the reference's headline feature)."""
    torch.manual_seed(0)
    spec = build("STFT", dict(n_fft=256, hop_length=64, trainable=True, output_format="Magnitude")).cuda()
    x = torch.randn(4, 4000, device="cuda")
    target = torch.rand(4, 129, 63, device="cuda")
    opt = torch.optim.SGD(spec.parameters(), lr=1e-4)
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss = ((spec(x) - target) ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < losses[0]
