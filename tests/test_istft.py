"""Inverse STFT (SURVEY.md §8f next #2): STFT.inverse / iSTFT against the reference
outputs recorded by tests/golden/make_golden.py, the fp64 oracle, and the reference's own
round-trip test (Installation/tests/test_stft.py:28-54: STFT -> inverse recovers x)."""
import pytest
import torch

from helpers import istft_input, oracle, ref_outputs, rel_errors
from cases import ISTFT_CASES, ISTFT_GRAD_CASES, loss_weights

import nnaudio_b200 as nb


def _module(n_fft, hop, win, kind):
    if kind == "roundtrip":
        return nb.STFT(n_fft=n_fft, hop_length=hop, window=win, iSTFT=True, verbose=False)
    return nb.iSTFT(n_fft=n_fft, hop_length=hop, window=win, verbose=False)


def _oracle(mod, kind, X, hop, length):
    if kind == "roundtrip":
        return oracle.istft(X, mod.kernel_cos_inv.cpu().numpy(), mod.kernel_sin_inv.cpu().numpy(),
                            mod.window_mask.cpu().numpy(), hop, True, True, length)
    return oracle.istft(X, mod.kernel_cos.cpu().numpy(), mod.kernel_sin.cpu().numpy(),
                        mod.window_mask.cpu().numpy(), hop, True, False, length)


@pytest.mark.parametrize("case", ISTFT_CASES, ids=[c[0] for c in ISTFT_CASES])
def test_oracle_istft_matches_reference(case):
    cid, n_fft, hop, win, kind, spec = case
    mod = _module(n_fft, hop, win, kind)
    X = istft_input(case)
    want = ref_outputs()[cid + "|y"]
    got = _oracle(mod, kind, X, hop, spec.get("length"))
    assert got.shape == want.shape
    emax, el2 = rel_errors(want.pick(got), want.values)
    assert emax < 2e-5 and el2 < 5e-6, (cid, emax, el2)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ISTFT_CASES, ids=[c[0] for c in ISTFT_CASES])
def test_cuda_istft_matches_reference_and_oracle(case):
    cid, n_fft, hop, win, kind, spec = case
    mod = _module(n_fft, hop, win, kind).cuda()
    X = istft_input(case)
    want = ref_outputs()[cid + "|y"]
    Xd = torch.from_numpy(X).cuda()
    with torch.no_grad():
        if kind == "roundtrip":
            y = mod.inverse(Xd, onesided=True, length=spec["length"])
        else:
            y = mod(Xd, onesided=False)
    torch.cuda.synchronize()
    got = y.cpu().numpy()
    assert got.shape == want.shape, "output length must follow the reference's slicing exactly"
    orc = _oracle(mod, kind, X, hop, spec.get("length"))
    for name, g, ref in (("reference", want.pick(got), want.values), ("oracle", got, orc)):
        emax, el2 = rel_errors(g, ref)
        assert emax < 1e-4 and el2 < 1e-4, (cid, name, emax, el2)


@pytest.mark.gpu
def test_stft_inverse_round_trip_recovers_waveform():
    """tests/test_stft.py:41-54 in the reference: randn(4, 16000), rtol 1e-5 / atol 1e-3."""
    x = torch.randn(4, 16000, device="cuda")
    for n_fft, hop in ((512, 128), (2048, 512)):
        st = nb.STFT(n_fft=n_fft, hop_length=hop, iSTFT=True, verbose=False).cuda()
        with torch.no_grad():
            y = st.inverse(st(x, output_format="Complex"), onesided=True, length=x.shape[-1])
        assert y.shape == x.shape
        assert torch.allclose(y, x, rtol=1e-5, atol=1e-3), (y - x).abs().max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ISTFT_GRAD_CASES, ids=[c[0] for c in ISTFT_GRAD_CASES])
def test_cuda_istft_spectrogram_gradient_matches_reference_autograd(case):
    """dL/dX through the inverse (reference: autograd through conv2d + fold, stft.py:15-63)."""
    cid, n_fft, hop, win, kind, spec = case
    mod = _module(n_fft, hop, win, kind).cuda()
    X = torch.from_numpy(istft_input(case)).cuda().requires_grad_(True)
    if kind == "roundtrip":
        y = mod.inverse(X, onesided=True, length=spec["length"])
    else:
        y = mod(X, onesided=False)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape))).cuda()
    (y * w).sum().backward()
    torch.cuda.synchronize()
    want = ref_outputs()[cid + "|dX"]
    got = X.grad.cpu().numpy()
    assert got.shape == want.shape
    emax, el2 = rel_errors(want.pick(got), want.values)
    assert emax < 1e-4 and el2 < 1e-4, (cid, emax, el2)


def test_inverse_requires_istft_flag_and_complex_input():
    st = nb.STFT(n_fft=256, verbose=False)
    with pytest.raises(NameError, match="iSTFT=True"):
        st.inverse(torch.zeros(1, 129, 10, 2))
    st2 = nb.STFT(n_fft=256, iSTFT=True, verbose=False)
    with pytest.raises(AssertionError, match="complex"):
        st2.inverse(torch.zeros(1, 129, 10))
    sd = nb.iSTFT(n_fft=256, verbose=False).state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        "kernel_sin": (256, 1, 256, 1), "kernel_cos": (256, 1, 256, 1), "window_mask": (1, 256, 1)}
