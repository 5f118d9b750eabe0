"""Dense filterbanks on the tensor cores (-m gpu): Gammatonegram (and any mel bank that is not banded) as
block-partial STFT -> bf16 hi/lo operand planes (FMT_PLANES epilogue) -> second tcgen05 contraction with the
re-indexed bank (FMT_REALPAIR), csrc/nnab_api.cu.  NNAB_FB_PLANES=1 selects it, 0 the round-1 path (fp32
(B, F, T) power spectrogram + CUDA-core filterbank GEMM).  Checked against the CPU oracle / the reference
fixtures at the 1e-4 bar, against the old path, and for bit-repeatability."""
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import record_error
from helpers import build, ref_outputs, rel_errors, run_oracle

pytestmark = pytest.mark.gpu


def _forward(mod, x, planes):
    os.environ["NNAB_FB_PLANES"] = "1" if planes else "0"
    try:
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y = mod(x)
        torch.cuda.synchronize()
    finally:
        os.environ.pop("NNAB_FB_PLANES", None)
    return y


CONFIGS = {
    "gammatone_default": ("Gammatonegram", dict(sr=22050), (2, 22050)),
    "gammatone_small": ("Gammatonegram", dict(sr=22050, n_fft=1024, n_bins=32, hop_length=256), (3, 8000)),
    "gammatone_odd_bins_hop_half": ("Gammatonegram", dict(sr=16000, n_fft=512, n_bins=33, hop_length=256), (2, 6000)),
    "gammatone_power1_constant_pad": ("Gammatonegram", dict(sr=22050, n_fft=2048, n_bins=64, power=1.0,
                                                            pad_mode="constant"), (1, 30000)),
}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_dense_bank_on_tensor_cores_matches_oracle_and_old_path(name):
    cls, ctor, shape = CONFIGS[name]
    mod = build(cls, ctor).cuda()
    xn = np.random.RandomState(11).standard_normal(shape).astype(np.float32)
    x = torch.from_numpy(xn).cuda()
    old = _forward(mod, x, False)
    new = _forward(mod, x, True)
    again = _forward(mod, x, True)
    assert new.shape == old.shape
    assert torch.equal(new, again), "no atomics on this path: two runs must be bit-identical"
    ref = run_oracle(cls, mod, xn, {})
    for tag, y in (("planes", new), ("old", old)):
        emax, el2 = rel_errors(y.cpu().numpy(), ref)
        record_error("fb_planes", f"{name}|{tag}|oracle", max_rel=emax, l2_rel=el2, tol=1e-4)
        assert emax < 1e-4 and el2 < 1e-4, (name, tag, emax, el2)
    emax, el2 = rel_errors(new.cpu().numpy(), old.cpu().numpy())
    assert emax < 5e-5 and el2 < 5e-5, (name, emax, el2)


def test_reference_fixture_gammatone_default():
    """The committed output of the unmodified reference (tests/golden/cases.py: gammatone_default)."""
    from cases import CASES, make_input
    from helpers import out_key

    cid, cls, ctor, inp, fwds = next(c for c in CASES if c[0] == "gammatone_default")
    mod = build(cls, ctor).cuda()
    y = _forward(mod, torch.from_numpy(make_input(inp)).cuda(), True)
    want = ref_outputs()[out_key(cid, fwds[0])]
    emax, el2 = rel_errors(want.pick(y.cpu().numpy()), want.values)
    assert emax < 1e-4 and el2 < 1e-4, (emax, el2)


def test_signed_dense_mel_bank():
    """A dense bank with negative weights (e.g. a trained mel basis): the real-GEMM output keeps the sign."""
    mod = build("MelSpectrogram", dict(sr=22050, n_fft=1024, hop_length=256, n_mels=40)).cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    with torch.no_grad():
        mod.mel_basis.copy_(torch.randn(mod.mel_basis.shape, generator=g, device="cuda") * 0.05)
    xn = np.random.RandomState(12).standard_normal((2, 9000)).astype(np.float32)
    x = torch.from_numpy(xn).cuda()
    new = _forward(mod, x, True)
    old = _forward(mod, x, False)
    ref = run_oracle("MelSpectrogram", mod, xn, {})
    assert (ref < 0).any()
    for y in (new, old):
        emax, el2 = rel_errors(y.cpu().numpy(), ref)
        assert emax < 1e-4 and el2 < 1e-4, (emax, el2)


def test_cfg2_shape_gammatone_planes_equals_old_path():
    mod = build("Gammatonegram", dict(sr=22050, n_fft=2048, n_bins=64, hop_length=512)).cuda()
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(64, 220500, generator=g, device="cuda")
    old = _forward(mod, x, False)
    new = _forward(mod, x, True)
    d = (new - old).abs().max().item() / old.abs().max().item()
    assert d < 5e-5, d
