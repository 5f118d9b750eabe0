"""bf16 / fp16 waveform inputs on the GPU (-m gpu; collected last).

Every bf16 and fp16 value is exact in fp32 and splits exactly into bf16 hi + lo, so a module called
on a 16-bit tensor must return exactly (torch.equal) what it returns on the fp32 copy of that tensor
on the same kernel path: fp16 runs the same three MMA terms on the same planes, bf16 drops only the
x_lo * w_hi term, whose operand is zero.  The executed-flop counter shows that drop (2/3 of the fp32
count on the block, dense and tall kernels), so the two-term path is the one being compared."""
import warnings

import pytest
import torch

from cases import CASES, CFP_CASES, make_input
from conftest import record_error
from helpers import build
from nnaudio_b200 import _C
from nnaudio_b200.host import HostPipeline, alloc_pinned

pytestmark = pytest.mark.gpu

DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
FWD = [(c[0], i) for c in CASES for i in range(len(c[4]))]


def _call(mod, x, kw=None):
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **(kw or {}))
    torch.cuda.synchronize()
    return y


def _diff(a, b):
    d = (a.double() - b.double()).abs()
    return float(d.max()), int((d != 0).sum())


@pytest.mark.parametrize("path", ["auto", "simt"])
@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("cid,i", FWD, ids=[f"{c}-{i}" for c, i in FWD])
def test_16bit_input_equals_its_fp32_copy(cid, i, dt, path, monkeypatch):
    case = next(c for c in CASES if c[0] == cid)
    _, cls, ctor, inp, fwds = case
    monkeypatch.setenv("NNAUDIO_B200_PATH", path)
    mod = build(cls, ctor).cuda()
    x16 = torch.from_numpy(make_input(inp)).cuda().to(DTYPES[dt])
    got = _call(mod, x16, fwds[i])
    want = _call(mod, x16.float(), fwds[i])
    assert got.dtype == torch.float32 and got.shape == want.shape
    dmax, n = _diff(got, want)
    record_error("x16_equal", f"{cid}-{i}|{dt}|{path}", max_abs=dmax, n_diff=n)
    assert torch.equal(got, want), (cid, i, dt, path, dmax, n)


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("case", CFP_CASES[:2], ids=[c[0] for c in CFP_CASES[:2]])
def test_cfp_16bit_input_equals_its_fp32_copy(case, dt):
    cid, cls, ctor, inp = case
    mod = build(cls, ctor).cuda()
    x16 = torch.from_numpy(make_input(inp)).cuda().to(DTYPES[dt])
    got, want = _call(mod, x16), _call(mod, x16.float())
    got = got if isinstance(got, tuple) else (got,)
    want = want if isinstance(want, tuple) else (want,)
    for g, w in zip(got, want):
        assert g.dtype == torch.float32
        assert torch.equal(g, w), (cid, dt, _diff(g, w))


# BASELINE-size workloads (bench.py WORKLOADS) in bf16: equality with the fp32 copy + run-to-run identity
BIG = {
    "cfg2": ("MelSpectrogram", dict(sr=22050, n_fft=2048, hop_length=512, n_mels=128), (64, 220500)),
    "stft2048": ("STFT", dict(n_fft=2048, hop_length=512, sr=22050, output_format="Magnitude"), (64, 220500)),
    "cfg3": ("CQT1992v2", dict(sr=44100, n_bins=84, bins_per_octave=12, fmin=32.7), (128, 441000)),
    "cfg4": ("CQT2010v2", dict(sr=22050, n_bins=88), (256, 661500)),
    "cfg5": ("MFCC", dict(sr=16000), (1024, 80000)),
    "gammatone": ("Gammatonegram", dict(sr=22050, n_fft=2048, hop_length=512, n_bins=64), (64, 220500)),
}


@pytest.mark.parametrize("name", sorted(BIG))
def test_full_size_bf16_equal_and_repeatable(name):
    cls, ctor, shape = BIG[name]
    mod = build(cls, ctor).cuda()
    x16 = torch.randn(*shape, generator=torch.Generator().manual_seed(11)).to(torch.bfloat16).cuda()
    a = _call(mod, x16).clone()
    junk = torch.randn(1 << 22, device="cuda")  # perturb allocator / L2 state between the repetitions
    b = _call(mod, x16).clone()
    del junk
    want = _call(mod, x16.float())
    dmax, n = _diff(a, want)
    record_error("x16_full_size", name, max_abs=dmax, n_diff=n)
    assert torch.equal(a, b), (name, "bf16 run twice", _diff(a, b))
    assert torch.equal(a, want), (name, dmax, n)


# one problem per tensor-core kernel family: executed MMA flops of bf16 input = 2/3 of fp32's
FLOP_CASES = {
    "block": ("STFT", dict(n_fft=2048, hop_length=512, output_format="Magnitude"), (4, 44100)),
    "dense": ("STFT", dict(n_fft=1024, hop_length=256, window="hamming", output_format="Complex"), (4, 44100)),
    "tall": ("CQT1992v2", dict(sr=44100, n_bins=84, bins_per_octave=12, fmin=32.7), (4, 88200)),
}


@pytest.mark.parametrize("kernel", sorted(FLOP_CASES))
def test_bf16_runs_two_of_three_mma_terms(kernel):
    cls, ctor, shape = FLOP_CASES[kernel]
    mod = build(cls, ctor).cuda()
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(3)).cuda()
    flops = {}
    _call(mod, x)  # packed bases built outside the counted calls
    _C.profile_enable(True)
    try:
        for dt, t in (("fp32", x), ("bf16", x.to(torch.bfloat16)), ("fp16", x.to(torch.float16))):
            _C.profile_read_exec_flops()
            _call(mod, t)
            flops[dt] = _C.profile_read_exec_flops()
            _C.profile_read()
    finally:
        _C.profile_enable(False)
    assert flops["fp32"] > 0
    assert 3.0 * flops["bf16"] == 2.0 * flops["fp32"], flops
    assert flops["fp16"] == flops["fp32"], flops


GRAD_CASES = [
    ("STFT", dict(n_fft=512, hop_length=128, output_format="Complex"), (2, 8000)),
    ("MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40), (2, 8000)),
    ("CQT1992v2", dict(sr=22050, fmin=220, n_bins=48, hop_length=256), (2, 16000)),
    ("CQT2010v2", dict(sr=22050, n_bins=84), (2, 32768)),
]


@pytest.mark.parametrize("dt", sorted(DTYPES))
@pytest.mark.parametrize("case", GRAD_CASES, ids=[c[0] for c in GRAD_CASES])
def test_input_gradient_of_16bit_input(case, dt):
    cls, ctor, shape = case
    dtype = DTYPES[dt]
    mod = build(cls, ctor).cuda()
    x16 = torch.randn(*shape, generator=torch.Generator().manual_seed(5)).to(dtype).cuda().requires_grad_()
    x32 = x16.detach().float().requires_grad_()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y16, y32 = mod(x16), mod(x32)
    w = torch.randn(y32.shape, generator=torch.Generator().manual_seed(6)).cuda()
    (y16 * w).sum().backward()
    (y32 * w).sum().backward()
    torch.cuda.synchronize()
    assert y16.dtype == torch.float32 and torch.equal(y16.detach(), y32.detach())
    assert x16.grad.dtype == dtype and x16.grad.shape == x16.shape
    got, want = x16.grad.float(), x32.grad.to(dtype).float()
    # the dX kernels accumulate with fp32 atomics: the fp32 gradients may differ in their last bits,
    # which can move the rounding to 16 bits by one unit
    ulp = 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11
    scale = float(x32.grad.abs().max())
    err = float(((got - want).abs() - 2 * ulp * want.abs()).max())
    record_error("x16_grad", f"{cls}|{dt}", max_abs_beyond_ulp=err, grad_max=scale)
    assert err <= 1e-5 * scale, (cls, dt, err, scale)


@pytest.mark.parametrize("dt", sorted(DTYPES))
def test_host_pipeline_16bit_input(dt):
    mod = build("MelSpectrogram", dict(sr=22050, n_fft=2048, hop_length=512, n_mels=128)).cuda()
    x_host, _ = alloc_pinned((13, 44100), dtype=DTYPES[dt], fill="randn")
    assert x_host.dtype == DTYPES[dt] and x_host.is_pinned()
    want = _call(mod, x_host.cuda().float())
    pipe = HostPipeline(mod, chunk_clips=4)
    for _ in range(2):
        y = pipe(x_host)
        torch.cuda.current_stream().synchronize()
        assert y.dtype == torch.float32 and y.is_pinned()
        assert torch.equal(y, want.cpu())


@pytest.mark.parametrize("dt", [torch.float64, torch.int16, torch.uint8])
def test_other_cuda_dtypes_raise_before_any_launch(dt):
    mod = build("STFT", dict(n_fft=512, hop_length=128)).cuda()
    _call(mod, torch.zeros(2, 8000, device="cuda"))  # the packed basis (one launch, cached) exists
    x = torch.zeros(2, 8000, dtype=dt, device="cuda")
    before = _C.launch_count()
    with pytest.raises(RuntimeError, match="float32, bfloat16 or float16"):
        _call(mod, x)
    assert _C.launch_count() == before
