"""CPU checks of bf16 / fp16 waveform inputs: which dtypes are accepted, that the modules hand the
16-bit tensor itself (not an fp32 copy) to the library with the matching nnab_dtype code and return
fp32, that input gradients come back in the input's dtype, and that the C ABI's *_ex entry points
reject an unknown dtype on the host.  The kernels themselves are checked on the GPU by
tests/test_zz_gpu_x16.py."""
import ctypes
import warnings

import pytest
import torch

import cpu_kernels
from helpers import build
from nnaudio_b200 import _C

X16 = (torch.bfloat16, torch.float16)

# module -> the _C forward wrapper its inference path calls
MODULES = [
    ("STFT", dict(n_fft=256, hop_length=64), "stft_forward"),
    ("MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40), "stft_filterbank_forward"),
    ("MFCC", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40), "mfcc_forward"),
    ("Gammatonegram", dict(sr=16000, n_fft=512, hop_length=128, n_bins=32), "stft_filterbank_forward"),
    ("CQT1992v2", dict(sr=22050, fmin=220, n_bins=24, hop_length=256), "cqt1992v2_forward"),
    ("CQT2010v2", dict(sr=22050, n_bins=24, fmin=220, earlydownsample=False), "cqt_pyramid_forward"),
    ("VQT", dict(sr=22050, n_bins=24, fmin=220, earlydownsample=False), "cqt_pyramid_forward"),
    ("CQT1992", dict(sr=22050, fmin=220, n_bins=24), "cqt1992v2_forward"),
    ("CQT2010", dict(sr=22050, n_bins=24, fmin=220, earlydownsample=False), "cqt_pyramid_forward"),
]


def _recording(monkeypatch, name, seen):
    fn = getattr(_C, name)

    def wrapper(x, *args, **kwargs):
        seen.append(_C.x_dtype_code(x.dtype))
        return fn(x, *args, **kwargs)

    monkeypatch.setattr(_C, name, wrapper)


def test_dtype_codes():
    assert _C.x_dtype_code(torch.float32) == _C.DTYPE_F32 == 0
    assert _C.x_dtype_code(torch.bfloat16) == _C.DTYPE_BF16 == 1
    assert _C.x_dtype_code(torch.float16) == _C.DTYPE_F16 == 2
    for dt in (torch.float64, torch.int16, torch.uint8):
        with pytest.raises(RuntimeError, match="float32, bfloat16 or float16"):
            _C.x_dtype_code(dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.int16, torch.uint8, torch.bfloat16])
def test_other_dtypes_and_cpu_tensors_raise_before_any_c_call(dt):
    mod = build("STFT", dict(n_fft=256, hop_length=64))
    x = torch.zeros(2, 4000, dtype=dt)
    before = _C.launch_count()
    with pytest.raises(RuntimeError):
        mod(x)
    assert _C.launch_count() == before


@pytest.mark.parametrize("dt", X16, ids=["bf16", "fp16"])
@pytest.mark.parametrize("cls,ctor,wrapper", MODULES, ids=[m[0] for m in MODULES])
def test_modules_pass_16bit_input_and_return_fp32(cls, ctor, wrapper, dt, monkeypatch):
    cpu_kernels.install(monkeypatch)
    seen = []
    _recording(monkeypatch, wrapper, seen)
    mod = build(cls, ctor)
    x = torch.randn(2, 8000, generator=torch.Generator().manual_seed(1)).to(dt)
    with torch.no_grad(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x)
        y32 = mod(x.float())
    assert seen == [_C.x_dtype_code(dt), _C.DTYPE_F32]
    assert y.dtype == torch.float32
    assert torch.equal(y, y32)  # the stand-ins compute in float64 from the exact fp32 values


@pytest.mark.parametrize("dt", X16, ids=["bf16", "fp16"])
@pytest.mark.parametrize("cls,ctor", [
    ("STFT", dict(n_fft=256, hop_length=64, output_format="Complex")),
    ("MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40)),
    ("CQT1992v2", dict(sr=22050, fmin=220, n_bins=24, hop_length=256)),
    ("CQT2010v2", dict(sr=22050, n_bins=24, fmin=220, earlydownsample=False)),
    ("CQT2010v2", dict(sr=22050, n_bins=24, fmin=220, trainable=True)),
])
def test_input_gradient_has_the_input_dtype(cls, ctor, dt, monkeypatch):
    cpu_kernels.install(monkeypatch)
    mod = build(cls, ctor)
    x = torch.randn(2, 8000, generator=torch.Generator().manual_seed(2)).to(dt).requires_grad_()
    x32 = x.detach().float().requires_grad_()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y, y32 = mod(x), mod(x32)
    assert y.dtype == torch.float32
    y.sum().backward()
    y32.sum().backward()
    assert x.grad.dtype == dt and x.grad.shape == x.shape
    assert torch.equal(x.grad, x32.grad.to(dt))


_EX = ["nnab_stft_forward_ex", "nnab_stft_filterbank_forward_ex", "nnab_mfcc_forward_ex",
       "nnab_cqt1992v2_forward_ex", "nnab_cqt_pyramid_forward_ex"]


@pytest.mark.parametrize("name", _EX)
def test_ex_argtypes_extend_the_fp32_entry_point(name):
    plain = _C.SIGNATURES[name[:-3]]
    res, args = _C.SIGNATURES[name]
    assert res is ctypes.c_int and args == plain[1] + [ctypes.c_int]
    assert getattr(_C.lib(), name).argtypes == args


def test_unknown_dtype_is_einval_on_the_host():
    """A well-formed call with an unknown x_dtype returns NNAB_EINVAL before any device work (with a
    valid dtype the same call on a GPU-less host would reach the device and fail there)."""
    lib = _C.lib()
    P = ctypes.c_void_p
    x = w = out = P(256)  # never dereferenced
    before = lib.nnab_launch_count()

    def stft(dt):
        return lib.nnab_stft_forward_ex(x, 4, 4000, 4000, w, w, None, 512, 257, 128, 1, 0, 0, 0.0, out, 32,
                                        None, 0, 0, None, dt)

    for dt in (3, -1, 99):
        assert stft(dt) == -1
        assert lib.nnab_stft_filterbank_forward_ex(x, 4, 4000, 4000, w, w, None, 512, 257, 128, 1, 0, 0.0,
                                                   2.0, w, 128, None, out, 32, None, 0, 0, None, dt) == -1
        assert lib.nnab_mfcc_forward_ex(x, 4, 4000, 4000, w, w, None, 512, 257, 128, 1, 0, 0.0, 2.0, w, 128,
                                        None, 1e-10, 1.0, 80.0, w, 20, out, 32, None, 0, 0, None, dt) == -1
        assert lib.nnab_cqt1992v2_forward_ex(x, 4, 4000, 4000, w, w, None, None, None, 24, 512, 128, 1, 0,
                                             None, 1.0, 0, 0.0, out, 32, None, 0, 0, None, dt) == -1
        banks = (P * 1)(256)
        widths = (ctypes.c_int32 * 1)(512)
        assert lib.nnab_cqt_pyramid_forward_ex(x, 4, 4000, 4000, 1, banks, banks, None, widths, 12, w, None,
                                               None, None, 1, 128, 0, 12, None, 1.0, 0, 0.0, out, 32, None,
                                               0, 0, None, dt) == -1
    assert lib.nnab_launch_count() == before
    if not torch.cuda.is_available():
        assert stft(_C.DTYPE_BF16) in (-2, -4)  # a valid dtype goes on to the device (and finds none)
