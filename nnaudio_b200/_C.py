"""ctypes binding of ``libnnab.so`` (C ABI in ``include/nnab.h``).

PyTorch is used only for device memory and the current CUDA stream; every
compute call goes through the C ABI with raw device pointers.  There is no
CPU / eager fallback: if the library is missing, or a tensor is not a CUDA
tensor of a supported dtype (fp32; waveform inputs also bf16 / fp16), the call
fails loudly.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnnab.so")

PAD_REFLECT, PAD_CONSTANT = 0, 1
FMT_MAGNITUDE, FMT_COMPLEX, FMT_PHASE_ANGLE, FMT_PHASE_UNIT = 0, 1, 2, 3
PATH_AUTO, PATH_SIMT, PATH_TCGEN05 = 0, 1, 2
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2  # nnab_dtype: element type of a waveform input

# waveform element types the forward entry points read (outputs stay fp32)
X_DTYPES = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float16: DTYPE_F16}

_PATH_NAMES = {"auto": PATH_AUTO, "simt": PATH_SIMT, "tcgen05": PATH_TCGEN05}

# every symbol include/nnab.h declares: (restype, argtypes)
_P = c_void_p
SIGNATURES = {
    "nnab_abi_version": (c_int, []),
    "nnab_strerror": (c_char_p, [c_int]),
    "nnab_last_cuda_error": (c_char_p, []),
    "nnab_launch_count": (c_uint64, []),
    "nnab_set_sm_reserve": (c_int, [c_int]),
    "nnab_profile_enable": (None, [c_int]),
    "nnab_profile_read": (c_int, [_P, _P]),
    "nnab_profile_read_exec_flops": (c_int, [_P]),
    "nnab_balanced_launch_count": (c_uint64, []),
    "nnab_pack_tile_n": (c_int, [c_int]),
    "nnab_packed_basis_bytes": (c_size_t, [c_int, c_int]),
    "nnab_pack_basis": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "nnab_stft_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int]),
    "nnab_stft_forward": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
         c_float, _P, c_int64, _P, c_size_t, c_int, _P],
    ),
    "nnab_filterbank_table_bytes": (c_size_t, [c_int]),
    "nnab_build_filterbank_table": (c_int, [_P, c_int, c_int, _P, _P, _P]),
    "nnab_filterbank_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "nnab_stft_filterbank_forward": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float,
         c_float, _P, c_int, _P, _P, c_int64, _P, c_size_t, c_int, _P],
    ),
    "nnab_mfcc_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "nnab_mfcc_forward": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float,
         c_float, _P, c_int, _P, c_float, c_float, c_float, _P, c_int, _P, c_int64, _P, c_size_t,
         c_int, _P],
    ),
    "nnab_cqt1992v2_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int]),
    "nnab_cqt1992v2_forward": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
         _P, c_float, c_int, c_float, _P, c_int64, _P, c_size_t, c_int, _P],
    ),
    "nnab_packed_istft_bytes": (c_size_t, [c_int, c_int]),
    "nnab_pack_istft_basis": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P]),
    "nnab_istft_workspace_bytes": (c_size_t, [c_int64, c_int, c_int64, c_int, c_int]),
    "nnab_istft_forward": (
        c_int,
        [_P, c_int64, c_int, c_int64, _P, _P, c_int, c_int, c_int, c_int64, _P, c_int64, _P,
         c_size_t, _P],
    ),
    "nnab_packed_adjoint_bytes": (c_size_t, [c_int, c_int]),
    "nnab_pack_adjoint_basis": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "nnab_framed_backward_input_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "nnab_framed_backward_input": (
        c_int,
        [_P, c_int64, c_int, c_int64, _P, c_int, c_int, c_int, c_int, _P, c_int64, _P, c_size_t, _P],
    ),
    "nnab_framed_backward_weight_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "nnab_framed_backward_weight": (
        c_int,
        [_P, _P, c_int64, c_int64, c_int64, c_int, c_int64, c_int, c_int, c_int, c_int, _P, _P,
         c_size_t, _P],
    ),
    "nnab_pack_basis_ex": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P]),
    "nnab_block_layout_ok": (c_int, [c_int, c_int]),
    "nnab_stream_write_value32": (c_int, [_P, _P, ctypes.c_uint32]),
    "nnab_stream_wait_value32_geq": (c_int, [_P, _P, ctypes.c_uint32]),
    "nnab_packed_block_bytes": (c_size_t, [c_int, c_int]),
    "nnab_pack_basis_block": (c_int, [c_int, c_int, _P, _P]),
    "nnab_debug_varn_plan": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "nnab_fir_decimate": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int, c_int, _P, c_int64, _P]),
    "nnab_fir_decimate_adjoint": (
        c_int, [_P, c_int64, c_int64, c_int64, _P, c_int, c_int, _P, c_int64, _P]),
    "nnab_packed_fir_bytes": (c_size_t, [c_int, c_int]),
    "nnab_pack_fir": (c_int, [_P, c_int, c_int, _P, _P]),
    "nnab_stft_forward_ex": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
         c_float, _P, c_int64, _P, c_size_t, c_int, _P, c_int],
    ),
    "nnab_stft_filterbank_forward_ex": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float,
         c_float, _P, c_int, _P, _P, c_int64, _P, c_size_t, c_int, _P, c_int],
    ),
    "nnab_mfcc_forward_ex": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float,
         c_float, _P, c_int, _P, c_float, c_float, c_float, _P, c_int, _P, c_int64, _P, c_size_t,
         c_int, _P, c_int],
    ),
    "nnab_cqt1992v2_forward_ex": (
        c_int,
        [_P, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
         _P, c_float, c_int, c_float, _P, c_int64, _P, c_size_t, c_int, _P, c_int],
    ),
    "nnab_cqt_pyramid_forward_ex": (
        c_int,
        [_P, c_int64, c_int64, c_int64, c_int, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_int, c_int,
         c_int, c_int, _P, c_float, c_int, c_float, _P, c_int64, _P, c_size_t, c_int, _P, c_int],
    ),
    "nnab_cqt_pyramid_workspace_bytes": (
        c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int, c_int]),
    "nnab_cqt_pyramid_forward": (
        c_int,
        [_P, c_int64, c_int64, c_int64, c_int, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_int, c_int,
         c_int, c_int, _P, c_float, c_int, c_float, _P, c_int64, _P, c_size_t, c_int, _P],
    ),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load ``libnnab.so`` once; raise (never fall back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: the CUDA extension must be built first "
                "(python -c 'import __graft_entry__ as g; g.build()' or "
                "nnaudio_b200/csrc/build.sh). nnaudio_b200 has no CPU fallback."
            )
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if a declared symbol is missing
            fn.restype = res
            fn.argtypes = args
        if handle.nnab_abi_version() != 1:
            raise ImportError("libnnab.so ABI version mismatch")
        _lib = handle
    return _lib


def default_path() -> int:
    """Kernel family selector; ``NNAUDIO_B200_PATH=auto|simt|tcgen05``."""
    return _PATH_NAMES[os.environ.get("NNAUDIO_B200_PATH", "auto").lower()]


def resolve_path(path) -> int:
    if path is None:
        return default_path()
    if isinstance(path, str):
        return _PATH_NAMES[path.lower()]
    return int(path)


def launch_count() -> int:
    return int(lib().nnab_launch_count())


def balanced_launch_count() -> int:
    """Tall-A CQT launches that ran the balanced (shared-tile) schedule since load."""
    return int(lib().nnab_balanced_launch_count())


def set_sm_reserve(n_sms: int) -> int:
    """Keep ``n_sms`` SMs out of the persistent kernels' grids (for a concurrent collective)."""
    return int(lib().nnab_set_sm_reserve(int(n_sms)))


def profile_enable(on: bool):
    lib().nnab_profile_enable(1 if on else 0)


def profile_read():
    """(summed ms, launches) of the framed-contraction kernel since the last read."""
    ms = ctypes.c_double(0.0)
    n = c_uint64(0)
    _check(lib().nnab_profile_read(ctypes.byref(ms), ctypes.byref(n)), "nnab_profile_read")
    return ms.value, int(n.value)


def profile_read_exec_flops() -> float:
    v = ctypes.c_double(0.0)
    _check(lib().nnab_profile_read_exec_flops(ctypes.byref(v)), "nnab_profile_read_exec_flops")
    return float(v.value)


def _check(rc: int, what: str):
    if rc != 0:
        L = lib()
        msg = L.nnab_strerror(rc).decode()
        if rc == -4:
            msg += ": " + L.nnab_last_cuda_error().decode()
        raise RuntimeError(f"{what} failed: {msg} (status {rc})")


def _dev_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on {t.device}: nnaudio_b200 runs only on CUDA (sm_100a) tensors; "
            "there is no CPU fallback"
        )
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32, got {t.dtype}")
    return t


def x_dtype_code(dtype: torch.dtype, name: str = "x") -> int:
    """nnab_dtype of a waveform input; RuntimeError for any dtype the kernels do not read."""
    code = X_DTYPES.get(dtype)
    if code is None:
        raise RuntimeError(f"{name} must be float32, bfloat16 or float16, got {dtype}")
    return code


def _dev_wave(t: torch.Tensor, name: str) -> int:
    """A CUDA waveform tensor (fp32, bf16 or fp16) -> its nnab_dtype code."""
    if isinstance(t, torch.Tensor) and t.dtype == torch.float32:
        _dev_f32(t, name)  # the fp32 inputs' check, as for every other tensor
        return DTYPE_F32
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(
            f"{name} is on {t.device}: nnaudio_b200 runs only on CUDA (sm_100a) tensors; "
            "there is no CPU fallback"
        )
    return x_dtype_code(t.dtype, name)


def _ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else None


def _stream(device) -> c_void_p:
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _workspace(nbytes: int, device):
    if nbytes <= 0:
        return None, 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return ws, nbytes


MAX_BATCH = 65535  # clips per C call (the pre-pass kernels put the clip index in gridDim.y)


# --------------------------------------------------------------------------- #
# caller-provided output buffers (multi-GPU gather: the kernels write straight into the slice of a
# symmetric-memory buffer; see nnaudio_b200.parallel)
# --------------------------------------------------------------------------- #
import threading as _threading

_OUT = _threading.local()


class output_into:
    """``with _C.output_into(buf): y = module(x)`` -- the forward call that runs inside writes its
    result into ``buf`` (a contiguous fp32 CUDA tensor of exactly the result's shape) instead of
    allocating one, and returns ``buf``.  Used once: the first matching allocation takes it."""

    def __init__(self, buf: torch.Tensor):
        self.buf = buf

    def __enter__(self):
        _OUT.buf = self.buf
        return self

    def __exit__(self, *exc):
        _OUT.buf = None
        return False


def _new_out(shape, device) -> torch.Tensor:
    buf = getattr(_OUT, "buf", None)
    if buf is not None and tuple(buf.shape) == tuple(shape) and buf.device == device \
            and buf.dtype == torch.float32 and buf.is_contiguous():
        _OUT.buf = None
        return buf
    return torch.empty(shape, dtype=torch.float32, device=device)


def _batch_chunked(fn):
    """Forward wrappers take any batch size: more than ``MAX_BATCH`` clips are run as several C
    calls on the same stream and concatenated (every op of the path is per-clip, including the
    MFCC ``top_db`` clamp)."""
    import functools

    @functools.wraps(fn)
    def wrapper(x, *args, **kwargs):
        if x.dim() != 2 or x.shape[0] <= MAX_BATCH:
            return fn(x, *args, **kwargs)
        return torch.cat([fn(x[i:i + MAX_BATCH], *args, **kwargs)
                          for i in range(0, x.shape[0], MAX_BATCH)], 0)

    return wrapper


def _rows(x: torch.Tensor):
    """(B, L) CUDA waveform (fp32, bf16 or fp16) with unit inner stride ->
    (tensor, B, L, pitch in elements, nnab_dtype code)."""
    code = _dev_wave(x, "x")
    if x.dim() != 2:
        raise ValueError("internal: expected (B, L)")
    if x.stride(-1) != 1 or (x.shape[0] > 1 and x.stride(0) < x.shape[1]):
        x = x.contiguous()
    pitch = x.stride(0) if x.shape[0] > 1 else x.shape[1]
    return x, x.shape[0], x.shape[1], pitch, code


# --------------------------------------------------------------------------- #
# basis packing (tcgen05 path)
# --------------------------------------------------------------------------- #
LAYOUT_DENSE, LAYOUT_GROUPS = 0, 3


def pack_basis(w_re: torch.Tensor, w_im: torch.Tensor, layout: int = LAYOUT_DENSE):
    """bf16 hi/lo split of an (F, K) fp32 basis pair in the TMA/UMMA layout, or
    ``None`` when the library has no tcgen05 kernel for it.  ``layout``: LAYOUT_GROUPS for long
    nested CQT banks (per-K-block-width / tall-A kernels)."""
    L = lib()
    F, K = w_re.shape
    nbytes = L.nnab_packed_basis_bytes(F, K)
    if nbytes == 0:
        return None
    packed = torch.empty(nbytes, dtype=torch.uint8, device=w_re.device)
    with torch.cuda.device(w_re.device):
        if layout == LAYOUT_DENSE:
            rc = L.nnab_pack_basis(_ptr(w_re), _ptr(w_im), F, K, _ptr(packed), _stream(w_re.device))
        else:
            rc = L.nnab_pack_basis_ex(_ptr(w_re), _ptr(w_im), F, K, int(layout), _ptr(packed),
                                      _stream(w_re.device))
        _check(rc, "nnab_pack_basis")
    return packed


def stream_write_value32(stream: torch.cuda.Stream, addr: int, value: int):
    """Stream-ordered 32-bit store to a (possibly peer-mapped) device address: a front-end memory
    operation, no kernel and no SM (cuStreamWriteValue32)."""
    _check(lib().nnab_stream_write_value32(ctypes.c_void_p(stream.cuda_stream), ctypes.c_void_p(addr),
                                           int(value) & 0xFFFFFFFF), "nnab_stream_write_value32")


def stream_wait_value32_geq(stream: torch.cuda.Stream, addr: int, value: int):
    """Work queued on ``stream`` after this waits until (int32)(*addr - value) >= 0 (cuStreamWaitValue32)."""
    _check(lib().nnab_stream_wait_value32_geq(ctypes.c_void_p(stream.cuda_stream), ctypes.c_void_p(addr),
                                              int(value) & 0xFFFFFFFF), "nnab_stream_wait_value32_geq")


def block_layout_ok(n_fft: int, hop: int) -> bool:
    return bool(lib().nnab_block_layout_ok(int(n_fft), int(hop)))


def pack_basis_block(w_re: torch.Tensor, hop: int):
    """Packed rows of the block-partial STFT kernel for an (F, n_fft) periodic-Hann DFT basis
    (the caller has checked the buffers with ``is_hann_dft``); generated analytically on the device."""
    L = lib()
    F, K = w_re.shape
    packed = torch.empty(L.nnab_packed_block_bytes(int(K), int(hop)), dtype=torch.uint8, device=w_re.device)
    with torch.cuda.device(w_re.device):
        _check(L.nnab_pack_basis_block(int(K), int(hop), _ptr(packed), _stream(w_re.device)),
               "nnab_pack_basis_block")
    return packed


def pack_fir(fir: torch.Tensor, dec: int):
    """Banded-Toeplitz bf16 hi/lo packing of a decimation FIR (tensor-core pyramid)."""
    L = lib()
    taps = fir.numel()
    packed = torch.empty(L.nnab_packed_fir_bytes(taps, dec), dtype=torch.uint8, device=fir.device)
    with torch.cuda.device(fir.device):
        _check(L.nnab_pack_fir(_ptr(fir), taps, dec, _ptr(packed), _stream(fir.device)),
               "nnab_pack_fir")
    return packed


def build_filterbank_table(fb: torch.Tensor):
    """Banded (<= 2 non-zeros per FFT bin) table of an (n_fb, F) filterbank for the
    fused tcgen05 epilogue, or ``None`` when the bank is denser (e.g. gammatone).
    Init-time: synchronises the current stream once."""
    L = lib()
    n_fb, F = fb.shape
    table = torch.empty(L.nnab_filterbank_table_bytes(F), dtype=torch.uint8, device=fb.device)
    max_nnz = ctypes.c_int(0)
    with torch.cuda.device(fb.device):
        _check(L.nnab_build_filterbank_table(_ptr(fb), n_fb, F, _ptr(table), ctypes.byref(max_nnz),
                                             _stream(fb.device)), "nnab_build_filterbank_table")
    return table if max_nnz.value <= 2 else None


# --------------------------------------------------------------------------- #
# forward calls
# --------------------------------------------------------------------------- #
@_batch_chunked
def stft_forward(x, wcos, wsin, packed, n_fft, hop, center, pad_mode, out_format, sqrt_eps,
                 path=None):
    L = lib()
    x, B, Ln, pitch, xdt = _rows(x)
    F = wcos.shape[0]
    pad = n_fft // 2 if center else 0
    T = (Ln + 2 * pad - n_fft) // hop + 1
    shape = (B, F, T, 2) if out_format == FMT_COMPLEX else (B, F, T)
    out = _new_out(shape, x.device)
    path = resolve_path(path)
    with torch.cuda.device(x.device):
        ws, wsb = _workspace(L.nnab_stft_workspace_bytes(B, Ln, n_fft, F, hop, int(center), path),
                             x.device)
        rc = L.nnab_stft_forward_ex(_ptr(x), B, Ln, pitch, _ptr(wcos), _ptr(wsin), _ptr(packed),
                                    n_fft, F, hop, int(center), pad_mode, out_format, sqrt_eps,
                                    _ptr(out), T, _ptr(ws), wsb, path, _stream(x.device), xdt)
    _check(rc, "nnab_stft_forward")
    return out


@_batch_chunked
def stft_filterbank_forward(x, wcos, wsin, packed, n_fft, hop, center, pad_mode, sqrt_eps, power,
                            fb, fb_table=None, path=None):
    L = lib()
    x, B, Ln, pitch, xdt = _rows(x)
    F = wcos.shape[0]
    n_fb = fb.shape[0]
    pad = n_fft // 2 if center else 0
    T = (Ln + 2 * pad - n_fft) // hop + 1
    out = _new_out((B, n_fb, T), x.device)
    path = resolve_path(path)
    with torch.cuda.device(x.device):
        ws, wsb = _workspace(
            L.nnab_filterbank_workspace_bytes(B, Ln, n_fft, F, hop, int(center), n_fb, path,
                                              int(fb_table is not None)),
            x.device)
        rc = L.nnab_stft_filterbank_forward_ex(
            _ptr(x), B, Ln, pitch, _ptr(wcos), _ptr(wsin), _ptr(packed), n_fft, F, hop,
            int(center), pad_mode, sqrt_eps, power, _ptr(fb), n_fb, _ptr(fb_table), _ptr(out), T,
            _ptr(ws), wsb, path, _stream(x.device), xdt)
    _check(rc, "nnab_stft_filterbank_forward")
    return out


@_batch_chunked
def mfcc_forward(x, wcos, wsin, packed, n_fft, hop, center, pad_mode, sqrt_eps, power, mel_basis,
                 amin, ref, top_db, dct, fb_table=None, path=None):
    L = lib()
    x, B, Ln, pitch, xdt = _rows(x)
    F = wcos.shape[0]
    n_mels = mel_basis.shape[0]
    n_mfcc = dct.shape[0]
    pad = n_fft // 2 if center else 0
    T = (Ln + 2 * pad - n_fft) // hop + 1
    out = _new_out((B, n_mfcc, T), x.device)
    path = resolve_path(path)
    with torch.cuda.device(x.device):
        ws, wsb = _workspace(
            L.nnab_mfcc_workspace_bytes(B, Ln, n_fft, F, hop, int(center), n_mels, path,
                                        int(fb_table is not None)), x.device)
        rc = L.nnab_mfcc_forward_ex(
            _ptr(x), B, Ln, pitch, _ptr(wcos), _ptr(wsin), _ptr(packed), n_fft, F, hop,
            int(center), pad_mode, sqrt_eps, power, _ptr(mel_basis), n_mels, _ptr(fb_table), amin, ref,
            -1.0 if top_db is None else float(top_db), _ptr(dct), n_mfcc, _ptr(out), T, _ptr(ws),
            wsb, path, _stream(x.device), xdt)
    _check(rc, "nnab_mfcc_forward")
    return out


@_batch_chunked
def cqt1992v2_forward(x, k_real, k_imag, packed, k_begin, k_end, hop, center, pad_mode, scale,
                      scale_all, out_format, sqrt_eps, path=None):
    """k_begin / k_end: host int32 numpy arrays (per-bin support) or None."""
    L = lib()
    x, B, Ln, pitch, xdt = _rows(x)
    n_bins, width = k_real.shape
    pad = width // 2 if center else 0
    T = (Ln + 2 * pad - width) // hop + 1
    shape = (B, n_bins, T) if out_format == FMT_MAGNITUDE else (B, n_bins, T, 2)
    out = _new_out(shape, x.device)
    path = resolve_path(path)
    kb = k_begin.ctypes.data_as(c_void_p) if k_begin is not None else None
    ke = k_end.ctypes.data_as(c_void_p) if k_end is not None else None
    with torch.cuda.device(x.device):
        ws, wsb = _workspace(
            L.nnab_cqt1992v2_workspace_bytes(B, Ln, width, n_bins, hop, int(center), path),
            x.device)
        rc = L.nnab_cqt1992v2_forward_ex(
            _ptr(x), B, Ln, pitch, _ptr(k_real), _ptr(k_imag), _ptr(packed), kb, ke, n_bins,
            width, hop, int(center), pad_mode, _ptr(scale), scale_all, out_format, sqrt_eps,
            _ptr(out), T, _ptr(ws), wsb, path, _stream(x.device), xdt)
    _check(rc, "nnab_cqt1992v2_forward")
    return out


@_batch_chunked
def cqt_pyramid_forward(x, banks_real, banks_imag, packed, lowpass, lowpass_packed, early_filter,
                        early_packed, early_factor, hop, pad_mode, n_bins, scale, scale_all,
                        out_format, sqrt_eps, T, path=None):
    """banks_*: lists (octave 0 = top) of (n_filters, width_i) fp32 CUDA tensors;
    packed: list of packed-basis tensors (or None entries) per octave."""
    L = lib()
    x, B, Ln, pitch, xdt = _rows(x)
    n_oct = len(banks_real)
    n_filters = banks_real[0].shape[0]
    re_arr = (c_void_p * n_oct)(*[t.data_ptr() for t in banks_real])
    im_arr = (c_void_p * n_oct)(*[t.data_ptr() for t in banks_imag])
    pk_arr = (c_void_p * n_oct)(*[(t.data_ptr() if t is not None else None) for t in packed])
    widths = (c_int32 * n_oct)(*[int(t.shape[1]) for t in banks_real])
    max_width = max(int(t.shape[1]) for t in banks_real)
    shape = (B, n_bins, T) if out_format == FMT_MAGNITUDE else (B, n_bins, T, 2)
    out = _new_out(shape, x.device)
    path = resolve_path(path)
    with torch.cuda.device(x.device):
        ws, wsb = _workspace(
            L.nnab_cqt_pyramid_workspace_bytes(B, Ln, n_oct, early_factor, max_width, hop, path),
            x.device)
        rc = L.nnab_cqt_pyramid_forward_ex(
            _ptr(x), B, Ln, pitch, n_oct, re_arr, im_arr, pk_arr, widths, n_filters,
            _ptr(lowpass), _ptr(lowpass_packed), _ptr(early_filter), _ptr(early_packed),
            early_factor, hop, pad_mode, n_bins, _ptr(scale),
            scale_all, out_format, sqrt_eps, _ptr(out), T, _ptr(ws), wsb, path, _stream(x.device),
            xdt)
    _check(rc, "nnab_cqt_pyramid_forward")
    return out


def pack_istft_basis(kernel_cos: torch.Tensor, kernel_sin: torch.Tensor, f_in: int, onesided: bool):
    """Tensor-core packing of the (n_fft, n_fft) inverse kernels; the mirroring of a
    one-sided spectrum (utils.py:63-70) is folded into the packed rows."""
    L = lib()
    n_fft = kernel_cos.shape[0]
    packed = torch.empty(L.nnab_packed_istft_bytes(n_fft, f_in), dtype=torch.uint8,
                         device=kernel_cos.device)
    with torch.cuda.device(kernel_cos.device):
        _check(L.nnab_pack_istft_basis(_ptr(kernel_cos), _ptr(kernel_sin), n_fft, f_in,
                                       int(onesided), _ptr(packed), _stream(kernel_cos.device)),
               "nnab_pack_istft_basis")
    return packed


def istft_forward(X, packed, window, n_fft, hop, center, length):
    """X (B, f_in, T, 2) fp32 CUDA -> waveform (B, out_len)."""
    L = lib()
    X = _dev_f32(X, "X")
    X = X if X.is_contiguous() else X.contiguous()
    B, f_in, T, _ = X.shape
    ola_len = n_fft + hop * (T - 1)
    pad = n_fft // 2
    offset = pad if center else 0
    want = length if length is not None else (ola_len - 2 * pad if center else ola_len)
    want = max(0, min(want, ola_len - offset))
    out = torch.empty((B, want), dtype=torch.float32, device=X.device)
    with torch.cuda.device(X.device):
        ws, wsb = _workspace(L.nnab_istft_workspace_bytes(B, f_in, T, n_fft, hop), X.device)
        rc = L.nnab_istft_forward(_ptr(X), B, f_in, T, _ptr(packed), _ptr(window), n_fft, hop,
                                  int(center), -1 if length is None else int(length), _ptr(out),
                                  want, _ptr(ws), wsb, _stream(X.device))
    _check(rc, "nnab_istft_forward")
    return out


def fir_decimate(x, fir, factor):
    """EXPERIMENTAL: y = conv1d(x, fir, stride=factor, padding=(taps-1)//2) for (B, L) rows."""
    L = lib()
    x, B, Ln, pitch, _ = _rows(_dev_f32(x, "x"))
    fir = _dev_f32(fir, "fir").reshape(-1).contiguous()
    taps = fir.numel()
    half = (taps - 1) // 2
    Ly = (Ln + 2 * half - taps) // factor + 1
    y = torch.empty((B, Ly), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _check(L.nnab_fir_decimate(_ptr(x), B, Ln, pitch, _ptr(fir), taps, int(factor), _ptr(y), Ly,
                                   _stream(x.device)), "nnab_fir_decimate")
    return y


def fir_decimate_adjoint(g, fir, factor, L_in):
    """EXPERIMENTAL: gradient of fir_decimate w.r.t. its input, (B, Ly) -> (B, L_in)."""
    L = lib()
    g, B, Ly, pitch, _ = _rows(_dev_f32(g, "grad"))
    fir = _dev_f32(fir, "fir").reshape(-1).contiguous()
    dx = torch.empty((B, L_in), dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        _check(L.nnab_fir_decimate_adjoint(_ptr(g), B, Ly, pitch, _ptr(fir), fir.numel(), int(factor),
                                           _ptr(dx), int(L_in), _stream(g.device)),
               "nnab_fir_decimate_adjoint")
    return dx


def pack_adjoint_basis(w_re: torch.Tensor, w_im: torch.Tensor):
    """W^T packing of an (F, K) forward basis pair for the input-gradient GEMM."""
    L = lib()
    F, K = w_re.shape
    packed = torch.empty(L.nnab_packed_adjoint_bytes(K, F), dtype=torch.uint8, device=w_re.device)
    with torch.cuda.device(w_re.device):
        _check(L.nnab_pack_adjoint_basis(_ptr(w_re), _ptr(w_im), F, K, _ptr(packed),
                                         _stream(w_re.device)), "nnab_pack_adjoint_basis")
    return packed


def framed_backward_input(g, packed_adj, K, hop, center, pad_mode, L_in):
    """g (B, F, T, 2) -> dx (B, L_in)."""
    L = lib()
    g = _dev_f32(g, "grad")
    g = g if g.is_contiguous() else g.contiguous()
    B, F, T, _ = g.shape
    dx = torch.empty((B, L_in), dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        ws, wsb = _workspace(
            L.nnab_framed_backward_input_workspace_bytes(B, L_in, K, F, hop, int(center)), g.device)
        rc = L.nnab_framed_backward_input(_ptr(g), B, F, T, _ptr(packed_adj), K, hop, int(center),
                                          pad_mode, _ptr(dx), L_in, _ptr(ws), wsb,
                                          _stream(g.device))
    _check(rc, "nnab_framed_backward_input")
    return dx


def framed_backward_weight(g, x, K, hop, center, pad_mode):
    """g (B, F, T, 2), x (B, L) -> (d w_re, d w_im), each (F, K)."""
    L = lib()
    g = _dev_f32(g, "grad")
    g = g if g.is_contiguous() else g.contiguous()
    x, B, Ln, pitch, _ = _rows(_dev_f32(x, "x"))
    _, F, T, _ = g.shape
    dw = torch.empty((2 * F, K), dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device):
        ws, wsb = _workspace(
            L.nnab_framed_backward_weight_workspace_bytes(B, Ln, K, F, hop, int(center)), g.device)
        rc = L.nnab_framed_backward_weight(_ptr(g), _ptr(x), B, Ln, pitch, F, T, K, hop,
                                           int(center), pad_mode, _ptr(dw), _ptr(ws), wsb,
                                           _stream(g.device))
    _check(rc, "nnab_framed_backward_weight")
    return dw[:F], -dw[F:]
