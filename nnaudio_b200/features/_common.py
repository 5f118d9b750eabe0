"""Host-side helpers shared by the feature modules (argument checks that raise
the reference's exception types *before* the C call, and the cache of
device-side packed bases)."""
from __future__ import annotations

import numpy as np
import torch

from .. import _C

PAD_MODES = {"reflect": _C.PAD_REFLECT, "constant": _C.PAD_CONSTANT}


def broadcast_dim(x: torch.Tensor) -> torch.Tensor:
    """utils.py:206-222 — accept (L), (B, L) or (B, 1, L); returns a (B, L) view
    (the reference inserts the singleton conv channel instead)."""
    if x.dim() == 2:
        return x
    if x.dim() == 1:
        return x[None, :]
    if x.dim() == 3:
        if x.shape[1] != 1:
            raise RuntimeError(
                f"expected input with 1 channel, got {x.shape[1]} channels (shape {tuple(x.shape)})"
            )
        return x[:, 0, :]
    raise ValueError("Only support input with shape = (batch, len) or shape = (len)")


def pad_mode_id(pad_mode: str) -> int:
    try:
        return PAD_MODES[pad_mode]
    except KeyError:
        raise ValueError(f"unsupported pad_mode {pad_mode!r}; use 'reflect' or 'constant'")


def forward_only_guard(module: torch.nn.Module, x: torch.Tensor, used=None):
    """For parameters without a dW path (trainable inverse kernels / window of iSTFT):
    refuse loudly rather than return a result whose parameters silently get no gradient.
    ``used``: the tensors this call reads (default: every parameter of the module)."""
    if not torch.is_grad_enabled():
        return
    tensors = module.parameters() if used is None else used
    if any(p.requires_grad for p in tensors):
        raise NotImplementedError(
            "nnaudio_b200: this module is forward-only for trainable kernels; run under "
            "torch.no_grad()"
        )


def wants_grad(module: torch.nn.Module, x: torch.Tensor) -> bool:
    """True when autograd needs a graph through this call (input and/or trainable bases)."""
    if not torch.is_grad_enabled():
        return False
    return x.requires_grad or any(p.requires_grad for p in module.parameters())


class FramedComplexFn(torch.autograd.Function):
    """Differentiable complex framed contraction ``(x, w_re, w_im) -> (B, F, T, 2)``:
    forward = the fused kernel; backward = ``nnab_framed_backward_input`` (GEMM with the
    transposed basis + overlap-add + padding adjoint) for ``x`` and
    ``nnab_framed_backward_weight`` (split-K GEMM over all frames) for the bases
    (the reference gets both from autograd through conv1d, stft.py:290-293).  A bf16 / fp16 ``x``
    runs the forward kernel on the 16-bit samples; its gradient is the fp32 one cast to ``x.dtype``,
    and the weight gradient reads ``x.float()``."""

    @staticmethod
    def forward(ctx, x, w_re, w_im, fwd, bwd_x, bwd_w):
        ctx.bwd_x, ctx.bwd_w = bwd_x, bwd_w
        ctx.in_shape = x.shape
        ctx.w_shape = w_re.shape
        ctx.save_for_backward(x)
        with torch.no_grad():
            return fwd(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        g = g.contiguous()
        dx = dre = dim = None
        if ctx.needs_input_grad[0]:
            dx = ctx.bwd_x(g, ctx.in_shape[-1]).reshape(ctx.in_shape).to(x.dtype)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dre, dim = ctx.bwd_w(g, x.float())
            dre, dim = dre.reshape(ctx.w_shape), dim.reshape(ctx.w_shape)
        return dx, dre, dim, None, None, None


class PerDeviceCache:
    """One cached value per device, rebuilt when its key changes.  Entries are (key, value) tuples
    replaced in one assignment and ``lookup`` returns the value it just read or built, so module
    replicas that share this object across threads and devices (``torch.nn.DataParallel`` copies
    ``__dict__`` shallowly) can neither hand each other a buffer of the wrong device nor evict each
    other's entry."""

    def __init__(self):
        self._entries = {}

    def lookup(self, device, key, build, keep=()):
        """``keep``: the tensors whose (data_ptr, _version) make up ``key``.  The entry holds a
        reference to them, so the allocator cannot hand their address to a *different* tensor while
        the entry is alive (a recomputed temporary, e.g. the folded v1 CQT bank, always has
        ``_version`` 0 and would otherwise alias a stale entry after an optimiser step)."""
        slot = str(device)
        entry = self._entries.get(slot)
        if entry is None or entry[0] != key:
            entry = (key, build(), tuple(keep))
            self._entries[slot] = entry
        return entry[1]


class AdjointBasis:
    """Cache of the W^T packing used by the input-gradient GEMM."""

    def __init__(self):
        self._cache = PerDeviceCache()

    def get(self, w_re: torch.Tensor, w_im: torch.Tensor):
        key = (w_re.data_ptr(), w_re._version, w_im.data_ptr(), w_im._version)
        return self._cache.lookup(w_re.device, key, lambda: _C.pack_adjoint_basis(w_re, w_im),
                                  keep=(w_re, w_im))


def is_hann_dft(w_re: torch.Tensor, w_im: torch.Tensor, atol: float = 1e-6) -> bool:
    """True when an (F, K) basis pair IS the one-sided DFT with a periodic Hann window of length K:
    ``w_re[k][n] = hann[n] cos(2 pi k n / K)``, ``w_im[k][n] = hann[n] sin(2 pi k n / K)``, F = K/2 + 1
    -- what ``create_fourier_kernels(freq_scale='no', window='hann', win_length=n_fft)`` builds
    (utils.py:241-393, stft.py:230-232).  Checked on the buffers themselves in float64, so loaded,
    trained, sliced (``freq_bins``), linear / log-spaced or differently windowed bases keep the dense
    kernel; only an exact match may use the block-partial layout, whose rows are generated
    analytically."""
    F, K = w_re.shape
    if F != K // 2 + 1 or K % 2 != 0 or w_im.shape != w_re.shape:
        return False
    n = torch.arange(K, device=w_re.device)
    hann = 0.5 - 0.5 * torch.cos(2.0 * torch.pi * n.to(torch.float64) / K)
    rows = max(1, (1 << 22) // K)          # <= 32 MB of float64 scratch per block of bins
    for k0 in range(0, F, rows):
        k = torch.arange(k0, min(F, k0 + rows), device=w_re.device)
        m = (k[:, None] * n[None, :]) % K  # exact phase reduction in integers before the trig call
        ang = (2.0 * torch.pi / K) * m.to(torch.float64)
        if ((torch.cos(ang) * hann) - w_re[k0:k0 + rows].double()).abs().max() > atol:
            return False
        if ((torch.sin(ang) * hann) - w_im[k0:k0 + rows].double()).abs().max() > atol:
            return False
    return True


class PackedBasis:
    """Cache of the (F, K) fp32 views and the bf16 hi/lo packed copy of a basis
    pair, invalidated when the source tensors change (load_state_dict, .to(),
    optimiser steps)."""

    def __init__(self):
        self._cache = PerDeviceCache()

    def get(self, w_re: torch.Tensor, w_im: torch.Tensor, groups: bool = False, block_hop: int = 0):
        """``groups``: long nested CQT bank -> 8-bin-group layout (per-K-block-width / tall-A kernels);
        ``block_hop``: STFT-family module -> block-partial layout when the buffers ARE the periodic-Hann
        DFT (checked here on the tensors)."""
        import os

        def build():
            # block-partial layout (default for the STFT family): the module computes a plain
            # one-sided STFT with hop ``block_hop`` and an output format the block kernel has an
            # epilogue for; the buffers must BE the periodic-Hann DFT (NNAUDIO_B200_BLOCK=0: off)
            if block_hop and os.environ.get("NNAUDIO_B200_BLOCK", "1") != "0" \
                    and _C.block_layout_ok(int(w_re.shape[1]), int(block_hop)) \
                    and is_hann_dft(w_re, w_im):
                return _C.pack_basis_block(w_re, int(block_hop))
            # long CQT banks (CQT1992v2): per-K-block MMA width, the default since round 2
            # (GPU-verified: reference chirp goldens + cfg3 full size; NNAUDIO_B200_VARN=0: dense)
            if groups and w_re.shape[0] <= 128 and w_re.shape[1] >= 4096 \
                    and os.environ.get("NNAUDIO_B200_VARN", "1") != "0":
                return _C.pack_basis(w_re, w_im, _C.LAYOUT_GROUPS)
            return _C.pack_basis(w_re, w_im)

        key = (w_re.data_ptr(), w_re._version, w_im.data_ptr(), w_im._version, groups, int(block_hop))
        return self._cache.lookup(w_re.device, key, build, keep=(w_re, w_im))


def as_matrix(buf: torch.Tensor) -> torch.Tensor:
    """(F, 1, K) conv-style buffer -> contiguous (F, K) fp32 CUDA view."""
    t = buf.detach()
    _C._dev_f32(t, "basis")
    t = t.reshape(t.shape[0], t.shape[-1])
    return t if t.is_contiguous() else t.contiguous()


def tap_support(bank_2d: np.ndarray):
    """Per-row [begin, end) of the non-zero taps of a (n_bins, width) bank
    (real and imaginary parts combined by the caller)."""
    nz = bank_2d != 0
    any_nz = nz.any(axis=1)
    first = nz.argmax(axis=1)
    last = bank_2d.shape[1] - nz[:, ::-1].argmax(axis=1)
    begin = np.where(any_nz, first, 0).astype(np.int32)
    end = np.where(any_nz, last, 0).astype(np.int32)
    return np.ascontiguousarray(begin), np.ascontiguousarray(end)


class FilterbankTable:
    """Cache of the banded-filterbank table used by the fused tcgen05 epilogue
    (rebuilt when the filterbank tensor changes; ``None`` for dense banks)."""

    def __init__(self):
        self._cache = PerDeviceCache()

    def get(self, fb: torch.Tensor):
        key = (fb.data_ptr(), fb._version)
        return self._cache.lookup(fb.device, key, lambda: _C.build_filterbank_table(fb), keep=(fb,))


class PackedFir:
    """Cache of the tensor-core packing of a decimation FIR buffer."""

    def __init__(self):
        self._cache = PerDeviceCache()

    def get(self, fir: torch.Tensor, dec: int):
        key = (fir.data_ptr(), fir._version, int(dec))
        return self._cache.lookup(fir.device, key, lambda: _C.pack_fir(fir, int(dec)), keep=(fir,))
