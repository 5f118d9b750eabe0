"""``CQT1992v2``, ``CQT2010v2`` and the ``CQT`` alias — drop-ins for
``nnAudio.features.cqt`` (cqt.py:561-803, :805-1139, :1142-1145).

Buffer names follow the reference, including its spelling ``lenghts``.
"""
from __future__ import annotations

import os
import warnings
from time import time

import numpy as np
import torch
import torch.nn as nn

from .. import _C, design
from ._common import (AdjointBasis, FramedComplexFn, PackedBasis, PackedFir, PerDeviceCache, as_matrix,
                      broadcast_dim, pad_mode_id, tap_support, wants_grad)

_FORMATS = {
    "Magnitude": _C.FMT_MAGNITUDE,
    "Complex": _C.FMT_COMPLEX,
    "Phase": _C.FMT_PHASE_UNIT,
}
_NORMALIZATIONS = ("librosa", "convolutional", "wrap")


def _check_format_and_norm(output_format, normalization_type):
    if normalization_type not in _NORMALIZATIONS:
        raise ValueError(
            "The normalization_type %r is not part of our current options." % normalization_type
        )
    if output_format not in _FORMATS:
        raise ValueError(
            f"output_format must be 'Magnitude', 'Complex' or 'Phase', got {output_format!r}"
        )


class _ScaleCache:
    """sqrt(lenghts) * factor on the device, recomputed when ``lenghts`` changes."""

    def __init__(self):
        self._cache = PerDeviceCache()

    def get(self, lenghts: torch.Tensor, factor: float):
        def build():
            s = torch.sqrt(lenghts.detach().float())
            return (s * factor if factor != 1 else s).contiguous()

        key = (lenghts.data_ptr(), lenghts._version, float(factor))
        return self._cache.lookup(lenghts.device, key, build)


class CQT1992v2(nn.Module):
    """Time-domain constant-Q transform with one wavelet bank spanning all bins
    (cqt.py:655-780).  ``forward(x, output_format=None,
    normalization_type='librosa')`` returns ``(B, n_bins, T)`` (Magnitude) or
    ``(B, n_bins, T, 2)`` (Complex = (real, imag); Phase = (cos, sin))."""

    def __init__(
        self,
        sr=22050,
        hop_length=512,
        fmin=32.70,
        fmax=None,
        n_bins=84,
        bins_per_octave=12,
        filter_scale=1,
        norm=1,
        window="hann",
        center=True,
        pad_mode="reflect",
        trainable=False,
        output_format="Magnitude",
        verbose=True,
    ):
        super().__init__()
        self.trainable = trainable
        self.hop_length = hop_length
        self.center = center
        self.pad_mode = pad_mode
        self.output_format = output_format

        Q = float(filter_scale) / (2 ** (1 / bins_per_octave) - 1)
        if verbose:
            print("Creating CQT kernels ...", end="\r")
        start = time()
        bank, self.kernel_width, lengths, freqs = design.cqt_bank(
            Q, sr, fmin, n_bins, bins_per_octave, norm, window, fmax
        )
        self.register_buffer("lenghts", torch.tensor(lengths).float())
        self.frequencies = freqs

        k_real = torch.tensor(bank.real).unsqueeze(1)
        k_imag = torch.tensor(bank.imag).unsqueeze(1)
        if trainable:
            self.register_parameter("cqt_kernels_real", nn.Parameter(k_real, requires_grad=True))
            self.register_parameter("cqt_kernels_imag", nn.Parameter(k_imag, requires_grad=True))
        else:
            self.register_buffer("cqt_kernels_real", k_real)
            self.register_buffer("cqt_kernels_imag", k_imag)

        self._packed = PackedBasis()
        self._scale = _ScaleCache()
        self._support = PerDeviceCache()
        if verbose:
            print("CQT kernels created, time used = {:.4f} seconds".format(time() - start))

    def _tap_support(self):
        """Host int32 [begin, end) of each wavelet's non-zero taps, from the
        *current* buffer contents (dense when the bank is trainable)."""
        if self.trainable:
            return None, None
        kr, ki = self.cqt_kernels_real, self.cqt_kernels_imag

        def build():
            both = (kr.detach()[:, 0, :] != 0) | (ki.detach()[:, 0, :] != 0)
            return tap_support(both.cpu().numpy())

        key = (kr.data_ptr(), kr._version, ki.data_ptr(), ki._version)
        return self._support.lookup(kr.device, key, build)

    def forward(self, x, output_format=None, normalization_type="librosa"):
        output_format = output_format or self.output_format
        _check_format_and_norm(output_format, normalization_type)
        x = broadcast_dim(x)
        pad = self.kernel_width // 2 if self.center else 0
        if self.center and self.pad_mode == "reflect" and x.shape[-1] <= pad:
            raise RuntimeError(
                "Padding size should be less than the corresponding input dimension, but got: "
                f"padding ({pad}, {pad}) at dimension 2 of input {tuple(x[:, None, :].shape)}"
            )
        if x.shape[-1] + 2 * pad < self.kernel_width:
            raise RuntimeError("Kernel size can't be greater than actual input size")

        k_real, k_imag = as_matrix(self.cqt_kernels_real), as_matrix(self.cqt_kernels_imag)
        packed = self._packed.get(k_real, k_imag,
                                  groups=(not self.trainable) and self.hop_length % 8 == 0)
        k_begin, k_end = self._tap_support()
        scale, scale_all = None, 1.0
        if normalization_type == "librosa":
            scale = self._scale.get(self.lenghts, 1.0)
        elif normalization_type == "wrap":
            scale_all = 2.0
        eps = 1e-8 if (self.trainable and output_format == "Magnitude") else 0.0
        if wants_grad(self, x):
            # un-normalised complex CQT through the fused kernel + dX / dW kernels; normalisation and
            # output format (cqt.py:752-780) composed in torch for autograd
            if not hasattr(self, "_adjoint"):
                self._adjoint = AdjointBasis()

            def fwd(t):
                return _C.cqt1992v2_forward(t, k_real, k_imag, packed, k_begin, k_end,
                                            self.hop_length, self.center,
                                            pad_mode_id(self.pad_mode), None, 1.0,
                                            _C.FMT_COMPLEX, 0.0)

            def bwd(g, L):
                return _C.framed_backward_input(g, self._adjoint.get(k_real, k_imag),
                                                self.kernel_width, self.hop_length, self.center,
                                                pad_mode_id(self.pad_mode), L)

            def bwd_w(g, xin):
                return _C.framed_backward_weight(g, xin, self.kernel_width, self.hop_length,
                                                 self.center, pad_mode_id(self.pad_mode))

            c = FramedComplexFn.apply(x, self.cqt_kernels_real, self.cqt_kernels_imag, fwd, bwd,
                                      bwd_w)
            if scale is not None:
                c = c * scale.view(1, -1, 1, 1)
            elif scale_all != 1.0:
                c = c * scale_all
            if output_format == "Complex":
                return c
            if output_format == "Magnitude":
                return torch.sqrt(c[..., 0].pow(2) + c[..., 1].pow(2) + eps)
            ang = torch.atan2(c[..., 1], c[..., 0])
            return torch.stack((torch.cos(ang), torch.sin(ang)), -1)
        return _C.cqt1992v2_forward(
            x, k_real, k_imag, packed, k_begin, k_end, self.hop_length, self.center,
            pad_mode_id(self.pad_mode), scale, scale_all, _FORMATS[output_format], eps,
        )


class CQT(CQT1992v2):
    """Alias of :class:`CQT1992v2` (cqt.py:1142-1145)."""

    pass


def _octave_plan(L, hop, widths, pad_mode):
    """Per-octave signal lengths of the ÷2 pyramid and whether the reference's
    reflect padding would fall back to zero padding (utils.py:505-517).
    Returns (T, fallback_flags) or raises like torch.cat would."""
    lens, hops, flags = [], [], []
    cur, h = L, hop
    for i, w in enumerate(widths):
        if i > 0:
            cur = (cur - 2) // 2 + 1 if cur >= 2 else 0
            h = h // 2
        lens.append(cur)
        hops.append(h)
        flags.append(pad_mode == "reflect" and w // 2 >= cur)
    if min(hops) <= 0 or min(lens) <= 0:
        raise RuntimeError(
            "CQT pyramid: hop_length or signal too small for the number of octaves "
            f"(lengths {lens}, hops {hops})"
        )
    Ts = [l // h + 1 for l, h in zip(lens, hops)]
    if len(set(Ts)) != 1:
        raise RuntimeError(
            f"Sizes of tensors must match except in dimension 1 (octave frame counts {Ts})"
        )
    return Ts[0], flags


class CQT2010v2(nn.Module):
    """Constant-Q transform by the resampling method: one top-octave bank reused
    over a ÷2 anti-aliased pyramid (cqt.py:901-1139).  Like the reference, the
    ``window`` and ``norm`` constructor arguments do not influence the bank
    (cqt.py:1023-1031 never forwards them)."""

    def __init__(
        self,
        sr=22050,
        hop_length=512,
        fmin=32.70,
        fmax=None,
        n_bins=84,
        filter_scale=1,
        bins_per_octave=12,
        norm=True,
        basis_norm=1,
        window="hann",
        pad_mode="reflect",
        earlydownsample=True,
        trainable=False,
        output_format="Magnitude",
        verbose=True,
    ):
        super().__init__()
        self.norm = norm
        self.hop_length = hop_length
        self.pad_mode = pad_mode
        self.n_bins = n_bins
        self.earlydownsample = earlydownsample
        self.trainable = trainable
        self.output_format = output_format

        Q = float(filter_scale) / (2 ** (1 / bins_per_octave) - 1)

        if verbose:
            print("Creating low pass filter ...", end="\r")
        start = time()
        lowpass = torch.tensor(design.lowpass_fir(0.50, 256, 0.001))
        self.register_buffer("lowpass_filter", lowpass[None, None, :])
        if verbose:
            print("Low pass filter created, time used = {:.4f} seconds".format(time() - start))

        n_filters = min(bins_per_octave, n_bins)
        self.n_octaves = int(np.ceil(float(n_bins) / bins_per_octave))
        if verbose:
            print("num_octave = ", self.n_octaves)

        # lowest bin of the top-octave bank (cqt.py:970-983)
        self.fmin_t = fmin * 2 ** (self.n_octaves - 1)
        remainder = n_bins % bins_per_octave
        if remainder == 0:
            fmax_t = self.fmin_t * 2 ** ((bins_per_octave - 1) / bins_per_octave)
        else:
            fmax_t = self.fmin_t * 2 ** ((remainder - 1) / bins_per_octave)
        self.fmin_t = fmax_t / 2 ** (1 - 1 / bins_per_octave)
        if fmax_t > sr / 2:
            raise ValueError(
                "The top bin {}Hz has exceeded the Nyquist frequency, \
                            please reduce the n_bins".format(
                    fmax_t
                )
            )

        if self.earlydownsample:
            if verbose:
                print("Creating early downsampling filter ...", end="\r")
            start = time()
            sr, self.hop_length, self.downsample_factor, early_fir = design.early_downsample_plan(
                sr, hop_length, fmax_t, Q, self.n_octaves
            )
            self.earlydownsample = early_fir is not None
            if verbose:
                if self.earlydownsample:
                    print("Can do early downsample, factor = ", self.downsample_factor)
                else:
                    print("No early downsampling is required, downsample_factor = ",
                          self.downsample_factor)
            self.register_buffer(
                "early_downsample_filter",
                torch.tensor(early_fir)[None, None, :] if early_fir is not None else None,
            )
            if verbose:
                print("Early downsampling filter created, \
                        time used = {:.4f} seconds".format(time() - start))
        else:
            self.downsample_factor = 1.0

        if verbose:
            print("Creating CQT kernels ...", end="\r")
        start = time()
        basis, self.n_fft, _, _ = design.cqt_bank(
            Q, sr, self.fmin_t, n_filters, bins_per_octave, norm=basis_norm, topbin_check=False
        )
        freqs = fmin * 2.0 ** (np.r_[0:n_bins] / np.double(bins_per_octave))
        self.frequencies = freqs
        lenghts = np.ceil(Q * sr / freqs)
        self.register_buffer("lenghts", torch.tensor(lenghts).float())

        self.basis = basis
        k_real = torch.tensor(basis.real).unsqueeze(1)
        k_imag = torch.tensor(basis.imag).unsqueeze(1)
        if trainable:
            self.register_parameter("cqt_kernels_real", nn.Parameter(k_real, requires_grad=True))
            self.register_parameter("cqt_kernels_imag", nn.Parameter(k_imag, requires_grad=True))
        else:
            self.register_buffer("cqt_kernels_real", k_real)
            self.register_buffer("cqt_kernels_imag", k_imag)
        if verbose:
            print("CQT kernels created, time used = {:.4f} seconds".format(time() - start))

        # kept for attribute parity (cqt.py:1065-1068); the kernels pad in-flight
        if self.pad_mode == "constant":
            self.padding = nn.ConstantPad1d(self.n_fft // 2, 0)
        elif self.pad_mode == "reflect":
            self.padding = nn.ReflectionPad1d(self.n_fft // 2)
        self._scale = _ScaleCache()
        self._packed = PackedBasis()

    def _banks(self):
        k_real, k_imag = as_matrix(self.cqt_kernels_real), as_matrix(self.cqt_kernels_imag)
        packed = self._packed.get(k_real, k_imag)  # one bank shared by every octave
        return [k_real] * self.n_octaves, [k_imag] * self.n_octaves, [packed] * self.n_octaves

    def _bank_tensors(self):
        """Per-octave (real, imag) bank tensors as autograd sees them (one shared, possibly
        trainable, bank: its gradient is the sum over the octaves)."""
        return [(self.cqt_kernels_real, self.cqt_kernels_imag)] * self.n_octaves

    def forward(self, x, output_format=None, normalization_type="librosa"):
        output_format = output_format or self.output_format
        _check_format_and_norm(output_format, normalization_type)
        x = broadcast_dim(x)
        return _pyramid_forward(self, x, output_format,
                                _v2_normalization(self, normalization_type, output_format))


def _v2_normalization(mod, normalization_type, output_format):
    """cqt.py:1112-1124 / vqt.py:190-200: (per-bin scale tensor or None, global factor, sqrt eps)."""
    scale, scale_all = None, 1.0
    dsf = float(mod.downsample_factor)
    if normalization_type == "librosa":
        scale = mod._scale.get(mod.lenghts, dsf)
    elif normalization_type == "wrap":
        scale_all = 2.0 * dsf
    else:
        scale_all = dsf
    eps = 1e-8 if (mod.trainable and output_format == "Magnitude") else 0.0
    return scale, scale_all, eps


def _pyramid_forward(mod, x, output_format, normalization):
    """Shared by CQT2010v2, VQT and CQT2010: plan the octave lengths on the host (for the
    reference's warnings / errors), then one C call.  ``normalization`` = (scale, scale_all, eps)."""
    scale, scale_all, eps = normalization
    banks_real, banks_imag, packed = mod._banks()
    early = mod.early_downsample_filter if mod.earlydownsample else None
    factor = int(mod.downsample_factor) if mod.earlydownsample else 1
    L = x.shape[-1]
    L0 = (L - 2) // factor + 1 if factor > 1 else L
    if factor > 1 and L < 2:
        raise RuntimeError("Kernel size can't be greater than actual input size")
    widths = [int(b.shape[1]) for b in banks_real]
    T, fallbacks = _octave_plan(L0, mod.hop_length, widths, mod.pad_mode)
    for i, fb in enumerate(fallbacks):
        if fb:
            warnings.warn(
                f"\ninput size = {(x.shape[0], 1, L0)}\tkernel size = {widths[i]}\n"
                "padding with reflection mode might not be the best choice, try using constant padding",
                UserWarning,
            )
    if wants_grad(mod, x):
        return _pyramid_forward_autograd(mod, x, output_format, fallbacks, factor, scale, scale_all,
                                         eps)
    lowpass = mod.lowpass_filter.detach().reshape(-1)
    early_flat = early.detach().reshape(-1) if early is not None else None
    for t in (lowpass, early_flat):
        if t is not None:
            _C._dev_f32(t, "filter")
    if not hasattr(mod, "_fir_packed"):
        mod._fir_packed = (PackedFir(), PackedFir())
    lowpass_packed = mod._fir_packed[0].get(lowpass, 2)
    early_packed = mod._fir_packed[1].get(early_flat, factor) if early_flat is not None else None
    return _C.cqt_pyramid_forward(
        x, banks_real, banks_imag, packed, lowpass, lowpass_packed, early_flat, early_packed,
        factor, mod.hop_length,
        pad_mode_id(mod.pad_mode), mod.n_bins, scale, scale_all, _FORMATS[output_format], eps, T,
    )


def _framed_complex_autograd(mod, tag, sig, w_re, w_im, hop, center, pad_mode):
    """One differentiable framed contraction ``sig (B, L) -> (B, F, T, 2)`` through the fused
    forward kernel and the dX / dW kernels; ``tag`` keys the packed-basis caches on ``mod``."""
    k_re, k_im = as_matrix(w_re), as_matrix(w_im)
    if w_re.grad_fn is not None or w_im.grad_fn is not None:
        # recomputed temporaries (the folded v1 bank under autograd): every call gets a fresh
        # tensor with _version 0 whose address the allocator may recycle from the previous step,
        # so a (data_ptr, _version) key cannot tell them apart -> pack per call, never cache.
        # The packing rides on the temporary itself (shared by the octaves of one forward, freed
        # with it).
        caches = w_re.__dict__.setdefault("_nnab_grad_caches", {})
        caches.setdefault(tag, (PackedBasis(), AdjointBasis()))
    else:
        caches = mod.__dict__.setdefault("_grad_caches", {})
        if tag not in caches:
            caches[tag] = (PackedBasis(), AdjointBasis())
    packed = caches[tag][0].get(k_re, k_im)
    width = int(k_re.shape[1])

    def fwd(t):
        return _C.cqt1992v2_forward(t, k_re, k_im, packed, None, None, hop, center, pad_mode,
                                    None, 1.0, _C.FMT_COMPLEX, 0.0)

    def bwd(g, L):
        return _C.framed_backward_input(g, caches[tag][1].get(k_re, k_im), width, hop, center,
                                        pad_mode, L)

    def bwd_w(g, xin):
        return _C.framed_backward_weight(g, xin, width, hop, center, pad_mode)

    return FramedComplexFn.apply(sig, w_re, w_im, fwd, bwd, bwd_w)


class _DecimateFn(torch.autograd.Function):
    """``conv1d(sig, fir, stride=n, padding=(taps-1)//2)`` (utils.py:73-100) with a gradient for
    ``sig``.  Forward: a one-row framed contraction on the zero-padded signal.  Backward: the
    adjoint of an n-fold decimating FIR is n interleaved stride-1 FIRs of ``dL/dy`` with the
    polyphase components ``h_p[q] = fir[n*q + p]`` — again a framed contraction (n rows,
    ceil(taps/n) taps, hop 1), so every input sample is written once instead of receiving
    ``taps`` atomics from an overlap-add."""

    @staticmethod
    def forward(ctx, sig, fir_row, zero_row, poly, n):
        taps = fir_row.shape[1]
        half = (taps - 1) // 2
        ctx.n, ctx.half, ctx.L, ctx.poly, ctx.dtype = n, half, sig.shape[-1], poly, sig.dtype
        padded = torch.nn.functional.pad(sig, (half, half))
        c = _C.cqt1992v2_forward(padded, fir_row, zero_row, None, None, None, n, False,
                                 _C.PAD_CONSTANT, None, 1.0, _C.FMT_COMPLEX, 0.0)
        return c[:, 0, :, 0].contiguous()

    @staticmethod
    def backward(ctx, g):
        n, half, L = ctx.n, ctx.half, ctx.L
        poly, poly_zero, packed = ctx.poly          # (n, Q) time-reversed polyphase rows, zeros
        Q = poly.shape[1]
        Lp = L + 2 * half
        M = (Lp + n - 1) // n                       # outputs per phase
        T = g.shape[-1]
        gp = torch.nn.functional.pad(g.contiguous(), (Q - 1, max(M - T, 0)))[:, : M + Q - 1]
        # hop 1: CUDA-core kernel by default; NNAUDIO_B200_DECIM_BWD=tc runs the 8 frame phases
        # of the tensor-core kernel instead
        use_tc = packed is not None and os.environ.get("NNAUDIO_B200_DECIM_BWD", "fir") == "tc"
        c = _C.cqt1992v2_forward(gp.contiguous(), poly, poly_zero, packed if use_tc else None, None,
                                 None, 1, False, _C.PAD_CONSTANT, None, 1.0, _C.FMT_COMPLEX, 0.0,
                                 path="tcgen05" if use_tc else "simt")
        d_padded = c[..., 0].permute(0, 2, 1).reshape(g.shape[0], M * n)   # [n*m + p] = phase p, m
        return d_padded[:, half:half + L].to(ctx.dtype).contiguous(), None, None, None, None


class _FirDecimateFn(torch.autograd.Function):
    """``nnab_fir_decimate`` / ``nnab_fir_decimate_adjoint``: one launch each way (GPU-verified round 2)."""

    @staticmethod
    def forward(ctx, sig, fir, n):
        ctx.fir, ctx.n, ctx.L = fir, n, sig.shape[-1]
        return _C.fir_decimate(sig, fir, n)

    @staticmethod
    def backward(ctx, g):
        return _C.fir_decimate_adjoint(g.contiguous(), ctx.fir, ctx.n, ctx.L), None, None


def _decimate_autograd(mod, tag, sig, fir, n):
    """Differentiable ``downsampling_by_n`` / ``_by_2`` stage of the training path.

    ``NNAUDIO_B200_DECIM_BWD`` picks the adjoint (CQT2010v2 32 x 30 s forward + backward, worst dX error
    of the pyramid cases vs the reference's autograd):
    ``fir`` (default since round 2) the dedicated CUDA-core FIR stage + adjoint kernel
    (``nnab_fir_decimate`` / ``nnab_fir_decimate_adjoint``: every input sample written once, no
    atomics) -- 2.96 ms, within the 1e-4 bar on every pyramid gradient case;
    ``simt`` polyphase FIRs on the framed CUDA-core kernel -- 42.0 ms, 6.1e-5; ``tc`` the same on the
    tensor-core kernel (8 frame phases) -- 30.1 ms, 6.1e-5; ``ola`` a K=1 adjoint GEMM + overlap-add
    atomics (256 atomics per input sample) -- 24.4 ms but 1.04e-4 on the Magnitude case, over the bar."""
    if os.environ.get("NNAUDIO_B200_DECIM_BWD", "fir") == "fir":
        return _FirDecimateFn.apply(sig, fir.detach().reshape(-1).contiguous(), int(n))
    if os.environ.get("NNAUDIO_B200_DECIM_BWD", "fir") == "ola":
        taps = fir.numel()
        w_re = fir.detach().reshape(1, taps)
        zeros = mod.__dict__.setdefault("_fir_zeros", {})
        if tag not in zeros or zeros[tag].shape != w_re.shape or zeros[tag].device != w_re.device:
            zeros[tag] = torch.zeros_like(w_re)
        half = (taps - 1) // 2
        padded = torch.nn.functional.pad(sig, (half, half))
        c = _framed_complex_autograd(mod, tag, padded, w_re, zeros[tag], n, False, _C.PAD_CONSTANT)
        return c[:, 0, :, 0].contiguous()
    cache = mod.__dict__.setdefault("_decim_cache", {})

    def build():
        taps = fir.numel()
        row = fir.detach().reshape(1, taps).contiguous()
        Q = (taps + n - 1) // n
        padded = torch.nn.functional.pad(row[0], (0, Q * n - taps))
        poly = padded.reshape(Q, n).t().flip(1).contiguous()      # poly[p, k] = fir[n*(Q-1-k) + p]
        poly_zero = torch.zeros_like(poly)
        return row, torch.zeros_like(row), (poly, poly_zero, _C.pack_basis(poly, poly_zero))

    key = (fir.data_ptr(), fir._version, int(n))
    row, zero_row, poly = cache.setdefault(tag, PerDeviceCache()).lookup(fir.device, key, build)
    return _DecimateFn.apply(sig, row, zero_row, poly, int(n))


def _pyramid_forward_autograd(mod, x, output_format, fallbacks, factor, scale, scale_all, eps):
    """cqt.py:1085-1139 / vqt.py:160-215 octave by octave with autograd-visible stages
    (training path; inference uses the single fused C call above).  A bf16 / fp16 input enters as
    its exact fp32 copy (the decimator stages are fp32); autograd casts its gradient back to x.dtype."""
    if x.dtype in (torch.bfloat16, torch.float16):
        x = x.float()
    if factor > 1:
        x = _decimate_autograd(mod, "early", x, mod.early_downsample_filter, factor)
    hop = mod.hop_length
    octaves = []
    cur = x
    for i, (w_re, w_im) in enumerate(mod._bank_tensors()):
        if i > 0:
            hop //= 2
            cur = _decimate_autograd(mod, "lowpass", cur, mod.lowpass_filter, 2)
        mode = _C.PAD_CONSTANT if fallbacks[i] else pad_mode_id(mod.pad_mode)
        octaves.insert(0, _framed_complex_autograd(mod, f"bank{i}", cur, w_re, w_im, hop, True,
                                                   mode))
    c = torch.cat(octaves, 1)[:, -mod.n_bins:]
    if scale is not None:  # sqrt(lenghts) * downsample_factor
        c = c * scale.view(1, -1, 1, 1)
    elif scale_all != 1.0:
        c = c * scale_all
    if output_format == "Complex":
        return c
    if output_format == "Magnitude":
        return torch.sqrt(c[..., 0].pow(2) + c[..., 1].pow(2) + eps)
    ang = torch.atan2(c[..., 1], c[..., 0])
    return torch.stack((torch.cos(ang), torch.sin(ang)), -1)
