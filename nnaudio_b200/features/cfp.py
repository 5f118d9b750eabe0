"""``Combined_Frequency_Periodicity`` / ``CFP`` — drop-ins for ``nnAudio.features.cfp``
(cfp.py:9-246 / 249-484; SURVEY.md §8f, the last "next" row).

What the reference computes per frame (cfp.py:137-180): an ``N = fs / fr``-point two-sided STFT with a
Blackman-Harris window of ``window_size`` samples (``torch.stft``), magnitude / ``|h|``, a power
non-linearity, then alternately ``Re FFT_N(.) / sqrt(N)`` + cut-off + power (generalised cepstrum ->
generalised spectrum -> ...), and finally two triangular log-frequency maps whose product is ``Z``.

B200 formulation — no FFT, three dense contractions on the tcgen05 framed kernel:

* **STFT stage.**  Only ``window_size`` of the ``N`` window samples are non-zero, so the frame is a
  framed contraction with ``K ~ window_size`` taps (not ``N``) against the one-sided windowed DFT rows
  ``h[m] e^{-2 pi i k (m + left) / N} / |h|``, ``k <= N/2``, hop and zero padding as ``torch.stft`` places
  them (``_stft_geometry``).  Magnitude comes out of the kernel's epilogue.
* **Cepstrum / spectrum stages.**  Every vector the reference transforms is real and (before its cut-off
  zeroing) symmetric, and only the real part of the FFT is kept, so a stage is the cosine transform
  ``out[q] = (1 / sqrt(N)) sum_n e[n] cos(2 pi n q / N)`` of the half vector ``e`` (length ``N//2 + 1``): a
  real GEMM (frames x (N/2+1)) . ((N/2+1) x (N/2+1)).  It runs on the complex framed kernel with frames as
  "clips of one hop": the first half of the output rows in the real bank, the second half in the
  imaginary bank.  The asymmetric cut-off of ``nonlinear_func`` (first ``c`` and LAST ``c`` entries of the
  full vector: index ``c`` survives, its mirror ``N - c`` does not) is folded into per-index input weights.
  The frame mean is removed before the contraction and restored analytically on ``q = 0``: the all-positive
  spectra carry a DC term ~1000x the cepstral values and the bf16 hi/lo split is relative to the terms.
* **Log-frequency maps**: the same real GEMM with the ``(Nest-1) x HighFreqIdx`` buffers.

Glue between the contractions (relu / pow / transposes) is elementwise torch on the same stream.
Forward only (the reference has no parameters here; gradients w.r.t. the waveform raise).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn

from .. import _C, design
from ._common import PerDeviceCache

EPSILON = 1e-8  # utils.py:20


def _round_up(a: int, m: int) -> int:
    return (a + m - 1) // m * m


def _stft_geometry(N: int, window_size: int):
    """Where ``torch.stft(n_fft=N, win_length=window_size, center=True)`` puts the window: zero-padded to
    ``N`` with ``left = (N - window_size) // 2`` zeros in front, frames centred by ``N // 2`` zeros of
    signal padding (cfp.py:138-147).  Frame ``t`` therefore reads ``x[t hop - d + m]``, ``d = N//2 - left``.
    The framed kernel centres by ``K // 2``: taps shifted ``j`` places into a ``K = 2 (d + j)`` wide bank
    (``K`` a multiple of 64) reproduce exactly that alignment and frame count ``L // hop + 1``."""
    if window_size > N:
        raise RuntimeError(f"stft: expected 0 < win_length <= n_fft, but got win_length={window_size}")
    left = (N - window_size) // 2
    d = N // 2 - left
    j = max(0, window_size - 2 * d)
    K = _round_up(2 * (d + j), 64)
    return left, K, K // 2 - d


class _RealGemm:
    """``(B, K_in, T) -> (B, F_out, T)`` product with a real ``(F_out, K_in)`` matrix on the complex framed
    kernel: every frame becomes one "hop" of a signal with ``hop = K = round_up(K_in, 64)``, output rows
    ``[0, Fh)`` ride in the real bank and rows ``[Fh, 2 Fh)`` (negated: the kernel returns ``-conv(x, w_im)``,
    cqt.py:749-750) in the imaginary bank."""

    def __init__(self):
        self._cache = PerDeviceCache()

    @staticmethod
    def _banks(mat: torch.Tensor):
        F_out, K_in = mat.shape
        Kp = _round_up(K_in, 64)
        Fh = (F_out + 1) // 2
        w_re = mat.new_zeros((Fh, Kp))
        w_im = mat.new_zeros((Fh, Kp))
        w_re[:, :K_in] = mat[:Fh]
        w_im[: F_out - Fh, :K_in] = -mat[Fh:]
        return w_re, w_im, _C.pack_basis(w_re, w_im)

    def __call__(self, v: torch.Tensor, F_out: int, key, matrix, keep=()) -> torch.Tensor:
        """``matrix()`` builds the fp32 ``(F_out, K_in)`` matrix on ``v.device``; it is called only when
        ``key`` (and ``keep``, the tensors it was derived from) is not the cached one."""
        w_re, w_im, packed = self._cache.lookup(v.device, key, lambda: self._banks(matrix()), keep=keep)
        B, K_in, T = v.shape
        Fh, Kp = w_re.shape
        rows = v.new_zeros((B, T, Kp))
        rows[:, :, :K_in] = v.transpose(1, 2)
        c = _C.cqt1992v2_forward(rows.view(B, T * Kp), w_re, w_im, packed, None, None, Kp, False,
                                 _C.PAD_CONSTANT, None, 1.0, _C.FMT_COMPLEX, 0.0)
        return torch.cat((c[..., 0], c[..., 1]), 1)[:, :F_out]


class _CFPBase(nn.Module):
    """Constructor, buffers and attributes shared by the two reference classes (cfp.py:66-117 = 304-355)."""

    def __init__(self, fr=2, fs=16000, hop_length=320, window_size=2049, fc=80, tc=1 / 1000,
                 g=[0.24, 0.6, 1], NumPerOct=48):
        super().__init__()
        self.window_size = window_size
        self.hop_length = hop_length

        ax = design.cfp_axes(fr, fs, fc, tc)
        self.N = ax["N"]
        self.f = ax["f"]
        self.pad_value = self.N - window_size
        self.register_buffer("h", torch.tensor(design.blackmanharris_window(window_size)).float())

        self.NumofLayer = np.size(g)
        self.g = g
        self.tc_idx = ax["tc_idx"]
        self.fc_idx = ax["fc_idx"]
        self.HighFreqIdx = ax["HighFreqIdx"]
        self.HighQuefIdx = ax["HighQuefIdx"]
        self.q = ax["q"]

        f2l, q2l = self.create_logfreq_matrix(self.f, self.q, fr, fc, tc, NumPerOct, fs)
        self.register_buffer("freq2logfreq_matrix", torch.tensor(f2l).float())
        self.register_buffer("quef2logfreq_matrix", torch.tensor(q2l).float())

        self._stft_bank = PerDeviceCache()
        self._cos_gemm = _RealGemm()
        self._freq_gemm = _RealGemm()
        self._quef_gemm = _RealGemm()

    def create_logfreq_matrix(self, f, q, fr, fc, tc, NumPerOct, fs):
        """cfp.py:195-246."""
        return design.cfp_logfreq_matrices(f, q, fr, fc, tc, NumPerOct, fs)

    # ---- index bookkeeping of the half-vector representation --------------------------------
    def _half(self) -> int:
        return self.N // 2 + 1

    def _mirror_count(self, device) -> torch.Tensor:
        """How many entries of the full length-N vector the half-vector index n stands for
        (1 for n = 0 and, N even, n = N/2; else 2)."""
        N, H = self.N, self._half()
        n = torch.arange(H, device=device)
        return 1.0 + ((n >= 1) & (n <= (N + 1) // 2 - 1)).to(torch.float32)

    def _cut_weights(self, cutoff, device):
        """``X[:, :, :c] = 0; X[:, :, -c:] = 0`` (cfp.py:182-193) on the full vector, seen from the half
        vector: ``keep_low[n]`` = entry n survives (this is also what the cropped outputs show),
        ``w_in[n]`` = surviving copies of entry n (n itself and its mirror N - n) = the weight with which
        it enters the next cosine transform.  ``c = 0`` zeroes everything, as ``X[:, :, -0:] = 0`` does."""
        N, H = self.N, self._half()
        c = int(cutoff)
        n = torch.arange(H, device=device)

        def kept(idx):
            if c == 0:
                return torch.zeros_like(idx, dtype=torch.bool)
            return (idx >= c) & (idx < N - c)

        has_up = (n >= 1) & (n <= (N + 1) // 2 - 1)
        keep_low = kept(n)
        w_in = keep_low.to(torch.float32) + (has_up & kept(N - n)).to(torch.float32)
        return keep_low.to(torch.float32), w_in

    # ---- the three contractions ---------------------------------------------------------------
    def _stft_magnitude(self, x: torch.Tensor) -> torch.Tensor:
        """``|STFT| / |h|`` for bins 0 .. N/2 -> (B, N//2 + 1, T), T = L // hop + 1 (cfp.py:138-150)."""
        h = self.h.detach()
        _C._dev_f32(h, "h")
        N, W, H = self.N, int(self.window_size), self._half()
        left, K, j = _stft_geometry(N, W)

        def build():
            k = torch.arange(H, device=h.device)
            m = torch.arange(W, device=h.device)
            phase = (k[:, None] * (m[None, :] + left)) % N  # exact reduction before the trig call
            ang = (2.0 * math.pi / N) * phase.to(torch.float64)
            win = h.double() / float(torch.norm(h))
            w_re = torch.zeros((H, K), dtype=torch.float32, device=h.device)
            w_im = torch.zeros((H, K), dtype=torch.float32, device=h.device)
            w_re[:, j:j + W] = (torch.cos(ang) * win).float()
            w_im[:, j:j + W] = (torch.sin(ang) * win).float()
            return w_re, w_im, _C.pack_basis(w_re, w_im)

        key = (h.data_ptr(), h._version, N, W)
        w_re, w_im, packed = self._stft_bank.lookup(h.device, key, build, keep=(h,))
        return _C.cqt1992v2_forward(x, w_re, w_im, packed, None, None, int(self.hop_length), True,
                                    _C.PAD_CONSTANT, None, 1.0, _C.FMT_MAGNITUDE, 0.0)

    def _cos_matrix(self, device) -> torch.Tensor:
        N, H = self.N, self._half()
        q = torch.arange(H, device=device)
        phase = (q[:, None] * q[None, :]) % N
        return (torch.cos((2.0 * math.pi / N) * phase.to(torch.float64)) / math.sqrt(N)).float()

    def _real_fft_half(self, v: torch.Tensor, w_in: torch.Tensor) -> torch.Tensor:
        """``Re FFT_N(full vector) / sqrt(N)`` on half vectors: (B, H, T) -> (B, H, T)
        (``rfft_fn(spec, 1, onesided=False)[:, :, :, 0] / np.sqrt(self.N)``, cfp.py:125-132)."""
        N = self.N
        ones = self._mirror_count(v.device)[None, :, None]
        e = v * w_in[None, :, None]
        mu = e.sum(1, keepdim=True) / N            # mean of the full vector; any value is exact in exact
        e = e - mu * ones                          # arithmetic: a constant only reaches q = 0
        out = self._cos_gemm(e, self._half(), ("cos", N), lambda: self._cos_matrix(v.device))
        out[:, 0] += mu[:, 0] * math.sqrt(N)
        return out

    def nonlinear_func(self, X, g, cutoff):
        """cfp.py:182-193 on a (B, H, T) half vector: returns the non-linearity with the LOW cut applied
        (what the reference's cropped outputs contain) — see ``_cut_weights`` for the mirrored cut."""
        keep_low, _ = self._cut_weights(cutoff, X.device)
        if g != 0:
            X = torch.relu(X) * keep_low[None, :, None]
            return X.pow(g)
        return torch.log(torch.relu(X) + EPSILON) * keep_low[None, :, None]

    def _CFP(self, spec):
        """cfp.py:119-135 on half vectors (B, H, T)."""
        spec = torch.relu(spec).pow(self.g[0])
        w_in = self._mirror_count(spec.device)
        if self.NumofLayer >= 2:
            for gc in range(1, self.NumofLayer):
                if np.remainder(gc, 2) == 1:
                    ceps = self.nonlinear_func(self._real_fft_half(spec, w_in), self.g[gc], self.tc_idx)
                    w_in = self._cut_weights(self.tc_idx, spec.device)[1]
                else:
                    spec = self.nonlinear_func(self._real_fft_half(ceps, w_in), self.g[gc], self.fc_idx)
                    w_in = self._cut_weights(self.fc_idx, spec.device)[1]
        return spec, ceps  # one layer only: UnboundLocalError, as in the reference

    def _maps(self, x: torch.Tensor, drop_edge_frames: bool):
        if not isinstance(x, torch.Tensor):
            raise TypeError("x must be a torch.Tensor")
        if x.dim() != 2:
            # torch.stft takes (L) or (B, L); the reference's transpose(1, 2) then needs the batch axis
            if x.dim() == 1:
                raise IndexError("Dimension out of range (expected to be in range of [-2, 1], but got 2)")
            raise RuntimeError(f"stft: expected a 1D or 2D tensor, but got {x.dim()}D tensor")
        if torch.is_grad_enabled() and x.requires_grad:
            raise NotImplementedError("nnaudio_b200: CFP is forward-only; run under torch.no_grad()")
        _C._dev_wave(x, "x")  # fp32, bf16 or fp16; the transform itself runs in fp32
        tfr0 = self._stft_magnitude(x)                       # (B, H, T)
        if drop_edge_frames:
            tfr0 = tfr0[:, :, 1:-1].contiguous()             # cfp.py:151-153
        B, H, T = tfr0.shape
        n_low = min(int(round(self.N / 2)), H)
        n_f, n_q = min(self.HighFreqIdx, n_low), min(self.HighQuefIdx, n_low)
        f2l, q2l = self.freq2logfreq_matrix.detach(), self.quef2logfreq_matrix.detach()
        if f2l.shape[1] != n_f or q2l.shape[1] != n_q:
            raise RuntimeError(f"size mismatch: the log-frequency maps expect {f2l.shape[1]} / {q2l.shape[1]} "
                               f"bins, the transform keeps {n_f} / {n_q}")
        if T == 0:
            empty = tfr0.new_zeros((B, f2l.shape[0], 0))
            return empty, empty.clone(), empty.clone(), empty.clone()
        tfr, ceps = self._CFP(tfr0)
        _C._dev_f32(f2l, "freq2logfreq_matrix")
        _C._dev_f32(q2l, "quef2logfreq_matrix")
        both = self._freq_gemm(torch.cat((tfr0[:, :n_f], tfr[:, :n_f]), 0), f2l.shape[0],
                               (f2l.data_ptr(), f2l._version), lambda: f2l, keep=(f2l,))
        tfrL0, tfrLF = both[:B], both[B:]
        tfrLQ = self._quef_gemm(ceps[:, :n_q], q2l.shape[0], (q2l.data_ptr(), q2l._version), lambda: q2l,
                                keep=(q2l,))
        self.t = np.arange(self.hop_length, np.ceil(len(x) / float(self.hop_length)) * self.hop_length,
                           self.hop_length)  # cfp.py:174-178 (len(x) is the batch size there too)
        return tfrLF * tfrLQ, tfrL0.contiguous(), tfrLF.contiguous(), tfrLQ


class Combined_Frequency_Periodicity(_CFPBase):
    """cfp.py:9-246: returns ``(Z, tfrL0, tfrLF, tfrLQ)``, each ``(B, Nest - 1, T - 2)`` — the first and
    last frame are discarded."""

    def forward(self, x):
        return self._maps(x, drop_edge_frames=True)


class CFP(_CFPBase):
    """cfp.py:249-484: returns ``Z`` only, ``(B, Nest - 1, T)`` with ``T = L // hop + 1`` like the other
    spectrogram classes."""

    def forward(self, x):
        return self._maps(x, drop_edge_frames=False)[0]
