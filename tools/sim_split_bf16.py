#!/usr/bin/env python
"""Predict, on the CPU, what the split-bf16 (x_hi*w_hi + x_lo*w_hi + x_hi*w_lo) tensor-core
forward does to a gradient test: the float64 stand-in kernels of tests/cpu_kernels.py run the
host-side autograd compositions, and the forward contraction is replaced by an emulation of the
three-term bf16 split.  Prints, per trainable-kernel case, the gradient error vs the exact
(float64) forward and vs the reference's autograd fixture.

Used in round 1 to explain a 1.6e-4 dW error on the GPU (ill-conditioned Magnitude loss on ~100
frames) without spending GPU time.  Test infrastructure only.

    python tools/sim_split_bf16.py [case-id-substring]
"""
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    sys.path.insert(0, p)

import torch  # noqa: E402

from helpers import build, ref_outputs, rel_errors  # noqa: E402
import cpu_kernels  # noqa: E402
from cases import WGRAD_CASES, loss_weights, make_input  # noqa: E402
from nnaudio_b200 import _C  # noqa: E402


def _split(v):
    hi = v.float().bfloat16().float()
    lo = (v.float() - hi).bfloat16().float()
    return hi.double(), lo.double()


def framed_split_bf16(x, w_re, w_im, hop, center, pad_mode):
    K = w_re.shape[1]
    xp = cpu_kernels._pad(x.float(), K // 2 if center else 0, pad_mode)
    xh, xl = _split(xp)

    def conv(a, b):
        return torch.nn.functional.conv1d(a[:, None, :], b[:, None, :], stride=hop)

    out = []
    for w, sign in ((w_re, 1.0), (w_im, -1.0)):
        wh, wl = _split(w)
        out.append(sign * (conv(xh, wh) + conv(xl, wh) + conv(xh, wl)))
    return torch.stack(out, -1)


def split_forward(x, k_real, k_imag, packed, kb, ke, hop, center, pad_mode, scale, scale_all, fmt,
                  eps, path=None):
    return framed_split_bf16(x, k_real, k_imag, hop, center, pad_mode).float()


class _Patch:
    def setattr(self, obj, name, value, raising=True):
        setattr(obj, name, value)


def grads(case, forward):
    cid, cls, ctor, inp, kw, names = case
    _C.cqt1992v2_forward = forward
    mod = build(cls, ctor)
    x = torch.from_numpy(make_input(inp))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = mod(x, **kw)
    w = torch.from_numpy(loss_weights(cid, tuple(y.shape)))
    (y * w).sum().backward()
    params = dict(mod.named_parameters())
    return {n: params[n].grad.numpy() for n in names}


def main():
    cpu_kernels.install(_Patch())
    want = sys.argv[1] if len(sys.argv) > 1 else ""
    for case in WGRAD_CASES:
        if want not in case[0] or case[1] not in ("CQT1992", "CQT2010", "CQT2010v2"):
            continue  # the modules whose training path goes through cqt1992v2_forward stand-ins
        approx = grads(case, split_forward)
        exact = grads(case, cpu_kernels.cqt1992v2_forward)
        for n in approx:
            e_exact = rel_errors(approx[n], exact[n])
            want = ref_outputs()[f"wgrad|{case[0]}|{n}"]
            e_ref = rel_errors(want.pick(approx[n]), want.values)
            print(f"{case[0]:18s} {n:18s} split-bf16 vs exact {e_exact[0]:.2e} / {e_exact[1]:.2e}   "
                  f"vs reference autograd {e_ref[0]:.2e} / {e_ref[1]:.2e}")


if __name__ == "__main__":
    main()
