"""Pins the CPU oracle (oracle/nnaudio_oracle.py) against
 (i) outputs of the unmodified reference on the cases of tests/golden/cases.py,
 (ii) the reference's OWN golden vectors, replayed exactly as its tests do
      (Installation/tests/test_cqt.py:94-262, rtol = atol = 1e-3)."""
import warnings

import numpy as np
import pytest

from helpers import (CASES, REF_GROUND_TRUTHS, SWEEP_CTOR, build, case_input, is_phase, make_input,
                     out_key, phase_to_unit, ref_ground_truths, ref_outputs, rel_errors, run_oracle)

# fp64 oracle vs the reference's fp32 arithmetic
TOL_MAX, TOL_L2 = 2e-5, 5e-6


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_matches_reference_outputs(case):
    cid, cls, ctor, inp, fwds = case
    mod = build(cls, ctor)
    x = case_input(cid, inp)
    for kw in fwds:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            got = run_oracle(cls, mod, x, kw)
        want = ref_outputs()[out_key(cid, kw)]
        if is_phase(kw):
            # phase of near-zero bins is ill-conditioned: compare where it is defined
            mag = run_oracle(cls, mod, x, dict(kw, output_format="Magnitude"))
            keep = want.pick(mag > 1e-3 * mag.max())
            g, w = phase_to_unit(cls, want.pick(got))[keep], phase_to_unit(cls, want.values)[keep]
            assert np.abs(g - w).max() < 2e-3, (cid, kw)
            continue
        emax, el2 = rel_errors(want.pick(got), want.values)
        tol_max = 4e-4 if cls == "MFCC" else TOL_MAX  # dB of tiny powers amplifies fp32 noise
        assert emax < tol_max and el2 < max(TOL_L2, tol_max / 4), (cid, kw, emax, el2)


@pytest.mark.parametrize("key", sorted(REF_GROUND_TRUTHS))
def test_oracle_matches_reference_ground_truths(key):
    cls, method, kw, transform = REF_GROUND_TRUTHS[key]
    mod = build(cls, SWEEP_CTOR)
    x = make_input(("chirp", method))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        y = run_oracle(cls, mod, x, kw)
    stored = ref_ground_truths()[key]
    y_full, y, gt = y, stored.pick(y), stored.values
    if transform is not None:
        # The goldens store log(X + eps).  Where X << eps the stored value is the
        # reference's own fp32 rounding noise amplified by 1/eps, so the log is
        # compared (at the reference's tolerance) where X carries signal, and the
        # linear magnitude is compared absolutely everywhere.
        eps = 1e-5 if transform == "log1e-5" else 1e-2
        lin_gt = np.exp(gt.astype(np.float64)) - eps
        assert np.abs(y - lin_gt).max() < 1e-5 * max(1.0, np.abs(lin_gt).max()) + 2e-3 * eps
        keep = y > 1e-2 * eps + 1e-5 * y_full.max()
        assert np.allclose(np.log(y[keep] + eps), gt[keep], rtol=1e-3, atol=1e-3)
        return
    if is_phase(kw):
        # the reference's phase golden holds cos/sin of atan2 on bins that are exactly
        # zero-energy in places; its own tolerance applies where energy exists
        mag = run_oracle(cls, mod, x, dict(kw, output_format="Magnitude"))
        keep = stored.pick(mag > 1e-4 * mag.max())
        assert np.allclose(y[keep], gt[keep], rtol=1e-3, atol=1e-3)
        return
    assert np.allclose(y, gt, rtol=1e-3, atol=1e-3), np.abs(y - gt).max()


def test_vqt_gamma0_equals_cqt2010v2_exactly():
    """Installation/tests/test_vqt.py:30-41: `(C2 == V2).all()`."""
    x = make_input(("randn", 50, (2, 32768)))
    c = run_oracle("CQT2010v2", build("CQT2010v2", dict(sr=22050)), x, dict(output_format="Magnitude"))
    v = run_oracle("VQT", build("VQT", dict(sr=22050, gamma=0)), x, dict(output_format="Magnitude"))
    assert (c == v).all()


def test_cfg1_matches_rfft_restatement_of_librosa():
    """SURVEY.md §8(c): librosa.stft restated as rfft(hann * frames) over a
    reflect-padded signal (librosa itself is not installed)."""
    from scipy.signal import get_window
    x = make_input(("randn", 0, (1, 16000)))
    mod = build("STFT", dict(n_fft=512, hop_length=256, sr=16000))
    got = run_oracle("STFT", mod, x, dict(output_format="Complex"))
    xp = np.pad(x[0].astype(np.float64), 256, mode="reflect")
    frames = np.lib.stride_tricks.sliding_window_view(xp, 512)[::256]
    spec = np.fft.rfft(frames * get_window("hann", 512, fftbins=True), axis=-1).T
    want = np.stack((spec.real, spec.imag), -1)[None]
    emax, el2 = rel_errors(got, want)
    assert emax < 1e-5 and el2 < 1e-5, (emax, el2)
