"""Parity cases shared by ``make_golden.py`` (runs the unmodified reference in the
build container) and the test-suite (runs the oracle and the CUDA path).

Inputs are regenerated from the spec (NumPy ``RandomState`` / ``scipy.signal.chirp``
are platform-stable), so only the reference OUTPUTS are stored in
``ref_outputs.npz``, and of each output only a fixed sample of its entries
(``sample_index``) plus its extreme entries, so that the stored files stay small.
"""
from __future__ import annotations

import zlib

import numpy as np
from scipy.signal import chirp

GOLDEN_SAMPLES = 2048  # entries kept of each stored reference array


def sample_index(key: str, shape, peaks=()) -> np.ndarray:
    """Sorted flat (C-order) indices of the entries of the reference array ``key`` that are stored: all
    of them for a small array, else ``GOLDEN_SAMPLES`` drawn with a seed derived from ``key``, plus
    ``peaks`` (the array's extremes, stored beside the values so that max-normalised errors use the full
    array's maximum)."""
    n = int(np.prod(shape))
    if n <= GOLDEN_SAMPLES:
        return np.arange(n)
    idx = np.random.RandomState(zlib.crc32(key.encode())).choice(n, GOLDEN_SAMPLES, replace=False)
    return np.union1d(idx, np.asarray(peaks, dtype=np.int64))


def array_peaks(a: np.ndarray) -> np.ndarray:
    """Flat indices of max |a|, max a and min a."""
    a = np.asarray(a).reshape(-1)
    return np.array([np.abs(a).argmax(), a.argmax(), a.argmin()], dtype=np.int64)


def pack_sampled(outputs: dict) -> dict:
    """{key: full array} -> the arrays of a sampled fixture file (values, shape and peaks per key)."""
    packed = {}
    for key, a in outputs.items():
        peaks = array_peaks(a)
        packed[key] = np.asarray(a, dtype=np.float32).reshape(-1)[sample_index(key, a.shape, peaks)]
        packed[key + "|shape"] = np.array(a.shape, dtype=np.int64)
        packed[key + "|peaks"] = peaks
    return packed


def istft_spectrogram(case, wsin=None, wcos=None) -> np.ndarray:
    """Spectrogram input of an ISTFT case: seeded noise ('module'), or the fp64 oracle STFT (rounded to
    fp32) of seeded noise with the bases ``wsin`` / ``wcos`` of the case's STFT module ('roundtrip')."""
    cid, n_fft, hop, win, kind, spec = case
    rng = np.random.RandomState(spec["seed"])
    if kind == "module":
        return rng.standard_normal(spec["shape"]).astype(np.float32)
    from nnaudio_oracle import stft

    x = rng.standard_normal(spec["shape"]).astype(np.float32)
    return stft(x, wsin, wcos, hop, center=True, pad_mode="reflect", output_format="Complex").astype(np.float32)


def make_input(spec) -> np.ndarray:
    kind = spec[0]
    if kind == "randn":
        _, seed, shape = spec
        return np.random.RandomState(seed).standard_normal(shape).astype(np.float32)
    if kind == "randn_decay":
        # clips with very different levels: exercises MFCC's per-clip top_db floor
        _, seed, shape = spec
        x = np.random.RandomState(seed).standard_normal(shape).astype(np.float32)
        gains = (10.0 ** (-np.arange(shape[0]))).astype(np.float32)[:, None]
        t = np.linspace(0, 1, shape[1], dtype=np.float32)[None, :]
        return (x * gains * np.exp(-6.0 * t)).astype(np.float32)
    if kind == "chirp":
        # the reference's own golden-vector input (tests/test_cqt.py:94-103)
        _, method = spec
        fs, t, f0, f1 = 44100, 1, 55, 22050
        s = np.linspace(0, t, fs * t)
        return chirp(s, f0, 1, f1, method=method).astype(np.float32)[None, :]
    raise ValueError(kind)


# id, class name, ctor kwargs, input spec, list of forward kwargs
CASES = [
    # ---- STFT (cfg1 of BASELINE.json first) --------------------------------
    ("stft_cfg1", "STFT", dict(n_fft=512, hop_length=256, sr=16000), ("randn", 0, (1, 16000)),
     [dict(output_format="Complex"), dict(output_format="Magnitude"), dict(output_format="Phase")]),
    ("stft_winlen_hamming", "STFT", dict(n_fft=512, win_length=400, hop_length=128, window="hamming"),
     ("randn", 1, (2, 4000)), [dict(output_format="Complex")]),
    ("stft_linear_bins", "STFT",
     dict(n_fft=256, freq_bins=80, freq_scale="linear", fmin=50, fmax=6000, sr=22050, hop_length=64),
     ("randn", 2, (2, 2000)), [dict(output_format="Complex")]),
    ("stft_log_nocenter_oddhop", "STFT",
     dict(n_fft=256, freq_bins=60, freq_scale="log", fmin=50, fmax=6000, sr=22050, hop_length=100,
          center=False),
     ("randn", 3, (1, 3000)), [dict(output_format="Magnitude")]),
    ("stft_constant_pad", "STFT", dict(n_fft=512, hop_length=128, pad_mode="constant"),
     ("randn", 4, (2, 3000)), [dict(output_format="Magnitude"), dict(output_format="Phase")]),
    ("stft_trainable_eps", "STFT", dict(n_fft=512, hop_length=128, trainable=True),
     ("randn", 5, (1, 3000)), [dict(output_format="Magnitude")]),
    ("stft_2048", "STFT", dict(n_fft=2048, hop_length=512), ("randn", 6, (1, 22050)),
     [dict(output_format="Magnitude")]),
    ("stft_default_hop_1d_input", "STFT", dict(n_fft=256, window="hann"), ("randn", 7, (1, 4000)),
     [dict(output_format="Complex")]),
    # ---- MelSpectrogram -----------------------------------------------------
    ("mel_small", "MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40),
     ("randn", 10, (2, 8000)), [dict()]),
    ("mel_cfg2_shape", "MelSpectrogram", dict(sr=22050, n_fft=2048, hop_length=512, n_mels=128),
     ("randn", 11, (2, 22050)), [dict()]),
    ("mel_htk_power1_winlen", "MelSpectrogram",
     dict(sr=16000, n_fft=1024, win_length=1000, hop_length=256, n_mels=64, power=1.0, htk=True,
          fmin=20, fmax=7600),
     ("randn", 12, (1, 8000)), [dict()]),
    # ---- MFCC ---------------------------------------------------------------
    ("mfcc_cfg5_shape", "MFCC", dict(sr=16000), ("randn_decay", 20, (3, 16000)), [dict()]),
    ("mfcc_small_no_topdb", "MFCC",
     dict(sr=22050, n_mfcc=13, n_fft=512, hop_length=160, n_mels=40, top_db=None),
     ("randn", 21, (2, 6000)), [dict()]),
    # ---- Gammatonegram ------------------------------------------------------
    ("gammatone_small", "Gammatonegram", dict(sr=22050, n_fft=1024, n_bins=32, hop_length=256),
     ("randn", 30, (2, 8000)), [dict()]),
    ("gammatone_default", "Gammatonegram", dict(sr=22050), ("randn", 31, (1, 22050)), [dict()]),
    # ---- CQT1992v2 ----------------------------------------------------------
    ("cqt1992v2_random", "CQT1992v2",
     dict(sr=22050, fmin=220, n_bins=48, bins_per_octave=12, hop_length=256),
     ("randn", 40, (2, 16000)),
     [dict(output_format="Complex"),
      dict(output_format="Magnitude", normalization_type="wrap"),
      dict(output_format="Phase", normalization_type="convolutional")]),
    ("cqt1992v2_nocenter", "CQT1992v2",
     dict(sr=22050, fmin=440, n_bins=24, hop_length=128, center=False, pad_mode="constant"),
     ("randn", 41, (1, 8000)), [dict(output_format="Magnitude")]),
    # ---- CQT2010v2 ----------------------------------------------------------
    ("cqt2010v2_random", "CQT2010v2", dict(sr=22050, n_bins=84), ("randn", 50, (2, 32768)),
     [dict(output_format="Magnitude"), dict(output_format="Complex")]),
    ("cqt2010v2_early_downsample", "CQT2010v2", dict(sr=44100, n_bins=72, fmin=32.7),
     ("randn", 51, (1, 40000)), [dict(output_format="Complex")]),
    ("cqt2010v2_reflect_fallback", "CQT2010v2", dict(sr=22050, n_bins=84),
     ("randn", 52, (1, 6000)), [dict(output_format="Complex")]),
    ("cqt2010v2_cfg4_bins88", "CQT2010v2", dict(sr=22050, n_bins=88), ("randn", 53, (1, 16384)),
     [dict(output_format="Magnitude"), dict(output_format="Phase", normalization_type="wrap")]),
    # ---- VQT ----------------------------------------------------------------
    ("vqt_gamma0", "VQT", dict(sr=22050, gamma=0), ("randn", 50, (2, 32768)),
     [dict(output_format="Magnitude")]),
    ("vqt_gamma5", "VQT", dict(sr=22050, gamma=5, n_bins=60), ("randn", 61, (1, 32768)),
     [dict(output_format="Complex")]),
    # ---- first-generation (frequency-domain) CQTs, SURVEY §8f next #3 ---------
    ("cqt1992_fmin220", "CQT1992", dict(sr=22050, fmin=220, n_bins=60), ("randn", 62, (2, 16384)),
     [dict(output_format="Magnitude"), dict(output_format="Complex", normalization_type="wrap"),
      dict(output_format="Phase", normalization_type="convolutional")]),
    ("cqt1992_nocenter_constant", "CQT1992",
     dict(sr=16000, fmin=110, n_bins=36, hop_length=256, center=False, pad_mode="constant"),
     ("randn", 63, (1, 12000)), [dict(output_format="Complex")]),
    ("cqt2010_default", "CQT2010", dict(sr=22050, n_bins=84), ("randn", 64, (2, 32768)),
     [dict(output_format="Magnitude"), dict(output_format="Complex", normalization_type="wrap"),
      dict(output_format="Phase", normalization_type="convolutional")]),
    ("cqt2010_early_downsample", "CQT2010", dict(sr=44100, n_bins=72, fmin=32.7),
     ("randn", 65, (1, 40000)), [dict(output_format="Complex")]),
]

# The reference's own golden vectors (Installation/tests/ground-truths/*.npy) and
# the test that loads each one (tests/test_cqt.py:94-262).
#   key in ref_ground_truths.npz -> (class, chirp method, forward kwargs, transform)
REF_GROUND_TRUTHS = {
    "log-sweep-cqt-1992-mag": ("CQT1992v2", "logarithmic", dict(output_format="Magnitude"), "log1e-5"),
    "log-sweep-cqt-1992-complex": ("CQT1992v2", "logarithmic", dict(output_format="Complex"), None),
    "log-sweep-cqt-1992-phase": ("CQT1992v2", "logarithmic", dict(output_format="Phase"), None),
    "linear-sweep-cqt-1992-mag": ("CQT1992v2", "linear", dict(output_format="Magnitude"), "log1e-5"),
    "linear-sweep-cqt-1992-complex": ("CQT1992v2", "linear", dict(output_format="Complex"), None),
    "linear-sweep-cqt-1992-phase": ("CQT1992v2", "linear", dict(output_format="Phase"), None),
    "log-sweep-cqt-2010-mag": ("CQT2010v2", "logarithmic", dict(output_format="Magnitude"), "log1e-2"),
    "log-sweep-cqt-2010-complex": ("CQT2010v2", "logarithmic", dict(output_format="Complex"), None),
    "linear-sweep-cqt-2010-mag": ("CQT2010v2", "linear", dict(output_format="Magnitude"), "log1e-2"),
    "linear-sweep-cqt-2010-complex": ("CQT2010v2", "linear", dict(output_format="Complex"), None),
}
SWEEP_CTOR = dict(sr=44100, fmin=55, n_bins=207, bins_per_octave=24)


# Inverse STFT cases (SURVEY.md §8f next #2): id, n_fft, hop, window, kind, spec
#   'roundtrip': X = STFT of x (istft_spectrogram), y = reference STFT(iSTFT=True).inverse(X, onesided=True,
#                length=L|None)
#   'module'   : y = reference iSTFT(...)(X_random, onesided=False)
ISTFT_CASES = [
    ("istft_roundtrip_512", 512, 128, "hann", "roundtrip", dict(seed=70, shape=(2, 4000), length=4000)),
    ("istft_roundtrip_1024_nolen", 1024, 256, "hamming", "roundtrip", dict(seed=71, shape=(2, 8000), length=None)),
    ("istft_roundtrip_2048", 2048, 512, "hann", "roundtrip", dict(seed=72, shape=(1, 22050), length=22050)),
    ("istft_module_256_full", 256, 64, "hann", "module", dict(seed=73, shape=(2, 256, 40, 2))),
]


# Constructor-only sweep: state_dict keys / shapes / sha256 of every buffer against the reference
# (no forward pass; widens the "buffers are bit-identical" drop-in claim beyond the CASES configs).
DESIGN_CASES = [
    ("d_stft_blackman_win300", "STFT", dict(n_fft=1024, win_length=300, hop_length=100, window="blackmanharris")),
    ("d_stft_gaussian_tuple", "STFT", dict(n_fft=512, window=("gaussian", 60))),
    ("d_stft_linear_fmin_fmax", "STFT", dict(n_fft=1024, freq_bins=200, freq_scale="linear", fmin=100, fmax=7000, sr=16000)),
    ("d_stft_log", "STFT", dict(n_fft=2048, freq_bins=120, freq_scale="log", fmin=55, fmax=8000, sr=22050)),
    ("d_stft_log2", "STFT", dict(n_fft=1024, freq_bins=96, freq_scale="log2", fmin=60, fmax=6000, sr=22050)),
    ("d_stft_istft_buffers", "STFT", dict(n_fft=256, hop_length=64, iSTFT=True, window="hamming")),
    ("d_istft_module", "iSTFT", dict(n_fft=512, hop_length=128, window="hann")),
    ("d_mel_htk_nonorm", "MelSpectrogram", dict(sr=16000, n_fft=400, hop_length=160, n_mels=64, htk=True, norm=None, fmin=60, fmax=7600)),
    ("d_mel_48k", "MelSpectrogram", dict(sr=48000, n_fft=4096, n_mels=256, fmin=20)),
    ("d_mel_power1", "MelSpectrogram", dict(sr=22050, n_fft=1024, n_mels=80, power=1.0, window="hamming")),
    ("d_mfcc_40", "MFCC", dict(sr=22050, n_mfcc=40, n_fft=2048, n_mels=128)),
    ("d_gammatone_96", "Gammatonegram", dict(sr=44100, n_fft=4096, n_bins=96, fmin=30, fmax=16000)),
    ("d_gammatone_small", "Gammatonegram", dict(sr=8000, n_fft=256, n_bins=16)),
    ("d_cqt1992v2_24bpo", "CQT1992v2", dict(sr=22050, fmin=55, n_bins=96, bins_per_octave=24, filter_scale=0.5)),
    ("d_cqt1992v2_norm2_hamming", "CQT1992v2", dict(sr=16000, fmin=110, n_bins=60, norm=2, window="hamming")),
    ("d_cqt1992v2_fmax", "CQT1992v2", dict(sr=22050, fmin=65.4, fmax=4000, bins_per_octave=12)),
    ("d_cqt2010v2_noearly_24bpo", "CQT2010v2", dict(sr=22050, n_bins=120, bins_per_octave=24, earlydownsample=False)),
    ("d_cqt2010v2_48k", "CQT2010v2", dict(sr=48000, n_bins=96, fmin=27.5, filter_scale=2)),
    ("d_vqt_gamma20_36bpo", "VQT", dict(sr=22050, n_bins=108, bins_per_octave=36, gamma=20)),
    ("d_vqt_noearly", "VQT", dict(sr=16000, n_bins=72, gamma=3, earlydownsample=False)),
    ("d_cqt1992_24bpo", "CQT1992", dict(sr=44100, fmin=220, n_bins=80, bins_per_octave=24)),
    ("d_cqt2010_24bpo", "CQT2010", dict(sr=44100, fmin=110, n_bins=160, bins_per_octave=24)),
]


# Forward outputs for the constructor sweep (default output format, one short clip each): CPU
# host-layer and oracle parity on configurations beyond CASES.  Length per class keeps the
# fixture small; GPU runs of these configurations are round-2 work.
def sweep_input(case_id: str, cls: str):
    length = {"STFT": 6000, "MelSpectrogram": 12000, "MFCC": 12000, "Gammatonegram": 12000,
              "CQT1992v2": 24000, "CQT2010v2": 40000, "VQT": 40000, "CQT1992": 24000, "CQT2010": 40000}[cls]
    seed = 2000 + sum(ord(c) for c in case_id) % 1000
    return ("randn", seed, (1, length))


SWEEP_FORWARD = [c for c in DESIGN_CASES if c[1] != "iSTFT"]


# Error-behaviour scenarios: what the reference raises (exception type) for malformed constructor
# arguments and inputs; recorded into ref_errors.json.  ("ctor",) | ("forward", shape, kwargs) |
# ("inverse", shape, kwargs)
ERROR_CASES = [
    ("e_stft_short_reflect", "STFT", dict(n_fft=512), ("forward", (1, 100), {})),
    ("e_stft_4d_input", "STFT", dict(n_fft=256), ("forward", (1, 1, 2, 4000), {})),
    ("e_stft_two_channels", "STFT", dict(n_fft=256), ("forward", (2, 2, 4000), {})),
    ("e_stft_inverse_without_flag", "STFT", dict(n_fft=256), ("inverse", (1, 129, 10, 2), {})),
    ("e_stft_inverse_3d", "STFT", dict(n_fft=256, iSTFT=True), ("inverse", (1, 129, 10), {})),
    ("e_istft_3d", "iSTFT", dict(n_fft=256), ("forward", (1, 256, 10), {})),
    ("e_mel_short_reflect", "MelSpectrogram", dict(sr=16000, n_fft=1024), ("forward", (2, 300), {})),
    ("e_cqt1992v2_nyquist", "CQT1992v2", dict(sr=8000, fmin=220, n_bins=84), ("ctor",)),
    ("e_cqt1992v2_short_reflect", "CQT1992v2", dict(sr=22050, fmin=220, n_bins=12), ("forward", (1, 100), {})),
    ("e_cqt1992v2_bad_norm", "CQT1992v2", dict(sr=22050, fmin=220, n_bins=12),
     ("forward", (1, 8000), dict(normalization_type="bogus"))),
    ("e_cqt2010v2_nyquist", "CQT2010v2", dict(sr=8000, n_bins=96), ("ctor",)),
    ("e_cqt2010v2_bad_norm", "CQT2010v2", dict(sr=22050, n_bins=24, fmin=220),
     ("forward", (1, 8000), dict(normalization_type="bogus"))),
    ("e_cqt2010v2_4d_input", "CQT2010v2", dict(sr=22050, n_bins=24, fmin=220), ("forward", (1, 1, 1, 8000), {})),
    ("e_vqt_nyquist", "VQT", dict(sr=8000, n_bins=96), ("ctor",)),
    ("e_cqt1992_nyquist", "CQT1992", dict(sr=8000, fmin=220, n_bins=84), ("ctor",)),
    ("e_cqt2010_nyquist", "CQT2010", dict(sr=8000, n_bins=96), ("ctor",)),
]


# Input-gradient cases (SURVEY.md §8f next #1, dX): loss = sum(out * w), w ~ N(0,1) seeded;
# the fixture holds the reference's x.grad (autograd through its conv1d path on CPU).
GRAD_CASES = [
    ("grad_stft_complex", "STFT", dict(n_fft=512, hop_length=128), ("randn", 80, (2, 4000)),
     dict(output_format="Complex")),
    ("grad_stft_magnitude", "STFT", dict(n_fft=512, hop_length=128), ("randn", 81, (2, 4000)),
     dict(output_format="Magnitude")),
    ("grad_stft_oddhop_constant", "STFT", dict(n_fft=256, hop_length=100, pad_mode="constant"),
     ("randn", 82, (1, 3000)), dict(output_format="Magnitude")),
    ("grad_mel", "MelSpectrogram", dict(sr=16000, n_fft=512, hop_length=128, n_mels=40),
     ("randn", 83, (2, 8000)), dict()),
    ("grad_mfcc", "MFCC", dict(sr=16000, n_fft=512, hop_length=160, n_mels=40, n_mfcc=13),
     ("randn", 84, (2, 6000)), dict()),
    ("grad_gammatone", "Gammatonegram", dict(sr=22050, n_fft=1024, n_bins=32, hop_length=256),
     ("randn", 85, (1, 8000)), dict()),
    ("grad_cqt1992v2_mag", "CQT1992v2", dict(sr=22050, fmin=220, n_bins=48, hop_length=256),
     ("randn", 86, (2, 16000)), dict(output_format="Magnitude")),
    ("grad_cqt1992v2_complex_wrap", "CQT1992v2",
     dict(sr=22050, fmin=440, n_bins=24, hop_length=128, center=False),
     ("randn", 87, (1, 8000)), dict(output_format="Complex", normalization_type="wrap")),
    # the /2 pyramid: gradients flow back through every FIR decimation stage
    ("grad_cqt2010v2_mag", "CQT2010v2", dict(sr=22050, n_bins=84), ("randn", 88, (2, 32768)),
     dict(output_format="Magnitude")),
    ("grad_cqt2010v2_early_complex", "CQT2010v2", dict(sr=44100, n_bins=72, fmin=32.7),
     ("randn", 89, (1, 65536)), dict(output_format="Complex", normalization_type="convolutional")),
    ("grad_cqt2010v2_reflect_fallback", "CQT2010v2", dict(sr=22050, n_bins=84),
     ("randn", 93, (1, 8192)), dict(output_format="Magnitude")),
    ("grad_cqt1992", "CQT1992", dict(sr=22050, fmin=220, n_bins=48, hop_length=256),
     ("randn", 99, (2, 12000)), dict(output_format="Magnitude")),
    ("grad_cqt2010", "CQT2010", dict(sr=22050, n_bins=60), ("randn", 100, (1, 32768)),
     dict(output_format="Complex")),
    ("grad_vqt_gamma5", "VQT", dict(sr=22050, gamma=5, n_bins=60), ("randn", 94, (1, 32768)),
     dict(output_format="Magnitude")),
]


# Trainable-kernel cases: the fixture holds the reference's gradients of the listed parameters.
WGRAD_CASES = [
    ("wgrad_stft", "STFT", dict(n_fft=256, hop_length=64, trainable=True), ("randn", 90, (3, 4000)),
     dict(output_format="Magnitude"), ["wsin", "wcos"]),
    ("wgrad_mel", "MelSpectrogram",
     dict(sr=16000, n_fft=256, hop_length=64, n_mels=20, trainable_mel=True, trainable_STFT=True),
     ("randn", 91, (2, 4000)), dict(), ["mel_basis", "stft.wsin", "stft.wcos"]),
    ("wgrad_cqt1992v2", "CQT1992v2",
     dict(sr=22050, fmin=880, n_bins=24, hop_length=128, trainable=True),
     ("randn", 92, (2, 8000)), dict(output_format="Magnitude"),
     ["cqt_kernels_real", "cqt_kernels_imag"]),
    # one trainable bank shared by all octaves: its gradient is the sum over the pyramid levels
    ("wgrad_cqt2010v2", "CQT2010v2", dict(sr=22050, n_bins=48, fmin=110, trainable=True),
     ("randn", 95, (2, 16384)), dict(output_format="Magnitude"),
     ["cqt_kernels_real", "cqt_kernels_imag"]),
]

WGRAD_CASES += [
    # gradients reach the reference's own parameters (DFT rows and spectral kernels) through the fold
    ("wgrad_cqt1992", "CQT1992",
     dict(sr=22050, fmin=880, n_bins=24, hop_length=128, trainable_STFT=True, trainable_CQT=True),
     ("randn", 101, (2, 6000)), dict(output_format="Magnitude"),
     ["wsin", "wcos", "cqt_kernels_real", "cqt_kernels_imag"]),
    # (4 x 32768 samples: d|c| = c/|c| is ill-conditioned where |c| ~ 0, so a Magnitude-loss
    # gradient summed over only ~100 frames amplifies any forward rounding — 1.6e-4 measured with
    # the split-bf16 forward on a (1, 16384) input vs 1.3e-5 with the fp32 CUDA-core forward)
    ("wgrad_cqt2010", "CQT2010", dict(sr=22050, n_bins=36, fmin=110, trainable_CQT=True),
     ("randn", 102, (4, 32768)), dict(output_format="Magnitude"),
     ["cqt_kernels_real", "cqt_kernels_imag"]),
]


# Gradients w.r.t. the spectrogram through the inverse STFT (reference autograd on CPU):
#   (id, n_fft, hop, window, kind, spec) as ISTFT_CASES; loss = sum(y * w)
ISTFT_GRAD_CASES = [
    ("grad_istft_onesided_512", 512, 128, "hann", "roundtrip", dict(seed=96, shape=(2, 4000), length=4000)),
    ("grad_istft_onesided_nolen", 256, 64, "hamming", "roundtrip", dict(seed=97, shape=(1, 3000), length=None)),
    ("grad_istft_module_full", 256, 64, "hann", "module", dict(seed=98, shape=(2, 256, 40, 2))),
]


def attribute_surface(module) -> dict:
    """JSON-able view of a module's public, non-tensor attributes (what user code reads:
    ``n_fft``, ``stride``, ``frequencies``, ``kernel_width`` ...).  Used on the reference by
    make_golden.py and on ours by tests/test_host_logic.py."""
    import torch

    base = set(vars(torch.nn.Module()))
    out = {}
    for k, v in vars(module).items():
        if k.startswith("_") or k in base:
            continue
        if isinstance(v, (bool, int, float, str, type(None))):
            out[k] = v
        elif isinstance(v, (np.floating, np.integer)):
            out[k] = float(v)
        elif isinstance(v, np.ndarray):
            out[k] = ["ndarray", list(v.shape), str(v.dtype), float(np.abs(v).sum())]
        elif isinstance(v, (list, tuple)):
            out[k] = [type(v).__name__, len(v)]
        else:
            out[k] = type(v).__name__
    return out


def loss_weights(case_id: str, shape) -> np.ndarray:
    seed = 1000 + sum(ord(c) for c in case_id) % 1000
    return np.random.RandomState(seed).standard_normal(shape).astype(np.float32)


def out_key(case_id: str, fwd_kwargs: dict) -> str:
    tag = "_".join(f"{k[:3]}-{v}" for k, v in sorted(fwd_kwargs.items()))
    return f"{case_id}|{tag}" if tag else case_id


# --------------------------------------------------------------------------- #
# Combined_Frequency_Periodicity / CFP (features/cfp.py) — fixtures from make_golden_cfp.py
# --------------------------------------------------------------------------- #
# id, class name, ctor kwargs, input spec
CFP_CASES = [
    ("cfp_default", "CFP", dict(), ("randn", 40, (2, 16000))),
    ("cfp_combined_default", "Combined_Frequency_Periodicity", dict(), ("randn", 41, (2, 8000))),
    ("cfp_fr4_four_layers", "CFP",
     dict(fr=4, hop_length=160, window_size=1025, g=[0.2, 0.5, 0.8, 1.0], NumPerOct=24), ("randn", 42, (3, 6000))),
    ("cfp_odd_n_log_layer", "Combined_Frequency_Periodicity", dict(fr=3, g=[0.3, 0], window_size=1500),
     ("randn", 43, (1, 7000))),
    ("cfp_fs22050_36_per_octave", "CFP",
     dict(fs=22050, fr=2, fc=55, tc=1 / 2000, NumPerOct=36, hop_length=256), ("randn", 44, (1, 5000))),
]
# constructor-only configurations (buffers + attributes)
CFP_DESIGN_CASES = [
    ("cfp_design_fr1", "CFP", dict(fr=1, fc=27.5, tc=1 / 4000, NumPerOct=60)),
    ("cfp_design_short_window", "Combined_Frequency_Periodicity", dict(window_size=513, hop_length=80, fc=110)),
]
# id, class, ctor, input shape: the exception type the reference raises
CFP_ERROR_CASES = [
    ("cfp_1d_input", "CFP", dict(), (4000,)),
    ("cfp_3d_input", "CFP", dict(), (1, 1, 4000)),
    ("cfp_single_layer", "CFP", dict(g=[0.5]), (1, 4000)),
    ("cfp_window_longer_than_n", "CFP", dict(fr=8, window_size=2049), (1, 4000)),
]
