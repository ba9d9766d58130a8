"""Shared helpers for the tests (input generators, tolerances)."""
import hashlib

import numpy as np

# north-star tolerance for float32 spectra: |X - Xref| <= ATOL*max|Xref| + RTOL*|Xref|
RTOL = 5e-5
ATOL = 5e-5
# north-star tolerance for ISTFT(STFT(x)) on the interior [nfft, n-nfft): relative L2
ROUNDTRIP_REL_L2 = 1e-5


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def noise(seed, n):
    """uniform(-1,1) float32 -- same generator as tests/golden/make_golden.py"""
    return np.random.default_rng(seed).uniform(-1.0, 1.0, n).astype(np.float32)


def spectra_close(x, ref, rtol=RTOL, atol=ATOL):
    """Returns (ok, worst budget fraction). Budget per bin = atol*max|ref| + rtol*|ref| (per frame row)."""
    x = np.asarray(x)
    ref = np.asarray(ref)
    assert x.shape == ref.shape, (x.shape, ref.shape)
    if ref.size == 0:
        return True, 0.0
    mx = np.abs(ref).max(axis=-1, keepdims=True)
    budget = atol * mx + rtol * np.abs(ref)
    err = np.abs(x.astype(np.complex128) - ref.astype(np.complex128)) if np.iscomplexobj(ref) else np.abs(
        x.astype(np.float64) - ref.astype(np.float64))
    zero = budget == 0
    frac = np.where(zero, np.where(err == 0, 0.0, np.inf), err / np.where(zero, 1, budget))
    return bool((frac <= 1.0).all()), float(frac.max())


def rel_l2(y, x):
    y = np.asarray(y, np.float64)
    x = np.asarray(x, np.float64)
    d = np.linalg.norm(x)
    return float(np.linalg.norm(y - x) / d) if d > 0 else float(np.linalg.norm(y - x))


def reflect_index(idx, n):
    """edge-inclusive reflection of any index into [0, n): ... 1 0 | 0 1 .. n-1 | n-1 n-2 ... (integer arithmetic)"""
    m = np.mod(idx, 2 * n)
    return np.where(m < n, m, 2 * n - 1 - m)


def stft_truth_f64(x, w, nfft, hop, frames=None, convention="valid"):
    """float64 STFT truth of x ([..., n]) in any of the four frame conventions: frame f starts at f*hop, or at
    f*hop - nfft/2 with edge-inclusive reflection for "center"; samples past either end are zero otherwise.
    frames defaults to the convention's frame count."""
    from oracle.oracle import num_frames
    x = np.asarray(x, np.float64)
    w = np.asarray(w, np.float64)
    n = x.shape[-1]
    if frames is None:
        frames = num_frames(n, nfft, hop, convention)
    if n == 0:
        return np.zeros(x.shape[:-1] + (frames, nfft // 2 + 1), np.complex128)
    idx = np.arange(nfft)[None, :] + hop * np.arange(frames)[:, None]
    if convention == "center":
        fr = x[..., reflect_index(idx - nfft // 2, n)]
    else:
        inside = idx < n
        fr = np.where(inside, x[..., np.where(inside, idx, 0)], 0.0)
    return np.fft.rfft(fr * w, axis=-1)


def istft_truth_f64(spec, w, nfft, hop, n_out):
    """float64 overlap-add of irfft(spec) * w ([..., frames, bins] -> [..., n_out]) and the float64 window-sum
    sum_f w(t - f*hop)^2 ([n_out]); frame f starts at sample f*hop, samples past n_out are dropped."""
    spec = np.asarray(spec)
    w = np.asarray(w, np.float64)
    frames = spec.shape[-2]
    span = max(n_out, (frames - 1) * hop + nfft if frames else 0)
    acc = np.zeros(spec.shape[:-2] + (span,))
    wsum = np.zeros(span)
    for f in range(frames):
        acc[..., f * hop:f * hop + nfft] += np.fft.irfft(spec[..., f, :].astype(np.complex128), nfft, axis=-1) * w
        wsum[f * hop:f * hop + nfft] += w * w
    return acc[..., :n_out], wsum[:n_out]
