"""Filterbank (mel) spectrogram restated in f64, on top of the f64 STFT (stft_reference.stft_f64): the oracle of
Spectrogram(mode="filterbank") / wfb_stft_create_filterbank.

    out[f][m] = L( sum_k F[m][k] |R_f[k]|^p ),   L(v) = v if scale == 0 else scale log2(max(v + offset, floor))

with F the f32 filter matrix the library was given (its values, in f64).

Bounds, per frame f and filter m, from the complex bound e_f of stft_reference (|X_f[k] - R_f[k]| <= e_f):
  * each bin's power lies in [max(|R| - e_f, 0)^p, (|R| + e_f)^p];
  * the filter sum of those intervals (weights of either sign) widened by the f32 arithmetic of the filter stage,
    (len_m + 2) 2^-24 sum_k |w_k| hi_k (len_m bins of the FMA chain, 2 for the power itself);
  * mapped through the monotone L, widened by MUFU.LG2's error (2^-21 absolute in log2, plus 2 ulp) and the f32
    rounding of v + offset and of the product with scale.
check_self is the tight form: the filter product of the same kernel's complex output, whose only error left is the
filter stage's own f32 arithmetic."""
import math

import numpy as np

from stft_reference import complex_bound, frames_f64, num_frames

U = 2.0 ** -24                        # f32 unit roundoff


def bands(filters):
    """The library's band of each filter: (first bin, bins) from the first to the last non-zero weight; (0, 0) if none."""
    out = []
    for row in np.asarray(filters, np.float32):
        nz = np.flatnonzero(row != 0)
        out.append((int(nz[0]), int(nz[-1] - nz[0] + 1)) if nz.size else (0, 0))
    return np.array(out, np.int64).reshape(-1, 2)


def apply_log(v, scale, offset, floor):
    v = np.asarray(v, np.float64)
    if scale == 0:
        return v
    return scale * np.log2(np.maximum(v + offset, floor))


def filterbank_f64(x, filters, fft_size, hop, window_type="hann", zero_padding=1, power=2, scale=0.0, offset=0.0,
                   floor=1e-10):
    """The filterbank spectrogram in f64, [..., frames, filters]."""
    z = np.fft.rfft(frames_f64(x, fft_size, hop, window_type, zero_padding), fft_size, axis=-1)
    p = np.abs(z) ** power
    return apply_log(p @ np.asarray(filters, np.float32).astype(np.float64).T, scale, offset, floor)


def _interval(lo_bin, hi_bin, w, lens, scale, offset, floor):
    """[lo, hi] of L(sum_k w_k P_k) for P_k in [lo_bin, hi_bin] (frames x bins), with the f32 slack above."""
    wp, wn = np.maximum(w, 0.0), np.minimum(w, 0.0)
    lo = lo_bin @ wp.T + hi_bin @ wn.T
    hi = hi_bin @ wp.T + lo_bin @ wn.T
    slack = (lens[None, :] + 2) * U * (hi_bin @ np.abs(w).T)
    lo, hi = lo - slack, hi + slack
    if scale == 0:
        return lo, hi
    # v + offset rounded in f32, then log2 (MUFU.LG2: 2^-21 absolute, 2 ulp), then one f32 multiply
    a_lo = np.maximum(np.maximum(lo + offset, 0.0) * (1 - 4 * U), floor)
    a_hi = np.maximum((hi + offset) * (1 + 4 * U), floor)
    l_lo, l_hi = np.log2(a_lo), np.log2(a_hi)
    d_lo = 2.0 ** -21 + 4 * U * np.abs(l_lo)
    d_hi = 2.0 ** -21 + 4 * U * np.abs(l_hi)
    a, b = scale * (l_lo - d_lo), scale * (l_hi + d_hi)                  # L is monotone for either sign of scale
    r_lo, r_hi = np.minimum(a, b), np.maximum(a, b)
    return r_lo - 2 * U * np.abs(r_lo), r_hi + 2 * U * np.abs(r_hi)


def _ratio(got, ref, lo, hi):
    err = np.abs(got - ref)
    allowed = np.where(got >= ref, hi - ref, ref - lo)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(err == 0, 0.0, err / allowed)


def _raise(ratio, got, ref, lo, hi, f0=0):
    bad = ratio > 1.0
    if bad.any():
        fi, m = np.argwhere(bad)[0]
        raise AssertionError(f"{int(bad.sum())} values outside the bound, first at frame {f0 + fi} filter {m}: got "
                             f"{got[fi, m]}, reference {(lo[fi, m], ref[fi, m], hi[fi, m])}; worst {ratio.max():.3g} x bound")


def check(got, x, filters, fft_size, hop, window_type="hann", zero_padding=1, power=2, scale=0.0, offset=0.0,
          floor=1e-10, chunk_values=1 << 22):
    """Assert `got` [frames, filters] against the f64 reference of the f32 signal x at every frame and filter, within
    the bounds above.  Returns the worst error as a fraction of its bound."""
    x = np.asarray(x, np.float32)
    got = np.asarray(got)
    w = np.asarray(filters, np.float32).astype(np.float64)
    lens = bands(filters)[:, 1].astype(np.float64)
    wsize = fft_size // zero_padding
    frames = num_frames(len(x), wsize, hop)
    assert got.shape == (frames, w.shape[0]), (got.shape, frames, w.shape)
    assert np.isfinite(got).all()
    step = max(1, chunk_values // (fft_size + w.size // 4 + 1))
    worst = 0.0
    for f0 in range(0, frames, step):
        f1 = min(frames, f0 + step)
        seg = frames_f64(x[f0 * hop: (f1 - 1) * hop + wsize], fft_size, hop, window_type, zero_padding)
        mag = np.abs(np.fft.rfft(seg, fft_size, axis=-1))
        e = complex_bound(fft_size) * np.linalg.norm(seg, axis=-1)[:, None]
        ref = apply_log(mag ** power @ w.T, scale, offset, floor)
        lo, hi = _interval(np.maximum(mag - e, 0.0) ** power, (mag + e) ** power, w, lens, scale, offset, floor)
        g = got[f0:f1].astype(np.float64)
        ratio = _ratio(g, ref, lo, hi)
        _raise(ratio, g, ref, lo, hi, f0)
        worst = max(worst, float(ratio.max()) if ratio.size else 0.0)
    return worst


def check_self(got, spectra, filters, power=2, scale=0.0, offset=0.0, floor=1e-10):
    """Assert `got` [frames, filters] against the f64 filter product of the complex output `spectra` [frames, bins, 2]
    of the same kernel on the same signal.  The kernel's per-bin power is fma(re, re, im im) in f32 (and its square
    root for p = 1): within 3 ulp of the f64 power of the same X, inside the (len_m + 2) slack."""
    s = np.asarray(spectra, np.float64)
    mag2 = s[..., 0] ** 2 + s[..., 1] ** 2
    p = mag2 if power == 2 else np.sqrt(mag2)
    w = np.asarray(filters, np.float32).astype(np.float64)
    lens = bands(filters)[:, 1].astype(np.float64)
    ref = apply_log(p @ w.T, scale, offset, floor)
    lo, hi = _interval(p * (1 - 3 * U), p * (1 + 3 * U), w, lens, scale, offset, floor)
    g = np.asarray(got, np.float64)
    ratio = _ratio(g, ref, lo, hi)
    _raise(ratio, g, ref, lo, hi)
    return float(ratio.max()) if ratio.size else 0.0


LOG_SCALES = {None: 0.0, "ln": math.log(2.0), "log10": math.log10(2.0), "db": 10.0 * math.log10(2.0)}


def log_scale(log, power):
    """The library's scale for Spectrogram(log=...): "db" is 10 log10 of a power and 20 log10 of a magnitude."""
    return LOG_SCALES[log] * (2.0 if log == "db" and power == 1 else 1.0)
