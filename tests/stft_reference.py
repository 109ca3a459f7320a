"""Forward STFT restated in f64: the independent oracle of the fused spectrogram kernels (k_stft, k_stft_span,
k_stft_pipe), next to the inverse one (istft_reference.py).

Vectorised over frames (sliding_window_view), so every frame and every bin of a long signal is checked, not a sample of
them.  It is pinned to the oracle's per-frame loop (oracle.spectrogram_reference) and to torch.stft(center=False) by
test_stft_f64.py on the CPU.

Bounds, per frame f and bin k, with e_f = 4 f32_bound(N) ||x_f w32||_2 (the factor 4: the oracle's Taylor-series
twiddles sit a few parity bounds from the true DFT, the yardstick test_gpu_fuzz.py uses as well):
    complex:  |got - R_f[k]| <= e_f
    dB:       v(max(|R| - e_f, 0)) - delta <= got <= v(|R| + e_f) + delta,   delta = DB_ABS + DB_DB / range
where v is the monotone magnitude -> [0, 1] map, so the interval is tight where |R| is large and widens only where f32
cannot resolve the bin.  DB_DB covers the MUFU.LG2 and f32 rounding of the dB step and DB_ABS the fast form's dropped
+1e-10 (at most 1e-6 of the output where the library takes it)."""
import math

import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

from oracle import window_function

DB_ABS = 2e-6          # normalised output units
DB_DB = 5e-5           # dB, divided by the range


def window32(window_type, wsize):
    """The window values the library stores: the f64 formula rounded to f32, returned in f64."""
    return window_function(window_type, wsize).astype(np.float32).astype(np.float64)


def num_frames(num_samples, wsize, hop):
    return (num_samples - wsize) // hop + 1


def frames_f64(x, fft_size, hop, window_type="hann", zero_padding=1):
    """Windowed frames x[fH + j] w32[j], j < window, f64 [..., frames, window] (x: [..., num_samples])."""
    wsize = fft_size // zero_padding
    x = np.asarray(x, np.float64)
    frames = num_frames(x.shape[-1], wsize, hop)
    if frames <= 0:
        raise ValueError("Audio too short for the given FFT size")
    seg = sliding_window_view(x, wsize, axis=-1)[..., : (frames - 1) * hop + 1: hop, :]
    return seg * window32(window_type, wsize)


def stft_f64(x, fft_size, hop, window_type="hann", zero_padding=1):
    """Complex STFT in f64 in the library's layout [..., frames, fft_size/2 + 1, 2]:
        R_f[k] = sum_{j < window} x[fH + j] w32[j] e^{-2 pi i jk / N},
    the frame zero-padded at its end to N = fft_size."""
    z = np.fft.rfft(frames_f64(x, fft_size, hop, window_type, zero_padding), fft_size, axis=-1)
    return np.stack([z.real, z.imag], axis=-1)


def db_value(mag, fft_size, gain=0.0, range_db=80.0):
    """magnitudeToDb + the gain/range normalisation (spectrogram.js:60-62, :343-352) of magnitudes |X|, in f64:
        v(m) = clip((20 log10(m / (N/2) + 1e-10) - (gain - range)) / range, 0, 1).
    Bins 0, 1 and 2 are zeroed separately (db_f64)."""
    db = 20.0 * np.log10(np.asarray(mag, np.float64) / (fft_size / 2) + 1e-10)
    return np.clip((db - (gain - range_db)) / range_db, 0.0, 1.0)


def db_f64(x, fft_size, hop, window_type="hann", zero_padding=1, gain=0.0, range_db=80.0):
    """The spectrogram in f64 [..., frames, fft_size/2 + 1]: db_value of |R|, bins 0, 1 and 2 exactly 0."""
    r = stft_f64(x, fft_size, hop, window_type, zero_padding)
    v = db_value(np.hypot(r[..., 0], r[..., 1]), fft_size, gain, range_db)
    v[..., :3] = 0.0
    return v


def complex_bound(n):
    """e_f / ||x_f w32||_2: 4 f32 parity bounds (2e-6 log2 N each)."""
    return 4 * 2e-6 * math.log2(n)


def check(got, x, fft_size, hop, window_type="hann", zero_padding=1, mode="db", gain=0.0, range_db=80.0,
          chunk_values=1 << 22):
    """Assert `got` ([frames, bins] in dB mode, [frames, bins, 2] complex) against the f64 reference of the f32 signal
    x at every frame and bin, within the bounds above.  Works through the frames in chunks so that long signals stay
    in bounded memory.  In dB mode also: values in [0, 1], no NaN, bins 0, 1 and 2 exactly 0.  Returns the worst error
    as a fraction of its bound (0 where every value is exact)."""
    x = np.asarray(x, np.float32)
    got = np.asarray(got)
    wsize = fft_size // zero_padding
    frames = num_frames(len(x), wsize, hop)
    bins = fft_size // 2 + 1
    assert got.shape == ((frames, bins) if mode == "db" else (frames, bins, 2)), (got.shape, frames, bins)
    assert not np.isnan(got).any()
    if mode == "db":
        assert got.min() >= 0.0 and got.max() <= 1.0, (got.min(), got.max())
        assert np.all(got[:, :3] == 0.0)
    step = max(1, chunk_values // (fft_size + bins * 2))
    worst = 0.0
    delta = DB_ABS + DB_DB / range_db
    for f0 in range(0, frames, step):
        f1 = min(frames, f0 + step)
        seg = frames_f64(x[f0 * hop: (f1 - 1) * hop + wsize], fft_size, hop, window_type, zero_padding)
        z = np.fft.rfft(seg, fft_size, axis=-1)
        e = complex_bound(fft_size) * np.linalg.norm(seg, axis=-1)[:, None]          # e_f per frame, [frames, 1]
        g = got[f0:f1].astype(np.float64)
        if mode == "db":
            m = np.abs(z)
            v = db_value(m, fft_size, gain, range_db)
            lo = db_value(np.maximum(m - e, 0.0), fft_size, gain, range_db) - delta
            hi = db_value(m + e, fft_size, gain, range_db) + delta
            v[:, :3] = lo[:, :3] = hi[:, :3] = 0.0
            # the error as a fraction of what the bound allows on its side of the reference value
            err = np.abs(g - v)
            allowed = np.where(g >= v, hi - v, v - lo)
        else:
            err = np.hypot(g[..., 0] - z.real, g[..., 1] - z.imag)
            allowed = np.broadcast_to(e, err.shape)
        with np.errstate(divide="ignore", invalid="ignore"):
            ratio = np.where(err == 0, 0.0, err / allowed)
        bad = ratio > 1.0
        if bad.any():
            fi, k = np.argwhere(bad)[0]
            ref = (lo[fi, k], v[fi, k], hi[fi, k]) if mode == "db" else (z[fi, k], e[fi, 0])
            raise AssertionError(f"{int(bad.sum())} values outside the bound, first at frame {f0 + fi} bin {k}: "
                                 f"got {got[f0 + fi, k]}, reference {ref}; worst {ratio.max():.3g} x bound")
        worst = max(worst, float(ratio.max()) if ratio.size else 0.0)
    return worst
