"""Inverse STFT restated in f64: the independent oracle of the fused inverse kernel (k_istft).

An extension with no reference counterpart, so it sits next to the tests rather than in oracle/ (whose restatements
are pinned to the reference); torch.istft(center=False) is its independent check (tests/test_istft.py)."""
import numpy as np

from oracle import window_function


def istft_reference(spectra, fft_size, hop, window_type="hann", zero_padding=1, irfft=None, num_samples=None):
    """Inverse of the complex spectrogram (an extension: the reference has no inverse), restated in f64 with the f32
    window values the forward applies.  Weighted overlap-add, the least-squares estimate:
        y_f = irfft(X_f) (1/N, real parts of DC and Nyquist), first `window` samples;
        x[t] = sum_f w[t-fH] y_f[t-fH] / D[t],  D[t] = sum_f w[t-fH]^2,  0 where D[t] < 1e-11.
    Returns (frames-1)*hop + window samples, or `num_samples` (>= that) with the rest 0.  `irfft` maps n+2 interleaved
    floats to n reals (default: numpy in f64).

    PARITY UNPINNED: nothing in the reference computes this; torch.istft(center=False) is the independent check."""
    spectra = np.asarray(spectra)
    frames = spectra.shape[0]
    wsize = fft_size // zero_padding
    w = window_function(window_type, wsize).astype(np.float32).astype(np.float64)
    length = (frames - 1) * hop + wsize
    out_len = length if num_samples is None else num_samples
    if out_len < length:
        raise ValueError("num_samples shorter than the frames reach")
    y = frames_c2r(spectra, fft_size, irfft)
    num = overlap_add(w * y[:, :wsize], hop)
    den = overlap_add(np.broadcast_to(w * w, (frames, wsize)), hop)
    x = np.zeros(out_len)
    ok = den >= 1e-11
    x[:length][ok] = num[ok] / den[ok]
    return x


def frames_c2r(spectra, fft_size, irfft=None):
    """y_f of every frame, f64 [frames][fft_size]: the 1/N inverse real transform using only the real parts of DC and
    Nyquist (numpy, or `irfft` per frame)."""
    spectra = np.asarray(spectra)
    if irfft is not None:
        return np.stack([np.asarray(irfft(np.asarray(s, np.float32).ravel()), np.float64) for s in spectra])
    z = spectra[..., 0].astype(np.float64) + 1j * spectra[..., 1].astype(np.float64)
    z[:, 0] = z[:, 0].real
    z[:, -1] = z[:, -1].real
    return np.fft.irfft(z, fft_size, axis=1)


def overlap_add(rows, hop):
    """sum_f rows[f] placed at sample f*hop, f64, (frames-1)*hop + width samples.  Every sample is summed from 0 in
    increasing frame order, so the result is bit for bit the per-frame loop `out[f*hop: f*hop + width] += rows[f]`."""
    rows = np.asarray(rows, np.float64)
    frames, width = rows.shape
    idx = (np.arange(frames)[:, None] * hop + np.arange(width)).ravel()
    return np.bincount(idx, weights=rows.ravel(), minlength=(frames - 1) * hop + width)
