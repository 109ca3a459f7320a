"""Batched spectrogram / STFT: the reference's batched caller, as one GPU launch.

Mirror of `generateSpectrogram({samples, sampleRate, fftContext, hopSize, windowType, zeroPadding,
gain, range})` in playground/src/spectrogram.js:270-372: same arguments (the FFT context is
replaced by `fftSize`), same returned fields, same numerics to f32 tolerance -- but the per-frame
JavaScript loop (slice, window, zero-pad, copy, run, magnitude, dB) is a single kernel over all
frames (csrc/wfb_kernels.cuh k_stft).

The inverse (Spectrogram.inverse, inverseSpectrogram) is an extension with no reference counterpart: the weighted
overlap-add of the frames' c2r outputs, fused into one kernel as well (k_istft).

Both directions also take a batch of equal-length signals ([B][num_samples], one launch for all of them); every
signal's result is exactly what the single-signal call gives for it.

Filterbank (mel) spectrograms (Spectrogram(mode="filterbank"), melSpectrogram, another extension) fuse |X|^p, a
filter matrix and an optional log into the same kernels: n_filters floats per frame leave the GPU, not the spectrum."""
from __future__ import annotations

import ctypes
import math

import numpy as np

from . import _cabi as C
from .contexts import _view


# L(v) = scale * log2(max(v + logOffset, logFloor)) for Spectrogram(mode="filterbank", log=...); "db" doubles for power 1
LOG_SCALES = {None: 0.0, "ln": math.log(2.0), "log10": math.log10(2.0), "db": 10.0 * math.log10(2.0)}


def _hz_to_mel(f, scale):
    f = np.asarray(f, np.float64)
    if scale == "htk":
        return 2595.0 * np.log10(1.0 + f / 700.0)
    # slaney: linear below 1 kHz (200/3 Hz per mel), logarithmic above
    lin = f / (200.0 / 3.0)
    return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1e-300) / 1000.0) / (math.log(6.4) / 27.0), lin)


def _mel_to_hz(m, scale):
    m = np.asarray(m, np.float64)
    if scale == "htk":
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
    return np.where(m >= 15.0, 1000.0 * np.exp((math.log(6.4) / 27.0) * (m - 15.0)), m * (200.0 / 3.0))


def mel_filterbank(fftSize, sampleRate, nMels, fMin=0.0, fMax=None, scale="htk", norm=None):
    """Triangular mel filters as float32 [nMels][fftSize/2+1], built in f64: nMels + 2 points equally spaced in mel
    from fMin to fMax (default sampleRate/2), filter m rising from point m to m+1 and falling to m+2 over the bin
    frequencies k sampleRate / fftSize.  scale "htk" or "slaney" (linear below 1 kHz); norm None or "slaney" (each filter
    scaled by 2 / its width in Hz).  torchaudio.functional.melscale_fbanks(...).T computes the same (it spaces the
    bins over [0, sampleRate // 2], the same frequencies for an even sampleRate)."""
    if scale not in ("htk", "slaney"):
        raise ValueError(f'scale must be "htk" or "slaney", got {scale!r}')
    if norm not in (None, "slaney"):
        raise ValueError(f'norm must be None or "slaney", got {norm!r}')
    fMax = sampleRate / 2.0 if fMax is None else float(fMax)
    freqs = np.arange(fftSize // 2 + 1, dtype=np.float64) * (sampleRate / fftSize)
    f_pts = _mel_to_hz(np.linspace(_hz_to_mel(fMin, scale), _hz_to_mel(fMax, scale), nMels + 2), scale)
    diff = np.diff(f_pts)
    slopes = f_pts[None, :] - freqs[:, None]
    down = -slopes[:, :-2] / diff[:-1]
    up = slopes[:, 2:] / diff[1:]
    fb = np.maximum(0.0, np.minimum(down, up))
    if norm == "slaney":
        fb *= 2.0 / (f_pts[2:] - f_pts[:-2])
    return np.ascontiguousarray(fb.T, np.float32)


class Spectrogram:
    """Reusable plan: fixed signal length / FFT size / hop / window.

    batch=None: one signal, buffers (num_samples,) -> (numFrames, numBins[, 2]).  batch=B: B signals of num_samples
    each, buffers (B, num_samples) -> (B, numFrames, numBins[, 2]); numFrames stays the count of one signal.

    mode="filterbank": out[f][m] = L(sum_k filters[m][k] |X_f[k]|^power), X_f the raw spectrum mode="complex" gives,
    filters a [nFilters][fftSize/2+1] matrix (mel_filterbank builds mel ones); buffers (numFrames, nFilters) or
    (B, numFrames, nFilters).  log: None (L(v) = v), "ln", "log10" or "db" (10 log10 of a power, 20 log10 of a
    magnitude: torchaudio's AmplitudeToDB with top_db=None), each of max(v + logOffset, logFloor).  gain and range are
    unused; there is no inverse."""

    def __init__(self, num_samples, fftSize, hopSize, windowType="hann", zeroPadding=1, gain=0.0, range=80.0,
                 mode="db", device=0, flags=0, *, batch=None, filters=None, power=2, log=None, logOffset=0.0,
                 logFloor=1e-10):
        if batch is not None and (isinstance(batch, bool) or int(batch) != batch or batch < 1):
            raise ValueError(f"batch must be None or an integer >= 1, got {batch!r}")
        self._lib = C.lib()
        if windowType not in C.WINDOWS:
            windowType = "hann"              # the JS falls back to hann for unknown names (:31)
        err = ctypes.c_int(0)
        nb = 1 if batch is None else int(batch)
        self.numFilters = 0
        if mode == "filterbank":
            if filters is None:
                raise ValueError('mode="filterbank" needs filters, a [nFilters][fftSize/2+1] matrix')
            f = np.ascontiguousarray(filters, np.float32)
            if f.ndim != 2 or f.shape[1] != int(fftSize) // 2 + 1:
                raise ValueError(f"filters must be [nFilters][{int(fftSize) // 2 + 1}], got shape {f.shape}")
            if log not in LOG_SCALES:
                raise ValueError(f"log must be one of {list(LOG_SCALES)}, got {log!r}")
            scale = LOG_SCALES[log] * (2.0 if log == "db" and power == 1 else 1.0)
            self._mode = C.STFT_FILTERBANK
            self._p = self._lib.wfb_stft_create_filterbank(
                int(fftSize), int(zeroPadding), int(hopSize), C.WINDOWS[windowType], int(num_samples), nb, f.shape[0],
                f.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), int(power), float(scale), float(logOffset),
                float(logFloor), int(device), int(flags), ctypes.byref(err))
        else:
            self._mode = C.STFT_COMPLEX if mode == "complex" else C.STFT_DB
            self._p = self._lib.wfb_stft_create_ex(int(fftSize), int(zeroPadding), int(hopSize), C.WINDOWS[windowType],
                                                   int(num_samples), nb, self._mode, float(gain), float(range),
                                                   int(device), int(flags), ctypes.byref(err))
        if not self._p:
            raise C.WatFFTError(err.value)
        self.numFilters = self._lib.wfb_stft_filters(self._p)
        self.fftSize, self.hopSize, self.windowSize = fftSize, hopSize, fftSize // zeroPadding
        self.numFrames = self._lib.wfb_stft_frames(self._p)
        self.numBins = self._lib.wfb_stft_bins(self._p)
        self.num_samples = num_samples
        self.batch = None if batch is None else int(batch)
        self._lead = () if batch is None else (self.batch,)

    def getInputBuffer(self):
        b = self._lib.wfb_stft_batch(self._p)
        return _view(self._lib.wfb_stft_host_samples(self._p), 4 * b * self.num_samples, np.float32).reshape(
            self._lead + (self.num_samples,))

    def getOutputBuffer(self):
        out = _view(self._lib.wfb_stft_host_output(self._p), self._lib.wfb_stft_output_bytes(self._p), np.float32)
        shape = {C.STFT_COMPLEX: (self.numFrames, self.numBins, 2), C.STFT_FILTERBANK: (self.numFrames, self.numFilters)}.get(
            self._mode, (self.numFrames, self.numBins))
        return out.reshape(self._lead + shape)

    def run(self):
        C.check(self._lib.wfb_stft_exec(self._p, C.EXEC_DEFAULT))

    def run_device(self, d_samples, d_out, stream=None):
        C.check(self._lib.wfb_stft_exec_device(self._p, ctypes.c_void_p(d_samples), ctypes.c_void_p(d_out),
                                               ctypes.c_void_p(stream) if stream else None))

    def inverse(self):
        """Signal from the complex spectra in getOutputBuffer() (weighted overlap-add, see inverseSpectrogram), written
        to getInputBuffer().  mode="complex" only (WatFFTError otherwise)."""
        C.check(self._lib.wfb_stft_exec_inverse(self._p, C.EXEC_DEFAULT))

    def inverse_device(self, d_spectra, d_samples, stream=None):
        C.check(self._lib.wfb_stft_exec_inverse_device(self._p, ctypes.c_void_p(d_spectra), ctypes.c_void_p(d_samples),
                                                       ctypes.c_void_p(stream) if stream else None))

    def algorithmic_bytes(self):
        return self._lib.wfb_stft_algorithmic_bytes(self._p)

    def dispose(self):
        if getattr(self, "_p", None):
            self._lib.wfb_stft_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.dispose()
        except Exception:
            pass


def generateSpectrogram(samples, sampleRate, fftSize, hopSize, windowType="hann", zeroPadding=1, gain=0.0, range=80.0,
                        device=0):
    """Same result object as the reference's generateSpectrogram (spectrogram.js:362-372).  2-D samples [B][T] are B
    signals in one launch: `data` is then [B][numFrames*numBins], row b equal to the 1-D call on samples[b], and the
    result also has "batch": B."""
    samples = np.ascontiguousarray(samples, np.float32)
    if samples.ndim not in (1, 2) or (samples.ndim == 2 and samples.shape[0] < 1):
        raise ValueError(f"samples must be [T] or [B][T] with B >= 1, got shape {samples.shape}")
    window = fftSize // zeroPadding
    n = samples.shape[-1]
    if (n - window) // hopSize + 1 <= 0 or n < window:
        raise ValueError("Audio too short for the given FFT size")          # spectrogram.js:299-301
    batch = samples.shape[0] if samples.ndim == 2 else None
    sp = Spectrogram(n, fftSize, hopSize, windowType, zeroPadding, gain, range, device=device, batch=batch)
    sp.getInputBuffer()[:] = samples
    sp.run()
    data = sp.getOutputBuffer().copy().reshape(samples.shape[:-1] + (-1,))
    out = {"data": data, "numFrames": sp.numFrames, "numBins": sp.numBins, "fftSize": fftSize,
           "windowSize": window, "hopSize": hopSize, "sampleRate": sampleRate}
    if batch is not None:
        out["batch"] = batch
    sp.dispose()
    return out


def inverseSpectrogram(spectra, fftSize, hopSize, windowType="hann", zeroPadding=1, device=0):
    """Signal from complex STFT frames ([frames][fftSize/2+1][2] float32, the layout of Spectrogram(mode="complex")):
    the least-squares / weighted overlap-add estimate that torch.istft(..., center=False) also computes,
        x[t] = sum_f w[t-f*hop] y_f[t-f*hop] / sum_f w[t-f*hop]^2   (0 where that sum is below 1e-11),
    y_f the 1/N-normalised c2r of frame f (real parts of DC and Nyquist).  Returns (frames-1)*hop + window float32
    samples; spectra left unmodified give back the analysed signal wherever a frame carries weight.
    A batch [B][frames][bins][2] gives [B][length], each row from that signal's frames alone, in one launch."""
    spectra = np.ascontiguousarray(spectra, np.float32)
    if (spectra.ndim not in (3, 4) or spectra.shape[-2] != fftSize // 2 + 1 or spectra.shape[-1] != 2 or
            min(spectra.shape[:-2]) < 1):
        raise ValueError(f"spectra must be [frames][{fftSize // 2 + 1}][2] or [B][frames][{fftSize // 2 + 1}][2], "
                         f"got {spectra.shape}")
    window = fftSize // zeroPadding
    frames = spectra.shape[-3]
    length = (frames - 1) * hopSize + window
    batch = spectra.shape[0] if spectra.ndim == 4 else None
    sp = Spectrogram(length, fftSize, hopSize, windowType, zeroPadding, mode="complex", device=device, batch=batch)
    try:
        assert sp.numFrames == frames
        sp.getOutputBuffer()[:] = spectra
        sp.inverse()
        return sp.getInputBuffer().copy()
    finally:
        sp.dispose()


def melSpectrogram(samples, sampleRate, fftSize, hopSize, nMels=128, windowType="hann", zeroPadding=1, fMin=0.0,
                   fMax=None, scale="htk", norm=None, power=2, log=None, logOffset=0.0, logFloor=1e-10, device=0):
    """Mel spectrogram in one launch, shaped like generateSpectrogram: `data` is [numFrames*nMels] (frame-major), or
    [B][numFrames*nMels] for samples [B][T] (then "batch": B).  The filters are mel_filterbank(fftSize, sampleRate,
    nMels, fMin, fMax, scale, norm); power and log as Spectrogram(mode="filterbank").  With the defaults this is
    torchaudio.transforms.MelSpectrogram(center=False) with the library's window."""
    samples = np.ascontiguousarray(samples, np.float32)
    if samples.ndim not in (1, 2) or (samples.ndim == 2 and samples.shape[0] < 1):
        raise ValueError(f"samples must be [T] or [B][T] with B >= 1, got shape {samples.shape}")
    window = fftSize // zeroPadding
    n = samples.shape[-1]
    if n < window:
        raise ValueError("Audio too short for the given FFT size")
    batch = samples.shape[0] if samples.ndim == 2 else None
    filters = mel_filterbank(fftSize, sampleRate, nMels, fMin, fMax, scale, norm)
    sp = Spectrogram(n, fftSize, hopSize, windowType, zeroPadding, mode="filterbank", filters=filters, power=power,
                     log=log, logOffset=logOffset, logFloor=logFloor, device=device, batch=batch)
    try:
        sp.getInputBuffer()[:] = samples
        sp.run()
        data = sp.getOutputBuffer().copy().reshape(samples.shape[:-1] + (-1,))
    finally:
        sp.dispose()
    out = {"data": data, "numFrames": sp.numFrames, "nMels": nMels, "fftSize": fftSize, "windowSize": window,
           "hopSize": hopSize, "sampleRate": sampleRate}
    if batch is not None:
        out["batch"] = batch
    return out
