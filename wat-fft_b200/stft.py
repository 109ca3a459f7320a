"""Batched spectrogram / STFT: the reference's batched caller, as one GPU launch.

Mirror of `generateSpectrogram({samples, sampleRate, fftContext, hopSize, windowType, zeroPadding,
gain, range})` in playground/src/spectrogram.js:270-372: same arguments (the FFT context is
replaced by `fftSize`), same returned fields, same numerics to f32 tolerance -- but the per-frame
JavaScript loop (slice, window, zero-pad, copy, run, magnitude, dB) is a single kernel over all
frames (csrc/wfb_kernels.cuh k_stft).

The inverse (Spectrogram.inverse, inverseSpectrogram) is an extension with no reference counterpart: the weighted
overlap-add of the frames' c2r outputs, fused into one kernel as well (k_istft).

Both directions also take a batch of equal-length signals ([B][num_samples], one launch for all of them); every
signal's result is exactly what the single-signal call gives for it."""
from __future__ import annotations

import ctypes

import numpy as np

from . import _cabi as C
from .contexts import _view


class Spectrogram:
    """Reusable plan: fixed signal length / FFT size / hop / window.

    batch=None: one signal, buffers (num_samples,) -> (numFrames, numBins[, 2]).  batch=B: B signals of num_samples
    each, buffers (B, num_samples) -> (B, numFrames, numBins[, 2]); numFrames stays the count of one signal."""

    def __init__(self, num_samples, fftSize, hopSize, windowType="hann", zeroPadding=1, gain=0.0, range=80.0,
                 mode="db", device=0, flags=0, *, batch=None):
        if batch is not None and (isinstance(batch, bool) or int(batch) != batch or batch < 1):
            raise ValueError(f"batch must be None or an integer >= 1, got {batch!r}")
        self._lib = C.lib()
        if windowType not in C.WINDOWS:
            windowType = "hann"              # the JS falls back to hann for unknown names (:31)
        err = ctypes.c_int(0)
        self._mode = C.STFT_COMPLEX if mode == "complex" else C.STFT_DB
        self._p = self._lib.wfb_stft_create_ex(int(fftSize), int(zeroPadding), int(hopSize), C.WINDOWS[windowType],
                                               int(num_samples), 1 if batch is None else int(batch), self._mode,
                                               float(gain), float(range), int(device), int(flags), ctypes.byref(err))
        if not self._p:
            raise C.WatFFTError(err.value)
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
        shape = (self.numFrames, self.numBins, 2) if self._mode == C.STFT_COMPLEX else (self.numFrames, self.numBins)
        return out.reshape(self._lead + shape)

    def run(self):
        C.check(self._lib.wfb_stft_exec(self._p, C.EXEC_DEFAULT))

    def run_device(self, d_samples, d_out, stream=None):
        C.check(self._lib.wfb_stft_exec_device(self._p, ctypes.c_void_p(d_samples), ctypes.c_void_p(d_out),
                                               ctypes.c_void_p(stream) if stream else None))

    def inverse(self):
        """Signal from the complex spectra in getOutputBuffer() (weighted overlap-add, see inverseSpectrogram), written
        to getInputBuffer().  mode="complex" only."""
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
