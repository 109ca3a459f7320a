"""watfft_b200 -- B200-native batched FFT engine behind wat-fft's context surface.

Python host mirror of the reference's JavaScript plugin API (index.js:69-178): the same factory
names, buffer accessors and forward()/inverse() semantics, each context gaining a `batch` count.
The JavaScript host proper lives in js/ (Node + N-API addon in napi/); this mirror exists because
the build image has no JS runtime, and binds the very same C ABI (include/watfft_b200.h).
"""
from . import _cabi
from ._cabi import WatFFTError, build
from .stft import Spectrogram, generateSpectrogram, inverseSpectrogram, mel_filterbank, melSpectrogram
from .contexts import (
    createFFT, createFFTf32, createRFFT, createRFFTf32,
    createFFTf32Split, createRFFTf32Split, SplitExportsFacade, ModuleExports, HostMemory, Plan,
    createFFTInstance, createFFTf32Instance, createRFFTInstance, createRFFTf32Instance, createFFTf32SplitInstance,
)

__all__ = [
    "createFFT", "createFFTf32", "createRFFT", "createRFFTf32",
    "createFFTf32Split", "createRFFTf32Split", "SplitExportsFacade", "ModuleExports", "HostMemory", "Plan",
    "createFFTInstance", "createFFTf32Instance", "createRFFTInstance", "createRFFTf32Instance", "createFFTf32SplitInstance",
    "Spectrogram", "generateSpectrogram", "inverseSpectrogram", "mel_filterbank", "melSpectrogram", "WatFFTError", "build", "_cabi",
]
