"""ctypes binding of include/watfft_b200.h (the same C ABI the N-API addon binds).

There is no fallback of any kind: if libwatfft_b200.so is missing the import of the
transform entry points raises, and every plan creation fails with WFB_ERR_NO_DEVICE when no
sm_100 device is present."""
from __future__ import annotations

import ctypes
import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
# WFB_LIB: A/B builds of the same library for tools/sweep.py (never a different implementation)
LIB_PATH = Path(os.environ["WFB_LIB"]) if os.environ.get("WFB_LIB") else HERE / "libwatfft_b200.so"

# enums of include/watfft_b200.h
C2C, R2C = 0, 1
F32, F64 = 0, 1
SPLIT, INTERLEAVED = 0, 1
FORWARD, INVERSE = 0, 1
STAGE_H2D, STAGE_D2H, SYNC, EXEC_DEFAULT = 1, 2, 4, 7
BUF_TIME, BUF_SPECTRUM = 0, 1
PLAN_NO_HOST_BUFFERS, PLAN_NO_DEVICE_BUFFERS = 1, 2
OPT_MAPPED_MAX_BYTES, OPT_STAGE_CHUNK_BYTES, OPT_STAGE_STREAMS, OPT_STAGE_RAMP = 0, 1, 2, 3
PATH_NONE, PATH_STAGED, PATH_PIPELINED, PATH_MAPPED = 0, 1, 2, 3
OK, ERR_NO_DEVICE, ERR_BAD_SIZE, ERR_BAD_ARG, ERR_UNSUPPORTED, ERR_ALLOC, ERR_CUDA, ERR_NO_HOST_BUFFERS = (
    0, -1, -2, -3, -4, -5, -6, -7)

# every symbol include/watfft_b200.h declares (tests/test_cabi.py checks the header against this list)
SYMBOLS = {
    "wfb_device_count": (ctypes.c_int, []),
    "wfb_require_b200": (ctypes.c_int, [ctypes.c_int]),
    "wfb_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "wfb_last_cuda_error": (ctypes.c_char_p, []),
    "wfb_size_range": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_int)] * 2),
    "wfb_plan_create": (ctypes.c_void_p, [ctypes.c_int] * 4 + [ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "wfb_plan_create_ex": (ctypes.c_void_p, [ctypes.c_int] * 4 + [ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                                                 ctypes.POINTER(ctypes.c_int)]),
    "wfb_plan_destroy": (None, [ctypes.c_void_p]),
    "wfb_host_in": (ctypes.c_void_p, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_host_out": (ctypes.c_void_p, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_host_buffer": (ctypes.c_void_p, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_host_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_device_buffer": (ctypes.c_void_p, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_exec": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "wfb_exec_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                       ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p]),
    "wfb_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "wfb_host_alloc": (ctypes.c_void_p, [ctypes.c_size_t]),
    "wfb_host_free": (None, [ctypes.c_void_p]),
    "wfb_exec_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                     ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]),
    "wfb_plan_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "wfb_plan_variant_count": (ctypes.c_int, [ctypes.c_void_p]),
    "wfb_plan_set_variant": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_plan_variant_name": (ctypes.c_char_p, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_plan_current_variant": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_plan_algorithmic_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "wfb_plan_set_option": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_long]),
    "wfb_plan_get_option": (ctypes.c_long, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_plan_last_path": (ctypes.c_int, [ctypes.c_void_p]),
    "wfb_stage_schedule": (ctypes.c_int, [ctypes.c_long, ctypes.c_size_t, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_long), ctypes.c_int]),
    "wfb_pcie_probe": (ctypes.c_int, [ctypes.c_int, ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]),
    "wfb_pcie_probe_open": (ctypes.c_int, [ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]),
    "wfb_pcie_probe_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]),
    "wfb_pcie_probe_close": (None, [ctypes.c_void_p]),
    "wfb_kernel_launch_count": (ctypes.c_ulonglong, []),
    "wfb_reference_twiddles": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.c_void_p] * 2),
    "wfb_stft_create": (ctypes.c_void_p, [ctypes.c_int] * 4 + [ctypes.c_long, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                           ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "wfb_stft_create_ex": (ctypes.c_void_p, [ctypes.c_int] * 4 + [ctypes.c_long, ctypes.c_long, ctypes.c_int, ctypes.c_float,
                                              ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "wfb_stft_create_filterbank": (ctypes.c_void_p, [ctypes.c_int] * 4 + [ctypes.c_long, ctypes.c_long, ctypes.c_int,
                                                      ctypes.POINTER(ctypes.c_float), ctypes.c_int] + [ctypes.c_float] * 3
                                   + [ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "wfb_stft_destroy": (None, [ctypes.c_void_p]),
    "wfb_stft_frames": (ctypes.c_long, [ctypes.c_void_p]),
    "wfb_stft_batch": (ctypes.c_long, [ctypes.c_void_p]),
    "wfb_stft_bins": (ctypes.c_int, [ctypes.c_void_p]),
    "wfb_stft_filters": (ctypes.c_int, [ctypes.c_void_p]),
    "wfb_stft_host_samples": (ctypes.c_void_p, [ctypes.c_void_p]),
    "wfb_stft_host_output": (ctypes.c_void_p, [ctypes.c_void_p]),
    "wfb_stft_output_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "wfb_stft_exec": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_stft_exec_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "wfb_stft_algorithmic_bytes": (ctypes.c_size_t, [ctypes.c_void_p]),
    "wfb_stft_exec_inverse": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "wfb_stft_exec_inverse_device": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
}
WINDOWS = {"hann": 0, "hamming": 1, "blackman": 2, "blackmanHarris": 3, "rectangular": 4}
STFT_DB, STFT_COMPLEX = 0, 1
STFT_FILTERBANK = 2      # the mode of a wfb_stft_create_filterbank handle (wfb_stft_create_ex rejects it)

_lib = None


class WatFFTError(RuntimeError):
    def __init__(self, code, detail=""):
        self.code = code
        msg = lib().wfb_strerror(code).decode()
        if code == ERR_CUDA or detail:
            msg += f" [{detail or lib().wfb_last_cuda_error().decode()}]"
        super().__init__(f"watfft_b200: {msg} (code {code})")


def build(verbose: bool = False) -> Path:
    """nvcc -gencode arch=compute_100a,code=sm_100a -> wat-fft_b200/libwatfft_b200.so (in-tree)."""
    subprocess.check_call(["make", "-C", str(HERE), "all"],
                          stdout=None if verbose else subprocess.DEVNULL)
    return LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                              "the B200 engine has no CPU fallback")
        L = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def check(code: int):
    if code != OK:
        raise WatFFTError(code)
