"""ctypes front-ends for the two CPU checkers (TEST INFRASTRUCTURE).

* ``Oracle``  -- oracle/libwatfft_oracle.so, the committed C restatement
  (watfft_oracle.c).  Always buildable (gcc only).
* ``WatRef``  -- oracle/_ref/libwatref.so, the reference's own WAT modules
  transpiled to C (wat2c.py).  Built in the authoring container where
  /root/reference exists; the prebuilt .so travels to the GPU box.

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs import
this module.  The product (wat-fft_b200/) never does.

Also holds the numpy restatements of the reference's test fixtures:
the double-rounding LCG of tests/dft-reference.js:187-190, mulberry32 of
benchmarks/lib/harness.js:99-108 and the O(N^2) f64 DFT of
tests/dft-reference.js:14-88.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "libwatfft_oracle.so"
WATREF_SO = HERE / "_ref" / "libwatref.so"

_c_f32p = ctypes.POINTER(ctypes.c_float)
_c_f64p = ctypes.POINTER(ctypes.c_double)


def reference_modules() -> Path | None:
    """``modules/`` of the wat-fft checkout named by $WATFFT_REFERENCE, or None when it is not set."""
    ref = os.environ.get("WATFFT_REFERENCE")
    return Path(ref) / "modules" if ref else None


def build(force: bool = False) -> None:
    """Compile the restatement and, when $WATFFT_REFERENCE names a wat-fft checkout, libwatref."""
    src = HERE / "watfft_oracle.c"
    if force or not ORACLE_SO.exists() or ORACLE_SO.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["make", "-C", str(HERE), "libwatfft_oracle.so"], stdout=subprocess.DEVNULL)
    mods = reference_modules()
    if mods is not None:
        if not mods.is_dir():
            raise FileNotFoundError(f"WATFFT_REFERENCE: {mods} is not a directory")
        newest = max(p.stat().st_mtime for p in [HERE / "wat2c.py", HERE / "watref_threads.c"])
        if force or not WATREF_SO.exists() or WATREF_SO.stat().st_mtime < newest:
            subprocess.check_call(["make", "-C", str(HERE), "ref", f"REFMODS={mods}"], stdout=subprocess.DEVNULL)


def _f32(a):
    return a.ctypes.data_as(_c_f32p)


def _f64(a):
    return a.ctypes.data_as(_c_f64p)


class Oracle:
    """The C restatement.  All methods take/return numpy arrays, one transform per call."""

    def __init__(self):
        if not ORACLE_SO.exists():
            build()
        self.lib = L = ctypes.CDLL(str(ORACLE_SO))
        L.wfo_fft_split_f32.argtypes = [ctypes.c_int, _c_f32p, _c_f32p, ctypes.c_int]
        L.wfo_rfft_split_f32.argtypes = [ctypes.c_int, _c_f32p, _c_f32p]
        L.wfo_irfft_split_f32.argtypes = [ctypes.c_int, _c_f32p, _c_f32p]
        L.wfo_fft_interleaved_f32.argtypes = [ctypes.c_int, _c_f32p, ctypes.c_int]
        L.wfo_fft_f64.argtypes = [ctypes.c_int, _c_f64p, ctypes.c_int]
        L.wfo_rfft_f64.argtypes = [ctypes.c_int, _c_f64p]
        L.wfo_irfft_f64.argtypes = [ctypes.c_int, _c_f64p, _c_f64p]
        L.wfo_dft_f64.argtypes = [ctypes.c_int, _c_f64p, _c_f64p, _c_f64p, _c_f64p, ctypes.c_int]
        L.wfo_twiddles_f32_split.argtypes = [ctypes.c_int, ctypes.c_int, _c_f32p, _c_f32p]
        L.wfo_twiddles_f32_dual.argtypes = [ctypes.c_int, ctypes.c_int, _c_f32p, _c_f32p]
        L.wfo_twiddles_f64.argtypes = [ctypes.c_int, ctypes.c_int, _c_f64p, _c_f64p]
        L.wfo_fft_split_f32_batch.argtypes = [ctypes.c_int, ctypes.c_int, _c_f32p, _c_f32p, ctypes.c_int]
        for f in ("wfo_fft_split_f32", "wfo_rfft_split_f32", "wfo_irfft_split_f32", "wfo_fft_interleaved_f32",
                  "wfo_fft_f64", "wfo_rfft_f64", "wfo_irfft_f64", "wfo_dft_f64", "wfo_twiddles_f32_split",
                  "wfo_twiddles_f32_dual", "wfo_twiddles_f64", "wfo_fft_split_f32_batch"):
            getattr(L, f).restype = None

    # -- transform 1
    def fft_split_f32(self, re, im, inverse=False):
        re = np.ascontiguousarray(re, np.float32).copy()
        im = np.ascontiguousarray(im, np.float32).copy()
        self.lib.wfo_fft_split_f32(re.size, _f32(re), _f32(im), int(inverse))
        return re, im

    # -- transform 2
    def rfft_split_f32(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.zeros(x.size + 2, np.float32)
        self.lib.wfo_rfft_split_f32(x.size, _f32(x), _f32(out))
        return out

    def irfft_split_f32(self, spec):
        spec = np.ascontiguousarray(spec, np.float32)
        n = spec.size - 2
        out = np.zeros(n, np.float32)
        self.lib.wfo_irfft_split_f32(n, _f32(spec), _f32(out))
        return out

    # -- transform 3
    def fft_interleaved_f32(self, data, inverse=False):
        d = np.ascontiguousarray(data, np.float32).copy()
        self.lib.wfo_fft_interleaved_f32(d.size // 2, _f32(d), int(inverse))
        return d

    # -- transform 4
    def fft_f64(self, data, inverse=False):
        d = np.ascontiguousarray(data, np.float64).copy()
        self.lib.wfo_fft_f64(d.size // 2, _f64(d), int(inverse))
        return d

    def rfft_f64(self, x):
        x = np.ascontiguousarray(x, np.float64)
        buf = np.zeros(x.size + 2, np.float64)
        buf[: x.size] = x
        self.lib.wfo_rfft_f64(x.size, _f64(buf))
        return buf

    def irfft_f64(self, spec):
        spec = np.ascontiguousarray(spec, np.float64)
        n = spec.size - 2
        out = np.zeros(n, np.float64)
        self.lib.wfo_irfft_f64(n, _f64(spec), _f64(out))
        return out

    def dft_f64(self, z, inverse=False):
        z = np.asarray(z, np.complex128)
        re, im = np.ascontiguousarray(z.real), np.ascontiguousarray(z.imag)
        ore, oim = np.zeros_like(re), np.zeros_like(im)
        self.lib.wfo_dft_f64(z.size, _f64(re), _f64(im), _f64(ore), _f64(oim), int(inverse))
        return ore + 1j * oim

    def twiddles(self, kind, n, count=None):
        count = n if count is None else count
        if kind == "f64":
            re, im = np.zeros(count), np.zeros(count)
            self.lib.wfo_twiddles_f64(n, count, _f64(re), _f64(im))
        else:
            re, im = np.zeros(count, np.float32), np.zeros(count, np.float32)
            getattr(self.lib, f"wfo_twiddles_f32_{kind}")(n, count, _f32(re), _f32(im))
        return re, im


# Memory maps of the reference modules (SURVEY.md Appendix A; the .wat headers).
SPLIT_IMAG_OFFSET = 32768


class WatRef:
    """The reference modules themselves (transpiled).  One instance == one linear memory per module,
    exactly like one WebAssembly.Instance; methods mirror the module exports."""

    MODULES = ("fft_combined", "fft_real_combined", "fft_real_f32_dual", "fft_split_native_f32",
               "fft_stockham_f32_dual")

    def __init__(self):
        if not WATREF_SO.exists():
            raise FileNotFoundError(f"{WATREF_SO} missing (build it with WATFFT_REFERENCE set to a wat-fft checkout)")
        self.lib = ctypes.CDLL(str(WATREF_SO))
        self.mem = {}
        for m in self.MODULES:
            pages = getattr(self.lib, f"watref_{m}_pages")
            pages.restype = ctypes.c_uint32
            self.mem[m] = np.zeros(pages() * 65536, np.uint8)

    @staticmethod
    def available() -> bool:
        return WATREF_SO.exists()

    def fn(self, module, export):
        f = getattr(self.lib, f"watref_{module}_{export}")
        f.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
        f.restype = None
        return f

    def call(self, module, export, n):
        self.fn(module, export)(self.mem[module].ctypes.data, n)

    def view(self, module, dtype, offset, count):
        item = np.dtype(dtype).itemsize
        return self.mem[module][offset: offset + count * item].view(dtype)

    # ---- the four transforms, with the module's own precompute -------
    def fft_split_f32(self, re, im, inverse=False):
        m, n = "fft_split_native_f32", len(re)
        self.view(m, np.float32, 0, n)[:] = re
        self.view(m, np.float32, SPLIT_IMAG_OFFSET, n)[:] = im
        self.call(m, "precompute_twiddles_split", n)
        self.call(m, "ifft_split" if inverse else "fft_split", n)
        return self.view(m, np.float32, 0, n).copy(), self.view(m, np.float32, SPLIT_IMAG_OFFSET, n).copy()

    def rfft_split_f32(self, x):
        m, n = "fft_split_native_f32", len(x)
        self.view(m, np.float32, 0, n)[:] = x
        self.call(m, "precompute_rfft_twiddles_split", n)
        self.call(m, "rfft_split", n)
        return self.view(m, np.float32, 0, n + 2).copy()

    def irfft_split_f32(self, spec):
        m, n = "fft_split_native_f32", len(spec) - 2
        self.view(m, np.float32, 0, n + 2)[:] = spec
        self.call(m, "precompute_rfft_twiddles_split", n)
        self.call(m, "irfft_split", n)
        return self.view(m, np.float32, 0, n).copy()

    def fft_interleaved_f32(self, data, inverse=False):
        m, n = "fft_stockham_f32_dual", len(data) // 2
        self.view(m, np.float32, 0, 2 * n)[:] = data
        self.call(m, "precompute_twiddles", n)
        self.call(m, "ifft" if inverse else "fft", n)
        return self.view(m, np.float32, 0, 2 * n).copy()

    def fft_f64(self, data, inverse=False):
        m, n = "fft_combined", len(data) // 2
        self.view(m, np.float64, 0, 2 * n)[:] = data
        self.call(m, "precompute_twiddles", n)
        self.call(m, "ifft" if inverse else "fft", n)
        return self.view(m, np.float64, 0, 2 * n).copy()

    def rfft_f64(self, x):
        m, n = "fft_real_combined", len(x)
        self.view(m, np.float64, 0, n)[:] = x
        self.call(m, "precompute_rfft_twiddles", n)
        self.call(m, "rfft", n)
        return self.view(m, np.float64, 0, n + 2).copy()

    def rfft_f32_dual(self, x):
        m, n = "fft_real_f32_dual", len(x)
        self.view(m, np.float32, 0, n)[:] = x
        self.call(m, "precompute_rfft_twiddles", n)
        self.call(m, "rfft", n)
        return self.view(m, np.float32, 0, n + 2).copy()

    def irfft_f32_dual(self, spec):
        m, n = "fft_real_f32_dual", len(spec) - 2
        self.view(m, np.float32, 0, n + 2)[:] = spec
        self.call(m, "precompute_rfft_twiddles", n)
        self.call(m, "irfft", n)
        return self.view(m, np.float32, 0, n).copy()

    # ---- threaded batch runner (CPU baseline) -------------------------
    def run_batch(self, module, precompute, run, n, in0, dst0=0, in1=None, dst1=0,
                  out0=None, src0=0, out1=None, src1=0, reps=1, threads=None):
        """rows of `in0` (2-D, C-contiguous) are copied to memory offset dst0 then `run(n)` is called;
        optional second plane and copy-out.  Returns wall seconds."""
        threads = threads or os.cpu_count() or 1
        f = self.lib.watref_run_batch
        f.restype = ctypes.c_double
        vp, sz, u32, lg = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_long
        f.argtypes = [vp, vp, u32, u32,
                      vp, sz, sz, u32, vp, sz, sz, u32,
                      vp, sz, sz, u32, vp, sz, sz, u32,
                      lg, lg, ctypes.c_int]

        def plane(a):
            if a is None:
                return None, 0, 0
            assert a.ndim == 2 and a.flags.c_contiguous
            return a.ctypes.data, a.shape[1] * a.itemsize, a.strides[0]

        pages = getattr(self.lib, f"watref_{module}_pages")
        pages.restype = ctypes.c_uint32
        fp = ctypes.cast(getattr(self.lib, f"watref_{module}_{precompute}"), vp)
        fr = ctypes.cast(getattr(self.lib, f"watref_{module}_{run}"), vp)
        i0, i1, o0, o1 = plane(in0), plane(in1), plane(out0), plane(out1)
        return f(fp, fr, pages(), n, i0[0], i0[1], i0[2], dst0, i1[0], i1[1], i1[2], dst1,
                 o0[0], o0[1], o0[2], src0, o1[0], o1[1], o1[2], src1, in0.shape[0], reps, threads)


class WatRefPool:
    """Persistent pthread pool over the transpiled reference modules (oracle/watref_threads.c): one private module
    memory per worker, `prepare()` = instantiate + precompute once per size (untimed, like
    benchmarks/lib/wat-contexts.js:110-131), `run()` = the timed memcpy-in + transform loop over the rows."""

    def __init__(self, ref: "WatRef", threads=None):
        self.ref, self.lib = ref, ref.lib
        vp, sz, u32, lg, dbl = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_long, ctypes.c_double
        L = self.lib
        L.watref_pool_create.restype, L.watref_pool_create.argtypes = vp, [ctypes.c_int]
        L.watref_pool_destroy.restype, L.watref_pool_destroy.argtypes = None, [vp]
        L.watref_pool_prepare.restype, L.watref_pool_prepare.argtypes = None, [vp, vp, u32, u32]
        L.watref_pool_run.restype = dbl
        L.watref_pool_run.argtypes = [vp, vp, u32, vp, sz, sz, u32, vp, sz, sz, u32, vp, sz, sz, u32, vp, sz, sz, u32, lg, lg]
        L.watref_pool_run_stft.restype = dbl
        L.watref_pool_run_stft.argtypes = [vp, vp, u32, vp, vp, ctypes.c_int, ctypes.c_int, lg, dbl, dbl, vp, lg]
        self.threads = threads or os.cpu_count() or 1
        self._p = L.watref_pool_create(self.threads)

    def _fn(self, module, export):
        return ctypes.cast(getattr(self.lib, f"watref_{module}_{export}"), ctypes.c_void_p)

    def prepare(self, module, precompute, n):
        pages = getattr(self.lib, f"watref_{module}_pages")
        pages.restype = ctypes.c_uint32
        self.lib.watref_pool_prepare(self._p, self._fn(module, precompute), pages(), n)

    def run(self, module, export, n, in0, dst0=0, in1=None, dst1=0, out0=None, src0=0, out1=None, src1=0, reps=1):
        """rows of in0 (2-D, C-contiguous) -> memory offset dst0, then export(n); optional copy-out.  Wall seconds."""
        def plane(a):
            if a is None:
                return None, 0, 0
            assert a.ndim == 2 and a.flags.c_contiguous
            return a.ctypes.data, a.shape[1] * a.itemsize, a.strides[0]
        i0, i1, o0, o1 = plane(in0), plane(in1), plane(out0), plane(out1)
        return self.lib.watref_pool_run(self._p, self._fn(module, export), n, i0[0], i0[1], i0[2], dst0, i1[0], i1[1], i1[2], dst1,
                                        o0[0], o0[1], o0[2], src0, o1[0], o1[1], o1[2], src1, in0.shape[0], reps)

    def run_stft(self, samples, fft_size, hop, window, gain, range_db, out, reps=1):
        """generateSpectrogram's per-frame loop (C port) around the module's rfft_split; prepare() must have been
        called with precompute_rfft_twiddles_split(fft_size).  Wall seconds."""
        assert samples.dtype == np.float32 and window.dtype == np.float64 and out.dtype == np.float32
        frames = (len(samples) - len(window)) // hop + 1
        assert out.size >= frames * (fft_size // 2 + 1)
        return self.lib.watref_pool_run_stft(self._p, self._fn("fft_split_native_f32", "rfft_split"), fft_size,
                                             samples.ctypes.data, window.ctypes.data, len(window), hop, frames,
                                             float(gain), float(range_db), out.ctypes.data, reps)

    def close(self):
        if self._p:
            self.lib.watref_pool_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ----------------------------------------------------------------------
# Reference fixtures restated
# ----------------------------------------------------------------------
def lcg_signal(n: int, seed: int) -> np.ndarray:
    """tests/dft-reference.js:187-190 / tools/accuracy_report.js:46-55.  The JS LCG runs in doubles:
    s*1103515245+12345 exceeds 2^53 and is ROUNDED before `& 0x7fffffff` (SURVEY F7)."""
    out = np.empty(n, np.float64)
    s = seed
    for i in range(n):
        x = float(s) * 1103515245.0 + 12345.0     # double arithmetic, rounds like JS
        s = (int(x) % (1 << 32)) & 0x7FFFFFFF      # ToInt32 then mask
        out[i] = s / 0x7FFFFFFF * 2.0 - 1.0
    return out


def mulberry32(seed: int):
    """benchmarks/lib/harness.js:99-108: returns a generator of uniform [0,1) doubles."""
    M = 0xFFFFFFFF
    state = seed & M

    def imul(a, b):
        return (a * b) & M

    def nxt():
        nonlocal state
        state = (state + 0x6D2B79F5) & M
        t = imul(state ^ (state >> 15), state | 1)
        t ^= (t + imul(t ^ (t >> 7), t | 61)) & M
        t &= M
        return ((t ^ (t >> 14)) & M) / 4294967296.0

    return nxt


def bench_complex_inputs(n: int, seed: int | None = None):
    """benchmarks/lib/wat-contexts.js:34-50 generateComplexInputs: re then im per element, seed = n."""
    rnd = mulberry32(n if seed is None else seed)
    re, im = np.empty(n), np.empty(n)
    for i in range(n):
        re[i] = rnd() * 2 - 1
        im[i] = rnd() * 2 - 1
    return re, im


def bench_real_inputs(n: int, seed: int | None = None):
    """benchmarks/lib/wat-contexts.js:52-68 generateRealInputs."""
    rnd = mulberry32(n if seed is None else seed)
    return np.array([rnd() * 2 - 1 for _ in range(n)])


def dft(z, inverse=False):
    """O(N^2) f64 DFT, tests/dft-reference.js:14-88 (numpy matrix form for small N)."""
    z = np.asarray(z, np.complex128)
    n = z.size
    k = np.arange(n)
    ang = (2.0 if inverse else -2.0) * np.pi * ((k[:, None] * k[None, :]) % n) / n
    out = (np.cos(ang) + 1j * np.sin(ang)) @ z
    return out / n if inverse else out


def real_dft(x):
    x = np.asarray(x, np.float64)
    return dft(x.astype(np.complex128))[: x.size // 2 + 1]


# ----------------------------------------------------------------------
# STFT / spectrogram front-end (SURVEY 8f-1): playground/src/spectrogram.js restated
# ----------------------------------------------------------------------
def window_function(window_type: str, n: int) -> np.ndarray:
    """WINDOW_FUNCTIONS, spectrogram.js:1-25 (evaluated in double, like the JS)."""
    i = np.arange(n, dtype=np.float64)
    x = 2 * np.pi * i / (n - 1)
    if window_type == "hamming":
        return 0.54 - 0.46 * np.cos(x)
    if window_type == "blackman":
        return 0.42 - 0.5 * np.cos(x) + 0.08 * np.cos(2 * x)
    if window_type == "blackmanHarris":
        return 0.35875 - 0.48829 * np.cos(x) + 0.14128 * np.cos(2 * x) - 0.01168 * np.cos(3 * x)
    if window_type == "rectangular":
        return np.ones(n)
    return 0.5 * (1 - np.cos(x))          # hann, also the fallback for unknown names (:31)


def spectrogram_reference(samples, fft_size, hop, window_type="hann", zero_padding=1, gain=0.0, range_db=80.0,
                          rfft=None, complex_out=False):
    """generateSpectrogram, spectrogram.js:281-360: per frame slice -> applyWindow (:27-38, product
    rounded to f32) -> zeroPad (:40-45) -> real FFT -> computeMagnitude (:47-58, rounded to f32) ->
    magnitudeToDb (:60-62) -> gain/range normalisation with the first 3 bins zeroed (:335-352).
    `rfft` is the f32 real transform (n reals -> n+2 interleaved floats).

    PARITY UNPINNED for everything but the transform: the reference loop is JavaScript and no JS engine exists in this
    image, so this restatement has no reference-run output behind it.  The r2c core it calls IS pinned (bit-identical to
    the transpiled reference module, tests/test_oracle_pinning.py); window / magnitude / dB / normalise are restated from
    the cited lines."""
    samples = np.asarray(samples, np.float32)
    wsize = fft_size // zero_padding
    bins = fft_size // 2 + 1
    frames = (len(samples) - wsize) // hop + 1
    if frames <= 0:
        raise ValueError("Audio too short for the given FFT size")
    w = window_function(window_type, wsize)
    out = np.zeros((frames, bins, 2) if complex_out else (frames, bins), np.float32)
    for f in range(frames):
        frame = samples[f * hop: f * hop + wsize]
        padded = np.zeros(fft_size, np.float32)
        padded[:wsize] = (frame.astype(np.float64) * w).astype(np.float32)
        spec = np.asarray(rfft(padded), np.float32)
        re, im = spec[0::2].astype(np.float64), spec[1::2].astype(np.float64)
        if complex_out:
            out[f, :, 0], out[f, :, 1] = re, im
            continue
        mag = np.sqrt(re * re + im * im).astype(np.float32).astype(np.float64)
        db = 20 * np.log10(mag / (fft_size / 2) + 1e-10)
        norm = np.clip((db - (gain - range_db)) / range_db, 0.0, 1.0)
        norm[:3] = 0.0
        out[f] = norm
    return out
