"""Uniform batched front-ends over the three implementations the restated reference suites run
against: the C restatement (oracle), the transpiled reference modules (watref) and the B200 engine
(gpu, through the public contexts == the C ABI).  All take 2-D arrays [batch, row]."""
import numpy as np


class _Loop:
    """Row-at-a-time adapter for the CPU checkers."""

    def __init__(self, impl):
        self.impl = impl

    def fft_split_f32(self, re, im, inverse=False):
        out = [self.impl.fft_split_f32(r, i, inverse) for r, i in zip(re, im)]
        return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])

    def fft_interleaved_f32(self, x, inverse=False):
        return np.stack([self.impl.fft_interleaved_f32(r, inverse) for r in x])

    def rfft_f32(self, x):
        return np.stack([self.impl.rfft_split_f32(r) for r in x])

    def irfft_f32(self, s):
        return np.stack([self.impl.irfft_split_f32(r) for r in s])

    def fft_f64(self, x, inverse=False):
        return np.stack([self.impl.fft_f64(r, inverse) for r in x])

    def rfft_f64(self, x):
        return np.stack([self.impl.rfft_f64(r) for r in x])


class OracleBackend(_Loop):
    name = "oracle"


class WatRefBackend(_Loop):
    """rfft_split needs n >= 32; below that the public f32 real context is backed by fft_real_f32_dual."""
    name = "watref"

    def rfft_f32(self, x):
        if x.shape[-1] < 32:
            return np.stack([self.impl.rfft_f32_dual(r) for r in x])
        return super().rfft_f32(x)

    def irfft_f32(self, s):
        if s.shape[-1] - 2 < 32:
            return np.stack([self.impl.irfft_f32_dual(r) for r in s])
        return super().irfft_f32(s)


class GpuBackend:
    """Batched calls through createFFT*/createRFFT* (pinned host buffers, H2D, kernel, D2H)."""
    name = "gpu"

    def __init__(self, wf):
        self.wf = wf

    def fft_split_f32(self, re, im, inverse=False):
        re, im = np.atleast_2d(re), np.atleast_2d(im)
        b, n = re.shape
        c = self.wf.createFFTf32Split(n, batch=b)
        c.getRealBuffer()[:] = np.asarray(re, np.float32).ravel()
        c.getImagBuffer()[:] = np.asarray(im, np.float32).ravel()
        c.inverse() if inverse else c.forward()
        out = c.getRealBuffer().reshape(b, n).copy(), c.getImagBuffer().reshape(b, n).copy()
        c.dispose()
        return out

    def _il(self, factory, x, inverse, dtype):
        x = np.atleast_2d(x)
        b, n2 = x.shape
        c = factory(n2 // 2, batch=b)
        c.getInputBuffer()[:] = np.asarray(x, dtype).ravel()
        c.inverse() if inverse else c.forward()
        out = c.getOutputBuffer().reshape(b, n2).copy()
        c.dispose()
        return out

    def fft_interleaved_f32(self, x, inverse=False):
        return self._il(self.wf.createFFTf32, x, inverse, np.float32)

    def fft_f64(self, x, inverse=False):
        return self._il(self.wf.createFFT, x, inverse, np.float64)

    def _r(self, factory, x, dtype):
        x = np.atleast_2d(x)
        b, n = x.shape
        c = factory(n, batch=b)
        c.getInputBuffer()[:] = np.asarray(x, dtype).ravel()
        c.forward()
        out = c.getOutputBuffer().reshape(b, n + 2).copy()
        c.dispose()
        return out

    def rfft_f32(self, x):
        return self._r(self.wf.createRFFTf32, x, np.float32)

    def rfft_f64(self, x):
        return self._r(self.wf.createRFFT, x, np.float64)

    def irfft_f32(self, s):
        s = np.atleast_2d(s)
        b, n = s.shape[0], s.shape[1] - 2
        c = self.wf.createRFFTf32(n, batch=b)
        c.getOutputBuffer()[:] = np.asarray(s, np.float32).ravel()
        c.inverse()
        out = c.getInputBuffer().reshape(b, n).copy()
        c.dispose()
        return out


class StoredWatRef:
    """Stand-in for oracle.WatRef where the transpiled reference modules are not built: answers with the outputs the
    reference modules produced for the stored inputs (tests/golden/watref_vectors.npz, tests/golden/make_fixtures.py)
    and raises LookupError for any other input."""

    SIZES = (4, 8, 16, 32, 64, 128, 256, 1024, 4096)

    def __init__(self):
        from pathlib import Path
        self.fix = np.load(Path(__file__).resolve().parent / "golden" / "watref_vectors.npz")

    def signals(self, n):
        """The stored inputs at size n: re, im (f32 split), il (f32 interleaved), d (f64 interleaved), xr (f64 real)."""
        import oracle as om
        if n not in self.SIZES:
            raise LookupError(f"no stored reference outputs at N={n}")
        re, im = self.fix[f"in_re_{n}"], self.fix[f"in_im_{n}"]
        il = np.empty(2 * n, np.float32)
        il[0::2], il[1::2] = re, im
        d = np.empty(2 * n)
        d[0::2], d[1::2] = om.lcg_signal(n, 12345 + n), om.lcg_signal(n, 54321 + n)
        return {"re": re, "im": im, "il": il, "d": d, "xr": self.fix[f"in_real_{n}"]}

    def _get(self, x, stored, key):
        if not np.array_equal(np.asarray(x), stored) or key not in self.fix:
            raise LookupError(f"{key}: input is not a stored one")
        return self.fix[key].copy()

    def fft_split_f32(self, re, im, inverse=False):
        n, tag = len(re), "inv" if inverse else "fwd"
        s = self.signals(n)
        self._get(im, s["im"], f"split_{tag}_im_{n}")
        return self._get(re, s["re"], f"split_{tag}_re_{n}"), self.fix[f"split_{tag}_im_{n}"].copy()

    def fft_interleaved_f32(self, data, inverse=False):
        n = len(data) // 2
        return self._get(data, self.signals(n)["il"], f"dual_{'inv' if inverse else 'fwd'}_{n}")

    def fft_f64(self, data, inverse=False):
        n = len(data) // 2
        return self._get(data, self.signals(n)["d"], f"f64_{'inv' if inverse else 'fwd'}_{n}")

    def rfft_split_f32(self, x):
        n = len(x)
        return self._get(x, self.signals(n)["xr"].astype(np.float32), f"rfft32_{n}")

    def irfft_split_f32(self, spec):
        n = len(spec) - 2
        self.signals(n)
        return self._get(spec, self.fix.get(f"rfft32_{n}"), f"irfft32_{n}")

    def rfft_f64(self, x):
        n = len(x)
        return self._get(x, self.signals(n)["xr"], f"rfft64_{n}")
