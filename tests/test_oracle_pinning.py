"""Pins the CPU oracle: (1) bit-for-bit against the transpiled reference modules where the
reference runs its general path, to rounding level on the hard-coded codelet sizes; (2) against
the committed fixtures generated from those modules (tests/golden/watref_vectors.npz), which is
what travels to the GPU box."""
from pathlib import Path

import numpy as np
import pytest

import oracle as om

FIX = np.load(Path(__file__).resolve().parent / "golden" / "watref_vectors.npz")
FIX_SIZES = [4, 8, 16, 32, 64, 128, 256, 1024, 4096]
ALL = [4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]


@pytest.mark.parametrize("n", ALL)
def test_oracle_bit_exact_vs_reference_modules(oracle, reference, n):
    """Random inputs through the transpiled modules when they are built; otherwise the inputs stored with the modules'
    outputs (tests/golden), which exist for FIX_SIZES."""
    watref = reference
    if isinstance(reference, om.WatRef):
        rng = np.random.default_rng(n)
        re = rng.uniform(-1, 1, n).astype(np.float32)
        im = rng.uniform(-1, 1, n).astype(np.float32)
        ds = [rng.uniform(-1, 1, 2 * n) for _ in range(2)]
        x32 = rng.uniform(-1, 1, n).astype(np.float32) if n >= 32 else None
        x64 = rng.uniform(-1, 1, n) if n >= 8 else None
    else:
        if n not in FIX_SIZES:
            pytest.skip(f"no stored reference outputs at N={n} (needs WATFFT_REFERENCE, a wat-fft checkout)")
        s = reference.signals(n)
        re, im, ds, x32, x64 = s["re"], s["im"], [s["d"], s["d"]], s["xr"].astype(np.float32), s["xr"]
    for inv in (False, True):
        a, b = oracle.fft_split_f32(re, im, inv), watref.fft_split_f32(re, im, inv)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), ("split", n, inv)
        x = np.empty(2 * n, np.float32)
        x[0::2], x[1::2] = re, im
        a, b = oracle.fft_interleaved_f32(x, inv), watref.fft_interleaved_f32(x, inv)
        if n in (8, 16):        # unrolled codelets (fft_stockham_f32_dual.wat:202-534): same maths, other op order
            assert np.max(np.abs(a - b)) <= 4e-7 * np.linalg.norm(x)
        else:
            assert np.array_equal(a, b), ("dual", n, inv)
        d = ds[inv]
        a, b = oracle.fft_f64(d, inv), watref.fft_f64(d, inv)
        if n == 16:             # $fft_16 codelet (fft_combined.wat:175-356)
            assert np.max(np.abs(a - b)) <= 4e-16 * np.linalg.norm(d)
        else:
            assert np.array_equal(a, b), ("f64", n, inv)
    if n >= 32:
        x = x32
        s = watref.rfft_split_f32(x)
        assert np.array_equal(oracle.rfft_split_f32(x), s), ("rfft32", n)
        assert np.array_equal(oracle.irfft_split_f32(s), watref.irfft_split_f32(s)), ("irfft32", n)
    if n >= 8:
        x = x64
        a, b = oracle.rfft_f64(x), watref.rfft_f64(x)
        if n in (8, 32):        # $rfft_8 / $rfft_32 fused codelets
            assert np.max(np.abs(a - b)) <= 8e-16 * np.linalg.norm(x)
        else:
            assert np.array_equal(a, b), ("rfft64", n)


@pytest.mark.parametrize("n", [32768 // 2, 16384])
def test_oracle_rfft_max_size(oracle, watref, n):
    x = np.random.default_rng(1).uniform(-1, 1, n).astype(np.float32)
    s = watref.rfft_split_f32(x)
    assert np.array_equal(oracle.rfft_split_f32(x), s)
    assert np.array_equal(oracle.irfft_split_f32(s), watref.irfft_split_f32(s))


@pytest.mark.parametrize("n", FIX_SIZES)
def test_oracle_vs_committed_fixtures(oracle, n):
    re, im, xr = FIX[f"in_re_{n}"], FIX[f"in_im_{n}"], FIX[f"in_real_{n}"]
    for inv, tag in ((False, "fwd"), (True, "inv")):
        a = oracle.fft_split_f32(re, im, inv)
        assert np.array_equal(a[0], FIX[f"split_{tag}_re_{n}"]) and np.array_equal(a[1], FIX[f"split_{tag}_im_{n}"])
        x = np.empty(2 * n, np.float32)
        x[0::2], x[1::2] = re, im
        assert np.max(np.abs(oracle.fft_interleaved_f32(x, inv) - FIX[f"dual_{tag}_{n}"])) <= 4e-7 * np.linalg.norm(x)
        d = np.empty(2 * n)
        d[0::2], d[1::2] = om.lcg_signal(n, 12345 + n), om.lcg_signal(n, 54321 + n)
        assert np.max(np.abs(oracle.fft_f64(d, inv) - FIX[f"f64_{tag}_{n}"])) <= 4e-16 * np.linalg.norm(d)
    if n >= 32:
        assert np.array_equal(oracle.rfft_split_f32(xr.astype(np.float32)), FIX[f"rfft32_{n}"])
        assert np.array_equal(oracle.irfft_split_f32(FIX[f"rfft32_{n}"]), FIX[f"irfft32_{n}"])
    if n >= 8:
        assert np.max(np.abs(oracle.rfft_f64(xr) - FIX[f"rfft64_{n}"])) <= 8e-16 * np.linalg.norm(xr)
    if 8 <= n <= 256:
        # rfft_split's algorithm (the restatement, any n >= 8) against the OTHER f32 real module of the
        # reference (fft_real_f32_dual, which backs createRFFTf32): different algorithm, f32 tolerance
        x32 = xr.astype(np.float32)
        s = oracle.rfft_split_f32(x32)
        assert np.max(np.abs(s - FIX[f"rfft32dual_{n}"])) <= 2e-6 * np.log2(n) * np.linalg.norm(x32)
        back = oracle.irfft_split_f32(FIX[f"rfft32dual_{n}"])
        assert np.max(np.abs(back - FIX[f"irfft32dual_{n}"])) <= 2e-6 * np.log2(n) * np.linalg.norm(FIX[f"rfft32dual_{n}"])


def test_lcg_matches_js_double_rounding():
    # SURVEY F7: the JS LCG runs in doubles; the exact-integer LCG diverges at the second draw
    s = om.lcg_signal(4, 12345 + 16)
    exact, st = [], 12345 + 16
    for _ in range(4):
        st = (st * 1103515245 + 12345) & 0x7FFFFFFF
        exact.append(st / 0x7FFFFFFF * 2 - 1)
    assert s[0] == exact[0] and not np.allclose(s[1:], exact[1:])
    assert np.all(np.abs(s) <= 1.0)


def test_mulberry32_known_values():
    # benchmarks/lib/harness.js:99-108 restated; first draws for seed 1024 are stable numbers in [0,1)
    r = om.mulberry32(1024)
    v = [r() for _ in range(3)]
    assert all(0.0 <= x < 1.0 for x in v) and len(set(v)) == 3
    re, im = om.bench_complex_inputs(16)
    assert re.shape == (16,) and np.all(np.abs(re) <= 1) and np.all(np.abs(im) <= 1)


def test_trig_accuracy_levels(oracle):
    # SURVEY Appendix B: max |twiddle - exact| = 6.5e-11 (f64), 5.3e-7..6.3e-7 (f32)
    for n in (16, 256, 4096):
        k = np.arange(n)
        re, im = oracle.twiddles("f64", n)
        err = np.max(np.abs((re + 1j * im) - np.exp(-2j * np.pi * k / n)))
        assert 1e-12 < err < 1.5e-10 or n == 16
        re, im = oracle.twiddles("split", n)
        err = np.max(np.abs((re.astype(np.float64) + 1j * im) - np.exp(-2j * np.pi * k / n)))
        assert err < 1.2e-6


@pytest.mark.parametrize("n", [1 << k for k in range(3, 15)])
def test_oracle_irfft_f64(oracle, n):
    """f64 c2r has no reference module (the restatement defines it), so it is pinned to the truth: numpy's inverse real DFT
    of an exact Hermitian half spectrum, and the inverse of the oracle's own rfft_f64, both at the level of the reference's
    Taylor-series f64 twiddles (~6.5e-11 each); the imaginary parts of DC and Nyquist are ignored, bit for bit."""
    rng = np.random.default_rng(n + 99)
    x = rng.uniform(-1, 1, n)
    s = np.fft.rfft(x)
    il = np.empty(n + 2)
    il[0::2], il[1::2] = s.real, s.imag
    y = oracle.irfft_f64(il)
    assert np.max(np.abs(y - np.fft.irfft(s, n))) < 2e-9
    assert np.max(np.abs(oracle.irfft_f64(oracle.rfft_f64(x)) - x)) < 2e-9
    g = il.copy()
    g[1], g[n + 1] = 123.0, -77.0
    assert np.array_equal(oracle.irfft_f64(g), y)
