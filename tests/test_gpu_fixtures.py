"""GPU engine vs the committed reference-module outputs (tests/golden/watref_vectors.npz) and the
size-independent properties of the domain at BASELINE.json's full batch sizes."""
import math
from pathlib import Path

import numpy as np
import pytest

import oracle as om
from conftest import f32_bound, f64_bound, rel_err

pytestmark = pytest.mark.gpu
FIX = np.load(Path(__file__).resolve().parent / "golden" / "watref_vectors.npz")
FIX_SIZES = [4, 8, 16, 32, 64, 128, 256, 1024, 4096]


@pytest.mark.parametrize("n", FIX_SIZES)
def test_gpu_vs_reference_module_fixtures(wf, n):
    re, im, xr = FIX[f"in_re_{n}"], FIX[f"in_im_{n}"], FIX[f"in_real_{n}"]
    xin = np.r_[re, im]
    for inv, tag in ((False, "fwd"), (True, "inv")):
        c = wf.createFFTf32Split(n)
        c.getRealBuffer()[:] = re
        c.getImagBuffer()[:] = im
        c.inverse() if inv else c.forward()
        got = np.r_[c.getRealBuffer(), c.getImagBuffer()]
        c.dispose()
        assert rel_err(got, np.r_[FIX[f"split_{tag}_re_{n}"], FIX[f"split_{tag}_im_{n}"]], xin) <= f32_bound(n)
        x = np.empty(2 * n, np.float32)
        x[0::2], x[1::2] = re, im
        c = wf.createFFTf32(n)
        c.getInputBuffer()[:] = x
        c.inverse() if inv else c.forward()
        assert rel_err(c.getOutputBuffer(), FIX[f"dual_{tag}_{n}"], x) <= f32_bound(n)
        c.dispose()
        d = np.empty(2 * n)
        d[0::2], d[1::2] = om.lcg_signal(n, 12345 + n), om.lcg_signal(n, 54321 + n)
        c = wf.createFFT(n)
        c.getInputBuffer()[:] = d
        c.inverse() if inv else c.forward()
        assert rel_err(c.getOutputBuffer(), FIX[f"f64_{tag}_{n}"], d) <= f64_bound(n)
        c.dispose()
    if n >= 32:
        c = wf.createRFFTf32(n)
        c.getInputBuffer()[:] = xr.astype(np.float32)
        c.forward()
        assert rel_err(c.getOutputBuffer(), FIX[f"rfft32_{n}"], xr) <= f32_bound(n)
        c.getOutputBuffer()[:] = FIX[f"rfft32_{n}"]
        c.inverse()
        assert rel_err(c.getInputBuffer(), FIX[f"irfft32_{n}"], FIX[f"rfft32_{n}"]) <= f32_bound(n)
        c.dispose()
    if n >= 8:
        c = wf.createRFFT(n)
        c.getInputBuffer()[:] = xr
        c.forward()
        assert rel_err(c.getOutputBuffer(), FIX[f"rfft64_{n}"], xr) <= f64_bound(n)
        c.dispose()
    if 8 <= n <= 256:
        # createRFFTf32 against the module that backs it in the reference (fft_real_f32_dual), N >= 8
        c = wf.createRFFTf32(n)
        c.getInputBuffer()[:] = xr.astype(np.float32)
        c.forward()
        assert rel_err(c.getOutputBuffer(), FIX[f"rfft32dual_{n}"], xr) <= f32_bound(n)
        c.getOutputBuffer()[:] = FIX[f"rfft32dual_{n}"]
        c.inverse()
        assert rel_err(c.getInputBuffer(), FIX[f"irfft32dual_{n}"], FIX[f"rfft32dual_{n}"]) <= f32_bound(n)
        c.dispose()


@pytest.mark.parametrize("n", [16, 256, 4096])
def test_full_size_properties_c2c(wf, oracle, n):
    """BASELINE config 2 at full size (1 GiB of input): rows checked against the oracle on a sample,
    linearity, and the fft->ifft round trip over the WHOLE batch."""
    import torch
    C = wf._cabi
    batch = (1 << 30) // (8 * n)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(n)
    re = torch.rand(batch * n, device=dev, generator=g) * 2 - 1
    im = torch.rand(batch * n, device=dev, generator=g) * 2 - 1
    ore, oim = torch.empty_like(re), torch.empty_like(im)
    plan = wf.Plan(C.C2C, C.F32, C.SPLIT, n, batch, 0, C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS)
    torch.cuda.synchronize()      # torch filled the inputs on ITS stream; the plan's stream is non-blocking
    plan.exec_device(C.FORWARD, (re.data_ptr(), im.data_ptr()), (ore.data_ptr(), oim.data_ptr()))
    plan.sync()
    for r in sorted({0, 1, batch // 2, batch - 1}):
        a, b = re[r * n:(r + 1) * n].cpu().numpy(), im[r * n:(r + 1) * n].cpu().numpy()
        er, ei = oracle.fft_split_f32(a, b)
        got = np.r_[ore[r * n:(r + 1) * n].cpu().numpy(), oim[r * n:(r + 1) * n].cpu().numpy()]
        assert rel_err(got, np.r_[er, ei], np.r_[a, b]) <= f32_bound(n), (n, r)
    # Parseval over the whole batch: sum |X|^2 = N * sum |x|^2
    e_t = float((re.double() ** 2).sum() + (im.double() ** 2).sum())
    e_f = float((ore.double() ** 2).sum() + (oim.double() ** 2).sum())
    assert abs(e_f / (n * e_t) - 1) < 1e-5
    # round trip in place over the whole batch
    plan.exec_device(C.INVERSE, (ore.data_ptr(), oim.data_ptr()), (ore.data_ptr(), oim.data_ptr()))
    plan.sync()
    assert float((ore - re).abs().max()) < 1e-4 and float((oim - im).abs().max()) < 1e-4
    plan.destroy()


@pytest.mark.parametrize("n", [64, 4096])
def test_full_size_properties_r2c(wf, oracle, n):
    import torch
    C = wf._cabi
    batch = (1 << 30) // (4 * n)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(n)
    x = torch.rand(batch * n, device=dev, generator=g) * 2 - 1
    spec = torch.empty(batch * (n + 2), device=dev)
    back = torch.empty_like(x)
    plan = wf.Plan(C.R2C, C.F32, 0, n, batch, 0, C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS)
    torch.cuda.synchronize()      # torch filled the inputs on ITS stream; the plan's stream is non-blocking
    plan.exec_device(C.FORWARD, (x.data_ptr(), None), (spec.data_ptr(), None))
    plan.exec_device(C.INVERSE, (spec.data_ptr(), None), (back.data_ptr(), None))
    plan.sync()
    for r in sorted({0, batch // 2, batch - 1}):
        a = x[r * n:(r + 1) * n].cpu().numpy()
        got = spec[r * (n + 2):(r + 1) * (n + 2)].cpu().numpy()
        assert rel_err(got, oracle.rfft_split_f32(a), a) <= f32_bound(n), (n, r)
    assert float((back - x).abs().max()) < 1e-4          # irfft(rfft(x)) = x over the whole batch
    plan.destroy()


@pytest.mark.parametrize("n", [256, 1024, 4096])
def test_full_size_properties_f64(wf, oracle, n):
    """BASELINE config 4 at full size (batch = 2^30 / 16N): f64 c2c rows against the oracle with the 1e-14*log2(N) bound,
    Parseval and the round trip over the whole batch; f64 r2c rows against the oracle, c2r(r2c(x)) = x over the whole batch."""
    import torch
    C = wf._cabi
    batch = (1 << 30) // (16 * n)
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(n)
    flags = C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS
    z = torch.rand(batch * 2 * n, device=dev, generator=g, dtype=torch.float64) * 2 - 1
    out = torch.empty_like(z)
    plan = wf.Plan(C.C2C, C.F64, C.INTERLEAVED, n, batch, 0, flags)
    torch.cuda.synchronize()      # torch filled the inputs on ITS stream; the plan's stream is non-blocking
    plan.exec_device(C.FORWARD, (z.data_ptr(), None), (out.data_ptr(), None))
    plan.sync()
    for r in sorted({0, 1, batch // 2, batch - 1}):
        a = z[r * 2 * n:(r + 1) * 2 * n].cpu().numpy()
        assert rel_err(out[r * 2 * n:(r + 1) * 2 * n].cpu().numpy(), oracle.fft_f64(a), a) <= f64_bound(n), (n, r)
    assert abs(float((out ** 2).sum()) / (n * float((z ** 2).sum())) - 1) < 1e-9
    plan.exec_device(C.INVERSE, (out.data_ptr(), None), (out.data_ptr(), None))         # in place
    plan.sync()
    assert float((out - z).abs().max()) < 1e-9          # (Taylor-series twiddles: the round trip is good to ~1e-10, not 1e-16)
    plan.destroy()
    x = z[: batch * n]
    spec = out[: batch * (n + 2)]
    back = torch.empty_like(x)
    plan = wf.Plan(C.R2C, C.F64, 0, n, batch, 0, flags)
    torch.cuda.synchronize()      # torch filled the inputs on ITS stream; the plan's stream is non-blocking
    plan.exec_device(C.FORWARD, (x.data_ptr(), None), (spec.data_ptr(), None))
    plan.exec_device(C.INVERSE, (spec.data_ptr(), None), (back.data_ptr(), None))
    plan.sync()
    for r in sorted({0, batch // 2, batch - 1}):
        a = x[r * n:(r + 1) * n].cpu().numpy()
        assert rel_err(spec[r * (n + 2):(r + 1) * (n + 2)].cpu().numpy(), oracle.rfft_f64(a), a) <= f64_bound(n), (n, r)
    assert float((back - x).abs().max()) < 1e-9
    plan.destroy()


@pytest.mark.parametrize("n", [8, 16, 32, 64, 256, 1024, 4096, 16384])
def test_c2r_f64_against_the_f64_dft(wf, n):
    """SURVEY 8f-4: f64 c2r has no reference implementation (parity unpinned by definition), so it is gated against the f64
    truth itself: for a Hermitian spectrum built by numpy from random x, c2r must return x (numpy.fft.irfft semantics, 1/n
    normalised), at every size and for a batch; the imaginary parts of DC and Nyquist are ignored like irfft_split does."""
    rng = np.random.default_rng(n)
    batch = 5
    x = rng.uniform(-1, 1, (batch, n))
    spec = np.fft.rfft(x, axis=-1)                        # exact (to 1e-16) Hermitian half spectra
    il = np.empty((batch, n + 2))
    il[:, 0::2], il[:, 1::2] = spec.real, spec.imag
    il[:, 1] = 123.0                                      # garbage in the DC / Nyquist imaginary parts must not matter
    il[:, n + 1] = -7.0
    c = wf.createRFFT(n, batch=batch)
    c.getOutputBuffer()[:] = il.ravel()
    c.inverse()
    got = c.getInputBuffer().reshape(batch, n).copy()
    c.dispose()
    # the c2r core multiplies by the Taylor-series twiddles of the reference's f64 modules (accurate to ~5e-11)
    assert np.max(np.abs(got - x)) < 2e-9 * math.log2(n)
    assert np.max(np.abs(got - np.fft.irfft(spec, n=n, axis=-1))) < 2e-9 * math.log2(n)


def test_sharded_context_single_device(wf):
    from watfft_b200.sharding import ShardedSplitFFT
    n, batch = 256, 19
    rng = np.random.default_rng(3)
    re = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
    im = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
    sh = ShardedSplitFFT(n, batch, devices=[0, 0, 0])     # three shards on one device: same code path
    sh.scatter(re, im)
    sh.run()
    gr, gi = sh.gather()
    sh.dispose()
    truth = np.fft.fft(re.astype(np.float64) + 1j * im, axis=-1)
    assert np.max(np.abs((gr + 1j * gi) - truth)) < 5e-3


def test_context_contract(wf):
    """Buffer lengths / aliasing per index.js:73-83,131-141; batch rows are independent."""
    n = 64
    c = wf.createFFTf32(n)
    assert c.getInputBuffer().size == 2 * n and c.getInputBuffer().ctypes.data == c.getOutputBuffer().ctypes.data
    c.dispose()
    r = wf.createRFFTf32(n)
    assert r.getInputBuffer().size == n and r.getOutputBuffer().size == n + 2
    assert r.getInputBuffer().ctypes.data == r.getOutputBuffer().ctypes.data       # same bytes at batch = 1
    r.dispose()
    rb = wf.createRFFTf32(n, batch=3)
    assert rb.getInputBuffer().size == 3 * n and rb.getOutputBuffer().size == 3 * (n + 2)
    rb.dispose()
    # row independence: changing row 1 must not change row 0's output
    x = np.random.default_rng(0).uniform(-1, 1, (2, 2 * n)).astype(np.float32)
    c2 = wf.createFFTf32(n, batch=2)
    c2.getInputBuffer()[:] = x.ravel()
    c2.forward()
    first = c2.getOutputBuffer().reshape(2, -1)[0].copy()
    x[1] = 0
    c2.getInputBuffer()[:] = x.ravel()
    c2.forward()
    assert np.array_equal(first, c2.getOutputBuffer().reshape(2, -1)[0])
    assert np.all(c2.getOutputBuffer().reshape(2, -1)[1] == 0)
    c2.dispose()


def test_exports_facade(wf):
    """The exports-shaped instance runs the reference's raw-export call sequence unchanged and SYNCHRONOUSLY: results are
    in `memory` on the line after the call (tests/fft_split_native.test.js:78-114)."""
    ex = wf.createFFTf32SplitInstance()
    assert wf.SplitExportsFacade is wf.ModuleExports
    n = 1024
    re = np.frombuffer(ex.memory.buffer, np.float32, n, ex.REAL_OFFSET)
    im = np.frombuffer(ex.memory.buffer, np.float32, n, ex.IMAG_OFFSET)
    rng = np.random.default_rng(1)
    a, b = rng.uniform(-1, 1, n).astype(np.float32), rng.uniform(-1, 1, n).astype(np.float32)
    re[:], im[:] = a, b
    ex.precompute_twiddles_split(n)
    ex.fft_split(n)
    truth = np.fft.fft(a.astype(np.float64) + 1j * b)
    assert np.max(np.abs((re + 1j * im) - truth)) < 5e-3
    ex.ifft_split(n)
    assert np.max(np.abs(re - a)) < 1e-4
    # precompute with a new n silently re-targets the instance (tests/boundary.test.js:304-332)
    ex.precompute_rfft_twiddles_split(64)
    x = np.frombuffer(ex.memory.buffer, np.float32, 66, 0)
    sig = rng.uniform(-1, 1, 64).astype(np.float32)
    x[:64] = sig
    ex.rfft_split(64)
    assert np.max(np.abs((x[0::2] + 1j * x[1::2]) - np.fft.rfft(sig.astype(np.float64)))) < 1e-4
    ex.irfft_split(64)
    assert np.max(np.abs(x[:64] - sig)) < 1e-5
    ex.dispose()


@pytest.mark.parametrize("factory,dtype,real", [("createFFTInstance", np.float64, False), ("createFFTf32Instance", np.float32, False),
                                                 ("createRFFTInstance", np.float64, True), ("createRFFTf32Instance", np.float32, True)])
def test_instance_factories(wf, factory, dtype, real):
    """index.js:28-58: the four low-level factories return raw module-shaped exports over one linear memory."""
    ex = getattr(wf, factory)()
    n = 256
    rng = np.random.default_rng(3)
    # (the reference's f64 twiddles are Taylor series good to ~5e-11, BASELINE.md section 1: neither the comparison with numpy
    #  nor the fft -> ifft round trip is exact to machine precision)
    tol = 1e-9 if dtype == np.float64 else 2e-4
    if real:
        ex.precompute_rfft_twiddles(n)
        buf = np.frombuffer(ex.memory.buffer, dtype, n + 2, 0)
        sig = rng.uniform(-1, 1, n).astype(dtype)
        buf[:n] = sig
        ex.rfft(n)
        assert np.max(np.abs((buf[0::2] + 1j * buf[1::2]) - np.fft.rfft(sig.astype(np.float64)))) < tol * n
        ex.irfft(n)                         # (f64: extension, the reference export is missing)
        assert np.max(np.abs(buf[:n] - sig)) < tol
    else:
        ex.precompute_twiddles(n)
        buf = np.frombuffer(ex.memory.buffer, dtype, 2 * n, 0)
        z = rng.uniform(-1, 1, 2 * n).astype(dtype)
        buf[:] = z
        ex.fft(n)
        assert np.max(np.abs((buf[0::2] + 1j * buf[1::2]) - np.fft.fft(z[0::2].astype(np.float64) + 1j * z[1::2]))) < tol * n
        ex.ifft(n)
        assert np.max(np.abs(buf - z)) < tol
    ex.dispose()


def test_context_exports_field(wf):
    """index.js:72-75: a context carries `exports`, the instance it runs on -- at batch = 1 the context's views ARE views of
    exports.memory and forward() IS exports.fft(size); dispose() is idempotent and later use raises."""
    n = 128
    ctx = wf.createFFT(n)
    ex = ctx.exports
    view = np.frombuffer(ex.memory.buffer, np.float64, 2 * n, 0)
    ctx.getInputBuffer()[:] = 0.0
    ctx.getInputBuffer()[0] = 1.0                       # impulse through the context's view ...
    assert view[0] == 1.0                               # ... is the instance's memory
    ex.fft(n)                                           # raw export call
    assert np.allclose(ctx.getOutputBuffer()[0::2], 1.0) and np.allclose(ctx.getOutputBuffer()[1::2], 0.0)
    ctx.inverse()
    assert abs(view[0] - 1.0) < 1e-15 and np.max(np.abs(view[1:])) < 1e-15
    ctx.dispose()
    ctx.dispose()
    with pytest.raises(RuntimeError):
        ctx.forward()
    with pytest.raises(RuntimeError):
        ctx.getInputBuffer()
    big = wf.createRFFTf32(64, batch=4)                 # batch > 1: exports is a module instance of its own
    e2 = big.exports
    e2.precompute_rfft_twiddles(64)
    np.frombuffer(e2.memory.buffer, np.float32, 64, 0)[:] = 1.0
    e2.rfft(64)
    assert abs(np.frombuffer(e2.memory.buffer, np.float32, 2, 0)[0] - 64.0) < 1e-4
    big.dispose()


def test_staged_pipeline_large_batch(wf, oracle):
    """wfb_exec with host buffers switches to the chunked multi-stream H2D/kernel/D2H pipeline for
    large batches; rows from every chunk (first, interior, last, ragged tail) must still be right."""
    n = 1024
    batch = 65536 + 3                       # 256 MiB per plane -> several 32 MiB chunks + ragged tail
    rng = np.random.default_rng(11)
    ctx = wf.createFFTf32Split(n, batch=batch)
    re, im = ctx.getRealBuffer().reshape(batch, n), ctx.getImagBuffer().reshape(batch, n)
    rows = [0, 1, 8191, 8192, 8193, 30000, batch - 4, batch - 1]
    src = {}
    re[:] = 0.0
    im[:] = 0.0
    for r in rows:
        src[r] = (rng.uniform(-1, 1, n).astype(np.float32), rng.uniform(-1, 1, n).astype(np.float32))
        re[r], im[r] = src[r]
    ctx.forward()
    for r in rows:
        er, ei = oracle.fft_split_f32(*src[r])
        assert rel_err(np.r_[re[r], im[r]], np.r_[er, ei], np.r_[src[r][0], src[r][1]]) <= f32_bound(n), r
    assert not re[2].any() and not im[40000].any()          # untouched rows stay zero
    ctx.inverse()
    for r in rows:
        assert np.max(np.abs(re[r] - src[r][0])) < 1e-4 and np.max(np.abs(im[r] - src[r][1])) < 1e-4
    ctx.dispose()
    # real transform: different input / output row strides through the same pipeline
    n = 4096
    batch = 20000 + 1
    rc = wf.createRFFTf32(n, batch=batch)
    t, s = rc.getInputBuffer().reshape(batch, n), rc.getOutputBuffer().reshape(batch, n + 2)
    t[:] = 0.0
    rows = [0, 2047, 2048, 9999, batch - 1]
    xs = {r: rng.uniform(-1, 1, n).astype(np.float32) for r in rows}
    for r in rows:
        t[r] = xs[r]
    rc.forward()
    for r in rows:
        assert rel_err(s[r], oracle.rfft_split_f32(xs[r]), xs[r]) <= f32_bound(n), r
    rc.inverse()
    for r in rows:
        assert np.max(np.abs(t[r] - xs[r])) < 1e-4
    rc.dispose()


def test_exec_device_misaligned_pointers_fall_back(wf, oracle):
    """Caller-supplied device pointers that are only 4- or 8-byte aligned must not reach the TMA /
    128-bit kernels: the plan serves them with the direct variant (same results)."""
    import torch
    C = wf._cabi
    n, batch = 1024, 33
    rng = np.random.default_rng(5)
    re = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
    im = rng.uniform(-1, 1, (batch, n)).astype(np.float32)
    dev = torch.device("cuda:0")
    pad = 1                                              # one float: 4-byte aligned, not 16
    d_re = torch.zeros(batch * n + 8, device=dev)
    d_im = torch.zeros(batch * n + 8, device=dev)
    o_re, o_im = torch.zeros_like(d_re), torch.zeros_like(d_im)
    d_re[pad:pad + batch * n] = torch.from_numpy(re.ravel()).to(dev)
    d_im[pad:pad + batch * n] = torch.from_numpy(im.ravel()).to(dev)
    plan = wf.Plan(C.C2C, C.F32, C.SPLIT, n, batch, 0, C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS)
    torch.cuda.synchronize()      # torch filled the inputs on ITS stream; the plan's stream is non-blocking
    assert "pipe" in plan.variants()[0]                  # the default would be a TMA kernel
    plan.exec_device(C.FORWARD, (d_re.data_ptr() + 4 * pad, d_im.data_ptr() + 4 * pad),
                     (o_re.data_ptr() + 4 * pad, o_im.data_ptr() + 4 * pad))
    plan.sync()
    gr = o_re[pad:pad + batch * n].cpu().numpy().reshape(batch, n)
    gi = o_im[pad:pad + batch * n].cpu().numpy().reshape(batch, n)
    for r in (0, 16, batch - 1):
        er, ei = oracle.fft_split_f32(re[r], im[r])
        assert rel_err(np.r_[gr[r], gi[r]], np.r_[er, ei], np.r_[re[r], im[r]]) <= f32_bound(n)
    assert float(o_re[0]) == 0.0 and float(o_re[pad + batch * n]) == 0.0     # nothing written outside
    plan.destroy()


MISALIGNED = [(kind, n) for kind, sizes in (("c2c f32 split", (16, 512, 8192)), ("c2c f32 interleaved", (16, 512, 8192)),
                                             ("c2c f64", (16, 512, 8192)), ("r2c f32", (16, 1024, 16384)),
                                             ("r2c f64", (16, 1024, 16384))) for n in sizes]


@pytest.mark.parametrize("kind,n", MISALIGNED)
def test_exec_device_misaligned_pointers_per_kind(wf, oracle, kind, n):
    """Caller pointers off the 16-byte grid by one scalar or one complex value, in every kind and both directions.  Split
    c2c is served one scalar off (the direct kernel reads scalars); interleaved c2c and r2c / c2r are served one complex
    value off (8 bytes in f32: the direct kernel; 16 bytes in f64: every variant) and refuse one scalar off with
    WFB_ERR_BAD_ARG, leaving the output untouched.  A served call matches the oracle on every row and writes nothing
    outside its output rows."""
    import torch
    C = wf._cabi
    dev = torch.device("cuda:0")
    f64, real, split = "f64" in kind, kind.startswith("r2c"), "split" in kind
    dt, tdt, elem = (np.float64, torch.float64, 8) if f64 else (np.float32, torch.float32, 4)
    batch, guard = 33, 4096                                   # guard: scalars before and after, a multiple of 16 bytes
    plan = wf.Plan(C.R2C if real else C.C2C, C.F64 if f64 else C.F32, C.SPLIT if split else C.INTERLEAVED, n, batch, 0,
                   C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS)
    rng = np.random.default_rng(n + 31)
    for direction in (C.FORWARD, C.INVERSE):
        inv = direction == C.INVERSE
        li, lo = ((n + 2, n) if inv else (n, n + 2)) if real else ((n, n) if split else (2 * n, 2 * n))
        x = [rng.uniform(-1, 1, (batch, li)).astype(dt) for _ in range(2 if split else 1)]
        for r in range(batch):
            if split:
                want = np.concatenate(oracle.fft_split_f32(x[0][r], x[1][r], inv))
            elif not real:
                want = (oracle.fft_f64 if f64 else oracle.fft_interleaved_f32)(x[0][r], inv)
            elif inv:
                want = (oracle.irfft_f64 if f64 else oracle.irfft_split_f32)(x[0][r])
            else:
                want = (oracle.rfft_f64 if f64 else oracle.rfft_split_f32)(x[0][r])
            if r == 0:
                ref = np.empty((batch, want.size))
            ref[r] = want
        for off, served in ((1, True),) if split else ((1, False), (2, True)):     # scalars off the 16-byte grid
            ins, outs = [], []
            for p in x:
                t = torch.zeros(2 * guard + batch * li, dtype=tdt, device=dev)
                t[guard + off:guard + off + batch * li] = torch.from_numpy(p.ravel()).to(dev)
                o = torch.empty(2 * guard + batch * lo, dtype=tdt, device=dev)
                o.view(torch.int32).fill_(0x5AA5C33C)
                o[guard + off:guard + off + batch * lo] = float("nan")
                ins.append(t)
                outs.append(o)
            before = [o.clone() for o in outs]
            at = lambda ts: tuple(t.data_ptr() + (guard + off) * elem for t in ts) + (None,) * (2 - len(ts))
            torch.cuda.synchronize()      # torch filled the buffers on ITS stream; the plan's stream is non-blocking
            tag = (kind, n, "inverse" if inv else "forward", f"{off * elem} bytes off")
            if not served:
                with pytest.raises(wf.WatFFTError) as e:
                    plan.exec_device(direction, at(ins), at(outs))
                assert e.value.code == C.ERR_BAD_ARG, tag
                plan.sync()
                assert all(torch.equal(o.view(torch.int32), b.view(torch.int32)) for o, b in zip(outs, before)), tag
                continue
            plan.exec_device(direction, at(ins), at(outs))
            plan.sync()
            for o, b in zip(outs, before):
                assert torch.equal(o[:guard + off].view(torch.int32), b[:guard + off].view(torch.int32)), (tag, "wrote before")
                assert torch.equal(o[guard + off + batch * lo:].view(torch.int32), b[guard + off + batch * lo:].view(torch.int32)), (tag, "wrote after")
            got = np.concatenate([o[guard + off:guard + off + batch * lo].cpu().numpy().reshape(batch, lo) for o in outs], axis=1)
            xin = np.concatenate(x, axis=1)
            for r in range(batch):
                assert rel_err(got[r], ref[r], xin[r]) <= (f64_bound(n) if f64 else f32_bound(n)), (tag, r)
    plan.destroy()
