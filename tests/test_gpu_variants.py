"""Every registered kernel variant of every plan, at every supported size, in every operation it has.

A plan holds all variants of its (kind, precision, layout, core size); each one is selectable (wfb_plan_set_variant) and
describes its launch as data (threads, rows per work item, shared memory, persistent flag), so a wrong record in one
variant shows only where that variant runs.  Per plan, every variant index runs:

* at batch 1 and at an odd batch of a few dozen rows (a ragged last tile, the packed-lane tail), every row against the
  CPU oracle at the north-star bound and against the f64 DFT (numpy) at the Taylor-twiddle level (relative to the
  time-domain row's norm in both real directions);
* the persistent variants also on a device-resident batch of about three tiles per resident CTA plus an odd remainder
  (tile claims from the counter, refill / drain of the stage buffers), sampled rows against both references;
* outputs pre-filled with NaN (a row never written cannot pass), guard regions of more than one tile before and after
  every output with a fixed bit pattern (a ragged tile stored whole would overwrite them), inputs bitwise unchanged;
* in place (the contexts' call shape): c2c at both small batches, r2c / c2r at batch 1, bitwise equal to out of place;
* c2r rows with garbage in Im X[0] and Im X[N/2], which the contract ignores: bitwise equal to the same row without;
* 2^k x gives bitwise 2^k F(x) (adds, multiplies and FMAs against fixed tables commute with exact scaling);
* f32: rows scaled by 2^-120, where twiddle products fall below 2^-126, against the oracle (IEEE subnormals): a kernel
  that flushes subnormals to zero misses the bound by an order of magnitude."""
import ctypes

import numpy as np
import pytest

from conftest import f32_bound, f64_bound

pytestmark = pytest.mark.gpu

C2C_SIZES = [1 << k for k in range(2, 14)]       # 4 .. 8192: wfb_size_range of every c2c plan (asserted below)
R2C_SIZES = [1 << k for k in range(3, 15)]       # 8 .. 16384
SMALL = 37                                       # odd, > 32: a ragged last tile for every variant
TARGET_BYTES = 96 << 20        # large batch, as test_gpu_multitile.py: >= 3 tiles of 16-32 KB for each of the <= 1776 resident CTAs
SAMPLES = 24                   # random rows of the large batch checked against the references (plus both ends and the middle)
GUARD_BITS = 0x5AA5C33C        # guard pattern (as float32: a large finite number; never a kernel output)
F64_DFT = 2e-9                 # f64 against the true DFT: the reference's Taylor-series f64 twiddles are good to ~6.5e-11
GARBAGE = (123.0, -77.0)       # Im X[0], Im X[N/2] of the c2r rows that carry garbage there

_worst = {}                    # (family, reference) -> worst error as a fraction of its bound, over the session


def _torch():
    import torch
    return torch, torch.device("cuda:0")


def _persistent(name):
    return "pipe" in name or "rpf" in name


class Family:
    """(kind, precision, layout) of a plan: row shapes, host references and the bounds of its checks."""

    def __init__(self, C, kind, precision, layout):
        self.C, self.kind, self.precision, self.layout = C, kind, precision, layout
        self.f64 = precision == C.F64
        self.dtype = np.float64 if self.f64 else np.float32
        self.real = kind == C.R2C
        self.split = not self.real and layout == C.SPLIT
        self.name = ("r2c" if self.real else "c2c") + (" f64" if self.f64 else " f32") + \
            ("" if self.real else " split" if self.split else " interleaved")
        self.ops = (("r2c", C.FORWARD), ("c2r", C.INVERSE)) if self.real else (("fwd", C.FORWARD), ("inv", C.INVERSE))
        self.bound = f64_bound if self.f64 else f32_bound
        self.dft_bound = (lambda n: F64_DFT) if self.f64 else (lambda n: 4 * f32_bound(n))
        self.scale_k = 200 if self.f64 else 20

    def row_lens(self, op, n):
        """per plane: (input row length, output row length) in scalars"""
        if self.real:
            return (n, n + 2) if op == "r2c" else (n + 2, n)
        return (n, n) if self.split else (2 * n, 2 * n)

    def planes(self):
        return 2 if self.split else 1

    def host_inputs(self, op, n, rows, rng):
        """input planes [rows, len] of the small batches; c2r rows come in pairs, the odd one with garbage in Im X[0], Im X[N/2]"""
        if not self.real:
            z = rng.uniform(-1, 1, (rows, 2 * n)).astype(self.dtype)
            return [z[:, :n].copy(), z[:, n:].copy()] if self.split else [z]
        if op == "r2c":
            return [rng.uniform(-1, 1, (rows, n)).astype(self.dtype)]
        s = np.fft.rfft(rng.uniform(-1, 1, (rows, n)), axis=-1)
        il = np.empty((rows, n + 2))
        il[:, 0::2], il[:, 1::2] = s.real, s.imag
        il = il.astype(self.dtype)
        for r in range(1, rows, 2):
            il[r] = il[r - 1]
            il[r, 1], il[r, n + 1] = GARBAGE
        return [il]

    def oracle_rows(self, oracle, op, n, planes):
        """the CPU restatement, row by row; rows are returned as the planes concatenated"""
        inv = op in ("inv", "c2r")
        out = []
        for r in range(planes[0].shape[0]):
            if self.split:
                o = np.concatenate(oracle.fft_split_f32(planes[0][r], planes[1][r], inv))
            elif not self.real:
                o = (oracle.fft_f64 if self.f64 else oracle.fft_interleaved_f32)(planes[0][r], inv)
            elif op == "r2c":
                o = (oracle.rfft_f64 if self.f64 else oracle.rfft_split_f32)(planes[0][r])
            else:
                o = (oracle.irfft_f64 if self.f64 else oracle.irfft_split_f32)(planes[0][r])
            out.append(np.asarray(o, np.float64))
        return np.stack(out)

    def dft_rows(self, op, n, planes):
        """the true transform in f64 (numpy), rows as the planes concatenated"""
        p = [np.asarray(a, np.float64) for a in planes]
        if self.real:
            if op == "r2c":
                s = np.fft.rfft(p[0], axis=-1)
                o = np.empty((p[0].shape[0], n + 2))
                o[:, 0::2], o[:, 1::2] = s.real, s.imag
                return o
            s = p[0][:, 0::2] + 1j * p[0][:, 1::2]
            s[:, 0], s[:, -1] = s[:, 0].real, s[:, -1].real           # the imaginary parts of DC and Nyquist are ignored
            return np.fft.irfft(s, n=n, axis=-1)
        z = p[0] + 1j * p[1] if self.split else p[0][:, 0::2] + 1j * p[0][:, 1::2]
        z = np.fft.ifft(z, axis=-1) if op == "inv" else np.fft.fft(z, axis=-1)
        if self.split:
            return np.concatenate([z.real, z.imag], axis=1)
        o = np.empty((z.shape[0], 2 * n))
        o[:, 0::2], o[:, 1::2] = z.real, z.imag
        return o


def _row_errors(got, ref, x):
    """max |got - ref| / ||x||_2 per row"""
    x = np.asarray(x, np.float64)
    return np.max(np.abs(np.asarray(got, np.float64) - ref), axis=1) / np.maximum(np.linalg.norm(x, axis=1), 1e-300)


class Guarded:
    """A device array of `rows` rows of `row_len` scalars with guard regions of more than one tile on both sides, filled
    with GUARD_BITS; `body` is the array itself (16-byte aligned: the guards are whole 256-byte blocks)."""

    def __init__(self, torch, dev, rows, row_len, dtype):
        elem = torch.tensor([], dtype=dtype).element_size()
        gbytes = (max(64 << 10, 4 * row_len * elem) + 255) // 256 * 256
        self.g, self.count, self.torch = gbytes // elem, rows * row_len, torch
        self.t = torch.empty(2 * self.g + self.count, dtype=dtype, device=dev)
        self.t.view(torch.int32).fill_(GUARD_BITS)
        self.body = self.t[self.g:self.g + self.count]

    def ptr(self):
        return self.body.data_ptr()

    def guards_intact(self):
        T = self.torch
        return bool(T.all(self.t[:self.g].view(T.int32) == GUARD_BITS)) and \
            bool(T.all(self.t[self.g + self.count:].view(T.int32) == GUARD_BITS))


def _ptrs(bufs):
    return tuple(b.data_ptr() if hasattr(b, "data_ptr") else b.ptr() for b in bufs) + (None,) * (2 - len(bufs))


def _launch(torch, plan, direction, ins, outs):
    torch.cuda.synchronize()      # torch filled the buffers on ITS stream; the plan's stream is non-blocking
    plan.exec_device(direction, _ptrs(ins), _ptrs(outs))
    plan.sync()


def _run_oop(torch, dev, fam, plan, op, direction, n, rows, d_in, tag):
    """out-of-place launch into NaN-poisoned, guarded outputs; checks guards, poison and the untouched input.
    Returns the output planes (device) as one [rows, sum of row lengths] host-comparable tensor list."""
    li, lo = fam.row_lens(op, n)
    outs = [Guarded(torch, dev, rows, lo, d_in[0].dtype) for _ in d_in]
    for o in outs:
        o.body.fill_(float("nan"))
    before = [t.clone() for t in d_in]
    _launch(torch, plan, direction, d_in, outs)
    for o in outs:
        assert o.guards_intact(), (tag, "wrote outside its output rows")
        assert not bool(torch.isnan(o.body).any()), (tag, "left output rows unwritten (NaN poison)")
    assert all(torch.equal(a, b) for a, b in zip(before, d_in)), (tag, "changed its out-of-place input")
    return [o.body.view(rows, lo) for o in outs]


def _check(fam, op, n, got, ref_o, ref_t, x, tag):
    """rows against the oracle and the true DFT; records the worst fraction of each bound.  Errors are relative to the
    input's norm, except for c2r: there they are relative to the time-domain row's (the output's), like r2c's.  (The
    half spectrum's norm is sqrt(N/2) times larger: against it f64 c2r could not tell the Taylor-series pre-process
    twiddles from correctly rounded ones.)"""
    x = ref_o if op == "c2r" else x
    eo = float(np.max(_row_errors(got, ref_o, x))) / fam.bound(n)
    et = float(np.max(_row_errors(got, ref_t, x))) / fam.dft_bound(n)
    assert eo <= 1.0, (tag, "oracle", eo)
    assert et <= 1.0, (tag, "dft", et)
    for key, e in (((fam.name, "oracle"), eo), ((fam.name, "dft"), et)):
        _worst[key] = max(_worst.get(key, 0.0), e)


def _cat(planes):
    return np.concatenate([p.cpu().numpy() if hasattr(p, "cpu") else p for p in planes], axis=1)


def _small_batch(oracle, fam, n, rng):
    """host inputs and references of the small batches (batch 1 runs row 0), once per plan: every variant gets the same"""
    small = {}
    for op, _ in fam.ops:
        planes = fam.host_inputs(op, n, SMALL, rng)
        entry = {"in": planes, "oracle": fam.oracle_rows(oracle, op, n, planes), "dft": fam.dft_rows(op, n, planes)}
        if not fam.f64:
            tiny = [p * np.float32(2.0 ** -120) for p in planes]
            entry["tiny"], entry["tiny_oracle"] = tiny, fam.oracle_rows(oracle, op, n, tiny)
        small[op] = entry
    return small


def _run_plan(wf, oracle, fam, n):
    torch, dev = _torch()
    C = wf._cabi
    lo_n, hi_n = ctypes.c_int(), ctypes.c_int()
    C.check(C.lib().wfb_size_range(fam.kind, fam.precision, fam.layout, lo_n, hi_n))
    sizes = R2C_SIZES if fam.real else C2C_SIZES
    assert (lo_n.value, hi_n.value) == (sizes[0], sizes[-1]), ("the size list must cover wfb_size_range", fam.name)
    flags = C.PLAN_NO_HOST_BUFFERS | C.PLAN_NO_DEVICE_BUFFERS
    rng = np.random.default_rng(n * 7 + fam.kind * 3 + fam.precision + 5 * fam.layout)
    small = _small_batch(oracle, fam, n, rng)

    plans = {b: wf.Plan(fam.kind, fam.precision, fam.layout, n, b, 0, flags) for b in (1, SMALL)}
    names = plans[SMALL].variants()
    count = C.lib().wfb_plan_variant_count(plans[SMALL]._p)
    assert names and plans[1].variants() == names
    ran = []
    for vi, vn in enumerate(names):
        for b in (1, SMALL):
            plans[b].set_variant(vi)
        for op, direction in fam.ops:
            ref = small[op]
            li, lo = fam.row_lens(op, n)
            for b in (1, SMALL):
                tag = (fam.name, n, vn, op, f"batch {b}")
                d_in = [torch.from_numpy(np.ascontiguousarray(p[:b])).to(dev).reshape(-1) for p in ref["in"]]
                out = _run_oop(torch, dev, fam, plans[b], op, direction, n, b, d_in, tag)
                got = _cat(out)
                _check(fam, op, n, got, ref["oracle"][:b], ref["dft"][:b], _cat([p[:b] for p in ref["in"]]), tag)
                if op == "c2r" and b > 1:          # Im X[0], Im X[N/2] are ignored: odd rows equal the even rows bitwise
                    assert np.array_equal(got[1::2], got[0:b - 1:2]), (tag, "c2r read Im X[0] or Im X[N/2]")
                if not fam.real or b == 1:        # in place, bitwise equal to out of place
                    bufs = [Guarded(torch, dev, b, max(li, lo), d_in[0].dtype) for _ in d_in]
                    for g, t in zip(bufs, d_in):
                        g.body.view(b, -1)[:, :li].copy_(t.view(b, li))
                    _launch(torch, plans[b], direction, bufs, bufs)
                    for g, o in zip(bufs, out):
                        assert g.guards_intact(), (tag, "in place: wrote outside its rows")
                        assert torch.equal(g.body.view(b, -1)[:, :lo], o), (tag, "in place differs from out of place")
                if b == SMALL:
                    for k in (fam.scale_k, -fam.scale_k):    # exact power-of-two scaling
                        s = 2.0 ** k
                        o2 = _run_oop(torch, dev, fam, plans[b], op, direction, n, b, [t * s for t in d_in], tag + (f"2^{k}",))
                        assert all(torch.equal(a, c * s) for a, c in zip(o2, out)), (tag, f"F(2^{k} x) != 2^{k} F(x) bitwise")
                    if not fam.f64:                  # subnormal twiddle products: no flush to zero
                        tin = [torch.from_numpy(p).to(dev).reshape(-1) for p in ref["tiny"]]
                        o3 = _cat(_run_oop(torch, dev, fam, plans[b], op, direction, n, b, tin, tag + ("2^-120",)))
                        tx = ref["tiny_oracle"] if op == "c2r" else _cat(ref["tiny"])
                        e = float(np.max(_row_errors(o3, ref["tiny_oracle"], tx))) / fam.bound(n)
                        assert e <= 1.0, (tag, "2^-120 rows against the oracle (flush to zero?)", e)
                        _worst[(fam.name, "oracle 2^-120")] = max(_worst.get((fam.name, "oracle 2^-120"), 0.0), e)
        ran.append(vi)
    for p in plans.values():
        p.destroy()

    # the persistent variants on a device-resident batch of several tiles per resident CTA, with a ragged last tile
    pers = [vi for vi, vn in enumerate(names) if _persistent(vn)]
    if pers:
        li0 = fam.row_lens(fam.ops[0][0], n)[0]
        batch = TARGET_BYTES // (li0 * fam.planes() * np.dtype(fam.dtype).itemsize) + 3
        tdt = torch.float64 if fam.f64 else torch.float32
        g = torch.Generator(device=dev)
        g.manual_seed(5000 + n)
        rows = sorted({0, 1, batch // 2, batch - 2, batch - 1} | set(rng.integers(0, batch, SAMPLES).tolist()))
        idx = torch.tensor(rows, device=dev)
        plan = wf.Plan(fam.kind, fam.precision, fam.layout, n, batch, 0, flags)
        assert plan.variants() == names
        for op, direction in fam.ops:
            li, lo = fam.row_lens(op, n)
            d_in = [torch.rand(batch * li, device=dev, generator=g, dtype=tdt) * 2 - 1 for _ in range(fam.planes())]
            host = [t.view(batch, li)[idx].cpu().numpy() for t in d_in]
            ref_o, ref_t = fam.oracle_rows(oracle, op, n, host), fam.dft_rows(op, n, host)
            for vi in pers:
                plan.set_variant(vi)
                tag = (fam.name, n, names[vi], op, f"batch {batch}")
                out = _run_oop(torch, dev, fam, plan, op, direction, n, batch, d_in, tag)
                _check(fam, op, n, _cat([o[idx] for o in out]), ref_o, ref_t, _cat(host), tag)
                del out
            del d_in
        plan.destroy()
        torch.cuda.empty_cache()
    assert ran == list(range(count)), ("every registered variant index runs", ran, count)
    print(f"\n{fam.name} N={n}: {len(ran)} of {len(names)} variants ran ({len(pers)} persistent, also at the large batch): "
          + ", ".join(names))
    print("  worst so far, as a fraction of the bound: "
          + "; ".join(f"{k[0]} {k[1]} {v:.3f}" for k, v in sorted(_worst.items()) if k[0] == fam.name))


@pytest.mark.parametrize("layout", ["split", "interleaved"])
@pytest.mark.parametrize("n", C2C_SIZES)
def test_c2c_f32_all_variants(wf, oracle, n, layout):
    C = wf._cabi
    _run_plan(wf, oracle, Family(C, C.C2C, C.F32, C.SPLIT if layout == "split" else C.INTERLEAVED), n)


@pytest.mark.parametrize("n", C2C_SIZES)
def test_c2c_f64_all_variants(wf, oracle, n):
    C = wf._cabi
    _run_plan(wf, oracle, Family(C, C.C2C, C.F64, C.INTERLEAVED), n)


@pytest.mark.parametrize("n", R2C_SIZES)
def test_real_f32_all_variants(wf, oracle, n):
    C = wf._cabi
    _run_plan(wf, oracle, Family(C, C.R2C, C.F32, 0), n)


@pytest.mark.parametrize("n", R2C_SIZES)
def test_real_f64_all_variants(wf, oracle, n):
    C = wf._cabi
    _run_plan(wf, oracle, Family(C, C.R2C, C.F64, 0), n)
