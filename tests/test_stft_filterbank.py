"""Filterbank (mel) spectrograms: wfb_stft_create_filterbank, Spectrogram(mode="filterbank"), mel_filterbank and
melSpectrogram.

CPU: mel_filterbank against torchaudio's melscale_fbanks, the f64 reference (filterbank_reference.py) against
torchaudio's MelSpectrogram and its bound against the oracle's own f32 transform, and every argument rule of the ABI.
GPU: every route (direct, span, pipe) at N = 64 ... 8192 at every frame and filter against the f64 reference, and
tightly against the filter product of the same route's complex output; filter shapes; batches bit-for-bit equal to
their single-signal runs; the kernel each route runs; device pointers; repeatability.

FB_F64_REPORT=<file> writes the worst error per route x flavour, as a fraction of its bound, as JSON."""
import ctypes
import json
import math
import os

import numpy as np
import pytest

import oracle as om
from filterbank_reference import bands, check, check_self, filterbank_f64, log_scale
from test_stft_f64 import MATRIX, _ns, _route, _signals

SR = 16000
# flavour -> (power, log, logOffset, logFloor)
FLAVOURS = {
    "p2_linear": (2, None, 0.0, 1e-10),
    "p1_linear": (1, None, 0.0, 1e-10),
    "p2_ln": (2, "ln", 0.0, 1e-10),
    "p1_log10": (1, "log10", 1e-6, 1e-10),
    "p2_log10": (2, "log10", 0.0, 1e-10),
    "p2_db": (2, "db", 0.0, 1e-10),
    "p1_db": (1, "db", 0.0, 1e-5),
}

_worst = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("FB_F64_REPORT")
    if path and _worst:
        with open(path, "w") as f:
            json.dump({k: round(v, 4) for k, v in sorted(_worst.items())}, f, indent=1)


def _record(key, ratio):
    _worst[key] = max(_worst.get(key, 0.0), ratio)


def _mel(wf, n_fft, n_mels=None, **kw):
    bins = n_fft // 2 + 1
    return wf.mel_filterbank(n_fft, SR, n_mels or min(80, bins - 1), **kw)


def _run(wf, x, n_fft, hop, filters, flavour, window="hann", zp=1, mode="filterbank"):
    power, log, off, floor = FLAVOURS[flavour]
    batch = x.shape[0] if x.ndim == 2 else None
    kw = dict(filters=filters, power=power, log=log, logOffset=off, logFloor=floor) if mode == "filterbank" else {}
    sp = wf.Spectrogram(x.shape[-1], n_fft, hop, window, zp, mode=mode, batch=batch, **kw)
    try:
        sp.getInputBuffer()[:] = x
        sp.run()
        return sp.getOutputBuffer().copy()
    finally:
        sp.dispose()


def _check(got, x, n_fft, hop, filters, flavour, window="hann", zp=1):
    power, log, off, floor = FLAVOURS[flavour]
    kw = dict(power=power, scale=log_scale(log, power), offset=off, floor=floor)
    if x.ndim == 1:
        return check(got, x, filters, n_fft, hop, window, zp, **kw)
    return max(check(got[b], x[b], filters, n_fft, hop, window, zp, **kw) for b in range(x.shape[0]))


def _check_self(got, spectra, filters, flavour):
    power, log, off, floor = FLAVOURS[flavour]
    kw = dict(power=power, scale=log_scale(log, power), offset=off, floor=floor)
    g, s = got.reshape((-1,) + got.shape[-1:]), spectra.reshape((-1,) + spectra.shape[-2:])
    return check_self(g, s, filters, **kw)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ------------------------------------------------------------------ CPU: mel filters and the reference
@pytest.mark.parametrize("scale", ["htk", "slaney"])
@pytest.mark.parametrize("norm", [None, "slaney"])
@pytest.mark.parametrize("n_fft,sr,n_mels,f_min,f_max", [(512, 16000, 40, 0.0, None), (1024, 22050, 80, 20.0, 8000.0),
                                                          (2048, 44100, 128, 0.0, 16000.0), (256, 8000, 64, 50.0, 3900.0)])
def test_mel_filterbank_matches_torchaudio(wf, scale, norm, n_fft, sr, n_mels, f_min, f_max):
    torch = pytest.importorskip("torch")
    F = pytest.importorskip("torchaudio.functional")
    ours = wf.mel_filterbank(n_fft, sr, n_mels, f_min, f_max, scale=scale, norm=norm)
    dtype = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)                               # torchaudio's construction, in f64
    try:
        ta = F.melscale_fbanks(n_fft // 2 + 1, f_min, f_max if f_max is not None else sr / 2, n_mels, sr, norm=norm,
                               mel_scale=scale).T.numpy()
    finally:
        torch.set_default_dtype(dtype)
    assert ours.dtype == np.float32 and ours.shape == (n_mels, n_fft // 2 + 1)
    assert np.all(ours >= 0)
    assert np.max(np.abs(ours - ta)) <= 2.0 ** -24 * float(np.abs(ta).max())   # f64 agreement, rounded to f32 once
    with pytest.raises(ValueError):
        wf.mel_filterbank(n_fft, sr, n_mels, scale="bark")
    with pytest.raises(ValueError):
        wf.mel_filterbank(n_fft, sr, n_mels, norm="max")


@pytest.mark.parametrize("power", [1, 2])
@pytest.mark.parametrize("n_fft,hop,window,scale,norm", [(256, 64, "hann", "htk", None), (512, 100, "hamming", "slaney", "slaney"),
                                                         (1024, 256, "blackman", "htk", "slaney")])
def test_reference_matches_torchaudio_melspectrogram(wf, power, n_fft, hop, window, scale, norm):
    torch = pytest.importorskip("torch")
    T = pytest.importorskip("torchaudio.transforms")
    x = _signals(2, 6 * n_fft + 3 * hop + 1, seed=n_fft + power)
    w = torch.from_numpy(om.window_function(window, n_fft).astype(np.float32).astype(np.float64))
    ms = T.MelSpectrogram(SR, n_fft=n_fft, win_length=n_fft, hop_length=hop, n_mels=64, window_fn=lambda n, **k: w,
                          power=float(power), center=False, norm=norm, mel_scale=scale).double()
    t = ms(torch.from_numpy(x.astype(np.float64))).transpose(1, 2).numpy()
    fb = wf.mel_filterbank(n_fft, SR, 64, scale=scale, norm=norm)
    ref = filterbank_f64(x, fb, n_fft, hop, window, power=power)
    assert t.shape == ref.shape
    # torchaudio's filters are f32 values computed in f32: agreement to f32 rounding of the weights
    assert np.max(np.abs(t - ref)) <= 1e-5 * np.max(np.abs(ref))


@pytest.mark.parametrize("n_fft,hop,zp", [(64, 16, 1), (256, 37, 2), (1024, 256, 1), (512, 128, 4)])
def test_reference_bound_holds_for_oracle(wf, oracle, n_fft, hop, zp):
    """The bound holds for the oracle's own f32 transform (its complex output through the f64 filter product), for
    every flavour, with mel filters and with negative weights (linear)."""
    x = _signals(1, 5 * n_fft + 7 * hop + 3, seed=n_fft + hop, amp=20.0)[0]
    x[: n_fft] = 0.0                                                     # silent frames
    rc = om.spectrogram_reference(x, n_fft, hop, "hann", zp, rfft=oracle.rfft_split_f32, complex_out=True)
    mag = np.hypot(rc[..., 0].astype(np.float64), rc[..., 1])
    mel = _mel(wf, n_fft)
    signed = np.random.default_rng(n_fft).standard_normal(mel.shape).astype(np.float32)
    for name, (power, log, off, floor) in FLAVOURS.items():
        for F in (mel, signed) if log is None else (mel,):
            scale = log_scale(log, power)
            v = (mag ** power) @ F.astype(np.float64).T
            got = (scale * np.log2(np.maximum(v + off, floor)) if scale else v).astype(np.float32)
            assert check(got, x, F, n_fft, hop, "hann", zp, power, scale, off, floor) <= 0.5, name


def test_reference_catches_errors(wf):
    n, hop = 256, 64
    x = _signals(1, 4 * n, seed=2)[0]
    F = _mel(wf, n)
    good = filterbank_f64(x, F, n, hop).astype(np.float32)
    assert check(good, x, F, n, hop) <= 1.0
    for f, m, v in ((3, 40, good[3, 40] * 1.001 + 1e-3), (1, 7, np.nan), (0, 9, -1.0)):
        bad = good.copy()
        bad[f, m] = v
        with pytest.raises(AssertionError):
            check(bad, x, F, n, hop)
    dbv = filterbank_f64(x, F, n, hop, scale=log_scale("db", 2)).astype(np.float32)
    check(dbv, x, F, n, hop, scale=log_scale("db", 2))
    dbv[2, 5] += 0.01
    with pytest.raises(AssertionError):
        check(dbv, x, F, n, hop, scale=log_scale("db", 2))
    assert bands(np.array([[0, 1, 0, 2, 0], [0, 0, 0, 0, 0], [3, 0, 0, 0, 4]], np.float32)).tolist() == [[1, 3], [0, 0], [0, 5]]


def test_create_filterbank_argument_checks(wf):
    C = wf._cabi
    lib = C.lib()
    err = ctypes.c_int(0)
    n = 512
    bins = n // 2 + 1
    good = np.ascontiguousarray(_mel(wf, n, 40))

    def create(fft=n, zp=1, hop=128, window=0, ns=16000, batch=1, nf=None, filters=good, power=2, scale=0.0, off=0.0,
               floor=1e-10):
        err.value = 0
        f = None if filters is None else np.ascontiguousarray(filters, np.float32)
        ptr = None if f is None else f.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
        p = lib.wfb_stft_create_filterbank(fft, zp, hop, window, ns, batch, (40 if f is None else f.shape[0]) if nf is None else nf, ptr, power,
                                           scale, off, floor, 0, 0, ctypes.byref(err))
        if p:
            lib.wfb_stft_destroy(p)
        return p

    for fft in (32, 100, 16384):
        assert not create(fft=fft) and err.value == C.ERR_BAD_SIZE
    big = np.zeros((bins + 1, bins), np.float32)
    bad_args = [dict(nf=0), dict(nf=-1), dict(filters=big), dict(filters=None), dict(power=0), dict(power=3),
                dict(scale=math.inf), dict(scale=math.nan), dict(scale=1.0, floor=0.0), dict(scale=1.0, floor=-1.0),
                dict(scale=1.0, floor=math.inf), dict(scale=1.0, floor=math.nan), dict(scale=1.0, off=-1e-3),
                dict(scale=1.0, off=math.inf), dict(scale=1.0, off=math.nan),
                dict(zp=3), dict(zp=n), dict(hop=0), dict(window=5), dict(window=-1), dict(ns=n - 1), dict(batch=0),
                dict(ns=1 << 40, batch=1 << 40)]
    for v in (math.nan, math.inf, -math.inf):
        f = good.copy()
        f[7, 100] = v
        bad_args.append(dict(filters=f))
    for kw in bad_args:
        assert not create(**kw) and err.value == C.ERR_BAD_ARG, kw
    # the input fits (2^52 bytes); the output, 2^10 signals of 2^40 frames of 4097 filters, does not
    assert not create(fft=8192, hop=1, ns=1 << 40, batch=1 << 10, filters=np.ones((4097, 4097), np.float32)) and \
        err.value == C.ERR_BAD_ARG
    # with log_scale 0, floor and offset are not looked at; a valid handle needs a device
    ok = [dict(), dict(scale=0.0, floor=-1.0, off=-5.0), dict(filters=np.ones((bins, bins), np.float32)), dict(power=1),
          dict(scale=-2.0, off=0.0, floor=1e-30), dict(filters=np.zeros((1, bins), np.float32))]
    on_gpu = lib.wfb_device_count() > 0 and lib.wfb_require_b200(0) == 0
    for kw in ok:
        p = create(**kw)
        assert (bool(p) and err.value == C.OK) if on_gpu else (not p and err.value == C.ERR_NO_DEVICE), kw
    assert lib.wfb_stft_filters(None) == 0
    with pytest.raises(ValueError):
        wf.Spectrogram(16000, n, 128, mode="filterbank")                              # no filters
    with pytest.raises(ValueError):
        wf.Spectrogram(16000, n, 128, mode="filterbank", filters=good[:, :-1])        # wrong width
    with pytest.raises(ValueError):
        wf.Spectrogram(16000, n, 128, mode="filterbank", filters=good, log="log2")
    with pytest.raises(ValueError):
        wf.melSpectrogram(np.zeros((2, 3, 4096), np.float32), SR, 256, 64)
    with pytest.raises(ValueError):
        wf.melSpectrogram(np.zeros(100, np.float32), SR, 256, 64)


def test_create_ex_still_rejects_the_filterbank_mode(wf):
    C = wf._cabi
    lib = C.lib()
    err = ctypes.c_int(0)
    for mode in (C.STFT_FILTERBANK, 3, -1):
        assert not lib.wfb_stft_create_ex(1024, 1, 256, 0, 16000, 1, mode, 0.0, 80.0, 0, 0, ctypes.byref(err))
        assert err.value == C.ERR_BAD_ARG


# ------------------------------------------------------------------ GPU: every route against f64
@pytest.mark.gpu
@pytest.mark.parametrize("flavour", list(FLAVOURS))
@pytest.mark.parametrize("n_fft,path", MATRIX)
def test_gpu_fb_matrix(wf, monkeypatch, n_fft, path, flavour):
    """Each route x flavour at every frame and filter: a batch of 3 with a ragged last tile, then one signal at zero
    padding 2 and another window (an odd hop on the direct kernel).  Against the f64 reference and, tightly, against
    the filter product of the same route's complex output."""
    _route(monkeypatch, path)
    i = (64, 128, 256, 512, 1024, 2048, 4096, 8192).index(n_fft)
    mel = _mel(wf, n_fft, scale="slaney" if i % 2 else "htk", norm="slaney" if i % 3 == 0 else None)
    hop = n_fft // 4
    x = _signals(3, _ns(n_fft, hop, 133), seed=n_fft + i)
    got = _run(wf, x, n_fft, hop, mel, flavour)
    assert got.shape == (3, (x.shape[1] - n_fft) // hop + 1, mel.shape[0])
    _record(f"{path}/{flavour}", _check(got, x, n_fft, hop, mel, flavour))
    spectra = _run(wf, x, n_fft, hop, None, flavour, mode="complex")
    _record(f"{path}/{flavour}/self", _check_self(got, spectra, mel, flavour))
    # one signal, zero padding 2, another window
    wsize = n_fft // 2
    hop = wsize // 2 + (path == "direct")
    x = _signals(1, _ns(wsize, hop, 61, mult4=False) + 1, seed=3 * n_fft)[0]
    window = ("hamming", "blackman", "blackmanHarris", "rectangular")[i % 4]
    got = _run(wf, x, n_fft, hop, mel, flavour, window, 2)
    _record(f"{path}/{flavour}", _check(got, x, n_fft, hop, mel, flavour, window, 2))


# ------------------------------------------------------------------ GPU: filter shapes
def _shapes(wf, n_fft):
    bins = n_fft // 2 + 1
    rng = np.random.default_rng(n_fft)
    edges = np.zeros((3, bins), np.float32)
    edges[0, :5] = [1.0, 0.5, 0.0, 0.25, 0.125]                           # touches bin 0 (an interior zero)
    edges[1, -4:] = [0.3, 0.0, 0.7, 1.0]                                 # touches bin M
    edges[2, bins // 2] = 2.0                                             # the middle bin alone
    zero = np.vstack([_mel(wf, n_fft, 8), np.zeros((1, bins), np.float32), _mel(wf, n_fft, 4)])
    return {
        "one": _mel(wf, n_fft, 1),
        "identity": np.eye(bins, dtype=np.float32),                      # num_filters = bins: the power spectrum itself
        "dense": rng.uniform(0.0, 1.0, (3, bins)).astype(np.float32),
        "edges": edges,
        "all_zero": zero,
        "negative": rng.standard_normal((16, bins)).astype(np.float32),
        "mel80": _mel(wf, n_fft, 80),
        "mel128": wf.mel_filterbank(n_fft, SR, 128, scale="slaney", norm="slaney"),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["one", "identity", "dense", "edges", "all_zero", "negative", "mel80", "mel128"])
@pytest.mark.parametrize("n_fft,path", [(512, "direct"), (512, "span"), (2048, "span"), (1024, "pipe"), (4096, "direct")])
def test_gpu_filter_shapes(wf, monkeypatch, n_fft, path, shape):
    _route(monkeypatch, path)
    F = _shapes(wf, n_fft)[shape]
    hop = n_fft // 4
    x = _signals(2, _ns(n_fft, hop, 37), seed=n_fft + len(shape))
    x[1, : 3 * n_fft] = 0.0                                              # silent frames
    flavours = ("p2_linear", "p1_linear") if shape == "negative" else ("p2_linear", "p1_db", "p2_log10", "p2_ln")
    for flavour in flavours:
        got = _run(wf, x, n_fft, hop, F, flavour)
        _record(f"{path}/{flavour}", _check(got, x, n_fft, hop, F, flavour))
        spectra = _run(wf, x, n_fft, hop, None, flavour, mode="complex")
        _check_self(got, spectra, F, flavour)
        if shape == "all_zero":
            power, log, off, floor = FLAVOURS[flavour]
            expect = np.float32(log_scale(log, power) * math.log2(max(off, floor))) if log else 0.0
            assert np.all(got[..., 8] == expect), (flavour, np.unique(got[..., 8]))
        if shape == "identity" and flavour == "p2_linear":
            s = spectra.astype(np.float64)
            assert np.allclose(got, s[..., 0] ** 2 + s[..., 1] ** 2, rtol=4 * 2.0 ** -24, atol=0)


# ------------------------------------------------------------------ GPU: batches
FB_BATCH = [(64, 16, 3), (256, 64, 3), (1024, 256, 3), (2048, 512, 3), (8192, 2048, 3), (1024, 100, 5)]


@pytest.mark.gpu
@pytest.mark.parametrize("mod4", [0, 1, 2, 3])
@pytest.mark.parametrize("n_fft,hop,batch", FB_BATCH)
def test_gpu_batch_rows_equal_single(wf, monkeypatch, n_fft, hop, batch, mod4):
    """Every row of a batch bit-for-bit its single-signal run on the same kernel: a batch whose num_samples is not a
    multiple of 4 takes the direct kernel, so its single runs are sent there too.  Two runs are bitwise equal."""
    _route(monkeypatch, "default")
    ns = n_fft + 6 * hop + 1
    ns += (mod4 - ns) % 4
    x = _signals(batch, ns, seed=n_fft + hop + mod4)
    x[batch // 2] = 0.0                                                  # a silent clip between loud ones
    x[-1] *= 1e3
    F = _mel(wf, n_fft)
    got = _run(wf, x, n_fft, hop, F, "p2_db")
    again = _run(wf, x, n_fft, hop, F, "p2_db")
    assert np.array_equal(_bits(got), _bits(again))
    if ns % 4 and hop % 4 == 0:
        _route(monkeypatch, "direct")
    single = np.stack([_run(wf, r, n_fft, hop, F, "p2_db") for r in x])
    assert np.array_equal(_bits(got), _bits(single))
    _record("batch/p2_db", _check(got, x, n_fft, hop, F, "p2_db"))


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,path", [(512, "span"), (1024, "span"), (2048, "span"), (256, "direct"), (512, "pipe")])
def test_gpu_many_short_clips(wf, monkeypatch, n_fft, path):
    """4194 clips of a few frames (the speech workload's shape at a smaller length), silent clips among them: every
    clip against the reference and bit-for-bit its own single run (sampled clips)."""
    _route(monkeypatch, path)
    hop = n_fft // 4
    ns = _ns(n_fft, hop, 3)
    x = _signals(4194, ns, seed=n_fft)
    x[::7] = 0.0
    F = _mel(wf, n_fft)
    got = _run(wf, x, n_fft, hop, F, "p2_log10")
    assert got.shape == (4194, 3, F.shape[0])
    expect = np.float32(log_scale("log10", 2) * math.log2(1e-10))
    assert np.all(got[::7] == expect)
    _record(f"{path}/p2_log10", _check(got[:500], x[:500], n_fft, hop, F, "p2_log10"))
    for b in (0, 1, 2000, 4193):
        assert np.array_equal(_bits(got[b]), _bits(_run(wf, x[b], n_fft, hop, F, "p2_log10")))


# ------------------------------------------------------------------ GPU: routing, device pointers, the Python entry
# torch.profiler in a process of its own: in a long pytest process that has already held many profiler sessions it was
# seen to report no CUDA events at all (an empty kernel set on every route while the kernels ran and their outputs were
# right), so the route check runs where the profiler starts fresh
_ROUTES_CHILD = r"""
import json, os, sys
sys.path[:0] = [sys.argv[1], sys.argv[2], os.path.join(sys.argv[2], "oracle")]
import torch
import watfft_b200 as wf
from test_stft_f64 import _kernels_run, _signals
from test_stft_filterbank import _mel, _run
torch.cuda.init()
ran = []
for path, n_fft, hop, ns, batch, nf in json.load(sys.stdin):
    # test_stft_f64._route's settings
    span = {"direct": "0", "span": "1", "pipe": "0"}.get(path)
    pipe = {"direct": str(1 << 30), "pipe": "64"}.get(path)
    for name, value in (("WFB_STFT_SPAN", span), ("WFB_STFT_PIPE_MIN_N", pipe)):
        if value is None:
            os.environ.pop(name, None)
        else:
            os.environ[name] = value
    x = _signals(batch, ns, seed=1)
    ran.append(sorted(_kernels_run(torch, lambda: _run(wf, x, n_fft, hop, _mel(wf, n_fft, nf), "p2_db"))))
print(json.dumps(ran))
"""


@pytest.mark.gpu
def test_gpu_kernel_routing(wf):
    """A filterbank handle runs the kernel a dB handle of the same geometry runs (torch.profiler); with 1 filter the
    span route still takes the span kernel (the narrow-row cases of test_gpu_span_narrow_rows_stay_in_bounds)."""
    import subprocess
    import sys
    from pathlib import Path
    pytest.importorskip("torch")
    sizes = (64, 128, 256, 512, 1024, 2048, 4096, 8192)
    cases = [(p, n, n // 4, _ns(n, n // 4, 40), 3, None, p) for n, p in MATRIX]
    cases += [("default", n, n // 4, _ns(n, n // 4, 40), 3, None,
               "span" if n in (1024, 2048) else "pipe" if n == 8192 else "direct") for n in sizes]
    cases += [("span", n, n // 4, _ns(n, n // 4, 3 * X + 1), 5, 1, "span") for n, X in ((256, 16), (1024, 8), (2048, 4))]
    here = Path(__file__).resolve().parent
    res = subprocess.run([sys.executable, "-c", _ROUTES_CHILD, str(here), str(here.parent)], text=True,
                         input=json.dumps([c[:6] for c in cases]), capture_output=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    ran = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [(c, r) for c, r in zip(cases, ran) if r != [c[6]]]
    assert len(ran) == len(cases) and not wrong, wrong


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 1024, 8192])
def test_gpu_device_pointers(wf, monkeypatch, n_fft):
    """run_device on a caller's stream with the samples at +0 ... +3 floats from 16-byte alignment and the output at
    +0 and +1 float (4-byte aligned: the bulk-copy kernels step aside)."""
    torch = pytest.importorskip("torch")
    _route(monkeypatch, "default")
    C = wf._cabi
    hop, batch = n_fft // 4, 3
    ns = _ns(n_fft, hop, 30)
    x = _signals(batch, ns, seed=n_fft + 1)
    F = _mel(wf, n_fft)
    stream = torch.cuda.Stream()
    power, log, off, floor = FLAVOURS["p2_db"]
    sp = wf.Spectrogram(ns, n_fft, hop, mode="filterbank", filters=F, power=power, log=log, logOffset=off,
                        logFloor=floor, flags=C.PLAN_NO_HOST_BUFFERS, batch=batch)
    shape = (batch, sp.numFrames, F.shape[0])
    out_len = int(np.prod(shape))
    for xo, oo in ((0, 0), (1, 0), (2, 0), (3, 0), (0, 1)):
        with torch.cuda.stream(stream):
            xin = torch.zeros(batch * ns + 4, dtype=torch.float32, device="cuda")
            xin[xo: xo + batch * ns] = torch.from_numpy(x.ravel()).cuda()
            out = torch.full((out_len + 4,), float("nan"), dtype=torch.float32, device="cuda")
        sp.run_device(xin.data_ptr() + 4 * xo, out.data_ptr() + 4 * oo, stream=stream.cuda_stream)
        stream.synchronize()
        o = out.cpu().numpy()
        assert np.isnan(o[:oo]).all() and np.isnan(o[oo + out_len:]).all()
        got = o[oo: oo + out_len].reshape(shape)
        _record("device/p2_db", _check(got, x, n_fft, hop, F, "p2_db"))
    sp.dispose()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 1024, 2048])
def test_gpu_span_narrow_rows_stay_in_bounds(wf, monkeypatch, n_fft):
    """The span kernel's result tile leaves as a bulk store of its 16-byte aligned interior plus plain stores of the
    floats before and after it.  With 1, 2 or 3 filters a ragged last tile can hold fewer floats than lie before the
    next 16-byte boundary: for 5 signals whose last tile has 1 ... 3 rows (so it starts at every output phase), every
    value is checked and NaN guards on both sides of a run_device output stay untouched.  That these geometries take
    the span kernel is checked by test_gpu_kernel_routing."""
    torch = pytest.importorskip("torch")
    C = wf._cabi
    _route(monkeypatch, "span")
    X = {256: 16, 1024: 8, 2048: 4}[n_fft]                              # span frames per tile
    hop, batch = n_fft // 4, 5
    for frames in (3 * X + 1, 3 * X + 2, 3 * X + 3):
        ns = _ns(n_fft, hop, frames)
        x = _signals(batch, ns, seed=n_fft + frames)
        for nf in (1, 2, 3):
            F = _mel(wf, n_fft, nf)
            sp = wf.Spectrogram(ns, n_fft, hop, mode="filterbank", filters=F, flags=C.PLAN_NO_HOST_BUFFERS, batch=batch)
            assert sp.numFrames == frames
            out_len = batch * frames * nf
            xin = torch.from_numpy(x.ravel()).cuda()
            out = torch.full((out_len + 64,), float("nan"), dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()
            sp.run_device(xin.data_ptr(), out.data_ptr() + 4 * 32)      # (16-byte aligned: the span route)
            torch.cuda.synchronize()
            sp.dispose()
            o = out.cpu().numpy()
            assert np.isnan(o[:32]).all() and np.isnan(o[32 + out_len:]).all(), (frames, nf)
            got = o[32: 32 + out_len].reshape(batch, frames, nf)
            _record("span/p2_linear", _check(got, x, n_fft, hop, F, "p2_linear"))


@pytest.mark.gpu
def test_gpu_python_entry_points(wf):
    """melSpectrogram for [T] and [B][T], shaped like generateSpectrogram; the output buffer's shape; no inverse."""
    n_fft, hop = 512, 128
    x = _signals(3, _ns(n_fft, hop, 20), seed=5)
    one = wf.melSpectrogram(x[0], SR, n_fft, hop, nMels=40, log="db")
    many = wf.melSpectrogram(x, SR, n_fft, hop, nMels=40, log="db")
    assert one["data"].shape == (20 * 40,) and many["data"].shape == (3, 20 * 40) and many["batch"] == 3
    assert one["numFrames"] == 20 and one["nMels"] == 40
    assert np.array_equal(_bits(one["data"]), _bits(many["data"][0]))
    F = wf.mel_filterbank(n_fft, SR, 40)
    check(one["data"].reshape(20, 40), x[0], F, n_fft, hop, scale=log_scale("db", 2))
    sp = wf.Spectrogram(x.shape[1], n_fft, hop, mode="filterbank", filters=F, batch=3)
    assert sp.getOutputBuffer().shape == (3, 20, 40) and sp.numFilters == 40
    with pytest.raises(wf.WatFFTError):
        sp.inverse()
    sp.dispose()
    db = wf.Spectrogram(x.shape[1], n_fft, hop)
    assert db.numFilters == 0
    db.dispose()
