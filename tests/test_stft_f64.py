"""Every forward STFT kernel at every frame and bin against the f64 STFT (tests/stft_reference.py).

The kernel matrix: N = 64 ... 8192 x flavour (fast dB, fast dB zero-padded, exact dB, complex) x every kernel that can
run at that N -- direct (k_stft), span (k_stft_span, N >= 256) and pipe (k_stft_pipe; the default at N = 8192, and at
any N with WFB_STFT_PIPE_MIN_N).  Then the edges where kernels go wrong (hops of 1, odd, = window and > window; windows
of 2 and 4 samples; one-frame signals; the span kernel's large-hop fallback; unaligned device pointers; silence, tiny
and huge signals; gain > 0), and the fast/exact dB switch around the floors where the fast form's dropped +1e-10 starts
to show.  Which kernel each case runs is checked with torch.profiler (test_gpu_kernel_routing).

The reference is pinned on the CPU to the oracle's per-frame loop and to torch.stft (the first tests here).

STFT_F64_REPORT=<file> writes the worst error per kernel x flavour, as a fraction of its bound, as JSON."""
import json
import math
import os
import re

import numpy as np
import pytest

import oracle as om
from stft_reference import check, complex_bound, db_f64, db_value, frames_f64, stft_f64

WINDOWS = ("hann", "hamming", "blackman", "blackmanHarris", "rectangular")
SIZES = (64, 128, 256, 512, 1024, 2048, 4096, 8192)
PATHS = ("direct", "span", "pipe")
# flavour -> (mode, zero padding of the first / second configuration, gain, range, amplitude of the loud tone)
FLAVOURS = {
    "fast": ("db", (1, 1), -6.0, 70.0, 1.0),
    "fast_pad": ("db", (2, 4), 6.0, 60.0, 40.0),          # gain > 0: the loud tone clips at 1
    "exact": ("db", (1, 2), -20.0, 200.0, 1.0),
    "complex": ("complex", (1, 4), 0.0, 80.0, 1.0),
}
SWITCH_FLOORS = (-150, -140, -130, -120, -100, -80)
SWITCH_RANGES = (20, 50, 80, 150)

_worst = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("STFT_F64_REPORT")
    if path and _worst:
        with open(path, "w") as f:
            json.dump({k: round(v, 4) for k, v in sorted(_worst.items())}, f, indent=1)


def _record(kernel, flavour, ratio):
    key = f"{kernel}/{flavour}"
    _worst[key] = max(_worst.get(key, 0.0), ratio)


def _exact_db(gain, range_db):
    """Whether the library takes the exact dB form (stft_flavour): where the fast form's dropped +1e-10 would
    lower the output at the floor by more than 1e-6."""
    floor = np.float32(gain) - np.float32(range_db)
    inv_range = float(np.float32(1.0) / np.float32(range_db))
    return 20 * math.log10(1 + 1e-10 * 10 ** (-float(floor) / 20)) * inv_range > 1e-6


def _route(monkeypatch, path):
    """direct: neither bulk-copy kernel; span: WFB_STFT_SPAN=1 (its own fallbacks as by default); pipe: the pipelined
    kernel at every N; default: the library's own choice."""
    span = {"direct": "0", "span": "1", "pipe": "0"}.get(path)
    pipe = {"direct": str(1 << 30), "pipe": "64"}.get(path)
    for name, value in (("WFB_STFT_SPAN", span), ("WFB_STFT_PIPE_MIN_N", pipe)):
        if value is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, value)


def _signals(batch, n, seed, amp=1.0):
    """Two tones (one of amplitude `amp`) and noise per row, rows at different levels."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 16000.0
    f = rng.uniform(200, 6000, (batch, 2))
    x = (amp * np.sin(2 * np.pi * f[:, :1] * t) + 0.3 * np.sin(2 * np.pi * f[:, 1:] * t) +
         0.1 * rng.standard_normal((batch, n)))
    return (x * np.geomspace(1.0, 3.0, batch)[:, None]).astype(np.float32)


def _ns(wsize, hop, frames, mult4=True):
    ns = wsize + (frames - 1) * hop
    return ns + (-ns) % 4 if mult4 else ns


def _run(wf, x, n_fft, hop, window, zp, mode, gain, range_db):
    batch = x.shape[0] if x.ndim == 2 else None
    sp = wf.Spectrogram(x.shape[-1], n_fft, hop, window, zp, gain, range_db, mode=mode, batch=batch)
    try:
        sp.getInputBuffer()[:] = x
        sp.run()
        return sp.getOutputBuffer().copy()
    finally:
        sp.dispose()


def _check_rows(got, x, n_fft, hop, window, zp, mode, gain, range_db):
    if x.ndim == 1:
        return check(got, x, n_fft, hop, window, zp, mode, gain, range_db)
    return max(check(got[b], x[b], n_fft, hop, window, zp, mode, gain, range_db) for b in range(x.shape[0]))


def _run_check(wf, x, n_fft, hop, window, zp, mode, gain, range_db, kernel, flavour):
    got = _run(wf, x, n_fft, hop, window, zp, mode, gain, range_db)
    _record(kernel, flavour, _check_rows(got, x, n_fft, hop, window, zp, mode, gain, range_db))
    return got


# ------------------------------------------------------------------ CPU: the reference, pinned
def _frames_loop(x, n_fft, hop, window, zp):
    """The obvious per-frame loop, for the vectorised form to agree with."""
    wsize = n_fft // zp
    w = om.window_function(window, wsize).astype(np.float32).astype(np.float64)
    frames = (len(x) - wsize) // hop + 1
    return np.stack([np.asarray(x[f * hop: f * hop + wsize], np.float64) * w for f in range(frames)])


@pytest.mark.parametrize("n_fft,hop,zp", [(64, 1, 1), (256, 37, 2), (512, 512, 4), (1024, 1100, 1), (256, 3, 128)])
def test_reference_frames_are_the_loop(n_fft, hop, zp):
    x = _signals(1, 6 * n_fft + 2 * hop + 5, seed=hop)[0]
    for window in WINDOWS:
        assert np.array_equal(frames_f64(x, n_fft, hop, window, zp), _frames_loop(x, n_fft, hop, window, zp))
    # a batch is its rows
    xb = _signals(3, 3 * n_fft + hop, seed=1)
    sb = stft_f64(xb, n_fft, hop, "hann", zp)
    for b in range(3):
        assert np.array_equal(sb[b], stft_f64(xb[b], n_fft, hop, "hann", zp))
    with pytest.raises(ValueError):
        frames_f64(x[: n_fft // zp - 1], n_fft, hop, "hann", zp)


@pytest.mark.parametrize("window", WINDOWS)
@pytest.mark.parametrize("n_fft,hop,zp,gain,range_db", [(64, 16, 1, 0.0, 80.0), (256, 37, 2, -6.0, 70.0),
                                                        (1024, 256, 4, 6.0, 60.0), (512, 100, 1, 0.0, 220.0),
                                                        (256, 64, 16, -20.0, 200.0)])
def test_reference_matches_oracle_loop(oracle, window, n_fft, hop, zp, gain, range_db):
    """The f64 STFT against the oracle's per-frame loop over its f32 transform, every frame: complex within the
    complex bound, dB inside the dB interval -- the same yardsticks the GPU tests use, so this also shows they hold
    for an f32 transform that is not the library's."""
    x = _signals(1, 5 * n_fft + 7 * hop + 3, seed=n_fft + hop, amp=20.0)[0]
    x[: n_fft] = 0.0                                                     # silent frames
    rc = om.spectrogram_reference(x, n_fft, hop, window, zp, rfft=oracle.rfft_split_f32, complex_out=True)
    assert check(rc, x, n_fft, hop, window, zp, "complex") <= 0.5
    rd = om.spectrogram_reference(x, n_fft, hop, window, zp, gain=gain, range_db=range_db, rfft=oracle.rfft_split_f32)
    check(rd, x, n_fft, hop, window, zp, "db", gain, range_db)
    # with an f64 transform the loop IS the reference, up to its f32 roundings of frame, spectrum and magnitude
    def rfft64(p):
        z = np.fft.rfft(np.asarray(p, np.float64))
        return np.stack([z.real, z.imag], -1).ravel()
    ref = stft_f64(x, n_fft, hop, window, zp)
    loop = om.spectrogram_reference(x, n_fft, hop, window, zp, rfft=rfft64, complex_out=True)
    scale = np.linalg.norm(frames_f64(x, n_fft, hop, window, zp), axis=-1)[:, None, None]
    assert np.all(np.abs(loop - ref) <= 1e-6 * scale + 1e-30)
    loop_db = om.spectrogram_reference(x, n_fft, hop, window, zp, gain=gain, range_db=range_db, rfft=rfft64)
    ref_db = db_f64(x, n_fft, hop, window, zp, gain, range_db)
    strong = np.hypot(ref[..., 0], ref[..., 1]) >= 1e-2 * scale[..., 0]     # bins f32 resolves to 1e-5 or better
    assert np.max(np.abs(loop_db - ref_db)[strong]) < 2e-6
    assert check(loop_db, x, n_fft, hop, window, zp, "db", gain, range_db) < 0.1


@pytest.mark.parametrize("window", WINDOWS)
@pytest.mark.parametrize("n_fft,hop", [(64, 1), (256, 37), (1024, 256), (8192, 3000)])
def test_reference_matches_torch_stft(window, n_fft, hop):
    """torch.stft(center=False) in f64, zero padding 1 only: torch centres a window shorter than n_fft, the library pads
    at the end of the frame."""
    torch = pytest.importorskip("torch")
    x = _signals(2, 4 * n_fft + 3 * hop + 1, seed=hop)
    w = torch.from_numpy(om.window_function(window, n_fft).astype(np.float32).astype(np.float64))
    t = torch.stft(torch.from_numpy(x.astype(np.float64)), n_fft, hop_length=hop, win_length=n_fft, window=w,
                   center=False, return_complex=True).transpose(1, 2).numpy()
    ref = stft_f64(x, n_fft, hop, window)
    assert t.shape == ref.shape[:-1]
    scale = np.linalg.norm(frames_f64(x, n_fft, hop, window), axis=-1)[..., None]
    assert np.all(np.abs(t - (ref[..., 0] + 1j * ref[..., 1])) <= 1e-13 * scale)


def test_db_value_and_bounds():
    n = 256
    half = n / 2
    assert db_value(0.0, n, 0.0, 80.0) == 0.0
    assert db_value(half, n, 0.0, 80.0) == 1.0                          # 0 dB at gain 0 is the ceiling
    assert abs(db_value(half * 1e-2, n, 0.0, 80.0) - 40 / 80) < 1e-8
    assert abs(db_value(0.0, n, 0.0, 220.0) - 20 / 220) < 1e-9            # silence sits on the +1e-10
    assert db_value(half * 4, n, 6.0, 60.0) == 1.0 and db_value(half * 1.5, n, 6.0, 60.0) < 1.0
    assert complex_bound(1024) == pytest.approx(8e-5)
    # a wrong bin, a NaN, a value above 1 and a nonzero bin 0 are all caught
    x = _signals(1, 4 * n, seed=2)[0]
    good = db_f64(x, n, 64).astype(np.float32)
    assert check(good, x, n, 64) <= 1.0
    for f, k, v in ((3, 40, good[3, 40] + 1e-3), (1, 7, np.nan), (0, 9, 1.5), (2, 0, 1e-7)):
        bad = good.copy()
        bad[f, k] = v
        with pytest.raises(AssertionError):
            check(bad, x, n, 64)
    c = stft_f64(x, n, 64).astype(np.float32)
    check(c, x, n, 64, mode="complex")
    c[5, 17, 1] += 2 * complex_bound(n) * np.linalg.norm(frames_f64(x, n, 64)[5])
    with pytest.raises(AssertionError):
        check(c, x, n, 64, mode="complex")


def test_fast_db_switch_rule():
    """The fast form stays on at the defaults (gain 0, range 80) and at every floor down to about -99 dB at range 80;
    deeper floors, and floors whose error is large against a small range, take the exact form."""
    assert not _exact_db(0.0, 80.0) and not _exact_db(-6.0, 70.0) and not _exact_db(6.0, 60.0)
    assert not _exact_db(-19.0, 80.0) and _exact_db(-20.0, 80.0)
    assert _exact_db(-20.0, 200.0) and _exact_db(0.0, 220.0)
    assert _exact_db(-100.0, 50.0) and not _exact_db(-30.0, 50.0)
    for floor in SWITCH_FLOORS:
        for r in SWITCH_RANGES:
            dev = 20 * math.log10(1 + 1e-10 * 10 ** (-floor / 20)) / r        # the fast form's error at the floor
            assert _exact_db(floor + r, r) == (dev > 1e-6)


# ------------------------------------------------------------------ GPU: the kernel matrix
MATRIX = [(n, p) for n in SIZES for p in PATHS if p != "span" or n >= 256]


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", list(FLAVOURS))
@pytest.mark.parametrize("n_fft,path", MATRIX)
def test_gpu_kernel_matrix(wf, monkeypatch, n_fft, path, flavour):
    """Each kernel x flavour at every frame and bin: a batch of 3 with a ragged last tile in every persistent kernel, a
    single signal at another window, hop and zero padding (an odd hop on the direct kernel), and 211 clips of 5 frames
    (N <= 2048).  Over the sizes of a kernel each flavour sees all five windows."""
    mode, zps, gain, range_db, amp = FLAVOURS[flavour]
    assert _exact_db(gain, range_db) == (flavour == "exact") or mode == "complex"
    _route(monkeypatch, path)
    i = [n for n in SIZES if path != "span" or n >= 256].index(n_fft)
    # 1. batch 3, num_samples % 4 == 0; 133 frames: not a whole number of tiles of any persistent kernel
    zp = zps[0]
    wsize = n_fft // zp
    hop = wsize // 4
    x = _signals(3, _ns(wsize, hop, 133), seed=n_fft + i, amp=amp)
    got = _run_check(wf, x, n_fft, hop, WINDOWS[i % 5], zp, mode, gain, range_db, path, flavour)
    if gain > 0:
        assert np.any(got == 1.0)
    # 2. one signal, another window and zero padding, hop window/2 (+1, odd, on the direct kernel)
    zp = zps[1]
    wsize = n_fft // zp
    hop = wsize // 2 + (path == "direct")
    x = _signals(1, _ns(wsize, hop, 61, mult4=False) + 1, seed=3 * n_fft, amp=amp)[0]
    _run_check(wf, x, n_fft, hop, WINDOWS[(i + 2) % 5], zp, mode, gain, range_db, path, flavour)
    # 3. 211 clips of 5 frames each: every clip's tile-to-signal mapping
    if n_fft <= 2048:
        zp = zps[0]
        wsize = n_fft // zp
        hop = wsize // 4
        x = _signals(211, _ns(wsize, hop, 5), seed=n_fft, amp=amp)
        _run_check(wf, x, n_fft, hop, WINDOWS[(i + 4) % 5], zp, mode, gain, range_db, path, flavour)


# ------------------------------------------------------------------ GPU: edges
# (id, n_fft, path, hop, zero padding, num_samples, window, batch, the kernel that runs)
def _edge(eid, n_fft, path, hop, zp, frames, window="hann", batch=1, kernel=None, ns=None):
    wsize = n_fft // zp
    ns = ns if ns is not None else _ns(wsize, hop, frames, mult4=batch > 1)
    return pytest.param(n_fft, path, hop, zp, ns, window, batch, kernel or path, id=eid)


EDGES = [
    _edge("hop1", 256, "direct", 1, 1, 3000),
    _edge("hop1-window2", 256, "direct", 1, 128, 500, "hamming"),
    _edge("odd-hop", 512, "direct", 37, 2, 300, "blackman", 3),
    _edge("odd-hop-8192-default", 8192, "default", 2049, 1, 9, "blackmanHarris", kernel="direct"),
    _edge("hop-eq-window", 1024, "direct", 1024, 1, 20, "hamming", 3),
    _edge("hop-gt-window", 2048, "direct", 1037, 2, 20, "blackman"),
    _edge("window4", 1024, "direct", 3, 256, 400, "hann", 3),
    _edge("window2-64", 64, "direct", 3, 32, 100, "hamming"),
    _edge("window2-8192-default", 8192, "default", 2, 4096, 50, "rectangular", kernel="direct"),
    _edge("one-frame", 256, "direct", 64, 1, 1),
    _edge("one-frame-tail", 4096, "direct", 1024, 1, 1, ns=4096 + 1023),
    _edge("span-hop-eq-window", 512, "span", 512, 1, 30, "rectangular", 3),
    _edge("span-hop-gt-window", 1024, "span", 1060, 1, 30, "hann", 3),
    _edge("span-hop4", 256, "span", 4, 1, 500, "blackmanHarris"),
    _edge("span-window4", 256, "span", 4, 64, 300, "hann", 3),
    _edge("span-one-frame", 1024, "span", 256, 1, 1, batch=3),
    _edge("span-one-frame-tail", 2048, "span", 512, 1, 1, ns=2048 + 511),
    _edge("span-big-hop-8192", 8192, "span", 17000, 1, 5),
    _edge("span-fallback-direct", 256, "span", 4096, 1, 6, kernel="direct"),
    _edge("span-fallback-pipe", 8192, "span", 20000, 1, 4, "hamming", 3, kernel="pipe"),
    _edge("pipe-hop-eq-window", 8192, "pipe", 8192, 1, 6, "hann", 3),
    _edge("pipe-hop-gt-window", 8192, "pipe", 4100, 2, 7, "blackman"),
    _edge("pipe-hop4", 128, "pipe", 4, 1, 700, "hamming"),
    _edge("pipe-window4", 512, "pipe", 4, 128, 300, "hann", 3),
    _edge("pipe-one-frame", 8192, "default", 2048, 1, 1, kernel="pipe"),
    _edge("pipe-one-frame-tail", 8192, "default", 2048, 1, 1, ns=8192 + 2047, kernel="pipe"),
    _edge("pipe-one-frame-64", 64, "pipe", 16, 1, 1, batch=3),
]
EDGE_FLAVOURS = {"fast": ("db", -6.0, 70.0), "exact": ("db", -20.0, 200.0), "complex": ("complex", 0.0, 80.0)}


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,path,hop,zp,ns,window,batch,kernel", EDGES)
def test_gpu_edges(wf, monkeypatch, n_fft, path, hop, zp, ns, window, batch, kernel):
    _route(monkeypatch, path)
    x = _signals(batch, ns, seed=ns + hop)
    if batch == 1:
        x = x[0]
    for flavour, (mode, gain, range_db) in EDGE_FLAVOURS.items():
        _run_check(wf, x, n_fft, hop, window, zp, mode, gain, range_db, kernel, flavour + ("_pad" if zp > 1 else ""))


SCALES = [(256, "direct"), (128, "pipe"), (1024, "span"), (1024, "direct"), (8192, "pipe"), (4096, "span")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,path", SCALES)
def test_gpu_levels(wf, monkeypatch, n_fft, path):
    """Exact zeros, a silent stretch inside a signal, signals scaled by 1e-6 (bins at and below the floor) and by 1e4
    (every bin at the ceiling), with gain > 0 and with a floor deep enough that silence sits on the +1e-10."""
    _route(monkeypatch, path)
    hop = n_fft // 4
    ns = _ns(n_fft, hop, 40)
    x = _signals(5, ns, seed=n_fft)
    x[0] = 0.0
    x[1, ns // 3: 2 * ns // 3] = 0.0
    x[2] *= 1e-6
    x[3] *= 1e4
    x[4] *= 1e-3
    # (floor -99 dB at range 80 is the deepest the fast form takes there; -98 dB at range 58 is already too deep)
    for mode, zp, gain, range_db in (("db", 1, 0.0, 80.0), ("db", 2, 6.0, 60.0), ("db", 1, -19.0, 80.0),
                                     ("db", 1, -40.0, 58.0), ("db", 1, 0.0, 220.0), ("db", 2, -60.0, 100.0),
                                     ("complex", 1, 0.0, 80.0), ("complex", 4, 0.0, 80.0)):
        flavour = mode if mode == "complex" else "exact" if _exact_db(gain, range_db) else "fast"
        flavour += "_pad" if zp > 1 else ""
        got = _run_check(wf, x, n_fft, hop, "hann", zp, mode, gain, range_db, path, flavour)
        if mode == "db":
            assert np.mean(got[3][:, 3:] == 1.0) > 0.9                      # 1e4: clipped at the ceiling
            silence = min(max((-200.0 - (gain - range_db)) / range_db, 0.0), 1.0)
            assert np.allclose(got[0][:, 3:], silence, rtol=0, atol=1e-5)   # exact zeros: the +1e-10, or the floor
        else:
            assert np.all(got[0] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 1024, 8192])
def test_gpu_device_pointers(wf, monkeypatch, n_fft):
    """run_device on a caller's stream with the samples at +0 ... +3 floats from 16-byte alignment and the output at +0
    and +2 floats (the latter turns the bulk-copy kernels off): every frame against the reference."""
    torch = pytest.importorskip("torch")
    _route(monkeypatch, "default")
    C = wf._cabi
    hop, batch = n_fft // 4, 3
    ns = _ns(n_fft, hop, 30)
    x = _signals(batch, ns, seed=n_fft + 1)
    stream = torch.cuda.Stream()
    for flavour, mode, gain, range_db in (("fast", "db", 0.0, 80.0), ("exact", "db", -20.0, 200.0),
                                          ("complex", "complex", 0.0, 80.0)):
        sp = wf.Spectrogram(ns, n_fft, hop, "hann", 1, gain, range_db, mode=mode, flags=C.PLAN_NO_HOST_BUFFERS,
                            batch=batch)
        shape = (batch, sp.numFrames, sp.numBins) + ((2,) if mode == "complex" else ())
        out_len = int(np.prod(shape))
        for xo, oo in ((0, 0), (1, 0), (2, 0), (3, 0), (0, 2)):
            with torch.cuda.stream(stream):
                xin = torch.zeros(batch * ns + 4, dtype=torch.float32, device="cuda")
                xin[xo: xo + batch * ns] = torch.from_numpy(x.ravel()).cuda()
                out = torch.full((out_len + 4,), float("nan"), dtype=torch.float32, device="cuda")
            assert xin.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0
            sp.run_device(xin.data_ptr() + 4 * xo, out.data_ptr() + 4 * oo, stream=stream.cuda_stream)
            stream.synchronize()
            o = out.cpu().numpy()
            assert np.isnan(o[:oo]).all() and np.isnan(o[oo + out_len:]).all()
            kernel = "device" if (xo, oo) != (0, 0) else {256: "direct", 1024: "span", 8192: "pipe"}[n_fft]
            _record(kernel, flavour, _check_rows(o[oo: oo + out_len].reshape(shape), x, n_fft, hop, "hann", 1, mode,
                                                 gain, range_db))
        sp.dispose()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,path,frames", [(256, "pipe", 100001), (8192, "default", 3001)])
def test_gpu_pipe_kernel_many_tiles(wf, monkeypatch, n_fft, path, frames):
    """The pipelined persistent kernel with several tiles per resident CTA and a ragged last tile: every frame against
    the reference, and the persistent schedule bitwise repeatable."""
    _route(monkeypatch, path)
    hop = n_fft // 4
    x = _signals(1, _ns(n_fft, hop, frames) + 3, seed=frames)[0]
    for flavour, mode, gain, range_db in (("fast", "db", -3.0, 75.0), ("complex", "complex", 0.0, 80.0)):
        got = _run_check(wf, x, n_fft, hop, "hann", 1, mode, gain, range_db, "pipe", flavour)
        assert got.shape[0] == frames
        again = _run(wf, x, n_fft, hop, "hann", 1, mode, gain, range_db)
        assert np.array_equal(got.view(np.uint32), again.view(np.uint32))


# ------------------------------------------------------------------ GPU: the fast / exact dB switch
@pytest.mark.gpu
@pytest.mark.parametrize("floor", SWITCH_FLOORS)
@pytest.mark.parametrize("n_fft,path", [(256, "direct"), (1024, "span"), (8192, "pipe")])
def test_gpu_fast_exact_switch(wf, monkeypatch, n_fft, path, floor):
    """White noise whose median |X|/(N/2) sits 3 dB above the floor, at ranges 20 ... 150: most bins are within a few dB
    of the floor, where the fast form's dropped +1e-10 is largest.  Every range must land inside the dB interval."""
    _route(monkeypatch, path)
    hop = n_fft // 4
    ns = _ns(n_fft, hop, 40)
    noise = np.random.default_rng(n_fft - floor).standard_normal(ns)
    r = stft_f64(noise, n_fft, hop)
    med = np.median(np.hypot(r[..., 3:, 0], r[..., 3:, 1])) / (n_fft / 2)
    x = (noise * 10 ** ((floor + 3) / 20) / med).astype(np.float32)
    failed = []
    for range_db in SWITCH_RANGES:
        gain = float(floor + range_db)
        got = _run(wf, x, n_fft, hop, "hann", 1, "db", gain, range_db)
        try:
            ratio = check(got, x, n_fft, hop, "hann", 1, "db", gain, range_db)
            _record(path, "exact" if _exact_db(gain, range_db) else "fast", ratio)
        except AssertionError as e:
            failed.append(f"range {range_db} (gain {gain}; the {'exact' if _exact_db(gain, range_db) else 'fast'} form "
                          f"is the one that fits): {e}")
    assert not failed, "\n".join(failed)


# ------------------------------------------------------------------ GPU: which kernel each case runs
def _kernels_run(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    found = {m.group(1) or "" for n in names for m in [re.search(r"k_stft(_span|_pipe)?(?=[<I])", n)] if m}
    return {{"": "direct", "_span": "span", "_pipe": "pipe"}[f] for f in found}


@pytest.mark.gpu
def test_gpu_kernel_routing(wf, monkeypatch):
    """The kernel the matrix and the edges name is the one that runs (kernel names from torch.profiler)."""
    torch = pytest.importorskip("torch")
    torch.cuda.init()
    cases = [(n, p, (n // 4, 1, _ns(n, n // 4, 133), "hann", 3), p) for n, p in MATRIX]
    cases += [(n, "default", (n // 4, 1, _ns(n, n // 4, 20), "hann", 1),
               "span" if n in (1024, 2048) else "pipe" if n == 8192 else "direct") for n in SIZES]
    cases += [(e.values[0], e.values[1], e.values[2:7], e.values[7]) for e in EDGES]
    # a batch whose rows are not 16-byte aligned leaves the bulk-copy kernels
    cases += [(1024, "span", (256, 1, _ns(1024, 256, 9) + 2, "hann", 3), "direct"),
              (8192, "default", (2048, 1, _ns(8192, 2048, 9) + 1, "hann", 3), "direct")]
    wrong = []
    for n_fft, path, (hop, zp, ns, window, batch), kernel in cases:
        _route(monkeypatch, path)
        x = _signals(batch, ns, seed=1)
        x = x if batch > 1 else x[0]
        ran = _kernels_run(torch, lambda: _run(wf, x, n_fft, hop, window, zp, "db", 0.0, 80.0))
        if ran != {kernel}:
            wrong.append((n_fft, path, hop, zp, ns, batch, kernel, sorted(ran)))
    assert not wrong, wrong
