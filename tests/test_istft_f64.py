"""Every inverse STFT kernel (k_istft, one instantiation per N = 64 ... 8192) at every sample against the f64 weighted
overlap-add (tests/istft_reference.py), within the per-sample bound of tests/test_istft.py.

The kernel matrix aims at each regime of the kernel's tiling.  `tiling` restates the host rule of
wfb_stft_exec_inverse_device; X, the frames one round computes, is read back from wfb_variants_f32_istft.cu.
  * Every N with every hop class: 1 (N <= 512: a halo of W - 1 recomputed frames); a hop whose halo is X frames or
    more, so a CTA's first rounds only fill the carry buffer (impossible at N = 64, where X = 64 > W - 1); W/4; an odd
    hop near W/2; W - 1; W; W + 1; 2W + 3 (zero gaps between frames).
  * Per hop class: 1, X - 1 and X + 1 frames and enough frames for 3 tiles plus a ragged last one; num_samples tails
    of 0 and H - 1; batch 1 and 3, every row checked.
  * Zero padding 1, 2, 4, N/4 and N/2 and the five windows spread over the cases: every N gets zero padding 1 and one
    above 1, and the matrix has tapered edges where 0 < D < 1e-11 (the output there must be exactly 0).  No sample may
    have its f64 D within a relative 1e-4 of the 1e-11 threshold, where the kernel's f32 D could fall on the other side.
Edges at every N: silence; garbage in Im X[0] and Im X[N/2]; spectra scaled by 2^-120 (subnormals must not flush) and by
2^100 (bit for bit the unscaled run, scaled); the round trip through the library's own forward; device pointers off
16-byte alignment between NaN guards; the overlap rejection; the lazily uploaded tables made on a caller's stream and
then used on the handle's own stream; bitwise repeatability; one kernel launch per call, and under torch.profiler one
distinct k_istft kernel per N.

The reference is pinned on the CPU first: its vectorised overlap-add is the per-frame loop bit for bit.

ISTFT_F64_REPORT=<file> writes the worst error per N, as a fraction of its bound, as JSON."""
import json
import os
import re
import subprocess
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

import oracle as om
from conftest import f32_bound
from istft_reference import frames_c2r, istft_reference, overlap_add
from test_istft import _bound, _check, _den, _round_trip, _signal

HERE = Path(__file__).resolve().parent
WINDOWS = ("hann", "hamming", "blackman", "blackmanHarris", "rectangular")
SIZES = (64, 128, 256, 512, 1024, 2048, 4096, 8192)
# frames per round of each N's k_istft instantiation (wfb_variants_f32_istft.cu; test_x_table_is_the_registry)
X_PER_N = {64: 64, 128: 32, 256: 16, 512: 8, 1024: 8, 2048: 4, 4096: 2, 8192: 2}
HOP_CLASSES = ("hop1", "halo", "quarter", "odd-half", "w-1", "w", "w+1", "gap")
SPECTRA_CAP = 64 << 20               # bytes of spectra per case
THRESHOLD = 1e-11                    # the kernel's (and the reference's) D below which a sample is 0

_worst = {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("ISTFT_F64_REPORT")
    if path and _worst:
        with open(path, "w") as f:
            json.dump({k: round(v, 4) for k, v in sorted(_worst.items(), key=lambda kv: (len(kv[0]), kv[0]))}, f,
                      indent=1)


def _record(key, ratio):
    _worst[key] = max(_worst.get(key, 0.0), ratio)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------ the tiling, restated
def tiling(n_fft, hop, wsize, num_samples):
    """wfb_stft_exec_inverse_device's tiles: a CTA owns tile_frames hops of output and recomputes the halo = ceil(W/H)
    - 1 frames before them; tile_frames + halo is a whole number of rounds of X frames, at least 11 halo and 16."""
    X = X_PER_N[n_fft]
    halo = -(-wsize // hop) - 1
    rounds = max(-(-11 * halo // X), -(-16 // X))
    tile_frames = rounds * X - halo
    span = tile_frames * hop
    return SimpleNamespace(X=X, halo=halo, rounds=rounds, tile_frames=tile_frames, tiles=-(-num_samples // span),
                           ragged=num_samples % span != 0)


def _hop(cls, wsize, X):
    return {"hop1": 1, "halo": max(1, wsize // (2 * X)), "quarter": max(1, wsize // 4), "odd-half": wsize // 2 | 1,
            "w-1": max(1, wsize - 1), "w": wsize, "w+1": wsize + 1, "gap": 2 * wsize + 3}[cls]


def _regime(cls, n_fft, hop, wsize):
    """Whether (hop, window size) puts the class in its regime."""
    t = tiling(n_fft, hop, wsize, wsize)
    return {"hop1": hop == 1 and t.halo == wsize - 1 >= 15,
            "halo": t.halo >= t.X and wsize >= 64,
            "quarter": hop > 1 and hop == wsize // 4 and t.halo == 3,
            "odd-half": hop > 1 and hop % 2 == 1 and t.halo == 1,
            "w-1": hop > 1 and hop == wsize - 1 and t.halo == 1,
            "w": hop == wsize and t.halo == 0,
            "w+1": hop == wsize + 1 and t.halo == 0,
            "gap": hop > 2 * wsize and t.halo == 0}[cls]


def _case(n_fft, cls):
    """(hop, zero padding, window) of one matrix case: the zero paddings 1, 2, 4, N/4, N/2 rotate over the classes and
    sizes, and a case takes the first of them from its place in the rotation that keeps it in its regime."""
    if cls == "hop1" and n_fft > 512:                                   # 3.5 tiles would pass the spectra cap
        return None
    i, j = SIZES.index(n_fft), HOP_CLASSES.index(cls)
    zps = (1, 2, 4, n_fft // 4, n_fft // 2)
    for k in range(5):
        zp = zps[(i + 2 * j + k) % 5]
        wsize = n_fft // zp
        hop = _hop(cls, wsize, X_PER_N[n_fft])
        if _regime(cls, n_fft, hop, wsize):
            window = WINDOWS[(i + j) % 5]
            if wsize <= 2 and window in ("hann", "blackman"):   # both are 0 (or -1.4e-17) at every sample of 2
                window = "hamming"
            return hop, zp, window
    return None


MATRIX = [(n, c) for n in SIZES for c in HOP_CLASSES if _case(n, c) is not None]


def _runs(n_fft, cls):
    """The runs of one matrix case: (frames, num_samples, batch, what the run must reach)."""
    hop, zp, _ = _case(n_fft, cls)
    wsize = n_fft // zp
    X = X_PER_N[n_fft]
    tf = tiling(n_fft, hop, wsize, wsize).tile_frames
    many = 3 * tf + tf // 2 + 1
    many_bytes = many * (n_fft // 2 + 1) * 8
    out = []
    for frames, tail, batch, reach in ((1, 0, 3, "one frame"), (1, hop - 1, 1, "one frame"),
                                       (X - 1, hop - 1, 3, "one round"), (X - 1, 0, 1, "one round"),
                                       (X + 1, 0, 3, "two rounds"), (X + 1, hop - 1, 1, "two rounds"),
                                       (many, (hop - 1) * (HOP_CLASSES.index(cls) % 2), 3 if 3 * many_bytes <= SPECTRA_CAP
                                        else 1, "many tiles")):
        out.append((frames, (frames - 1) * hop + wsize + tail, batch, reach))
    return out


def _reached(reach, n_fft, hop, wsize, frames, ns):
    t = tiling(n_fft, hop, wsize, ns)
    return {"one frame": frames == 1,
            "one round": frames == max(1, t.X - 1) and frames < t.X,
            "two rounds": t.X < frames <= 2 * t.X,
            "many tiles": t.tiles >= 4 and t.ragged and frames > 3 * t.tile_frames}[reach]


# ------------------------------------------------------------------ helpers
def _random_spectra(shape, n_fft, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(tuple(shape) + (n_fft // 2 + 1, 2)).astype(np.float32)


def _subnormal_allowance(frames, n_fft, hop, window, zp, num_samples):
    """What subnormal arithmetic adds to the bound: an f32 result below 2^-126 is rounded to a multiple of 2^-149, an
    absolute error of up to 2^-150 whatever the result's size.  Each y_f sample picks up about sqrt(N) of them in the
    c2r, weighted by |w|; each w * y product and each sum adds one more; dividing by D carries them to the output:
        2^-149 (sqrt(N) sum_f |w| + frames covering t) / D[t].
    Near a tapered edge, where D is small, this is far larger than the relative bound.  A plain f32 overlap-add on the
    CPU (scipy's f32 irfft, numpy f32 sums) reaches 0.44 of bound + allowance at 2^-120, and 2.4 / 5.7 times the bound
    alone at N = 2048 (hann) / 8192 (blackman): the same figures k_istft gives."""
    wsize = n_fft // zp
    w = np.abs(om.window_function(window, wsize).astype(np.float32).astype(np.float64))
    den = _den(frames, n_fft, hop, window, zp)
    ok = den >= THRESHOLD
    reach = overlap_add(np.sqrt(n_fft) * np.broadcast_to(w, (frames, wsize)) + 1.0, hop)
    out = np.zeros(num_samples)
    out[:len(den)][ok] = 2.0 ** -149 * reach[ok] / den[ok]
    return out


def _check_rows(got, spectra, n_fft, hop, window, zp, key=None, factor=1.0, subnormal=False):
    """Every row of `got` against the f64 reference of its spectra, within `factor` * the bound (plus the subnormal
    allowance, for spectra scaled into the subnormal range); the worst fraction of the bound is recorded under `key`.
    Also: no sample's D lies within a relative 1e-4 of the threshold, and where 0 < D < threshold the output is 0 like
    everywhere else outside the live samples (_check)."""
    got = got.reshape((-1, got.shape[-1]))
    spectra = spectra.reshape((-1,) + spectra.shape[-3:])
    frames = spectra.shape[1]
    den = _den(frames, n_fft, hop, window, zp)
    assert not np.any(np.abs(den - THRESHOLD) <= 1e-4 * THRESHOLD)
    live = np.zeros(got.shape[-1], bool)
    live[:len(den)] = den >= THRESHOLD
    worst = 0.0
    for b in range(got.shape[0]):
        ref = istft_reference(spectra[b], n_fft, hop, window, zp, num_samples=got.shape[-1])
        bound = _bound(spectra[b], n_fft, hop, window, zp, ref)
        if subnormal:
            bound = bound + _subnormal_allowance(frames, n_fft, hop, window, zp, got.shape[-1])
        _check(got[b], ref, bound, n_fft, hop, window, zp, frames, factor)
        if live.any():
            worst = max(worst, float(np.max(np.abs(got[b][live].astype(np.float64) - ref[live]) / bound[live])))
    if key is not None:
        _record(key, worst / factor)
    return worst


def _handle(wf, ns, n_fft, hop, window, zp, batch, **kw):
    return wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex", batch=None if batch == 1 else batch, **kw)


def _inverse(wf, spectra, ns, n_fft, hop, window, zp, repeat=False):
    """The inverse of spectra [frames][bins][2] or [B][frames][bins][2] through Spectrogram.inverse(), one kernel launch
    per call; with `repeat`, a second call on the same handle must give the same bits."""
    lib = wf._cabi.lib()
    batch = 1 if spectra.ndim == 3 else spectra.shape[0]
    sp = _handle(wf, ns, n_fft, hop, window, zp, batch)
    try:
        assert sp.numFrames == spectra.shape[-3]
        sp.getOutputBuffer()[:] = spectra.reshape(sp.getOutputBuffer().shape)
        before = lib.wfb_kernel_launch_count()
        sp.inverse()
        assert lib.wfb_kernel_launch_count() == before + 1
        got = sp.getInputBuffer().copy()
        if repeat:
            sp.inverse()
            assert np.array_equal(_bits(sp.getInputBuffer()), _bits(got))
        return got
    finally:
        sp.dispose()


# ------------------------------------------------------------------ CPU: the reference and the matrix, pinned
def _ola_loop(rows, hop):
    rows = np.asarray(rows, np.float64)
    out = np.zeros((rows.shape[0] - 1) * hop + rows.shape[1])
    for f in range(rows.shape[0]):
        out[f * hop: f * hop + rows.shape[1]] += rows[f]
    return out


def _istft_loop(spectra, n_fft, hop, window, zp, num_samples):
    """The reference as a per-frame loop, for the vectorised form to agree with."""
    wsize = n_fft // zp
    w = om.window_function(window, wsize).astype(np.float32).astype(np.float64)
    y = frames_c2r(spectra, n_fft)
    frames = spectra.shape[0]
    num = np.zeros((frames - 1) * hop + wsize)
    den = np.zeros_like(num)
    for f in range(frames):
        num[f * hop: f * hop + wsize] += w * y[f, :wsize]
        den[f * hop: f * hop + wsize] += w * w
    x = np.zeros(num_samples)
    ok = den >= THRESHOLD
    x[:len(num)][ok] = num[ok] / den[ok]
    return x


@pytest.mark.parametrize("n_fft,hop,zp,frames", [(64, 1, 1, 200), (256, 37, 2, 41), (128, 3, 32, 17), (512, 512, 1, 5),
                                                 (1024, 1100, 4, 6), (64, 7, 1, 1), (8192, 1024, 1, 12)])
def test_vectorised_reference_is_the_loop(n_fft, hop, zp, frames):
    wsize = n_fft // zp
    spectra = _random_spectra((frames,), n_fft, seed=hop + frames).astype(np.float64)
    ns = (frames - 1) * hop + wsize + hop // 2
    rows = np.random.default_rng(frames).standard_normal((frames, wsize))
    assert np.array_equal(overlap_add(rows, hop), _ola_loop(rows, hop))
    for window in WINDOWS:
        w = om.window_function(window, wsize).astype(np.float32).astype(np.float64)
        assert np.array_equal(istft_reference(spectra, n_fft, hop, window, zp, num_samples=ns),
                              _istft_loop(spectra, n_fft, hop, window, zp, ns))
        assert np.array_equal(_den(frames, n_fft, hop, window, zp), _ola_loop(np.tile(w * w, (frames, 1)), hop))
        norms = np.linalg.norm(frames_c2r(spectra, n_fft), axis=1)
        acc = _ola_loop(np.abs(w)[None, :] * (f32_bound(n_fft) * norms)[:, None], hop)
        ref = istft_reference(spectra, n_fft, hop, window, zp, num_samples=ns)
        bound = _bound(spectra, n_fft, hop, window, zp, ref)
        den = _ola_loop(np.tile(w * w, (frames, 1)), hop)
        ok = den >= THRESHOLD
        expect = np.full(ns, np.inf)
        expect[:len(den)][ok] = acc[ok] / den[ok]
        expect += 4 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
        assert np.array_equal(bound, expect)


def test_x_table_is_the_registry():
    """X per N is the frames_per_round of the registered k_istft instantiations: a re-tuned X fails here instead of
    quietly moving the matrix off its regimes."""
    src = (HERE.parent / "wat-fft_b200" / "csrc" / "wfb_variants_f32_istft.cu").read_text()
    body = src[src.index("variants_istft()"):]
    found = {2 * int(m.group(1)): int(m.group(2)) for m in re.finditer(r"\bV\(\s*\w+?_(\d+)\s*,\s*(\d+)\s*,", body)}
    assert found == X_PER_N


def test_tiling_rule():
    """Hand-worked tiles of the host rule."""
    t = tiling(1024, 256, 1024, 10 * 256 + 1024)                       # halo 3: rounds max(ceil(33/8), 2) = 5
    assert (t.halo, t.rounds, t.tile_frames, t.tiles, t.ragged) == (3, 5, 37, 1, True)
    t = tiling(64, 1, 64, 3000)                                        # halo 63: rounds ceil(693/64) = 11
    assert (t.halo, t.rounds, t.tile_frames, t.tiles) == (63, 11, 641, 5)
    t = tiling(8192, 8192, 8192, 64 * 8192)                            # no halo: 16 frames per tile
    assert (t.halo, t.rounds, t.tile_frames, t.tiles, t.ragged) == (0, 8, 16, 4, False)
    # a halo of X frames or more cannot happen at N = 64
    assert all(tiling(64, h, w, w).halo < 64 for w in (2, 4, 16, 32, 64) for h in range(1, w + 1))


def test_matrix_reaches_every_regime():
    """Every case of the GPU matrix is in its regime, every run reaches what it is for, every N has every hop class it
    can have with zero padding 1 and above 1, the matrix spans all five zero paddings and windows, the spectra of a run
    stay under the cap, and somewhere a tapered edge gives 0 < D < 1e-11 (which the kernel must still output as 0)."""
    zps, windows, tiny_d = set(), set(), []
    for n_fft in SIZES:
        classes = [c for n, c in MATRIX if n == n_fft]
        assert classes == [c for c in HOP_CLASSES if (c != "hop1" or n_fft <= 512) and (c != "halo" or n_fft > 64)]
        n_zps = set()
        for cls in classes:
            hop, zp, window = _case(n_fft, cls)
            wsize = n_fft // zp
            assert _regime(cls, n_fft, hop, wsize)
            n_zps.add(zp)
            windows.add(window)
            for frames, ns, batch, reach in _runs(n_fft, cls):
                assert _reached(reach, n_fft, hop, wsize, frames, ns), (n_fft, cls, reach)
                assert batch * frames * (n_fft // 2 + 1) * 8 <= SPECTRA_CAP
                den = _den(frames, n_fft, hop, window, zp)
                assert not np.any(np.abs(den - THRESHOLD) <= 1e-4 * THRESHOLD)
                if np.any((den > 0) & (den < THRESHOLD)):
                    tiny_d.append((n_fft, cls))
        assert 1 in n_zps and max(n_zps) > 1, (n_fft, n_zps)
        zps |= {{1: "1", 2: "2", 4: "4", n_fft // 4: "N/4", n_fft // 2: "N/2"}[z] for z in n_zps}
    assert zps == {"1", "2", "4", "N/4", "N/2"} and windows == set(WINDOWS)
    assert tiny_d


# ------------------------------------------------------------------ GPU: the kernel matrix
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,cls", MATRIX)
def test_gpu_kernel_matrix(wf, n_fft, cls):
    """One hop class at one N: 1, X - 1, X + 1 and 3.5 tiles' worth of frames, tails 0 and H - 1, batch 1 and 3, every
    sample of every row against f64; the many-tile run twice, bit for bit."""
    hop, zp, window = _case(n_fft, cls)
    for k, (frames, ns, batch, reach) in enumerate(_runs(n_fft, cls)):
        spectra = _random_spectra((batch, frames), n_fft, seed=n_fft * 7919 + hop * 31 + k)
        got = _inverse(wf, spectra if batch > 1 else spectra[0], ns, n_fft, hop, window, zp, repeat=reach == "many tiles")
        assert got.shape == ((batch, ns) if batch > 1 else (ns,))
        _check_rows(got, spectra, n_fft, hop, window, zp, key=str(n_fft))


# ------------------------------------------------------------------ GPU: edge inputs
def _edge_geometry(n_fft):
    """Hop W/4 + 1 at zero padding 1, two tiles and a ragged third, a tail of 3 samples."""
    hop = n_fft // 4 + 1
    t = tiling(n_fft, hop, n_fft, n_fft)
    frames = 2 * t.tile_frames + t.X + 1
    return hop, frames, (frames - 1) * hop + n_fft + 3


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", SIZES)
def test_gpu_edge_inputs(wf, n_fft):
    """Silence gives exact zeros; Im X[0] and Im X[N/2] are ignored bit for bit; spectra at 2^-120 stay within the
    scaled bound (a flush of subnormals to zero would not); spectra at 2^100 neither overflow nor round differently:
    the output is the unscaled output times 2^100, bit for bit."""
    hop, frames, ns = _edge_geometry(n_fft)
    window = WINDOWS[SIZES.index(n_fft) % 5]
    t = tiling(n_fft, hop, n_fft, ns)
    assert t.tiles >= 3 and t.ragged
    spectra = _random_spectra((3, frames), n_fft, seed=n_fft + 5)
    spectra[1, frames // 3: frames // 2] = 0.0                          # silent frames inside a signal
    silence = _inverse(wf, np.zeros_like(spectra), ns, n_fft, hop, window, 1)
    assert np.all(_bits(silence) == 0)                                  # +0.0 everywhere
    clean = _inverse(wf, spectra, ns, n_fft, hop, window, 1)
    _check_rows(clean, spectra, n_fft, hop, window, 1, key=str(n_fft))
    dirty = spectra.copy()
    rng = np.random.default_rng(n_fft)
    dirty[..., 0, 1] = rng.uniform(-1e3, 1e3, dirty.shape[:2])
    dirty[..., -1, 1] = rng.uniform(-1e3, 1e3, dirty.shape[:2])
    assert np.array_equal(_bits(_inverse(wf, dirty, ns, n_fft, hop, window, 1)), _bits(clean))
    small = spectra * np.float32(2.0 ** -120)                          # many of them subnormal
    tiny = _inverse(wf, small, ns, n_fft, hop, window, 1)
    assert np.count_nonzero(tiny) > 0.9 * np.count_nonzero(clean)
    _check_rows(tiny, small, n_fft, hop, window, 1, key=f"{n_fft}/subnormal", subnormal=True)
    # and against the unscaled run, scaled: within both runs' bounds
    scaled_clean = clean.astype(np.float64) * 2.0 ** -120
    tol = np.stack([_bound(spectra[b], n_fft, hop, window, 1, clean[b].astype(np.float64)) for b in range(3)])
    tol = 2 * (tol * 2.0 ** -120 + _subnormal_allowance(frames, n_fft, hop, window, 1, ns))
    live = np.isfinite(tol)
    assert np.all(np.abs(tiny.astype(np.float64) - scaled_clean)[live] <= tol[live])
    huge = _inverse(wf, spectra * np.float32(2.0 ** 100), ns, n_fft, hop, window, 1)
    assert np.all(np.isfinite(huge))
    assert np.array_equal(_bits(huge), _bits(clean * np.float32(2.0 ** 100)))


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", SIZES)
def test_gpu_round_trip(wf, n_fft):
    """The library's forward (mode complex) then the inverse, zero padding 1 and 2, two windows: the signal back within
    twice the inverse's bound wherever a frame carries weight, 0 elsewhere."""
    i = SIZES.index(n_fft)
    for zp, window in ((1, WINDOWS[i % 5]), (2, WINDOWS[(i + 3) % 5])):
        wsize = n_fft // zp
        hop = wsize // 4
        frames = 2 * tiling(n_fft, hop, wsize, wsize).tile_frames + 3
        x = _signal((frames - 1) * hop + wsize + hop // 2, seed=n_fft + zp)
        spectra, got = _round_trip(wf, x, n_fft, hop, window, zp)
        assert spectra.shape[0] == frames
        den = _den(frames, n_fft, hop, window, zp)
        live = np.zeros(len(x), bool)
        live[:len(den)] = den >= THRESHOLD
        ref = np.where(live, x.astype(np.float64), 0.0)
        bound = _bound(spectra, n_fft, hop, window, zp, ref)
        _check(got, ref, bound, n_fft, hop, window, zp, frames, factor=2.0)
        _record(f"{n_fft}/round_trip", float(np.max(np.abs(got[live] - ref[live]) / (2 * bound[live]))))


# ------------------------------------------------------------------ GPU: device pointers, streams, launches
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", SIZES)
def test_gpu_device_pointers(wf, n_fft):
    """A fresh handle's first inverse is inverse_device on a caller's stream, with the spectra 8 bytes past 16-byte
    alignment and the samples at +1 float between NaN guards; it uploads the tables there.  inverse() on the handle's
    own stream follows at once and must wait for that upload: both give the same bits, and so does a third call with
    the samples at +3 floats.  Spectra that overlap the output are rejected before the device is touched."""
    torch = pytest.importorskip("torch")
    C = wf._cabi
    lib = C.lib()
    hop, frames, ns = _edge_geometry(n_fft)
    batch, window = 2, WINDOWS[(SIZES.index(n_fft) + 1) % 5]
    spectra = _random_spectra((batch, frames), n_fft, seed=n_fft + 9)
    sp = _handle(wf, ns, n_fft, hop, window, 1, batch)
    sp.getOutputBuffer()[:] = spectra
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        spec_buf = torch.zeros(spectra.size + 2, dtype=torch.float32, device="cuda")
        spec_buf[2:] = torch.from_numpy(spectra.ravel()).cuda()
        outs = [torch.full((batch * ns + oo + 5,), float("nan"), dtype=torch.float32, device="cuda") for oo in (1, 3)]
    assert spec_buf.data_ptr() % 16 == 0 and all(o.data_ptr() % 16 == 0 for o in outs)
    before = lib.wfb_kernel_launch_count()
    sp.inverse_device(spec_buf.data_ptr() + 8, outs[0].data_ptr() + 4, stream=stream.cuda_stream)
    sp.inverse()                                                        # the handle's stream: waits for the tables
    host = sp.getInputBuffer().copy()
    sp.inverse_device(spec_buf.data_ptr() + 8, outs[1].data_ptr() + 12, stream=stream.cuda_stream)
    stream.synchronize()
    assert lib.wfb_kernel_launch_count() == before + 3
    for oo, out in zip((1, 3), outs):
        o = out.cpu().numpy()
        assert np.isnan(o[:oo]).all() and np.isnan(o[oo + batch * ns:]).all()
        assert np.array_equal(_bits(o[oo: oo + batch * ns].reshape(batch, ns)), _bits(host))
    _check_rows(host, spectra, n_fft, hop, window, 1, key=str(n_fft))
    # spectra that start inside the last signal's samples; output that starts inside the spectra
    for s, d in ((outs[0].data_ptr() + 8 * ((batch - 1) * ns // 2), outs[0].data_ptr()),
                 (spec_buf.data_ptr() + 8, spec_buf.data_ptr() + 8 + 4 * (spectra.size - 1))):
        with pytest.raises(wf.WatFFTError) as e:
            sp.inverse_device(s, d, stream=stream.cuda_stream)
        assert e.value.code == C.ERR_BAD_ARG
    assert lib.wfb_kernel_launch_count() == before + 3
    sp.dispose()


# torch.profiler in a process of its own (see test_stft_filterbank.test_gpu_kernel_routing: a long test process that has
# held many profiler sessions can stop reporting kernel events)
_KERNELS_CHILD = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[2], sys.argv[2] + "/oracle"]
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
import watfft_b200 as wf
torch.cuda.init()
ran = []
for n_fft in json.load(sys.stdin):
    hop, frames = n_fft // 4, 40
    sp = wf.Spectrogram((frames - 1) * hop + n_fft, n_fft, hop, "hann", mode="complex")
    sp.getOutputBuffer()[:] = np.random.default_rng(n_fft).standard_normal(sp.getOutputBuffer().shape)
    sp.inverse()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sp.inverse()
        torch.cuda.synchronize()
    sp.dispose()
    ran.append(sorted({e.name for e in prof.events() if "k_istft" in e.name}))
print(json.dumps(ran))
"""


@pytest.mark.gpu
def test_gpu_kernels_run(wf):
    """Under torch.profiler each N runs exactly one k_istft kernel, and the eight sizes run eight different ones."""
    pytest.importorskip("torch")
    res = subprocess.run([sys.executable, "-c", _KERNELS_CHILD, str(HERE), str(HERE.parent)], text=True,
                         input=json.dumps(list(SIZES)), capture_output=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    ran = json.loads(res.stdout.strip().splitlines()[-1])
    for n_fft, names in zip(SIZES, ran):
        print(f"N = {n_fft}: {names}")
    assert len(ran) == len(SIZES) and all(len(names) == 1 for names in ran), ran
    assert len({names[0] for names in ran}) == len(SIZES)
