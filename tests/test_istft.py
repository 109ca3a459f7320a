"""Inverse STFT (extension: the reference has no inverse): the weighted overlap-add of the complex spectrogram's frames,
fused into one kernel (k_istft) behind Spectrogram.inverse() / inverseSpectrogram().

Oracle: tests/istft_reference.py, the contract restated in f64 with the f32 window values -- PARITY UNPINNED (no
reference run behind it); torch.istft(center=False) checks the formula independently on the CPU."""
import ctypes

import numpy as np
import pytest

import oracle as om
from conftest import f32_bound
from istft_reference import frames_c2r, istft_reference, overlap_add
from stft_reference import stft_f64

WINDOWS = ("hann", "hamming", "blackman", "blackmanHarris", "rectangular")


def _f32_window(window, wsize):
    return om.window_function(window, wsize).astype(np.float32).astype(np.float64)


def _den(frames, n_fft, hop, window, zp):
    wsize = n_fft // zp
    w = _f32_window(window, wsize)
    return overlap_add(np.broadcast_to(w * w, (frames, wsize)), hop)


def _bound(spectra, n_fft, hop, window, zp, ref):
    """Per-sample bound: the repository's c2r metric (f32_bound(N) * ||y_f||_2 per frame) carried through the weighted
    overlap-add, plus 4 ulp of the result."""
    wsize = n_fft // zp
    w = np.abs(_f32_window(window, wsize))
    norms = np.linalg.norm(frames_c2r(spectra, n_fft), axis=1)
    frames = spectra.shape[0]
    acc = overlap_add(w * (f32_bound(n_fft) * norms)[:, None], hop)
    den = _den(frames, n_fft, hop, window, zp)
    out = np.full(len(ref), np.inf)
    ok = den >= 1e-11
    out[:len(den)][ok] = acc[ok] / den[ok]
    return out + 4 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)


def _check(got, ref, bound, n_fft, hop, window, zp, frames, factor=1.0):
    """`got` within `factor` * bound where a frame carries weight; exactly 0 elsewhere and past the frames."""
    den = _den(frames, n_fft, hop, window, zp)
    live = np.zeros(len(got), bool)
    live[:len(den)] = den >= 1e-11
    err = np.abs(got.astype(np.float64) - ref)
    assert np.all(err[live] <= factor * bound[live]), float(np.max(err[live] / bound[live]))
    assert np.all(got[~live] == 0.0)


def _random_spectra(frames, n_fft, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((frames, n_fft // 2 + 1, 2)).astype(np.float32)


# ------------------------------------------------------------------ CPU: the restatement
@pytest.mark.parametrize("window", ["hamming", "rectangular"])
@pytest.mark.parametrize("hop", [64, 128, 37])
def test_reference_matches_torch_istft(window, hop):
    torch = pytest.importorskip("torch")
    n_fft, frames = 256, 23
    spectra = _random_spectra(frames, n_fft, seed=hop).astype(np.float64)     # not Hermitian-consistent
    ref = istft_reference(spectra, n_fft, hop, window)
    z = torch.from_numpy(spectra[..., 0] + 1j * spectra[..., 1]).T.contiguous()
    w = torch.from_numpy(_f32_window(window, n_fft))
    t = torch.istft(z, n_fft, hop_length=hop, win_length=n_fft, window=w, center=False).numpy()
    assert t.shape == ref.shape == ((frames - 1) * hop + n_fft,)
    assert np.max(np.abs(t - ref)) <= 1e-12, np.max(np.abs(t - ref))


@pytest.mark.parametrize("zp", [1, 2, 4])
@pytest.mark.parametrize("window", WINDOWS)
def test_reference_round_trip_f64(window, zp):
    n_fft, hop = 256, 40
    wsize = n_fft // zp
    for h in (hop // zp, wsize + 5):                        # overlapping frames, then gaps between frames
        ns = 20 * h + wsize + h // 2
        x = np.random.default_rng(zp).uniform(-1, 1, ns)
        spectra = stft_f64(x, n_fft, h, window, zp)
        frames = spectra.shape[0]
        got = istft_reference(spectra, n_fft, h, window, zp, num_samples=ns)
        den = _den(frames, n_fft, h, window, zp)
        live = np.zeros(ns, bool)
        live[:len(den)] = den >= 1e-11
        # f64 rounding, amplified where the window weight is small (the division by D near tapered edges)
        assert np.all(np.abs(got[live] - x[live]) <= 1e-13 * (1 + 1 / np.sqrt(den[live[:len(den)]]))), window
        assert np.all(got[~live] == 0.0) and len(den) < ns
        if window in ("hann", "blackman"):
            assert not live[0] and not live[len(den) - 1]   # the window edges carry no weight
        if h > wsize:
            assert not live[wsize: h].any()


# ------------------------------------------------------------------ GPU
def _gpu_inverse(wf, spectra, ns, n_fft, hop, window, zp):
    sp = wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex")
    assert sp.numFrames == spectra.shape[0]
    sp.getOutputBuffer()[:] = spectra
    sp.inverse()
    out = sp.getInputBuffer().copy()
    sp.dispose()
    return out


PARITY = [(64, 16, "hann", 1), (256, 64, "hamming", 1), (1024, 100, "blackman", 1), (1024, 256, "hann", 2),
          (4096, 1024, "blackmanHarris", 4), (8192, 2048, "rectangular", 1), (512, 37, "hann", 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,window,zp", PARITY)
def test_gpu_inverse_matches_reference(wf, n_fft, hop, window, zp):
    wsize = n_fft // zp
    ns = 3 * n_fft + 5 * hop + 11
    frames = (ns - wsize) // hop + 1
    spectra = _random_spectra(frames, n_fft, seed=n_fft + hop)
    got = _gpu_inverse(wf, spectra, ns, n_fft, hop, window, zp)
    ref = istft_reference(spectra, n_fft, hop, window, zp, num_samples=ns)
    _check(got, ref, _bound(spectra, n_fft, hop, window, zp, ref), n_fft, hop, window, zp, frames)


def _signal(n, seed):
    t = np.arange(n) / 16000.0
    rng = np.random.default_rng(seed)
    return (0.6 * np.sin(2 * np.pi * (200 + 1500 * t) * t) + 0.05 * rng.uniform(-1, 1, n)).astype(np.float32)


def _round_trip(wf, x, n_fft, hop, window, zp):
    sp = wf.Spectrogram(len(x), n_fft, hop, window, zp, mode="complex")
    sp.getInputBuffer()[:] = x
    sp.run()
    spectra = sp.getOutputBuffer().copy()
    sp.inverse()
    got = sp.getInputBuffer().copy()
    sp.dispose()
    return spectra, got


@pytest.mark.gpu
@pytest.mark.parametrize("zp", [1, 2, 4])
@pytest.mark.parametrize("window", WINDOWS)
def test_gpu_round_trip(wf, window, zp):
    n_fft = 1024
    hop = n_fft // zp // 4
    x = _signal(40 * hop + n_fft // zp + hop // 2, seed=zp)
    spectra, got = _round_trip(wf, x, n_fft, hop, window, zp)
    frames = spectra.shape[0]
    den = _den(frames, n_fft, hop, window, zp)
    live = np.zeros(len(x), bool)
    live[:len(den)] = den >= 1e-11
    ref = np.where(live, x.astype(np.float64), 0.0)
    _check(got, ref, _bound(spectra, n_fft, hop, window, zp, ref), n_fft, hop, window, zp, frames, factor=2.0)


MANY = [(64, 1, "hann", 1), (256, 64, "hann", 1), (512, 128, "hamming", 2), (1024, 256, "blackman", 1),
        (2048, 512, "hann", 1), (4096, 1024, "hann", 1), (8192, 2048, "hann", 1),
        (256, 256, "rectangular", 1), (512, 600, "hann", 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,window,zp", MANY)
def test_gpu_many_tiles(wf, n_fft, hop, window, zp):
    """Thousands of frames over many CTAs with a ragged last tile: hop 1 (a halo of W - 1 frames per tile), hop = W with
    the rectangular window (plain c2r frames side by side), hop > W (zero gaps); parity against the oracle and bitwise
    repeatability."""
    wsize = n_fft // zp
    frames = 3001 if n_fft <= 1024 else 1201
    ns = (frames - 1) * hop + wsize + max(hop - 1, 0) // 2
    spectra = _random_spectra(frames, n_fft, seed=frames + hop)
    sp = wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex")
    assert sp.numFrames == frames
    sp.getOutputBuffer()[:] = spectra
    sp.inverse()
    got = sp.getInputBuffer().copy()
    sp.inverse()
    again = sp.getInputBuffer().copy()
    sp.dispose()
    assert np.array_equal(got.view(np.uint32), again.view(np.uint32))
    ref = istft_reference(spectra, n_fft, hop, window, zp, num_samples=ns)
    _check(got, ref, _bound(spectra, n_fft, hop, window, zp, ref), n_fft, hop, window, zp, frames)
    if hop == wsize and window == "rectangular":
        y = frames_c2r(spectra, n_fft)[:, :wsize].ravel()
        assert np.max(np.abs(got[:len(y)] - y)) <= f32_bound(n_fft) * np.max(np.linalg.norm(frames_c2r(spectra, n_fft), axis=1))


@pytest.mark.gpu
def test_gpu_device_path(wf):
    torch = pytest.importorskip("torch")
    n_fft, hop, window = 1024, 256, "hann"
    ns = 200 * hop + n_fft + 7
    sp = wf.Spectrogram(ns, n_fft, hop, window, mode="complex", flags=wf._cabi.PLAN_NO_HOST_BUFFERS)
    frames, bins = sp.numFrames, sp.numBins
    spectra = _random_spectra(frames, n_fft, seed=11)
    ref = istft_reference(spectra, n_fft, hop, window, num_samples=ns)
    bound = _bound(spectra, n_fft, hop, window, 1, ref)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        spec_buf = torch.zeros(spectra.size + 2, dtype=torch.float32, device="cuda")
        spec_buf[2:] = torch.from_numpy(spectra.ravel()).cuda(non_blocking=False)    # 8 bytes past 16-byte alignment
        out_buf = torch.full((ns + 4,), float("nan"), dtype=torch.float32, device="cuda")
    assert (spec_buf.data_ptr() + 8) % 16 == 8 and (out_buf.data_ptr() + 4) % 16 == 4
    sp.inverse_device(spec_buf.data_ptr() + 8, out_buf.data_ptr() + 4, stream=stream.cuda_stream)
    stream.synchronize()
    o = out_buf.cpu().numpy()
    assert np.isnan(o[0]) and np.all(np.isnan(o[ns + 1:]))                           # nothing outside the samples
    _check(o[1: ns + 1], ref, bound, n_fft, hop, window, 1, frames)
    with pytest.raises(wf.WatFFTError) as e:
        sp.inverse_device(spec_buf.data_ptr() + 4, out_buf.data_ptr(), stream=stream.cuda_stream)
    assert e.value.code == wf._cabi.ERR_BAD_ARG
    for a, b in ((0, out_buf.data_ptr()), (spec_buf.data_ptr(), 0)):
        with pytest.raises(wf.WatFFTError) as e:
            sp.inverse_device(a, b)
        assert e.value.code == wf._cabi.ERR_BAD_ARG
    sp.dispose()
    db = wf.Spectrogram(ns, n_fft, hop, window)                         # magnitudes in dB have no inverse
    with pytest.raises(wf.WatFFTError) as e:
        db.inverse()
    assert e.value.code == wf._cabi.ERR_UNSUPPORTED
    with pytest.raises(wf.WatFFTError):
        db.inverse_device(spec_buf.data_ptr(), out_buf.data_ptr())
    db.dispose()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,window,zp", [(512, 128, "hann", 1), (2048, 300, "blackmanHarris", 2)])
def test_gpu_inverse_spectrogram(wf, n_fft, hop, window, zp):
    wsize = n_fft // zp
    frames = 97
    spectra = _random_spectra(frames, n_fft, seed=3)
    got = wf.inverseSpectrogram(spectra, n_fft, hop, window, zp)
    length = (frames - 1) * hop + wsize
    assert got.shape == (length,) and got.dtype == np.float32
    via_handle = _gpu_inverse(wf, spectra, length, n_fft, hop, window, zp)
    assert np.array_equal(got.view(np.uint32), via_handle.view(np.uint32))
    with pytest.raises(ValueError):
        wf.inverseSpectrogram(spectra[:, :-1], n_fft, hop, window, zp)
