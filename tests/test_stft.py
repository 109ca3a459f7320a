"""Batched STFT front-end (SURVEY 8f-1): the reference's spectrogram loop
(playground/src/spectrogram.js:281-360) restated in oracle/oracle.py and fused into one kernel.

Parity status: the r2c core of the oracle is pinned (bit-identical to the transpiled reference module); the window /
magnitude / dB / normalise stage is a restatement with no reference-run output behind it (the reference loop is
JavaScript; no JS engine in this image) -- PARITY UNPINNED for that stage."""
import numpy as np
import pytest

import oracle as om
from conftest import f32_bound
from stft_reference import check


def _signal(n, rate=16000.0, seed=0):
    t = np.arange(n) / rate
    rng = np.random.default_rng(seed)
    chirp = np.sin(2 * np.pi * (200 + 1500 * t) * t)
    return (0.6 * chirp + 0.3 * np.sin(2 * np.pi * 3000 * t) + 0.05 * rng.uniform(-1, 1, n)).astype(np.float32)


# ------------------------------------------------------------------ CPU: the restatement itself
def test_window_functions():
    for name in ("hann", "hamming", "blackman", "blackmanHarris", "rectangular", "nonsense"):
        w = om.window_function(name, 64)
        assert w.shape == (64,) and np.all(w <= 1.0 + 1e-12)
        assert np.allclose(w, w[::-1])                       # all symmetric
    assert om.window_function("hann", 8)[0] == 0.0 and abs(om.window_function("hamming", 8)[0] - 0.08) < 1e-12
    assert np.array_equal(om.window_function("nonsense", 16), om.window_function("hann", 16))


def test_reference_spectrogram_tone(oracle, watref):
    rate, n_fft, hop = 16000.0, 256, 64
    t = np.arange(4096) / rate
    x = np.sin(2 * np.pi * 2000.0 * t).astype(np.float32)
    s = om.spectrogram_reference(x, n_fft, hop, "hann", rfft=oracle.rfft_split_f32)
    assert s.shape == ((4096 - 256) // 64 + 1, 129) and s.dtype == np.float32
    assert np.all(s[:, :3] == 0.0) and s.min() >= 0.0 and s.max() <= 1.0
    assert np.all(np.argmax(s, axis=1) == round(2000.0 / rate * n_fft))       # bin 32
    # the same loop over the reference's own module gives the same picture
    s2 = om.spectrogram_reference(x, n_fft, hop, "hann", rfft=watref.rfft_split_f32)
    assert np.max(np.abs(s - s2)) < 1e-5
    with pytest.raises(ValueError):
        om.spectrogram_reference(x[:100], n_fft, hop, rfft=oracle.rfft_split_f32)


# ------------------------------------------------------------------ GPU parity
@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,window,zp", [(64, 16, "hann", 1), (256, 64, "hamming", 1), (1024, 100, "blackman", 1),
                                                 (1024, 256, "hann", 2), (4096, 1024, "blackmanHarris", 4),
                                                 (8192, 2048, "rectangular", 1), (512, 37, "hann", 1)])
def test_gpu_spectrogram_matches_reference_loop(wf, oracle, n_fft, hop, window, zp):
    x = _signal(3 * n_fft + 5 * hop + 11, seed=n_fft)
    ref = om.spectrogram_reference(x, n_fft, hop, window, zp, gain=-6.0, range_db=70.0, rfft=oracle.rfft_split_f32)
    got = wf.generateSpectrogram(x, 16000.0, n_fft, hop, window, zp, gain=-6.0, range=70.0)
    assert got["numFrames"] == ref.shape[0] and got["numBins"] == ref.shape[1] == n_fft // 2 + 1
    assert got["windowSize"] == n_fft // zp and got["fftSize"] == n_fft and got["hopSize"] == hop
    g = got["data"].reshape(ref.shape)
    assert np.all(g[:, :3] == 0.0)
    # normalised dB in [0,1]: f32 rounding of |X| moves a value by ~1e-6; bins at the clip edges by a bit more
    assert np.max(np.abs(g - ref)) < 2e-4, np.max(np.abs(g - ref))
    # raw spectra of the windowed frames, against the oracle's r2c of the same frames
    sp = wf.Spectrogram(len(x), n_fft, hop, window, zp, mode="complex")
    sp.getInputBuffer()[:] = x
    sp.run()
    gc = sp.getOutputBuffer().copy()
    sp.dispose()
    rc = om.spectrogram_reference(x, n_fft, hop, window, zp, rfft=oracle.rfft_split_f32, complex_out=True)
    wsize = n_fft // zp
    w = om.window_function(window, wsize)
    for f in sorted({0, ref.shape[0] // 2, ref.shape[0] - 1}):
        frame = (x[f * hop: f * hop + wsize].astype(np.float64) * w).astype(np.float32)
        err = np.max(np.abs(gc[f].astype(np.float64) - rc[f])) / np.linalg.norm(frame)
        assert err <= f32_bound(n_fft), (f, err)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,zp", [(256, 64, 1), (1024, 256, 2)])
def test_gpu_spectrogram_deep_floor_uses_exact_db(wf, oracle, n_fft, hop, zp):
    """A deep floor sees the reference's +1e-10 epsilon (spectrogram.js:60-62): where dropping it would move the output
    at the floor by more than 1e-6 (floors below about -99 dB at range 80), the kernel switches from the fast
    10*log10(|X|^2) form to the exact 20*log10(|X|/(N/2) + 1e-10) one.  A signal with exact zeros exercises it."""
    x = _signal(6 * n_fft, seed=7)
    x[: 2 * n_fft] = 0.0                                   # silent frames: magnitude 0 -> -200 dB
    ref = om.spectrogram_reference(x, n_fft, hop, "hann", zp, gain=0.0, range_db=220.0, rfft=oracle.rfft_split_f32)
    got = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hann", zp, gain=0.0, range=220.0)
    g = got["data"].reshape(ref.shape)
    assert abs(float(g[0, 5]) - (220.0 - 200.0) / 220.0) < 1e-4      # silence sits on the epsilon, not on the floor
    assert np.max(np.abs(g - ref)) < 2e-4, np.max(np.abs(g - ref))
    # and the fast path (floor at -70 dB) agrees with the same reference loop on the same signal
    ref2 = om.spectrogram_reference(x, n_fft, hop, "hann", zp, gain=0.0, range_db=70.0, rfft=oracle.rfft_split_f32)
    got2 = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hann", zp, gain=0.0, range=70.0)
    assert np.max(np.abs(got2["data"].reshape(ref2.shape) - ref2)) < 2e-4


@pytest.mark.gpu
def test_gpu_spectrogram_errors_and_long_signal(wf, oracle):
    with pytest.raises(ValueError):
        wf.generateSpectrogram(np.zeros(100, np.float32), 16000.0, 1024, 256)
    with pytest.raises(wf.WatFFTError):
        wf.Spectrogram(100000, 1000, 256)                    # not a power of two
    with pytest.raises(wf.WatFFTError):
        wf.Spectrogram(100000, 32, 8)                        # below the supported FFT sizes
    # one launch over ~15k frames; spot-check frames against the loop
    x = _signal(1 << 20, seed=3)
    got = wf.generateSpectrogram(x, 16000.0, 1024, 64)
    frames = got["numFrames"]
    assert frames == ((1 << 20) - 1024) // 64 + 1
    g = got["data"].reshape(frames, 513)
    for f in (0, 1, frames // 2, frames - 1):
        ref = om.spectrogram_reference(x[f * 64: f * 64 + 1024], 1024, 64, rfft=oracle.rfft_split_f32)
        assert np.max(np.abs(g[f] - ref[0])) < 2e-4


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,zp", [(256, 1), (256, 2), (512, 1), (512, 2), (1024, 1), (1024, 2), (2048, 1), (4096, 1), (4096, 4), (8192, 1)])
def test_span_kernel_many_tiles(wf, monkeypatch, n_fft, zp):
    """The span-staged persistent kernel with enough frames that every CTA loops over several tiles and the last tile is
    ragged: every frame against the f64 STFT, the whole picture against the direct kernel (different core plan, same
    contract), and bitwise repeatability of the persistent schedule."""
    hop = n_fft // zp // 4
    frames_wanted = 9001 if n_fft <= 1024 else 3001
    ns = (frames_wanted - 1) * hop + n_fft // zp + 3
    x = _signal(ns, seed=n_fft + zp)
    monkeypatch.setenv("WFB_STFT_SPAN", "1")
    got = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hann", zp, gain=-3.0, range=75.0)
    again = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hann", zp, gain=-3.0, range=75.0)
    monkeypatch.setenv("WFB_STFT_SPAN", "0")
    direct = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hann", zp, gain=-3.0, range=75.0)
    f, b = got["numFrames"], got["numBins"]
    assert f == frames_wanted and b == n_fft // 2 + 1
    g, d = got["data"].reshape(f, b), direct["data"].reshape(f, b)
    assert np.array_equal(g, again["data"].reshape(f, b))
    assert np.max(np.abs(g - d)) < 2e-4
    check(g, x, n_fft, hop, "hann", zp, "db", gain=-3.0, range_db=75.0)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 512, 1024])
def test_span_kernel_complex_output(wf, oracle, monkeypatch, n_fft):
    hop = n_fft // 4
    ns = 4000 * hop + n_fft
    x = _signal(ns, seed=5)
    monkeypatch.setenv("WFB_STFT_SPAN", "1")
    sp = wf.Spectrogram(ns, n_fft, hop, "blackman", mode="complex")
    sp.getInputBuffer()[:] = x
    sp.run()
    g = sp.getOutputBuffer().copy()
    sp.dispose()
    w = om.window_function("blackman", n_fft)
    for fr in (0, 3, 2000, g.shape[0] - 1):
        frame = (x[fr * hop: fr * hop + n_fft].astype(np.float64) * w).astype(np.float32)
        ref = oracle.rfft_split_f32(frame).reshape(-1, 2)
        assert np.max(np.abs(g[fr] - ref)) <= f32_bound(n_fft) * np.linalg.norm(frame), fr
