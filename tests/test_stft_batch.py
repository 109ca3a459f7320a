"""Batched STFT and inverse STFT: B equal-length signals per handle (wfb_stft_create_ex, Spectrogram(batch=B)).

The gate is bitwise equality with single-signal runs of each row: the single-signal kernels are checked against the
oracle and torch.istft by test_stft.py / test_istft.py.  Both sides run the same kernel: a batch takes the bulk-copy
kernels only when num_samples % 4 == 0, so where the batch falls back and the single run does not, the rows are compared
within the single-signal bounds instead (2e-4 on dB, f32_bound(N) * ||frame|| on complex)."""
import ctypes

import numpy as np
import pytest

import oracle as om
from conftest import f32_bound
from istft_reference import istft_reference
from test_istft import _bound, _check, _den

WINDOWS = ("hann", "hamming", "blackman", "blackmanHarris", "rectangular")


def _signals(batch, n, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 16000.0
    f = rng.uniform(200, 4000, (batch, 1))
    return (0.6 * np.sin(2 * np.pi * f * t) + 0.1 * rng.uniform(-1, 1, (batch, n))).astype(np.float32)


def _ns(wsize, hop, frames_wanted, mod4):
    ns = wsize + (frames_wanted - 1) * hop + 1
    return ns + (mod4 - ns) % 4


def _bulk_kernel(n_fft, span_on):
    """Whether a 16-byte aligned single-signal run takes a bulk-copy kernel (span from N = 256, pipe at N = 8192)."""
    return (span_on and n_fft >= 256) or n_fft >= 8192


def _same_kernel(n_fft, hop, wsize, ns, batch, span_on):
    if batch == 1 or ns % 4 == 0 or hop % 4 or wsize % 4:
        return True
    return not _bulk_kernel(n_fft, span_on)


def _forward_single(wf, x2d, n_fft, hop, window, zp, mode, gain=-6.0, rng_db=70.0):
    sp = wf.Spectrogram(x2d.shape[1], n_fft, hop, window, zp, gain, rng_db, mode=mode)
    rows = []
    for x in x2d:
        sp.getInputBuffer()[:] = x
        sp.run()
        rows.append(sp.getOutputBuffer().copy())
    sp.dispose()
    return np.stack(rows)


def _forward_batch(wf, x2d, n_fft, hop, window, zp, mode, gain=-6.0, rng_db=70.0):
    sp = wf.Spectrogram(x2d.shape[1], n_fft, hop, window, zp, gain, rng_db, mode=mode, batch=x2d.shape[0])
    assert sp.getInputBuffer().shape == x2d.shape
    sp.getInputBuffer()[:] = x2d
    sp.run()
    out = sp.getOutputBuffer().copy()
    sp.dispose()
    return out


def _inverse_single(wf, spectra, ns, n_fft, hop, window, zp):
    sp = wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex")
    rows = []
    for s in spectra:
        sp.getOutputBuffer()[:] = s
        sp.inverse()
        rows.append(sp.getInputBuffer().copy())
    sp.dispose()
    return np.stack(rows)


def _inverse_batch(wf, spectra, ns, n_fft, hop, window, zp):
    sp = wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex", batch=spectra.shape[0])
    assert sp.getOutputBuffer().shape == spectra.shape
    sp.getOutputBuffer()[:] = spectra
    sp.inverse()
    out = sp.getInputBuffer().copy()
    sp.dispose()
    return out


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _assert_rows(got, single, x2d, n_fft, hop, wsize, mode, bitwise):
    assert got.shape == single.shape
    if bitwise:
        assert np.array_equal(_bits(got), _bits(single))
    elif mode == "db":
        assert np.max(np.abs(got - single)) < 2e-4
    else:
        w = om.window_function("hann", wsize)
        for b in range(got.shape[0]):
            for f in range(got.shape[1]):
                frame = (x2d[b, f * hop: f * hop + wsize].astype(np.float64) * w).astype(np.float32)
                err = np.max(np.abs(got[b, f].astype(np.float64) - single[b, f]))
                assert err <= 2 * f32_bound(n_fft) * np.linalg.norm(frame), (b, f)


# ------------------------------------------------------------------ CPU
def test_create_ex_argument_checks(wf):
    C = wf._cabi
    lib = C.lib()
    err = ctypes.c_int(0)

    def create(ns, batch, fft=1024, hop=256, mode=C.STFT_DB):
        err.value = 0
        return lib.wfb_stft_create_ex(fft, 1, hop, 0, ns, batch, mode, 0.0, 80.0, 0, 0, ctypes.byref(err))

    for batch in (0, -1):
        assert not create(16000, batch) and err.value == C.ERR_BAD_ARG
    assert not create(1 << 40, 1 << 40) and err.value == C.ERR_BAD_ARG              # batch x num_samples x 4 overflows
    # the input fits, the output (hop 1: ~num_samples frames of 4097 complex bins) does not
    assert not create(1 << 20, 1 << 30, fft=8192, hop=1, mode=C.STFT_COMPLEX) and err.value == C.ERR_BAD_ARG
    assert not create(100, 3) and err.value == C.ERR_BAD_ARG                          # shorter than the window, as before
    p = create(16000, 8)
    if lib.wfb_device_count() > 0 and lib.wfb_require_b200(0) == 0:
        assert p and lib.wfb_stft_batch(p) == 8 and lib.wfb_stft_frames(p) == (16000 - 1024) // 256 + 1
        lib.wfb_stft_destroy(p)
    else:
        assert not p and err.value == C.ERR_NO_DEVICE
    with pytest.raises(ValueError):
        wf.Spectrogram(16000, 1024, 256, batch=0)
    with pytest.raises(ValueError):
        wf.Spectrogram(16000, 1024, 256, batch=2.5)


def test_shape_errors_before_the_device(wf):
    with pytest.raises(ValueError):
        wf.generateSpectrogram(np.zeros((2, 3, 4096), np.float32), 16000.0, 256, 64)
    with pytest.raises(ValueError):
        wf.generateSpectrogram(np.zeros((0, 4096), np.float32), 16000.0, 256, 64)
    with pytest.raises(ValueError):
        wf.generateSpectrogram(np.zeros((3, 100), np.float32), 16000.0, 256, 64)        # too short
    for bad in ((2, 5, 128, 2), (2, 5, 129, 3), (0, 5, 129, 2), (2, 0, 129, 2), (1, 2, 5, 129, 2)):
        with pytest.raises(ValueError):
            wf.inverseSpectrogram(np.zeros(bad, np.float32), 256, 64)


@pytest.mark.parametrize("window,hop", [("hamming", 64), ("rectangular", 37), ("hamming", 100)])
def test_torch_istft_batch_matches_reference_rows(window, hop):
    """torch.istft(center=False) over a batch [B, bins, frames] against istft_reference row by row: the batched
    independent check of the oracle the single-signal inverse is gated on."""
    torch = pytest.importorskip("torch")
    n_fft, frames, batch = 256, 19, 5
    rng = np.random.default_rng(hop)
    spectra = rng.standard_normal((batch, frames, n_fft // 2 + 1, 2))
    z = torch.from_numpy(spectra[..., 0] + 1j * spectra[..., 1]).transpose(1, 2).contiguous()
    w = torch.from_numpy(om.window_function(window, n_fft).astype(np.float32).astype(np.float64))
    t = torch.istft(z, n_fft, hop_length=hop, win_length=n_fft, window=w, center=False).numpy()
    assert t.shape == (batch, (frames - 1) * hop + n_fft)
    for b in range(batch):
        ref = istft_reference(spectra[b], n_fft, hop, window)
        assert np.max(np.abs(t[b] - ref)) <= 1e-12


# ------------------------------------------------------------------ GPU: forward
FWD = [(64, 16, 1, 3), (64, 7, 2, 64), (256, 64, 1, 3), (256, 37, 4, 3), (1024, 256, 1, 3), (1024, 128, 2, 64),
       (1024, 101, 1, 3), (2048, 512, 1, 3), (2048, 128, 4, 1), (8192, 2048, 1, 3), (8192, 1024, 2, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["db", "complex"])
@pytest.mark.parametrize("mod4", [0, 1, 2, 3])
@pytest.mark.parametrize("n_fft,hop,zp,batch", FWD)
def test_gpu_forward_rows_equal_single(wf, oracle, monkeypatch, n_fft, hop, zp, batch, mod4, mode):
    monkeypatch.delenv("WFB_STFT_SPAN", raising=False)
    wsize = n_fft // zp
    ns = _ns(wsize, hop, 7, mod4)
    x = _signals(batch, ns, seed=n_fft + hop + mod4)
    got = _forward_batch(wf, x, n_fft, hop, "hann", zp, mode)
    single = _forward_single(wf, x, n_fft, hop, "hann", zp, mode)
    frames = (ns - wsize) // hop + 1
    bins = n_fft // 2 + 1
    assert got.shape == ((batch, frames, bins, 2) if mode == "complex" else (batch, frames, bins))
    span_default = n_fft in (1024, 2048)
    _assert_rows(got, single, x, n_fft, hop, wsize, mode, _same_kernel(n_fft, hop, wsize, ns, batch, span_default))
    if not _same_kernel(n_fft, hop, wsize, ns, batch, span_default) and n_fft < 8192:
        monkeypatch.setenv("WFB_STFT_SPAN", "0")                         # both sides on the direct kernel: bitwise
        assert np.array_equal(_bits(_forward_batch(wf, x, n_fft, hop, "hann", zp, mode)),
                              _bits(_forward_single(wf, x, n_fft, hop, "hann", zp, mode)))
    # sampled frames of the first, middle and last signal against the reference loop
    w = om.window_function("hann", wsize)
    for b in sorted({0, batch // 2, batch - 1}):
        for f in sorted({0, frames // 2, frames - 1}):
            seg = x[b, f * hop: f * hop + wsize]
            if mode == "db":
                ref = om.spectrogram_reference(seg, n_fft, hop, "hann", zp, gain=-6.0, range_db=70.0,
                                               rfft=oracle.rfft_split_f32)
                assert np.max(np.abs(got[b, f] - ref[0])) < 2e-4, (b, f)
            else:
                frame = (seg.astype(np.float64) * w).astype(np.float32)
                ref = om.spectrogram_reference(seg, n_fft, hop, "hann", zp, rfft=oracle.rfft_split_f32, complex_out=True)
                err = np.max(np.abs(got[b, f].astype(np.float64) - ref[0])) / np.linalg.norm(frame)
                assert err <= f32_bound(n_fft), (b, f, err)


@pytest.mark.gpu
@pytest.mark.parametrize("span", ["1", None])
@pytest.mark.parametrize("n_fft,hop,zp", [(64, 16, 1), (256, 64, 1), (1024, 256, 1), (2048, 512, 2), (8192, 2048, 1)])
def test_gpu_no_leakage_between_signals(wf, monkeypatch, n_fft, hop, zp, span):
    """Silent signals between loud ones: their rows must be exactly the silent single-signal rows, forward in both modes
    and inverse.  A span, tile or overlap-add that crosses a signal boundary shows up here."""
    if span is None:
        monkeypatch.delenv("WFB_STFT_SPAN", raising=False)
    else:
        monkeypatch.setenv("WFB_STFT_SPAN", span)
    wsize = n_fft // zp
    batch = 9
    ns = _ns(wsize, hop, 37, 0) + 2 * hop                                 # a tail past the last frame, bulk-copy aligned
    x = np.zeros((batch, ns), np.float32)
    loud = np.arange(1, batch, 2)
    x[loud] = 1e3 * _signals(len(loud), ns, seed=1)
    zero = np.zeros((1, ns), np.float32)
    for mode in ("db", "complex"):
        got = _forward_batch(wf, x, n_fft, hop, "hann", zp, mode)
        silent = _forward_single(wf, zero, n_fft, hop, "hann", zp, mode)[0]
        for b in range(0, batch, 2):
            assert np.array_equal(_bits(got[b]), _bits(silent)), (mode, b)
        for b in loud:
            assert np.any(got[b] != silent)
    # inverse: loud spectra around all-zero ones; every zero row stays exactly 0 end to end
    frames = (ns - wsize) // hop + 1
    spectra = np.zeros((batch, frames, n_fft // 2 + 1, 2), np.float32)
    spectra[loud] = 1e3 * np.random.default_rng(2).standard_normal((len(loud), frames, n_fft // 2 + 1, 2))
    back = _inverse_batch(wf, spectra, ns, n_fft, hop, "hann", zp)
    assert np.all(back[0::2] == 0.0)
    assert np.array_equal(_bits(back[loud]), _bits(_inverse_single(wf, spectra[loud], ns, n_fft, hop, "hann", zp)))


@pytest.mark.gpu
@pytest.mark.parametrize("span", ["1", None])
@pytest.mark.parametrize("n_fft", [256, 512, 1024, 2048, 8192])
def test_gpu_many_short_clips(wf, monkeypatch, n_fft, span):
    """Thousands of clips of a few frames: per-signal tiles ragged in every persistent kernel, one-frame clips, and
    bitwise repeatability of the persistent schedule."""
    if span is None:
        monkeypatch.delenv("WFB_STFT_SPAN", raising=False)
    else:
        monkeypatch.setenv("WFB_STFT_SPAN", span)
    hop = n_fft // 4
    clips = 3000 if n_fft <= 1024 else 600
    for ns in (n_fft + 5 * hop + 4, n_fft + 5 * hop + 3, n_fft):         # 6 frames (aligned / not), exactly one frame
        x = _signals(clips, ns, seed=ns)
        for mode in ("db", "complex"):
            got = _forward_batch(wf, x, n_fft, hop, "hann", 1, mode)
            again = _forward_batch(wf, x, n_fft, hop, "hann", 1, mode)
            assert np.array_equal(_bits(got), _bits(again))
            pick = np.unique(np.r_[0, 1, np.random.default_rng(ns).integers(0, clips, 14), clips - 1])
            single = _forward_single(wf, x[pick], n_fft, hop, "hann", 1, mode)
            _assert_rows(got[pick], single, x[pick], n_fft, hop, n_fft, mode,
                         _same_kernel(n_fft, hop, n_fft, ns, clips, span == "1" or n_fft in (1024, 2048)))
    ns = n_fft + 5 * hop + 4
    frames = 6
    spectra = np.random.default_rng(n_fft).standard_normal((clips, frames, n_fft // 2 + 1, 2)).astype(np.float32)
    back = _inverse_batch(wf, spectra, ns, n_fft, hop, "hann", 1)
    assert np.array_equal(_bits(back), _bits(_inverse_batch(wf, spectra, ns, n_fft, hop, "hann", 1)))
    pick = [0, clips // 3, clips - 1]
    assert np.array_equal(_bits(back[pick]), _bits(_inverse_single(wf, spectra[pick], ns, n_fft, hop, "hann", 1)))


# ------------------------------------------------------------------ GPU: inverse
INV = [(64, 1, "hann", 1, 3), (256, 256, "rectangular", 1, 5), (512, 600, "hann", 1, 3), (1024, 256, "blackman", 1, 4),
       (2048, 300, "blackmanHarris", 2, 3), (8192, 2048, "hann", 1, 2), (512, 37, "hamming", 4, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,window,zp,batch", INV)
def test_gpu_inverse_rows_equal_single(wf, n_fft, hop, window, zp, batch):
    wsize = n_fft // zp
    frames = 41 if hop > 1 else 700
    ns = (frames - 1) * hop + wsize + (hop - 1) // 2                     # a tail past the last frame (none at hop 1)
    spectra = np.random.default_rng(n_fft + hop).standard_normal((batch, frames, n_fft // 2 + 1, 2)).astype(np.float32)
    got = _inverse_batch(wf, spectra, ns, n_fft, hop, window, zp)
    assert got.shape == (batch, ns)
    assert np.array_equal(_bits(got), _bits(_inverse_single(wf, spectra, ns, n_fft, hop, window, zp)))
    assert np.all(got[:, (frames - 1) * hop + wsize:] == 0.0)
    b = batch - 1
    ref = istft_reference(spectra[b], n_fft, hop, window, zp, num_samples=ns)
    _check(got[b], ref, _bound(spectra[b], n_fft, hop, window, zp, ref), n_fft, hop, window, zp, frames)


@pytest.mark.gpu
@pytest.mark.parametrize("zp", [1, 2, 4])
@pytest.mark.parametrize("window", WINDOWS)
def test_gpu_batch_round_trip(wf, window, zp):
    n_fft, batch = 1024, 4
    wsize = n_fft // zp
    hop = wsize // 4
    ns = 30 * hop + wsize + hop // 2 + 2
    x = _signals(batch, ns, seed=zp)
    sp = wf.Spectrogram(ns, n_fft, hop, window, zp, mode="complex", batch=batch)
    sp.getInputBuffer()[:] = x
    sp.run()
    spectra = sp.getOutputBuffer().copy()
    sp.inverse()
    got = sp.getInputBuffer().copy()
    sp.dispose()
    frames = spectra.shape[1]
    den = _den(frames, n_fft, hop, window, zp)
    live = np.zeros(ns, bool)
    live[:len(den)] = den >= 1e-11
    for b in range(batch):
        ref = np.where(live, x[b].astype(np.float64), 0.0)
        _check(got[b], ref, _bound(spectra[b], n_fft, hop, window, zp, ref), n_fft, hop, window, zp, frames, factor=2.0)
    assert np.array_equal(_bits(got), _bits(_inverse_single(wf, spectra, ns, n_fft, hop, window, zp)))


# ------------------------------------------------------------------ GPU: device paths and the C ABI
@pytest.mark.gpu
def test_gpu_device_paths(wf, monkeypatch):
    torch = pytest.importorskip("torch")
    monkeypatch.delenv("WFB_STFT_SPAN", raising=False)
    C = wf._cabi
    n_fft, hop, batch = 1024, 256, 5
    ns = _ns(n_fft, hop, 40, 0)
    x = _signals(batch, ns, seed=21)
    stream = torch.cuda.Stream()
    for mode in ("db", "complex"):
        sp = wf.Spectrogram(ns, n_fft, hop, "hann", mode=mode, flags=C.PLAN_NO_HOST_BUFFERS, batch=batch)
        vw = 2 if mode == "complex" else 1
        out_len = batch * sp.numFrames * sp.numBins * vw
        with torch.cuda.stream(stream):
            xin = torch.zeros(batch * ns + 1, dtype=torch.float32, device="cuda")
            xin[1:] = torch.from_numpy(x.ravel()).cuda()                          # 4 bytes past 16-byte alignment
            out = torch.full((out_len + 2,), float("nan"), dtype=torch.float32, device="cuda")
        sp.run_device(xin.data_ptr() + 4, out.data_ptr() + 8, stream=stream.cuda_stream)
        stream.synchronize()
        o = out.cpu().numpy()
        assert np.isnan(o[:2]).all()
        got = o[2:].reshape((batch, sp.numFrames, sp.numBins) + ((2,) if mode == "complex" else ()))
        # the unaligned batch runs the direct kernel: the single rows on the direct kernel agree bit for bit
        monkeypatch.setenv("WFB_STFT_SPAN", "0")
        assert np.array_equal(_bits(got), _bits(_forward_single(wf, x, n_fft, hop, "hann", 1, mode, 0.0, 80.0)))
        monkeypatch.delenv("WFB_STFT_SPAN")
        if mode == "db":
            with pytest.raises(wf.WatFFTError) as e:
                sp.inverse_device(out.data_ptr(), xin.data_ptr())
            assert e.value.code == C.ERR_UNSUPPORTED
        else:
            spectra = got.copy()
            with torch.cuda.stream(stream):
                spec_buf = torch.zeros(spectra.size + 2, dtype=torch.float32, device="cuda")
                spec_buf[2:] = torch.from_numpy(spectra.ravel()).cuda()               # 8 bytes past 16-byte alignment
                back = torch.full((batch * ns + 2,), float("nan"), dtype=torch.float32, device="cuda")
            sp.inverse_device(spec_buf.data_ptr() + 8, back.data_ptr() + 4, stream=stream.cuda_stream)
            stream.synchronize()
            b = back.cpu().numpy()
            assert np.isnan(b[0]) and np.isnan(b[-1])
            single = _inverse_single(wf, spectra, ns, n_fft, hop, "hann", 1)
            assert np.array_equal(_bits(b[1:-1].reshape(batch, ns)), _bits(single))
            # spectra that start inside the LAST signal's samples overlap the batch's output range
            with pytest.raises(wf.WatFFTError) as e:
                sp.inverse_device(back.data_ptr() + 4 * (batch - 1) * ns, back.data_ptr())
            assert e.value.code == C.ERR_BAD_ARG
        sp.dispose()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_gpu_create_ex_batch1_is_create(wf, mode):
    C = wf._cabi
    lib = C.lib()
    n_fft, hop, ns = 2048, 512, 48000 + 3
    x = _signals(1, ns, seed=4)[0]
    err = ctypes.c_int(0)
    outs = []
    for make in (lambda: lib.wfb_stft_create(n_fft, 1, hop, 1, ns, mode, -3.0, 75.0, 0, 0, ctypes.byref(err)),
                 lambda: lib.wfb_stft_create_ex(n_fft, 1, hop, 1, ns, 1, mode, -3.0, 75.0, 0, 0, ctypes.byref(err))):
        p = make()
        assert p, err.value
        assert lib.wfb_stft_batch(p) == 1
        nbytes = lib.wfb_stft_output_bytes(p)
        ctypes.memmove(lib.wfb_stft_host_samples(p), x.ctypes.data, 4 * ns)
        C.check(lib.wfb_stft_exec(p, C.EXEC_DEFAULT))
        outs.append(np.ctypeslib.as_array((ctypes.c_uint32 * (nbytes // 4)).from_address(lib.wfb_stft_host_output(p))).copy())
        assert lib.wfb_stft_algorithmic_bytes(p) == 4 * ns + nbytes
        lib.wfb_stft_destroy(p)
    assert np.array_equal(outs[0], outs[1])


@pytest.mark.gpu
def test_gpu_python_batch_entry_points(wf):
    n_fft, hop, batch = 512, 128, 6
    x = _signals(batch, 16000, seed=8)
    got = wf.generateSpectrogram(x, 16000.0, n_fft, hop, "hamming", 2, gain=-3.0, range=75.0)
    assert got["batch"] == batch and got["data"].shape == (batch, got["numFrames"] * got["numBins"])
    for b in range(batch):
        one = wf.generateSpectrogram(x[b], 16000.0, n_fft, hop, "hamming", 2, gain=-3.0, range=75.0)
        assert "batch" not in one and one["numFrames"] == got["numFrames"]
        assert np.array_equal(_bits(got["data"][b]), _bits(one["data"]))
    spectra = np.random.default_rng(5).standard_normal((batch, 50, n_fft // 2 + 1, 2)).astype(np.float32)
    back = wf.inverseSpectrogram(spectra, n_fft, hop, "hann", 1)
    assert back.shape == (batch, 49 * hop + n_fft)
    for b in range(batch):
        assert np.array_equal(_bits(back[b]), _bits(wf.inverseSpectrogram(spectra[b], n_fft, hop, "hann", 1)))
    sp = wf.Spectrogram(16000, n_fft, hop, batch=3)
    assert sp.batch == 3 and sp.getInputBuffer().shape == (3, 16000)
    assert sp.getOutputBuffer().shape == (3, sp.numFrames, sp.numBins)
    assert sp.algorithmic_bytes() == 3 * (4 * 16000 + 4 * sp.numFrames * sp.numBins)
    sp.dispose()
    sp = wf.Spectrogram(16000, n_fft, hop)
    assert sp.batch is None and sp.getInputBuffer().shape == (16000,) and sp.getOutputBuffer().ndim == 2
    sp.dispose()
