"""
STFT, Welch and inverse STFT with frames longer than one CTA's shared memory (float32 nfft >= 2^14, float64 >= 2^13):
the long-frame route of csrc/qi_stft.cu (frame means, multi-pass FFTs of frame pairs, Hermitian split / pair gather).

CPU tier: the public entry points on the emulator runtime against the float64 oracle (scipy's algorithm, any frame
length), at the bounds of the tile-route tests (test_emul_api.py: float64 1e-12, float32 3e-6); the C ABI directly
(workspace sizes, chunking, error codes); the new kernels under AddressSanitizer.
GPU tier (-m gpu): large records on the B200.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import qi_oracle as orc

FS = 800.0
HERE = os.path.dirname(os.path.abspath(__file__))
TOL = {"float64": 1e-12, "float32": 3e-6}


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - b)) / np.max(np.abs(b)))


def record(n, channels=2, seed=0):
    """noise + an offset + a 60 Hz tone"""
    k = np.arange(n)
    rng = np.random.default_rng(seed)
    return rng.standard_normal((channels, n)) + 3.0 + np.cos(2 * np.pi * 60.0 / FS * k)


@pytest.fixture(scope="module")
def emul():
    from quantum_inferno_b200 import _runtime
    from tests.emul.emul_runtime import EmulRuntime
    with _runtime.use_runtime(EmulRuntime()) as rt:
        yield rt


# ----------------------------------------------------------------------------- CPU tier
@pytest.mark.parametrize("seg,ov,nfft,dtype", [
    (8192, 4096, 8192, "float64"),
    (16384, 8192, 16384, "float64"), (16384, 8192, 16384, "float32"),
    (10000, 3000, 16384, "float64"), (10000, 3000, 16384, "float32")])   # padding to nfft, hop not a divisor
def test_styx_fft_long_frames(emul, seg, ov, nfft, dtype):
    from quantum_inferno_b200 import styx_fft
    x = record(70000)
    f0, t0, z0 = orc.stft_complex_pow2(x, FS, seg, ov, nfft)
    f, t, z = styx_fft.stft_complex_pow2(x, FS, seg, ov, nfft, dtype=dtype)
    assert np.array_equal(f, f0) and np.allclose(t, t0)
    assert z.shape == z0.shape and rel(z, z0) < TOL[dtype]
    _, _, g0 = orc.gtx_complex_pow2(x, FS, seg, overlap_points=ov, nfft_points=nfft)
    _, _, g = styx_fft.gtx_complex_pow2(x, FS, seg, overlap_points=ov, nfft_points=nfft, dtype=dtype)
    assert g.shape == g0.shape and rel(g, g0) < TOL[dtype]
    _, p0 = orc.welch_power_pow2(x, FS, seg, nfft, ov)
    _, p = styx_fft.welch_power_pow2(x, FS, seg, nfft, ov, dtype=dtype)
    assert p.shape == p0.shape and rel(p, p0) < TOL[dtype]


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_stft_from_sig_long_window(emul, dtype):
    """band_order_nth=24, octaves_below_center=8 asks for an 8192-point frame by itself"""
    from quantum_inferno_b200 import styx_fft
    x = record(70000)[0]
    z0, b0, t0, f0 = orc.stft_from_sig(x, FS, 24, octaves_below_center=8)
    assert z0.shape[0] == 8192 // 2 + 1
    z, b, t, f = styx_fft.stft_from_sig(x, FS, 24, octaves_below_center=8, dtype=dtype)
    assert np.array_equal(f, f0) and np.allclose(t, t0)
    assert z.shape == z0.shape and rel(z, z0) < TOL[dtype]


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_short_time_fft_long_segment(emul, dtype):
    """utilities/short_time_fft at segment 16384: stft_tukey, spectrogram_tukey, and ShortTimeFFT.stft with detr=None and
    a non-zero phase_shift against scipy's own ShortTimeFFT"""
    from scipy import signal
    from quantum_inferno_b200.utilities import short_time_fft as stf
    x = record(70000)[0]
    seg, ov = 16384, 8192
    f0, t0, m0 = orc.stft_tukey(x, FS, 0.25, seg, ov)
    f, t, mag = stf.stft_tukey(x, FS, 0.25, seg, ov, dtype=dtype)
    assert np.array_equal(f, f0) and np.allclose(t, t0) and mag.shape == m0.shape and rel(mag, m0) < TOL[dtype]
    _, _, s0 = orc.spectrogram_tukey(x, FS, 0.25, seg, ov)
    _, _, sp = stf.spectrogram_tukey(x, FS, 0.25, seg, ov, dtype=dtype)
    assert sp.shape == s0.shape and rel(sp, s0) < TOL[dtype]
    obj = stf.get_stft_object_tukey(FS, 0.25, seg, ov, dtype=dtype)
    ref = signal.ShortTimeFFT(win=obj.win, hop=obj.hop, fs=FS, mfft=obj.mfft, fft_mode="onesided")
    for shift in (1000, -3):
        obj.phase_shift = ref.phase_shift = shift
        z0 = ref.stft(x)
        z = obj.stft(x)
        assert z.shape == z0.shape and rel(z, z0) < TOL[dtype], shift


def test_istft_round_trip_long_segment(emul):
    """istft_tukey of the segment-16384 STFT gives the record back within 1e-14 (the reference's round-trip bound), and
    matches the oracle's inverse of the same spectrum"""
    from quantum_inferno_b200.utilities import short_time_fft as stf
    x = record(70000)[0]
    seg = 16384
    obj = stf.get_stft_object_tukey(FS, 0.25, seg, seg // 2, "magnitude")
    spec = obj.stft(x)
    ts, xr = stf.istft_tukey(spec, FS, 0.25, seg, seg // 2, "magnitude")
    ts0, xr0 = orc.istft_tukey(spec, FS, 0.25, seg, seg // 2, "magnitude")
    assert np.array_equal(ts, ts0) and xr.shape == xr0.shape
    assert rel(xr, xr0) < 1e-14
    n = min(len(xr), len(x))                       # the last half-filled window lies past the record
    assert n > len(x) - seg and rel(xr[:n], x[:n]) < 1e-14


def _c_stft(rt, x, nperseg, hop, nfft, n_frames, pad_left, dt, ws_bytes, roll=0, psd=False, ws=True):
    from quantum_inferno_b200 import _lib
    lib = rt.lib
    C, N = x.shape
    code = _lib.QI_F64 if dt == "float64" else _lib.QI_F32
    xs = rt.asarray(x, dt)
    win = rt.asarray(np.hanning(nperseg), dt)
    out = None if psd else rt.zeros((C, nfft // 2 + 1, n_frames), "complex128" if dt == "float64" else "complex64")
    acc = rt.zeros((C, nfft // 2 + 1), "float64") if psd else None
    buf = rt.workspace(ws_bytes) if ws else None
    rc = lib.qi_stft(rt.ptr(xs), C, N, N, rt.ptr(win), nperseg, hop, nfft, n_frames, pad_left, 0.5, 1, roll, code,
                     rt.ptr(out), rt.ptr(acc), rt.ptr(buf), ws_bytes, None)
    return rc, (acc if psd else out)


def test_c_abi_one_entry_per_direction_workspace_and_chunking(emul):
    """qi_stft with and without a workspace, and the workspace sizes of both directions"""
    from quantum_inferno_b200 import _lib
    lib = emul.lib
    # every size the one-CTA kernels take needs no forward workspace, and the inverse only its slices
    assert lib.qi_stft_workspace_bytes(3, 100, 8192, _lib.QI_F32) == 0
    assert lib.qi_stft_workspace_bytes(3, 100, 4096, _lib.QI_F64) == 0
    assert lib.qi_stft_workspace_bytes(3, 100, 16384, _lib.QI_F32) == 3 * 50 * (16384 * 8 + 8)
    assert lib.qi_stft_workspace_bytes(3, 101, 8192, _lib.QI_F64) == 3 * 51 * (8192 * 16 + 16)
    for nfft, code, real in ((8192, _lib.QI_F32, 4), (4096, _lib.QI_F64, 8), (512, _lib.QI_F64, 8)):
        assert lib.qi_istft_workspace_bytes(3, 100, 1000, nfft, code) == 3 * 100 * 1000 * real
    assert lib.qi_istft_workspace_bytes(3, 100, 9000, 16384, _lib.QI_F32) > 3 * 100 * 9000 * 4

    x = record(50000, channels=2, seed=3)
    geom = dict(nperseg=12000, hop=5000, nfft=16384, n_frames=11, pad_left=6000)
    for dt in ("float64", "float32"):
        code = _lib.QI_F64 if dt == "float64" else _lib.QI_F32
        full = lib.qi_stft_workspace_bytes(2, geom["n_frames"], geom["nfft"], code)
        least = lib.qi_stft_workspace_bytes(2, 2, geom["nfft"], code)
        assert 0 < least < full
        rc, z_full = _c_stft(emul, x, dt=dt, ws_bytes=full, roll=77, **geom)
        assert rc == 0
        z_full = z_full.copy()
        # one pair per channel per chunk, and a chunk size that leaves a partial last chunk: the same bits
        for nbytes in (least, 2 * least + 5):
            rc, z = _c_stft(emul, x, dt=dt, ws_bytes=nbytes, roll=77, **geom)
            assert rc == 0 and np.array_equal(z, z_full), nbytes
        rc, p_full = _c_stft(emul, x, dt=dt, ws_bytes=full, psd=True, **geom)
        p_full = p_full.copy()
        rc2, p = _c_stft(emul, x, dt=dt, ws_bytes=least, psd=True, **geom)
        assert rc == 0 and rc2 == 0 and np.allclose(p, p_full, rtol=1e-13, atol=0)
        rc, _ = _c_stft(emul, x, dt=dt, ws_bytes=least - 1, **geom)
        assert rc == -2                                                             # QI_ERR_WORKSPACE
        rc, _ = _c_stft(emul, x, dt=dt, ws_bytes=0, ws=False, **geom)
        assert rc == -4                                                             # QI_ERR_UNSUPPORTED
        # no workspace at all
        win = emul.asarray(np.hanning(16384), dt)
        xs = emul.asarray(x, dt)
        out = emul.empty((2, 8193, 5), "complex128" if dt == "float64" else "complex64")
        assert lib.qi_stft(emul.ptr(xs), 2, 50000, 50000, emul.ptr(win), 16384, 8192, 16384, 5, 8192, 1.0, 1, 0, code,
                           emul.ptr(out), None, None, 0, None) == -4


def test_non_pow2_nfft_still_refused(emul):
    from quantum_inferno_b200 import styx_fft
    with pytest.raises(ValueError):
        styx_fft.stft_complex_pow2(record(40000), FS, 12000, nfft_points=12288)


def test_long_frame_route_under_address_sanitizer(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not installed")
    env = dict(os.environ, TMPDIR=str(tmp_path))
    run = subprocess.run(["bash", os.path.join(HERE, "emul", "asan_check.sh"),
                          os.path.join(HERE, "emul", "stft_long_driver.py")],
                         capture_output=True, text=True, env=env, timeout=900)
    text = run.stdout + run.stderr
    assert run.returncode == 0, text[-3000:]
    assert "AddressSanitizer" not in text, text[-3000:]
    assert "runtime error:" not in text, text[-3000:]
    assert "asan run done" in run.stdout, text[-3000:]


# ----------------------------------------------------------------------------- GPU tier
@pytest.fixture(scope="module")
def cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from quantum_inferno_b200 import _runtime
    _runtime._runtime = None
    assert _runtime.get_runtime().name == "cuda"
    return torch


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("nfft", [1 << 14, 1 << 16])
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_gpu_welch_long_frames(cuda, nfft, dtype):
    torch = cuda
    from quantum_inferno_b200 import styx_fft
    x = record(1 << 22, channels=16, seed=5)
    xd = torch.from_numpy(x).to(device="cuda", dtype=getattr(torch, dtype))
    _, p = styx_fft.welch_power_pow2(xd, FS, nfft, dtype=dtype)
    assert tuple(p.shape) == (16, nfft // 2 + 1)
    for ch in (0, 11):
        _, p0 = orc.welch_power_pow2(x[ch], FS, nfft)
        assert rel(_np(p[ch]), p0) < TOL[dtype], ch


@pytest.mark.gpu
def test_gpu_stft_long_frames(cuda):
    torch = cuda
    from quantum_inferno_b200 import styx_fft
    x = record(1 << 22, channels=4, seed=6)
    nfft = 1 << 15
    for dtype in ("float32", "float64"):
        xd = torch.from_numpy(x).to(device="cuda", dtype=getattr(torch, dtype))
        _, _, z = styx_fft.stft_complex_pow2(xd, FS, nfft, dtype=dtype)
        for ch in (0, 3):
            z0 = orc.stft_complex_pow2(x[ch], FS, nfft)[2]
            zz = _np(z[ch])
            assert zz.shape == z0.shape and rel(zz, z0) < TOL[dtype], (dtype, ch)


@pytest.mark.gpu
def test_gpu_stft_three_passes(cuda):
    """nfft = 2^21 takes three passes"""
    torch = cuda
    from quantum_inferno_b200 import styx_fft
    x = record(1 << 23, channels=1, seed=7)
    nfft = 1 << 21
    xd = torch.from_numpy(x).to(device="cuda")
    _, _, z = styx_fft.stft_complex_pow2(xd, FS, nfft, dtype="float64")
    z0 = orc.stft_complex_pow2(x[0], FS, nfft)[2]
    assert tuple(z.shape[1:]) == z0.shape and rel(_np(z[0]), z0) < 1e-12
    _, p = styx_fft.welch_power_pow2(xd, FS, nfft, dtype="float64")
    assert rel(_np(p[0]), orc.welch_power_pow2(x[0], FS, nfft)[1]) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3])
def test_gpu_long_frames_on_slices(cuda, k):
    """x[k:k+N] of a device buffer: the same complex output bits as an aligned copy"""
    torch = cuda
    from quantum_inferno_b200 import styx_fft
    x = record(1 << 20, channels=2, seed=8)
    for dtype, nfft in (("float32", 1 << 14), ("float64", 1 << 13)):
        tdt = getattr(torch, dtype)
        base = torch.empty(x.size + 8, dtype=tdt, device="cuda")
        s = base[k:k + x.size].view(*x.shape)
        s.copy_(torch.from_numpy(x).to(tdt))
        assert s.data_ptr() % 16 == (k * s.element_size()) % 16
        _, _, z = styx_fft.stft_complex_pow2(s, FS, nfft, dtype=dtype)
        _, _, za = styx_fft.stft_complex_pow2(torch.from_numpy(x).to(device="cuda", dtype=tdt), FS, nfft, dtype=dtype)
        assert torch.equal(z, za), dtype


@pytest.mark.gpu
def test_gpu_short_time_fft_round_trip(cuda):
    """ShortTimeFFT at segment 2^16 on device buffers: stft, istft back to the record"""
    torch = cuda
    from quantum_inferno_b200.utilities import short_time_fft as stf
    x = record(1 << 21, channels=2, seed=9)
    seg = 1 << 16
    obj = stf.get_stft_object_tukey(FS, 0.25, seg, seg // 2, "magnitude")
    xd = torch.from_numpy(x).to("cuda")
    spec = obj.stft(xd)
    assert spec.is_cuda
    k1 = int((spec.shape[-1] - 1) * obj.hop)
    xr = obj.istft(spec, k1=k1)
    assert xr.is_cuda and tuple(xr.shape) == (2, k1)
    n = min(k1, x.shape[1])
    assert rel(_np(xr)[:, :n], x[:, :n]) < 1e-14
    ts0, xr0 = orc.istft_tukey(_np(spec[1]), FS, 0.25, seg, seg // 2, "magnitude")
    assert rel(_np(xr[1]), xr0) < 1e-14
