"""The 2048-point level-convolution kernel (qi_mr_level2k.cuh) against a float64 numpy overlap-save of the same band
tables, on the CPU emulator (no GPU), independently of the planner and of how the block transform is factored: level-0 power and complex rows, the deeper-level complex rows and the demodulated
envelope rows of the half-size inverse transforms, with odd block counts (the last pair holds one block) and an odd
band count on the envelope path (the last pass holds one band).  Random band tables exercise every bin of the
bit-reversed spectrum the kernel multiplies, not only a smooth Gabor response."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
EMUL = os.path.join(HERE, "emul")
SRC = os.path.join(HERE, "..", "quantum_inferno_b200", "csrc")
F = 2048
HALO = 16           # MR_HALO of qi_mr_expand.cuh
TOL = 1e-6          # relative L2 per row: float32 rounding of a reordered transform


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    subprocess.run([os.path.join(EMUL, "build_emul.sh")], check=True, capture_output=True)
    so = str(tmp_path_factory.mktemp("l2k") / "level2k_harness.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-DQI_EMUL", "-I" + EMUL, "-I" + SRC, "-x", "c++",
                    os.path.join(EMUL, "level2k_harness.cpp"), "-x", "none", os.path.join(EMUL, "build", "cuda_emul.o"),
                    "-lpthread", "-o", so], check=True)
    lib = ctypes.CDLL(so)
    lib.l2k_run.restype = ctypes.c_int
    i64, i32, vp = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p
    lib.l2k_run.argtypes = [vp, i64, i32, i64, i32, i32, i64, i64, i64, i64, i32, i32, vp, vp, i32, vp, vp, vp, i64, vp]
    return lib


def brev11():
    p = np.arange(F)
    r = np.zeros(F, dtype=np.int64)
    for bit in range(11):
        r |= ((p >> bit) & 1) << (10 - bit)
    return r


def ptr(a):
    return None if a is None else a.ctypes.data


def run(lib, *, x, x_halo, q_first, level, env, n_points, n_level, n_out, n_blocks, wk, tables, demod,
        ppc=1, power=False, complex_out=False, w_stride=0):
    nb = tables.shape[0]
    x = np.ascontiguousarray(x, dtype=np.float32)
    tab = np.ascontiguousarray(tables, dtype=np.complex64)
    dm = np.ascontiguousarray(demod, dtype=np.int32)
    out_p = np.zeros((nb, n_points), np.float32) if power else None
    out_c = np.zeros((nb, n_points), np.complex64) if complex_out else None
    wbuf = np.zeros(max(1, nb * w_stride), np.complex64)
    bsum = np.zeros(nb, np.float64)
    rc = lib.l2k_run(ptr(x), x.size, x_halo, q_first, level, env, n_points, n_level, n_out, n_blocks, wk, nb, ptr(tab),
                     ptr(dm), ppc, ptr(out_p), ptr(out_c), ptr(wbuf), w_stride, ptr(bsum))
    assert rc == 0
    return out_p, out_c, wbuf.reshape(nb, -1) if w_stride else None, bsum


def blocks_y(x, x_halo, q_first, n_blocks, wk, tables):
    """float64 overlap-save: y[b, blk, n] = IFFT_F(FFT_F(block) * K_b) * F (the kernel's inverse is unnormalised), with
    the tables stored in bit-reversed bin order."""
    V, half = F - wk, wk // 2
    kspec = tables.astype(np.complex128)[:, np.argsort(brev11())]     # natural bin order
    xs = x.astype(np.float64)
    ys = np.empty((tables.shape[0], n_blocks, F), np.complex128)
    for blk in range(n_blocks):
        k = q_first + blk * V - half + x_halo + np.arange(F)
        seg = np.where((k >= 0) & (k < xs.size), xs[np.clip(k, 0, xs.size - 1)], 0.0)
        ys[:, blk] = np.fft.ifft(np.fft.fft(seg)[None, :] * kspec, axis=1) * F
    return ys


def rel_rows(a, e):
    return np.linalg.norm(a - e, axis=-1) / np.linalg.norm(e, axis=-1)


def random_case(seed, nb, n_x):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(n_x)
    tables = (rng.standard_normal((nb, F)) + 1j * rng.standard_normal((nb, F))) / F
    return x, tables


@pytest.mark.parametrize("ppc", [1, 2])
def test_level0_power_and_complex(harness, ppc):
    n, wk, nb = 8192, 400, 3
    V, half = F - wk, wk // 2
    n_blocks = -(-n // V)                                              # 5: the last pair holds one block
    assert n_blocks % 2 == 1
    x, tables = random_case(1, nb, n)
    p, c, _, bsum = run(harness, x=x, x_halo=0, q_first=0, level=0, env=0, n_points=n, n_level=n, n_out=n,
                        n_blocks=n_blocks, wk=wk, tables=tables, demod=np.zeros(nb), ppc=ppc, power=True,
                        complex_out=True)
    ys = blocks_y(x, 0, 0, n_blocks, wk, tables)
    ref = ys[:, :, half:half + V].reshape(nb, -1)[:, :n]
    assert np.all(rel_rows(c, ref) < TOL), rel_rows(c, ref)
    assert np.all(rel_rows(p, np.abs(ref) ** 2) < TOL), rel_rows(p, np.abs(ref) ** 2)
    assert np.allclose(bsum, np.sum(np.abs(ref) ** 2, axis=1), rtol=1e-5)


def test_deep_level_complex_rows(harness):
    """level >= 1 without envelopes (the complex-TFR mode): the decimated complex output w_b, halo included."""
    n, level, wk, nb = 8192, 1, 600, 2
    n_level = n >> level
    V, half = F - wk, wk // 2
    n_out = n_level + 2 * HALO
    n_blocks = -(-n_out // V)                                          # 3
    assert n_blocks % 2 == 1
    x, tables = random_case(2, nb, n_level + 2 * HALO)
    _, _, w, bsum = run(harness, x=x, x_halo=HALO, q_first=-HALO, level=level, env=0, n_points=n, n_level=n_level,
                        n_out=n_out, n_blocks=n_blocks, wk=wk, tables=tables, demod=np.zeros(nb), w_stride=n_out)
    ys = blocks_y(x, HALO, -HALO, n_blocks, wk, tables)
    ref = ys[:, :, half:half + V].reshape(nb, -1)[:, :n_out]
    assert np.all(rel_rows(w, ref) < TOL), rel_rows(w, ref)
    assert np.allclose(bsum, np.sum(np.abs(ref[:, HALO:HALO + n_level]) ** 2, axis=1), rtol=1e-5)


@pytest.mark.parametrize("nb", [3, 4])
def test_envelope_rows(harness, nb):
    """levels >= 1, envelope bands: w(q) = y(2q) exp(-2 pi i demod q / 64) from the folded 1024-point inverse."""
    n, level, wk = 8192, 1, 600
    n_level = n >> level
    V, half = F - wk, wk // 2
    Vh, hh = V // 2, half // 2
    n_w = n_level // 2 + 2 * HALO
    n_out = n_level + 2 * HALO
    n_blocks = -(-n_out // V)                                          # 3
    assert n_blocks % 2 == 1
    x, tables = random_case(3 + nb, nb, n_level + 2 * HALO)
    demod = np.arange(nb) * 11 + 5
    _, _, w, bsum = run(harness, x=x, x_halo=HALO, q_first=-HALO, level=level, env=1, n_points=n, n_level=n_level,
                        n_out=n_out, n_blocks=n_blocks, wk=wk, tables=tables, demod=demod, w_stride=n_w)
    ys = blocks_y(x, HALO, -HALO, n_blocks, wk, tables)[:, :, 0::2]   # the even samples of each block
    ref = ys[:, :, hh:hh + Vh].reshape(nb, -1)[:, :n_w]
    q = np.arange(n_w) - HALO
    ref = ref * np.exp(-2j * np.pi * ((demod[:, None] * q[None, :]) % 64) / 64)
    assert np.all(rel_rows(w, ref) < TOL), rel_rows(w, ref)
    assert np.allclose(bsum, np.sum(np.abs(ref[:, HALO:HALO + n_level // 2]) ** 2, axis=1), rtol=1e-5)
