"""
Records that do not start on a 16-byte boundary.  A CUDA tensor slice such as ``x[k:k + N]`` or
``x[k:k + C * N].view(C, N)`` reaches the C ABI as it is, ``k * itemsize`` bytes past the allocation's alignment; a
kernel that reads it with vector loads faults on the device (misaligned address, and the CUDA context is lost).

CPU tier: tests/emul/alignment_driver.py runs every public entry point with its inputs at element offsets k = 1, 2, 3
(float32 / complex64) and k = 1 (float64) -- every residue mod 16 a slice can have -- against the emulator built with
AddressSanitizer and -fsanitize=alignment (tests/emul/asan_check.sh), in one subprocess: the emulator library is cached
per process, and a sanitizer abort must not take pytest with it.  Each case holds the offset call to the float64 oracle
at the family's usual tolerance and to the aligned call (bit-identical where the same kernels run).

GPU tier (-m gpu): the multirate paths, exact CWT and STFT on real CUDA slices of a 2^20-sample record.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.emul.alignment_driver import C_ABI_CASE, CASES

HERE = os.path.dirname(os.path.abspath(__file__))
FS = 800.0


def _sanitizer_available():
    if shutil.which("g++") is None:
        return False
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    return os.path.isabs(asan) and os.path.exists(asan)


@pytest.fixture(scope="module")
def alignment_results(tmp_path_factory):
    """{case: (status, message)} from the sanitized driver.  A case that aborts the process (sanitizer report) is
    recorded with the report, and the cases after it run in a fresh process."""
    if not _sanitizer_available():
        pytest.skip("no g++ / libasan")
    env = dict(os.environ, TMPDIR=str(tmp_path_factory.mktemp("align")))
    script = [os.path.join(HERE, "emul", "asan_check.sh"), os.path.join(HERE, "emul", "alignment_driver.py")]
    results, pending = {}, list(CASES) + [C_ABI_CASE]
    while pending:
        run = subprocess.run(["bash"] + script + pending, capture_output=True, text=True, env=env, timeout=1800)
        started = None
        for line in run.stdout.splitlines():
            parts = line.split(" ", 3)
            if len(parts) < 3 or parts[0] != "CASE":
                continue
            if parts[2] == "START":
                started = parts[1]
            else:
                results[parts[1]] = (parts[2], parts[3] if len(parts) > 3 else "")
                started = None
        out = run.stdout + run.stderr
        reports = [ln for ln in out.splitlines() if "runtime error:" in ln or "AddressSanitizer" in ln]
        if started is not None:                    # the process died inside this case
            results[started] = ("ABORT", "\n".join(reports) or out[-3000:])
        elif run.returncode != 0 or reports or "alignment run done" not in run.stdout:
            for name in pending:
                results.setdefault(name, ("ERROR", out[-3000:]))
        pending = [name for name in pending if name not in results]
    return results


@pytest.mark.parametrize("case", list(CASES))
def test_offset_input(alignment_results, case):
    status, message = alignment_results[case]
    assert status == "PASS", message


def test_multirate_c_abi_rejects_misaligned_records(alignment_results):
    """qi_cwt_multirate called directly (alignment_driver.c_abi_case, in the sanitized subprocess): records 4, 8 and
    12 bytes off a 16-byte boundary and a stride of N + 2 samples are QI_ERR_ARG; 16 bytes off with a stride of N + 4 runs."""
    status, message = alignment_results[C_ABI_CASE]
    assert status == "PASS", message


# ----------------------------------------------------------------------------- GPU tier: real CUDA slices
GPU_N = 1 << 20


def _synth(n, seed):
    k = np.arange(n)
    chirp = 0.5 * np.cos(2 * np.pi * (1.0 * k / FS + 0.5 * (199.0 / (n / FS)) * (k / FS) ** 2))
    return np.cos(2 * np.pi * 60.0 / FS * k) + chirp + np.random.default_rng(seed).standard_normal(n) / 16.0


@pytest.fixture(scope="module")
def gpu_record():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    from quantum_inferno_b200 import _runtime
    _runtime._runtime = None
    assert _runtime.get_runtime().name == "cuda"
    x = np.ascontiguousarray(np.stack([_synth(GPU_N, 1), _synth(GPU_N, 2)[::-1]]))
    return torch, x


def _slice(torch, x, k, dtype):
    """base[k:k + C*N].view(C, N): the record k elements past the allocation's (256-byte aligned) start."""
    base = torch.empty(x.size + 8, dtype=dtype, device="cuda")
    s = base[k:k + x.size].view(*x.shape)
    s.copy_(torch.from_numpy(x).to(dtype))
    assert s.data_ptr() % 16 == (k * s.element_size()) % 16
    return s


def _aligned(torch, x, dtype):
    return torch.from_numpy(x).to(device="cuda", dtype=dtype)


def _np(t):
    return t.detach().cpu().numpy()


ORACLE_BANDS = (0, 1, 10, 30, 47)           # 0 and 1: record-long truncated atoms (the multirate edge rows)
_SPECTRUM = {}


def _oracle_band(x, band, freq):
    """Complex CWT row of record 0 from the float64 oracle (single bands at full size, as test_gpu_parity.py does)."""
    from oracle import qi_oracle as orc
    if "xf" not in _SPECTRUM:
        _SPECTRUM["xf"] = np.fft.fft(x[0], 2 * x.shape[1])
    return orc.cwt_band(_SPECTRUM["xf"], 3, x.shape[1], freq[band], FS)


@pytest.mark.gpu
@pytest.mark.parametrize("truncated", ["multirate", "exact"])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_gpu_multirate_entropy_on_slices(gpu_record, k, truncated):
    """The headline call on a misaligned slice: the same power plane as on an aligned copy, bit for bit, the same sums
    and entropy up to the order of atomic additions, and single bands against the oracle at the float32 tolerance
    (1e-4 relative L2 on power)."""
    torch, x = gpu_record
    from quantum_inferno_b200 import cwt_entropy
    kw = dict(dtype="float32", method="multirate", truncated_bands=truncated)
    r = cwt_entropy.cwt_power_entropy(3, _slice(torch, x, k, torch.float32), FS, **kw)
    a = cwt_entropy.cwt_power_entropy(3, _aligned(torch, x, torch.float32), FS, **kw)
    assert torch.equal(r.power, a.power)
    # the fp64 sums are accumulated with atomics: equal up to the order of the additions, and so is the information
    # plane normalised by their total (the bounds of test_gpu_parity.py::test_host_pipelined_equals_resident)
    assert torch.allclose(r.info, a.info, rtol=0, atol=1e-5)
    assert torch.allclose(r.band_power, a.band_power, rtol=1e-12) and torch.allclose(r.total_power, a.total_power, rtol=1e-12)
    assert torch.allclose(r.band_entropy_bits, a.band_entropy_bits, rtol=0, atol=1e-9)
    assert torch.allclose(r.power.double().sum(-1), r.band_power, rtol=1e-5)
    for band in ORACLE_BANDS:
        row = np.abs(_oracle_band(x, band, r.frequency_hz)) ** 2
        p = _np(r.power[0, band]).astype(np.float64)
        assert np.linalg.norm(p - row) / np.linalg.norm(row) < 1e-4, band
        assert abs(float(r.band_power[0, band]) - row.sum()) / row.sum() < 1e-4, band


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3])
def test_gpu_multirate_complex_on_slices(gpu_record, k):
    torch, x = gpu_record
    from quantum_inferno_b200 import styx_cwt
    f, _, c = styx_cwt.cwt_complex_any_scale_pow2(3, _slice(torch, x, k, torch.float32), FS, dtype="float32",
                                                  method="multirate")
    _, _, ca = styx_cwt.cwt_complex_any_scale_pow2(3, _aligned(torch, x, torch.float32), FS, dtype="float32",
                                                   method="multirate")
    assert torch.equal(c, ca)
    for band in ORACLE_BANDS:
        row = _oracle_band(x, band, f)
        got = _np(c[0, band])
        assert np.linalg.norm(np.abs(got) ** 2 - np.abs(row) ** 2) / np.linalg.norm(np.abs(row) ** 2) < 1e-4, band


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 3])
def test_gpu_exact_cwt_and_stft_on_slices(gpu_record, k):
    """Exact CWT (float32, single bands against the oracle as in test_gpu_parity.py::test_cwt_band_limited_routes_large)
    and the STFT with 512 / 1024 / 2048-point and generic frames (tests/test_emul_api.py::test_stft_interior_fused_path)."""
    torch, x = gpu_record
    from oracle import qi_oracle as orc
    from quantum_inferno_b200 import styx_cwt, styx_fft
    s = _slice(torch, x, k, torch.float32)
    f, _, c = styx_cwt.cwt_complex_any_scale_pow2(3, s, FS, dtype="float32")
    _, _, ca = styx_cwt.cwt_complex_any_scale_pow2(3, _aligned(torch, x, torch.float32), FS, dtype="float32")
    assert torch.equal(c, ca)
    for band in ORACLE_BANDS:
        row = _oracle_band(x, band, f)
        noise = orc.reference_axis_phase_noise(3, x.shape[1], f[band], FS)
        assert np.max(np.abs(_np(c[0, band]) - row)) / np.max(np.abs(row)) < 2e-5 + noise, band
    xs = x[:, : 1 << 16]
    s = _slice(torch, xs, k, torch.float32)
    for geom in ((512, None, None), (1024, None, None), (2048, None, None), (200, 150, 256)):
        _, _, z = styx_fft.stft_complex_pow2(s, FS, *geom, alpha=0.25, dtype="float32")
        _, _, za = styx_fft.stft_complex_pow2(_aligned(torch, xs, torch.float32), FS, *geom, alpha=0.25, dtype="float32")
        assert torch.equal(z, za), geom
        z0 = orc.stft_complex_pow2(xs, FS, *geom, alpha=0.25)[2]
        zz = _np(z)
        assert zz.shape == z0.shape and np.max(np.abs(zz - z0)) / np.max(np.abs(z0)) < 3e-6, geom
