"""TEST INFRASTRUCTURE: the long-frame STFT route (frames too long for one CTA: frame means, forward passes with the
frame-pair gather, Hermitian split and Welch sums; pair gather, inverse passes with the dual-window sink) once per
dtype, small records, for tests/emul/asan_check.sh (AddressSanitizer + alignment build of the CPU emulator)."""
import os
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..", "..")))
import numpy as np  # noqa: E402
from tests.emul.emul_runtime import EmulRuntime  # noqa: E402
from quantum_inferno_b200 import _lib, _runtime, styx_fft  # noqa: E402
from quantum_inferno_b200.utilities import short_time_fft as stf  # noqa: E402

FS = 800.0
rng = np.random.default_rng(0)
with _runtime.use_runtime(EmulRuntime()) as rt:
    x = rng.standard_normal((2, 30000)) + 1.0
    for dt in ("float64", "float32"):
        # hop not a divisor of the segment, zero padding to nfft, an odd frame count (the last pair half empty)
        f, t, z = styx_fft.stft_complex_pow2(x, FS, 10000, 3000, 16384, dtype=dt)
        print("stft", dt, z.shape, flush=True)
        f, p = styx_fft.welch_power_pow2(x, FS, 16384, dtype=dt)
        print("welch", dt, p.shape, flush=True)
        obj = stf.get_stft_object_tukey(FS, 0.25, 16384, 8192, dtype=dt)
        obj.phase_shift = 3
        s = obj.stft(x[0])
        xr = obj.istft(s, k1=20000)
        print("tukey round trip", dt, s.shape, xr.shape, flush=True)
    # the smallest workspace: one frame pair per channel, a chunk per pair
    lib = rt.lib
    code = _lib.QI_F64
    win = rt.asarray(np.hanning(16384), "float64")
    n_frames = 5
    ws_min = lib.qi_stft_workspace_bytes(2, 2, 16384, code)
    ws = rt.workspace(ws_min)
    out = rt.empty((2, 8193, n_frames), "complex128")
    acc = rt.empty((2, 8193), "float64")
    rc = lib.qi_stft(rt.ptr(x), 2, 30000, 30000, rt.ptr(win), 16384, 6000, 16384, n_frames, 8192, 1.0, 1, 5, code,
                     rt.ptr(out), rt.ptr(acc), rt.ptr(ws), ws_min, None)
    print("minimum workspace", rc, flush=True)
    assert rc == 0
print("asan run done")
