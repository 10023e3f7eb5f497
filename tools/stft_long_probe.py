"""
Timing of the long-frame STFT route (frames too long for one CTA: csrc/qi_stft.cu, multi-pass FFTs of frame pairs) on
16 x 2^24 samples resident in HBM, float32 and float64, nfft = 2^13 .. 2^20 with nperseg = nfft and 50 % overlap:
  * Welch (the fp64 |X|^2 accumulator only, scipy.signal.welch's frames: no boundary extension);
  * the complex STFT (scipy.signal.stft's frames: nperseg / 2 zeros at both ends, padded to whole hops).
CUDA-event time per call after warm-up, algorithmic bytes (complex output + one read of the record; Welch: the record)
and GB/s, and the fraction of the 6547 GB/s copy peak of DESIGN.md.  The card's name, power limit and SM clock come from
a read-only nvidia-smi query in the same run.

It also times the one-CTA tile kernel at its largest size (float32 2^13, float64 2^12) against the long-frame route
forced at the same size: a variant of the STFT library built into a temporary directory with QI_STFT_TILE_MAX_NFFT=2048.

    python tools/stft_long_probe.py            # markdown table on stdout
"""
import ctypes
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from quantum_inferno_b200 import _lib, _plan, _runtime  # noqa: E402

C, N = 16, 1 << 24
PEAK_GBPS = 6547.0
CSRC = os.path.join(ROOT, "quantum_inferno_b200", "csrc")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi unavailable"


def forced_long_lib():
    """libqi_stft with every frame longer than 2048 points on the long-frame route (temporary directory)"""
    out = os.path.join(tempfile.mkdtemp(prefix="qi_stft_long_"), "libqi_stft_forced.so")
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                    "--expt-relaxed-constexpr", "-shared", "-DQI_STFT_TILE_MAX_NFFT=2048", "-I", CSRC,
                    os.path.join(CSRC, "qi_stft.cu"), os.path.join(CSRC, "qi_capi.cu"), "-o", out],
                   check=True, capture_output=True)
    lib = ctypes.CDLL(out)
    for name in ("qi_stft", "qi_stft_workspace_bytes"):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SIGNATURES[name]
    return lib


class Case:
    def __init__(self, rt, lib, x, dt, nfft, welch):
        self.rt, self.lib, self.x, self.nfft, self.welch = rt, lib, x, nfft, welch
        self.code = _runtime.DTYPE_CODE[dt]
        hop = nfft // 2
        self.n_frames, self.pad_left, _ = _plan.stft_frames(N, nfft, nfft - hop, boundary_zeros=not welch,
                                                            padded=not welch)
        K = nfft // 2 + 1
        win = _plan.periodic_window("tukey", 0.25, nfft)
        self.win = torch.from_numpy(win).to(device=x.device, dtype=x.dtype)
        cdt = torch.complex64 if dt == "float32" else torch.complex128
        self.out = None if welch else torch.empty((C, K, self.n_frames), dtype=cdt, device=x.device)
        self.acc = torch.empty((C, K), dtype=torch.float64, device=x.device) if welch else None
        full = lib.qi_stft_workspace_bytes(C, self.n_frames, nfft, self.code)
        least = lib.qi_stft_workspace_bytes(C, 2, nfft, self.code)
        self.ws_bytes = min(full, max(1 << 30, least))           # as _driver.stft
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=x.device) if self.ws_bytes else None
        self.route = "tile" if full == 0 else "long"
        isz = x.element_size()
        self.bytes = C * N * isz + (0 if welch else C * K * self.n_frames * 2 * isz)

    def __call__(self):
        p = lambda t: None if t is None else t.data_ptr()              # noqa: E731
        rc = self.lib.qi_stft(p(self.x), C, N, N, p(self.win), self.nfft, self.nfft // 2, self.nfft, self.n_frames,
                              self.pad_left, 1.0, 1, 0, self.code, p(self.out), p(self.acc), p(self.ws),
                              self.ws_bytes, self.rt.stream())
        assert rc == 0, rc


def time_ms(fn, warm=2, reps=10):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def row(label, dt, nfft, case, ms):
    gbps = case.bytes / ms / 1e6
    return (f"| {label} | {dt} | 2^{nfft.bit_length() - 1} | {case.route} | {case.n_frames} | {ms:.3f} | "
            f"{case.bytes / 1e9:.3f} | {gbps:.0f} | {gbps / PEAK_GBPS:.3f} |")


def main():
    rt = _runtime.get_runtime()
    lib = rt.lib
    print(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)")
    print(f"record: {C} x 2^{N.bit_length() - 1} samples, nperseg = nfft, 50 % overlap, detrend, Tukey(0.25) window")
    print()
    header = ("| call | dtype | nfft | route | frames | ms | algorithmic GB | GB/s | of 6547 GB/s |\n"
              "|---|---|---|---|---|---|---|---|---|")
    print(header)
    forced = forced_long_lib()
    cross = []
    for dt in ("float32", "float64"):
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.randn((C, N), generator=g, dtype=getattr(torch, dt), device="cuda") + 3.0
        for welch in (True, False):
            for m in range(13, 21):
                case = Case(rt, lib, x, dt, 1 << m, welch)
                print(row("welch" if welch else "stft", dt, 1 << m, case, time_ms(case)), flush=True)
                del case
                torch.cuda.empty_cache()
            # the tile kernel at its largest size against the long-frame route at the same size
            top = 1 << 13 if dt == "float32" else 1 << 12
            for which, L in (("tile", lib), ("long (forced)", forced)):
                case = Case(rt, L, x, dt, top, welch)
                cross.append(row(("welch" if welch else "stft") + f" {which}", dt, top, case, time_ms(case)))
                del case
                torch.cuda.empty_cache()
        del x
        torch.cuda.empty_cache()
    print()
    print("Largest tile size, both routes:")
    print()
    print(header)
    for r in cross:
        print(r)


if __name__ == "__main__":
    main()
