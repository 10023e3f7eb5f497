"""TEST INFRASTRUCTURE: every public entry point with its input record k elements past a 256-byte boundary, for
tests/test_input_alignment.py (run through tests/emul/asan_check.sh, i.e. against the emulator built with AddressSanitizer
and -fsanitize=alignment).

On the device a slice such as ``x[2:2 + N]`` reaches the C ABI at an offset of ``2 * itemsize`` bytes; the plain emulator
runtime always copies into a 256-byte aligned buffer, so no other CPU test sees such a record.  ``OffsetRuntime`` does
what the slice does.  Each case compares the offset call with the float64 oracle (or the golden vectors) at the
tolerance the family's existing test uses, and with the aligned call: bit-identical where the same kernels run.

A last case calls qi_cwt_multirate directly with misaligned records: it must refuse them before any kernel runs.

Usage: alignment_driver.py [case ...]   (no argument: every case).  One line per case on stdout:
``CASE <id> START``, then ``CASE <id> PASS`` or ``CASE <id> FAIL <message>``; an alignment or memory error aborts the
process after START."""
import functools
import os
import sys
import traceback

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from oracle import qi_oracle as orc  # noqa: E402
from quantum_inferno_b200 import _runtime, cwt_entropy, styx_cwt, styx_fft, styx_stx, tfr_info  # noqa: E402
from quantum_inferno_b200.utilities import picker, sampling  # noqa: E402
from quantum_inferno_b200.utilities import short_time_fft as stf  # noqa: E402
from tests.emul.emul_runtime import EmulRuntime  # noqa: E402

FS = 800.0
GOLDEN = os.path.join(ROOT, "tests", "golden")


class OffsetRuntime(EmulRuntime):
    """Inputs start ``k * itemsize`` bytes past a 256-byte boundary, as a slice ``base[k:k + n]`` of a device
    allocation does.  Outputs and scratch stay 256-byte aligned, as they are from the caching allocator."""

    def __init__(self, k):
        super().__init__()
        self.k = int(k)
        self.offset_inputs = 0

    def asarray(self, x, dtype):
        shape = tuple(int(s) for s in np.shape(x))
        dt = np.dtype(dtype)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dt.itemsize
        off = self.k * dt.itemsize
        raw = self._aligned((nbytes + off,), np.uint8)
        out = raw[off:off + nbytes].view(dt).reshape(shape)
        out[...] = np.asarray(x)
        self.offset_inputs += 1
        return out


@functools.lru_cache(maxsize=None)
def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - b)) / np.max(np.abs(b)))


def l2(a, b):
    return float(np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b))


def synth(n, seed=0):
    k = np.arange(n)
    chirp = 0.5 * np.cos(2 * np.pi * (1.0 * k / FS + 0.5 * (199.0 / (n / FS)) * (k / FS) ** 2))
    return np.cos(2 * np.pi * 60.0 / FS * k) + chirp + np.random.default_rng(seed).standard_normal(n) / 16.0


X2 = np.stack([synth(1 << 13, 1), synth(1 << 13, 2)[::-1]])          # two records: the second one at stride N
X3000 = synth(3000, 3)


@functools.lru_cache(maxsize=None)
def cwt_ref(n):
    return orc.cwt_complex_any_scale_pow2(3, X3000 if n == 3000 else X2[0], FS)


@functools.lru_cache(maxsize=None)
def cwt_entropy_ref(c):
    return orc.cwt_power_entropy(3, X2[c], FS)


@functools.lru_cache(maxsize=None)
def stx_ref(c):
    return orc.stx_complex_any_scale_pow2(3, X2[c], FS)


# ----------------------------------------------------------------------------- families
# Each family: run(dtype) -> dict of outputs (numpy), check(out, dtype) against the oracle, and which outputs must be
# bit-identical to the aligned call ("same", default all).  Where the alignment of an input selects another kernel
# (qi_pick.cu 128-bit subsample loads), that output is left to the oracle check.  "order" gives the tolerance of outputs
# accumulated with fp64 atomics, or normalised by such a sum: they equal the aligned call's up to the order of the
# additions.
FAMILIES = {}


def family(name, dtypes, same=None, order=None):
    def deco(cls):
        cls.name, cls.dtypes, cls.same, cls.order = name, dtypes, same, order or (lambda key, dt: None)
        FAMILIES[name] = cls
        return cls
    return deco


def entropy_out(r):
    return dict(power=r.power, info=r.info, band_power=r.band_power, total=r.total_power,
                band_entropy=r.band_entropy_bits)


# band and total power are fp64 atomic sums; the information plane is normalised by that total and the entropy sums are
# atomic too (tests/test_gpu_parity.py::test_host_pipelined_equals_resident holds them to the same bounds)
def entropy_order(key, dt):
    return dict(band_power=dict(rtol=1e-12, atol=0.0), total=dict(rtol=1e-12, atol=0.0),
                info=dict(rtol=0.0, atol=1e-5), band_entropy=dict(rtol=0.0, atol=1e-9)).get(key)


def normalised_order(*prefixes):
    """Outputs whose keys start with one of ``prefixes`` are planes divided by an fp64 sum that several CTAs add up
    with atomics (the total of qi_power_reduce over the rows, the sum of squares of qi_tdr_marginal): the quotient may
    round the other way.  The others must be bit-identical."""
    def order(key, dt):
        if not str(key).startswith(prefixes):
            return None
        return dict(rtol=1e-12, atol=1e-12) if dt == "float64" else dict(rtol=1e-6, atol=1e-6)
    return order


def check_mr_entropy(out):
    """tests/test_emul_api.py::test_multirate_fused_path."""
    for c in range(2):
        ref = cwt_entropy_ref(c)
        assert l2(out["power"][c], ref["power"]) < 2e-5
        assert abs(float(out["band_entropy"][c].sum()) - ref["entropy_bits"]) < 1e-4
        assert np.max(np.abs(out["band_power"][c] - ref["band_sum"]) / ref["band_sum"].max()) < 1e-5
        assert abs(out["total"][c] - ref["total"]) / ref["total"] < 1e-5
        per_band = np.linalg.norm(out["power"][c] - ref["power"], axis=1) / np.linalg.norm(ref["power"], axis=1)
        assert per_band.max() < 5e-5, per_band.max()


@family("mr_entropy_edge_rows", ("float32",), order=entropy_order)
class MrEntropyEdge:
    """The fused multirate path with the truncated (edge) rows on the fast path: edge_load reads the record."""
    @staticmethod
    def run(dt):
        return entropy_out(cwt_entropy.cwt_power_entropy(3, X2, FS, dtype=dt, method="multirate",
                                                         truncated_bands="multirate"))

    @staticmethod
    def check(out, dt):
        from quantum_inferno_b200 import _plan, scales_dyadic
        n = X2.shape[1]
        freq = scales_dyadic.log_frequency_hz_from_fft_points(frequency_sample_hz=FS, fft_points=n, scale_order=3)
        bands, _, _, _ = _plan.gabor_bands(3, n, freq, FS, "norm", dt)
        assert np.count_nonzero(bands["analytic"] == 0) > 0              # the table does have edge rows
        check_mr_entropy(out)


@family("mr_entropy_exact_truncated", ("float32",), order=entropy_order)
class MrEntropyExactTrunc:
    """Multirate without the fused information pass, the truncated rows recomputed by the exact path."""
    @staticmethod
    def run(dt):
        return entropy_out(cwt_entropy.cwt_power_entropy(3, X2, FS, dtype=dt, method="multirate",
                                                         truncated_bands="exact"))

    @staticmethod
    def check(out, dt):
        check_mr_entropy(out)


@family("mr_complex", ("float32",))
class MrComplex:
    @staticmethod
    def run(dt):
        f, t, c = styx_cwt.cwt_complex_any_scale_pow2(3, X2[0], FS, dtype=dt, method="multirate")
        return dict(f=f, c=c)

    @staticmethod
    def check(out, dt):
        """tests/test_emul_api.py::test_multirate_complex_output."""
        fr, _, cr = cwt_ref(1 << 13)
        c = out["c"]
        assert c.dtype == np.complex64 and np.array_equal(out["f"], fr)
        assert np.max(np.abs(c - cr)) / np.max(np.abs(cr)) < 5e-5
        assert np.linalg.norm(np.abs(c) ** 2 - np.abs(cr) ** 2) / np.linalg.norm(np.abs(cr) ** 2) < 2e-5


def cwt_exact_family(n):
    @family(f"cwt_exact_{n}", ("float32", "float64"))
    class CwtExact:
        @staticmethod
        def run(dt):
            f, t, c = styx_cwt.cwt_complex_any_scale_pow2(3, X3000 if n == 3000 else X2[0], FS, dtype=dt)
            return dict(f=f, c=c)

        @staticmethod
        def check(out, dt):
            """tests/test_emul_api.py::test_cwt_band_limited_routes: every band against the oracle."""
            fr, _, cr = cwt_ref(n)
            assert np.array_equal(out["f"], fr)
            err = np.max(np.abs(out["c"] - cr), axis=1) / np.max(np.abs(cr), axis=1)
            assert err.max() < (1e-10 if dt == "float64" else 2e-5), err.max()


cwt_exact_family(1 << 13)
cwt_exact_family(3000)


def stx_family(name, method, dtypes):
    @family(name, dtypes)
    class Stx:
        @staticmethod
        def run(dt):
            f, t, c = styx_stx.stx_complex_any_scale_pow2(3, X2, FS, dtype=dt, method=method)
            return dict(f=f, c=c)

        @staticmethod
        def check(out, dt):
            for ch in range(2):
                f0, _, c0 = stx_ref(ch)
                c = out["c"][ch]
                assert np.array_equal(out["f"], f0)
                if method == "multirate":          # tests/test_emul_api.py::test_stx_multirate
                    assert np.linalg.norm(c - c0) / np.linalg.norm(c0) < 1e-5
                    assert max(np.linalg.norm(c[b] - c0[b]) / np.linalg.norm(c0[b]) for b in range(len(f0))) < 2e-5
                else:                              # tests/_extra_checks.py::check_stx_band_limited_routes
                    err = np.max(np.abs(c - c0), axis=-1) / np.max(np.abs(c0), axis=-1)
                    assert err.max() < (1e-10 if dt == "float64" else 2e-5), err.max()


stx_family("stx_plain", "plain", ("float32", "float64"))
stx_family("stx_band_limited", "exact", ("float32", "float64"))
stx_family("stx_multirate", "multirate", ("float32",))


@family("stx_power_entropy", ("float32", "float64"), order=entropy_order)
class StxEntropy:
    @staticmethod
    def run(dt):
        return entropy_out(cwt_entropy.stx_power_entropy(3, X2, FS, dtype=dt))

    @staticmethod
    def check(out, dt):
        """tests/_extra_checks.py::check_stx_power_entropy."""
        tol_p, tol_bits = (1e-10, 1e-9) if dt == "float64" else (1e-4, 1e-3)
        for ch in range(2):
            p_ref = np.abs(stx_ref(ch)[2]) ** 2
            s_ref = p_ref.sum()
            pdf = p_ref / s_ref
            info_ref = -np.log2(pdf + np.finfo(np.float64).eps)
            assert l2(out["power"][ch], p_ref) < tol_p
            assert abs(float(out["total"][ch]) - s_ref) / s_ref < tol_p
            assert abs(float(out["band_entropy"][ch].sum()) - float(np.sum(pdf * info_ref))) < tol_bits
            strong = p_ref > 1e-3 * p_ref.max()
            info = np.asarray(out["info"][ch], dtype=np.float64)
            assert np.max(np.abs(info - info_ref)[strong]) < (1e-8 if dt == "float64" else 1e-3)


STFT_GEOMETRIES = ((512, None, None), (1024, None, None), (2048, None, None), (200, 150, 256))
X_STFT = np.random.default_rng(0).standard_normal((2, 12000)) + 3.0 + np.cos(2 * np.pi * 60 / FS * np.arange(12000))


@functools.lru_cache(maxsize=None)
def stft_ref(seg, ov, nfft):
    return orc.stft_complex_pow2(X_STFT, FS, seg, ov, nfft, alpha=0.25)


@family("stft", ("float32", "float64"))
class Stft:
    """512 / 1024 / 2048-point frames (compile-time instantiations) and one generic geometry."""
    @staticmethod
    def run(dt):
        return {g: styx_fft.stft_complex_pow2(X_STFT, FS, *g, alpha=0.25, dtype=dt)[2] for g in STFT_GEOMETRIES}

    @staticmethod
    def check(out, dt):
        """tests/test_emul_api.py::test_stft_interior_fused_path."""
        for g in STFT_GEOMETRIES:
            z0 = stft_ref(*g)[2]
            assert out[g].shape == z0.shape and rel(out[g], z0) < (1e-12 if dt == "float64" else 3e-6), g


@family("stft_tukey", ("float32", "float64"))
class StftTukey:
    """stft_tukey on the record, istft_tukey on the (complex) spectrum: both inputs at the offset."""
    @staticmethod
    def run(dt):
        g = golden("stft_tukey")
        out = {}
        for i, (m, ov, alpha) in enumerate(g["cases"]):
            scal = None if str(g["case_scaling"][i]) == "none" else str(g["case_scaling"][i])
            out[f"mag{i}"] = stf.stft_tukey(g["x"], FS, alpha, int(m), int(ov), scal, str(g["case_padding"][i]),
                                            dtype=dt)[2]
            out[f"xr{i}"] = stf.istft_tukey(g[f"c{i}_spec"], FS, alpha, int(m), int(ov), scal, dtype=dt)[1]
        return out

    @staticmethod
    def check(out, dt):
        """tests/test_emul_api.py::test_short_time_fft_tukey."""
        g = golden("stft_tukey")
        for i in range(len(g["cases"])):
            assert rel(out[f"mag{i}"], g[f"c{i}_mag"]) < (1e-12 if dt == "float64" else 2e-5), i
            assert np.max(np.abs(out[f"xr{i}"] - g[f"c{i}_xr"])) < (1e-14 if dt == "float64" else 2e-5), i


@family("shannon", ("float32", "float64"), order=normalised_order("glob_", "tdr_"))
class Shannon:
    @staticmethod
    def run(dt):
        p = golden("info")["power"]
        out = {}
        for tag, obj in (("glob", tfr_info.shannon_stft_from_tfr_power(p, dtype=dt)),
                         ("ptime", tfr_info.ShannonStftPerTime(p, dtype=dt)),
                         ("pfreq", tfr_info.ShannonStftPerFreq(p, dtype=dt))):
            out.update({f"{tag}_info": obj.info, f"{tag}_bits": obj.shannon_bits, f"{tag}_isnr": obj.isnr,
                        f"{tag}_esnr": obj.esnr})
        tdr, _ = tfr_info.shannon_tdr_fft(golden("info")["x1024"], dtype=dt)
        out.update(tdr_info=tdr.info, tdr_ent=tdr.entropy, tdr_marg=tdr.marginal)
        return out

    @staticmethod
    def check(out, dt):
        """tests/test_emul_api.py::test_tfr_info (float32: the total bits, as that test does)."""
        g = golden("info")
        if dt == "float32":
            assert abs(float(out["glob_bits"].sum()) - float(g["glob_bits"].sum())) < 1e-3
            return
        for tag in ("glob", "ptime", "pfreq"):
            assert np.max(np.abs(out[f"{tag}_info"] - g[tag + "_info"])) < 1e-10
            assert rel(out[f"{tag}_bits"], g[tag + "_bits"]) < 1e-12
            assert np.max(np.abs(out[f"{tag}_isnr"] - g[tag + "_isnr"])) < 1e-10
            assert rel(out[f"{tag}_esnr"], g[tag + "_esnr"]) < 1e-12
        assert np.max(np.abs(out["tdr_info"] - g["tdr_info"])) < 1e-10 and rel(out["tdr_ent"], g["tdr_ent"]) < 1e-12
        assert rel(out["tdr_marg"], g["tdr_marg"]) < 1e-13


SUB_FACTORS = (2, 4, 8, 16, 32, 64, 128, 129, 1000)
P_SUB = np.random.default_rng(9).standard_normal((3, 5 * 1024 + 72))
P_SUB[0, 1000] = np.nan
P_SUB[1, 2049] = np.inf
P_SUB[2, 64:128] = -3.5


@family("subsample", ("float32", "float64"), same=lambda key: not key.endswith("average"))
class Subsample:
    """Every method; power-of-two factors on 16-byte aligned rows take the 128-bit loads of qi_pick.cu, other rows
    the scalar kernels: the average (a sum) is held to the oracle's tolerance, the selections are exact."""
    @staticmethod
    def run(dt):
        return {f"{f}_{m}": sampling.subsample_2d(P_SUB.astype(dt), f, m) for f in SUB_FACTORS
                for m in ("average", "median", "max", "min", "nth")}

    @staticmethod
    def check(out, dt):
        """tests/_pick_checks.py::check_subsample_vector_path / check_subsample_vs_oracle."""
        p = P_SUB.astype(dt)
        for f in SUB_FACTORS:
            for m in ("median", "max", "min", "nth"):
                want = orc.subsample_2d(p, f, m)
                assert out[f"{f}_{m}"].dtype == want.dtype and np.array_equal(out[f"{f}_{m}"], want, equal_nan=True), (f, m)
            a, b = out[f"{f}_average"], orc.subsample_2d(p, f, "average")
            assert a.shape == b.shape and a.dtype == b.dtype
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isinf(a), np.isinf(b))
            ok = np.isfinite(b)
            assert np.allclose(a[ok], b[ok], rtol=2e-6 if dt == "float32" else 1e-13,
                               atol=1e-7 if dt == "float32" else 1e-15), f


N_PICK = 30000
X_PICK = np.round(np.random.default_rng(11).standard_normal(N_PICK) * 8.0) / 8.0 + 4.0 * np.sin(np.arange(N_PICK) * 2e-3)
PICK_CASES = (("log2", 6, 0.001), ("amplitude", 2, 0.05), ("log2", 1, 1.0))


@family("find_peaks_with_bits", ("float64",))
class Peaks:
    @staticmethod
    def run(dt):
        return {c: picker.find_peaks_with_bits(X_PICK.astype(dt), 1000.0, *c) for c in PICK_CASES}

    @staticmethod
    def check(out, dt):
        """tests/_pick_checks.py::check_picker_vs_oracle: the same peak indices."""
        for c in PICK_CASES:
            assert np.array_equal(out[c], orc.find_peaks_with_bits(X_PICK, 1000.0, *c)), c


@family("butterworth", ("float32", "float64"))
class Butter:
    @staticmethod
    def run(dt):
        from tests._iir_checks import BA_CALLS
        x = golden("iir")["x"].astype(dt)
        if dt == "float32":
            return dict(lowpass_100=styx_fft.butter_lowpass(x, FS, 100.0))
        return {name: call(styx_fft, x) for name, call in BA_CALLS.items()}

    @staticmethod
    def check(out, dt):
        """tests/_iir_checks.py::check_butter_golden."""
        from tests._iir_checks import _judge, peak_rel
        g = golden("iir")
        if dt == "float32":
            assert out["lowpass_100"].dtype == np.float32 and peak_rel(out["lowpass_100"], g["lowpass_100_truth"]) < 3e-7
            return
        for name, y in out.items():
            _judge(y, g[f"{name}_ref"], g[f"{name}_truth"], name)


@family("decimate_timeseries", ("float64",))
class Decimate:
    @staticmethod
    def run(dt):
        return {q: sampling.decimate_timeseries(golden("synth")["x"], q) for q in (2, 4, 10)}

    @staticmethod
    def check(out, dt):
        """tests/_synth_checks.py::check_decimate_golden."""
        for q, y in out.items():
            want = golden("synth")[f"dec_{q}"]
            assert y.shape == want.shape and rel(y, want) < 1e-11, q


@family("shannon_fft_bluestein", ("float64",))
class Bluestein:
    @staticmethod
    def run(dt):
        ff = tfr_info.ShannonFFT(X3000[:777], dtype=dt)
        return dict(sig=ff.sig, marginal=ff.marginal, info=ff.info)

    @staticmethod
    def check(out, dt):
        """tests/_extra_checks.py::check_shannon_1d_all_attributes (777 samples, the Bluestein route)."""
        ref = orc.shannon_fft(X3000[:777])
        assert rel(out["sig"], ref.sig) < 1e-10 and rel(out["marginal"], ref.marginal) < 1e-10
        assert np.max(np.abs(out["info"] - ref.info)) < 1e-9


# ----------------------------------------------------------------------------- cases
def offsets(dt):
    """Element offsets: every residue mod 16 that a slice of this dtype can have."""
    return (1,) if dt == "float64" else (1, 2, 3)


CASES = {f"{fam.name}-{dt}-k{k}": (fam, dt, k) for fam in FAMILIES.values() for dt in fam.dtypes for k in offsets(dt)}
C_ABI_CASE = "qi_cwt_multirate_c_abi"


def c_abi_case():
    """qi_cwt_multirate reads the record with 128-bit loads: a record that is not 16-byte aligned, or a stride that is
    not a multiple of 4 samples, is an argument error (a fault on the device); an aligned one at any other offset runs."""
    from quantum_inferno_b200 import _lib, _plan, scales_dyadic
    QI_OK, QI_ERR_ARG = 0, -1                      # include/qi_b200.h
    rt = EmulRuntime()
    C, N = 2, 1 << 13
    freq = scales_dyadic.log_frequency_hz_from_fft_points(frequency_sample_hz=FS, fft_points=N, scale_order=3)
    bands = np.ascontiguousarray(_plan.multirate_bands(3, N, freq, FS, "norm")[0], dtype=_lib.MR_BAND)
    B = len(bands)
    nbytes = rt.lib.qi_cwt_multirate_workspace_bytes(C, N, bands.ctypes.data, B)
    ws = rt.workspace(nbytes)
    base = rt.zeros((C * (N + 4) + 16,), "float32")
    base[: C * (N + 4)] = np.random.default_rng(0).standard_normal(C * (N + 4))
    power = rt.empty((C, B, N), "float32")

    def call(first, stride):
        return rt.lib.qi_cwt_multirate(rt.ptr(base) + 4 * first, C, N, stride, bands.ctypes.data, B, rt.ptr(power),
                                       None, None, None, None, None, None, 0.0, 0, rt.ptr(ws), nbytes, rt.stream())

    for first in (1, 2, 3):                        # 4, 8, 12 bytes past a 256-byte boundary
        assert call(first, N) == QI_ERR_ARG, first
    assert call(0, N + 2) == QI_ERR_ARG, "stride N + 2"                  # the second record 8 bytes off
    assert call(4, N + 4) == QI_OK                                       # 16 bytes off, stride 4 samples past N: runs
    assert np.all(np.isfinite(power)) and np.all(power.sum(axis=2) > 0)


@functools.lru_cache(maxsize=None)
def aligned_call(name, dt):
    with _runtime.use_runtime(EmulRuntime()):
        return FAMILIES[name].run(dt)


def run_case(fam, dt, k):
    want = aligned_call(fam.name, dt)
    rt = OffsetRuntime(k)
    with _runtime.use_runtime(rt):
        got = fam.run(dt)
    assert rt.offset_inputs > 0, "no input went through the offset runtime"
    fam.check(got, dt)
    for key, a in got.items():
        b = want[key]
        assert a.shape == b.shape and a.dtype == b.dtype, key
        tol = fam.order(key, dt)
        if tol is not None:
            assert np.allclose(a, b, **tol), f"{key}: differs from the aligned call"
        elif fam.same is None or fam.same(str(key)):
            assert np.array_equal(a, b, equal_nan=True), f"{key}: differs from the aligned call"


def main(names):
    for name in names or list(CASES) + [C_ABI_CASE]:
        print(f"CASE {name} START", flush=True)
        try:
            if name == C_ABI_CASE:
                c_abi_case()
            else:
                run_case(*CASES[name])
        except Exception as e:  # noqa: BLE001 -- reported per case, the next case still runs
            msg = (f"{type(e).__name__}: {e}" + " | " + traceback.format_exc().strip().splitlines()[-3]).replace("\n", " ")
            print(f"CASE {name} FAIL {msg}", flush=True)
        else:
            print(f"CASE {name} PASS", flush=True)
    print("alignment run done", flush=True)


if __name__ == "__main__":
    main(sys.argv[1:])
