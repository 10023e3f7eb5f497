"""
ctypes binding of libqi_b200.so (C ABI declared in include/qi_b200.h).

There is deliberately no fallback: if the shared library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C quantum_inferno_b200/csrc``) ``load()`` raises
``RuntimeError``.
"""
import ctypes
import os

import numpy as np

QI_F32, QI_F64 = 0, 1
QI_CONV_LINEAR_SAME, QI_CONV_CIRC_CORR = 0, 1
QI_CONV_PLAIN_ONLY = 0x100
SUBSAMPLE_METHOD_CODE = {"nth": 0, "average": 1, "median": 2, "max": 3, "min": 4}
QI_ABI_VERSION = 5
QI_N_CATEGORIES = 7
CATEGORY_NAMES = ("fft_fwd", "inv_first", "inv_mid", "inv_last", "info", "stft", "other")

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libqi_b200.so")

# numpy mirror of `QiAtomBand`
ATOM_BAND = np.dtype([("omega", "<f8"), ("p_re", "<f8"), ("p_im", "<f8"), ("amp", "<f8"),
                      ("analytic", "<i4"), ("reserved", "<i4")], align=True)

STX_BAND = np.dtype([("sigma", "<f8"), ("shift", "<i8")], align=True)
MR_BAND = np.dtype([("omega", "<f8"), ("scale", "<f8"), ("amp", "<f8"), ("level", "<i4"), ("reserved", "<i4")],
                   align=True)

QI_IIR_BA, QI_IIR_SOS, QI_IIR_MAX_STATE = 0, 1, 16
IIR_FILTER = np.dtype([("form", "<i4"), ("n_coef", "<i4"), ("b", "<f8", (17,)), ("a", "<f8", (17,)),
                       ("sos", "<f8", (8, 6)), ("zi", "<f8", (16,))], align=True)

_c_vp, _c_i64, _c_int, _c_sz, _c_dbl = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_size_t, ctypes.c_double

# name -> (restype, argtypes); every symbol include/qi_b200.h declares
SIGNATURES = {
    "qi_abi_version": (_c_int, []),
    "qi_error_string": (ctypes.c_char_p, [_c_int]),
    "qi_last_cuda_error": (ctypes.c_char_p, []),
    "qi_launch_count": (_c_i64, []),
    "qi_profile_enable": (_c_int, [_c_int]),
    "qi_profile_read": (_c_int, [_c_vp, _c_vp]),
    "qi_fft_c2c": (_c_int, [_c_vp, _c_vp, _c_i64, _c_int, _c_int, _c_int, _c_vp]),
    "qi_cwt_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int, _c_int, _c_int, _c_int, _c_int]),
    "qi_cwt_fft": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_dbl, _c_int, _c_int,
                            _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_int, _c_vp]),
    "qi_atoms_time": (_c_int, [_c_vp, _c_int, _c_i64, _c_dbl, _c_int, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_abs_log2": (_c_int, [_c_vp, _c_i64, _c_int, _c_int, _c_int, _c_dbl, _c_vp, _c_vp]),
    "qi_cwt_multirate_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_vp, _c_int]),
    "qi_cwt_multirate": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp,
                                  _c_vp, _c_vp, _c_dbl, _c_int, _c_vp, _c_sz, _c_vp]),
    "qi_stx_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int, _c_int, _c_int]),
    "qi_stx_fft": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_int,
                            _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_int, _c_vp]),
    "qi_stx_multirate_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_vp, _c_int]),
    "qi_stx_multirate": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_stft": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_dbl, _c_int,
                         _c_int, _c_int, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_stft_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int, _c_int]),
    "qi_istft_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int, _c_int, _c_int]),
    "qi_istft": (_c_int, [_c_vp, _c_i64, _c_i64, _c_vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_i64, _c_i64, _c_i64,
                          _c_i64, _c_int, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_power_reduce": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "qi_shannon": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_int, _c_vp, _c_dbl, _c_dbl,
                            _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "qi_power_bits": (_c_int, [_c_vp, _c_i64, _c_i64, _c_int, _c_vp, _c_dbl, _c_vp, _c_vp]),
    "qi_tdr_marginal": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_vp, _c_vp, _c_vp]),
    "qi_rfft": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_stx_windows_workspace_bytes": (_c_sz, [_c_int]),
    "qi_stx_windows": (_c_int, [_c_vp, _c_int, _c_i64, _c_int, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_subsample": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_i64, _c_int, _c_int, _c_vp, _c_i64, _c_vp]),
    "qi_extrema": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_int, _c_vp, _c_vp]),
    "qi_local_maxima": (_c_int, [_c_vp, _c_i64, _c_int, _c_dbl, _c_int, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp]),
    "qi_select_peaks_by_distance": (_c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_vp]),
    "qi_filtfilt_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int, _c_int]),
    "qi_filtfilt": (_c_int, [_c_vp, _c_i64, _c_i64, _c_i64, _c_vp, _c_int, _c_dbl, _c_int, _c_vp, _c_vp, _c_sz, _c_vp]),
    "qi_synth_chirp": (_c_int, [_c_i64, _c_i64, _c_i64, _c_i64, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _c_int, _c_int, _c_vp, _c_vp,
                                _c_vp]),
    "qi_divide": (_c_int, [_c_vp, _c_i64, _c_int, _c_dbl, _c_vp, _c_vp]),
}


def bind(lib):
    """Attach restype/argtypes for every exported entry point; raises AttributeError if one is missing."""
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load():
    """Return the bound CUDA library, loading it on first use."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"quantum_inferno_b200: CUDA library {LIB_PATH} is not built; there is no CPU fallback. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo root.")
        lib = bind(ctypes.CDLL(LIB_PATH))
        if lib.qi_abi_version() != QI_ABI_VERSION:
            raise RuntimeError("quantum_inferno_b200: libqi_b200.so ABI version mismatch; rebuild it")
        _lib = lib
    return _lib


def check(lib, code, what):
    """Map a QI_ERR_* return code to the exception the Python API promises."""
    if code == 0:
        return
    msg = lib.qi_error_string(code).decode()
    if code == -3:
        raise RuntimeError(f"{what}: {msg}: {lib.qi_last_cuda_error().decode()}")
    if code in (-1, -2):
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: {msg}")
