"""
Thin drivers: marshal host-side plans and device buffers into the C-ABI calls of libqi_b200.so.
Everything here enqueues work on the current CUDA stream and returns device buffers.
"""
import ctypes

import numpy as np

from . import _lib
from ._runtime import COMPLEX_OF, DTYPE_CODE, get_runtime

# bytes of scratch we are willing to spend on batching several bands per launch
WORKSPACE_TARGET_BYTES = 8 << 30
EPS64 = float(np.finfo(np.float64).eps)
EPS32 = float(np.finfo(np.float32).eps)


def _as_2d(rt, sig, dt):
    """Accept [N] or [C, N]; returns (device buffer [C, N], was_1d)."""
    x = rt.asarray(sig, dt)
    if x.ndim == 1:
        return rt.reshape(x, (1, x.shape[0])), True
    if x.ndim != 2:
        raise ValueError("sig_wf must be 1-D [points] or 2-D [channels, points]")
    return x, False


def _group_for(lib_fn_bytes, n_bands, target=WORKSPACE_TARGET_BYTES):
    """Largest bands-per-launch whose workspace stays under `target` (at least 1)."""
    group = n_bands
    while group > 1 and lib_fn_bytes(group) > target:
        group = max(1, group // 2)
    return group


def cwt_fft(sig, bands, fs, dt, conv_mode=_lib.QI_CONV_LINEAR_SAME, want_complex=True, want_power=False,
            want_band_sum=False, rt=None, out_complex=None, out_power=None, band_sum=None, plain_only=False):
    """Run qi_cwt_fft.  sig: device [C, N]; bands: numpy ATOM_BAND table.  Returns dict of device buffers
    (complex [C,B,N], power [C,B,N], band_sum [C,B] float64).  plain_only=True keeps every band on the three
    full-length passes (the band-limited routes of csrc/qi_cwt_fast.cuh off: for comparisons)."""
    rt = rt or get_runtime()
    lib = rt.lib
    if plain_only:
        conv_mode |= _lib.QI_CONV_PLAIN_ONLY
    C, N = int(sig.shape[0]), int(sig.shape[1])
    bands = np.ascontiguousarray(bands, dtype=_lib.ATOM_BAND)
    B = len(bands)
    n_tab = int(np.count_nonzero(bands["analytic"] == 0))
    code = DTYPE_CODE[dt]

    def ws_bytes(group):
        return lib.qi_cwt_workspace_bytes(C, N, B, n_tab, group, conv_mode, code)

    group = _group_for(ws_bytes, B)
    nbytes = ws_bytes(group)
    ws = rt.workspace(nbytes)
    if want_complex and out_complex is None:
        out_complex = rt.empty((C, B, N), COMPLEX_OF[dt])
    if want_power and out_power is None:
        out_power = rt.empty((C, B, N), dt)
    if want_band_sum and band_sum is None:
        band_sum = rt.empty((C, B), "float64")
    rc = lib.qi_cwt_fft(rt.ptr(sig), C, N, N, bands.ctypes.data, B, float(fs), conv_mode, code,
                        rt.ptr(out_complex), rt.ptr(out_power), rt.ptr(band_sum), rt.ptr(ws), nbytes, group,
                        rt.stream())
    _lib.check(lib, rc, "qi_cwt_fft")
    return {"complex": out_complex, "power": out_power, "band_sum": band_sum}


def atoms_time(bands, n_points, fs, dt, xtime=None, rt=None):
    """Time-domain atoms [B, n_points] complex (qi_atoms_time)."""
    rt = rt or get_runtime()
    lib = rt.lib
    bands = np.ascontiguousarray(bands, dtype=_lib.ATOM_BAND)
    B = len(bands)
    out = rt.empty((B, n_points), COMPLEX_OF[dt])
    ws = rt.workspace(max(4096, 128 * B))
    xt = None if xtime is None else rt.asarray(np.asarray(xtime, dtype=np.float64), "float64")
    rc = lib.qi_atoms_time(bands.ctypes.data, B, int(n_points), float(fs), DTYPE_CODE[dt], rt.ptr(xt), rt.ptr(out),
                           rt.ptr(ws), max(4096, 128 * B), rt.stream())
    _lib.check(lib, rc, "qi_atoms_time")
    return out


def stx_fft(sig, bands, dt, want_complex=True, want_power=False, want_band_sum=False, rt=None, method="exact",
            out_power=None):
    """Run qi_stx_fft (method="exact": band-limited voices where the window allows, full-length passes otherwise;
    method="plain": full-length passes for every band) or qi_stx_multirate (method="multirate": float32, records of
    2^m >= 4096 samples, decimated voices + packed polyphase interpolation)."""
    rt = rt or get_runtime()
    lib = rt.lib
    C, N = int(sig.shape[0]), int(sig.shape[1])
    bands = np.ascontiguousarray(bands, dtype=_lib.STX_BAND)
    B = len(bands)
    code = DTYPE_CODE[dt]
    if method == "multirate":
        if dt != "float32" or want_band_sum or N < 4096:
            raise ValueError("method='multirate' needs dtype float32, records of 2^m >= 4096 samples and no band sums")
        nbytes = lib.qi_stx_multirate_workspace_bytes(C, N, bands.ctypes.data, B)
        ws = rt.workspace(nbytes)
        out_c = rt.empty((C, B, N), COMPLEX_OF[dt]) if want_complex else None
        out_p = rt.empty((C, B, N), dt) if want_power else None
        rc = lib.qi_stx_multirate(rt.ptr(sig), C, N, N, bands.ctypes.data, B, rt.ptr(out_c), rt.ptr(out_p), rt.ptr(ws),
                                  nbytes, rt.stream())
        _lib.check(lib, rc, "qi_stx_multirate")
        return {"complex": out_c, "power": out_p, "band_sum": None}
    if method not in ("exact", "plain"):
        raise ValueError("method must be 'exact', 'plain' or 'multirate'")

    def ws_bytes(group):
        return lib.qi_stx_workspace_bytes(C, N, B, group, code)

    group = _group_for(ws_bytes, B)
    nbytes = ws_bytes(group)
    ws = rt.workspace(nbytes)
    out_c = rt.empty((C, B, N), COMPLEX_OF[dt]) if want_complex else None
    out_p = (out_power if out_power is not None else rt.empty((C, B, N), dt)) if want_power else None
    bsum = rt.empty((C, B), "float64") if want_band_sum else None
    rc = lib.qi_stx_fft(rt.ptr(sig), C, N, N, bands.ctypes.data, B, code, rt.ptr(out_c), rt.ptr(out_p), rt.ptr(bsum),
                        rt.ptr(ws), nbytes, -group if method == "plain" else group, rt.stream())
    _lib.check(lib, rc, "qi_stx_fft")
    return {"complex": out_c, "power": out_p, "band_sum": bsum}


def stx_windows(bands, n_points, dt, rt=None):
    rt = rt or get_runtime()
    lib = rt.lib
    bands = np.ascontiguousarray(bands, dtype=_lib.STX_BAND)
    B = len(bands)
    out = rt.empty((B, n_points), COMPLEX_OF[dt])
    nbytes = max(4096, lib.qi_stx_windows_workspace_bytes(B))
    ws = rt.workspace(nbytes)
    rc = lib.qi_stx_windows(bands.ctypes.data, B, int(n_points), DTYPE_CODE[dt], rt.ptr(out), rt.ptr(ws), nbytes,
                            rt.stream())
    _lib.check(lib, rc, "qi_stx_windows")
    return out


def stft(sig, window, nperseg, hop, nfft, n_frames, pad_left, scale, dt, detrend=True, psd=False, rt=None, roll=0):
    """sig: device [C, N]; window: numpy float64 [nperseg].  Returns complex [C, nfft/2+1, n_frames]
    (psd=False) or the fp64 accumulator [C, nfft/2+1] of sum_frames |X|^2 (psd=True).  roll: see qi_stft."""
    rt = rt or get_runtime()
    lib = rt.lib
    C, N = int(sig.shape[0]), int(sig.shape[1])
    K = nfft // 2 + 1
    win = rt.asarray(np.asarray(window, dtype=np.float64), dt)
    out = None if psd else rt.empty((C, K, n_frames), COMPLEX_OF[dt])
    acc = rt.empty((C, K), "float64") if psd else None
    rc = lib.qi_stft(rt.ptr(sig), C, N, N, rt.ptr(win), int(nperseg), int(hop), int(nfft), int(n_frames),
                     int(pad_left), float(scale), 1 if detrend else 0, int(roll), DTYPE_CODE[dt], rt.ptr(out),
                     rt.ptr(acc), rt.stream())
    _lib.check(lib, rc, "qi_stft")
    return acc if psd else out


def istft(spec, dual_win, nperseg, hop, nfft, roll, first_start, frame_lo, frame_hi, k0, n_out, dt, rt=None):
    """spec: device complex [C, nfft/2+1, P]; dual_win: numpy float64 [nperseg].  Returns real [C, n_out]: the
    overlap-add of frames [frame_lo, frame_hi) restricted to samples k0 .. k0 + n_out - 1 (see qi_istft)."""
    rt = rt or get_runtime()
    lib = rt.lib
    C, P = int(spec.shape[0]), int(spec.shape[2])
    dwin = rt.asarray(np.asarray(dual_win, dtype=np.float64), dt)
    out = rt.empty((C, int(n_out)), dt)
    nbytes = lib.qi_istft_workspace_bytes(C, P, int(nperseg), DTYPE_CODE[dt])
    ws = rt.workspace(nbytes)
    rc = lib.qi_istft(rt.ptr(spec), C, P, rt.ptr(dwin), int(nperseg), int(hop), int(nfft), int(roll), int(first_start),
                      int(frame_lo), int(frame_hi), int(k0), int(n_out), DTYPE_CODE[dt], rt.ptr(out), rt.ptr(ws), nbytes,
                      rt.stream())
    _lib.check(lib, rc, "qi_istft")
    return out


def power_reduce(power, dt, rows=False, cols=False, total=False, maximum=False, rt=None):
    """power: device [M, F, T].  Returns dict with requested fp64 buffers row_sum[M,F], col_sum[M,T], total[M], max[M]."""
    rt = rt or get_runtime()
    lib = rt.lib
    M, F, T = (int(s) for s in power.shape)
    rs = rt.empty((M, F), "float64") if rows else None
    cs = rt.empty((M, T), "float64") if cols else None
    tt = rt.empty((M,), "float64") if total else None
    mx = rt.empty((M,), "float64") if maximum else None
    rc = lib.qi_power_reduce(rt.ptr(power), M, F, T, DTYPE_CODE[dt], rt.ptr(rs), rt.ptr(cs), rt.ptr(tt), rt.ptr(mx),
                             rt.stream())
    _lib.check(lib, rc, "qi_power_reduce")
    return {"row_sum": rs, "col_sum": cs, "total": tt, "max": mx}


def shannon(power, dt, mode, norm, deg_free, eps=EPS64, planes=("info", "bits", "isnr", "esnr"), entropy_sum=False,
            rt=None, out_info=None):
    rt = rt or get_runtime()
    lib = rt.lib
    M, F, T = (int(s) for s in power.shape)
    out = {k: (rt.empty((M, F, T), dt) if (k in planes and not (k == "info" and out_info is not None)) else None)
           for k in ("pdf", "info", "bits", "isnr", "esnr")}
    if out_info is not None:
        out["info"] = out_info
    es = rt.empty((M, F), "float64") if entropy_sum else None
    rc = lib.qi_shannon(rt.ptr(power), M, F, T, DTYPE_CODE[dt], int(mode), rt.ptr(norm), float(eps), float(deg_free),
                        rt.ptr(out["pdf"]), rt.ptr(out["info"]), rt.ptr(out["bits"]), rt.ptr(out["isnr"]), rt.ptr(out["esnr"]), rt.ptr(es),
                        rt.stream())
    _lib.check(lib, rc, "qi_shannon")
    out["entropy_sum"] = es
    return out


def power_bits(power, dt, max_value, eps=EPS64, rt=None):
    """power: device [M, ...]; max_value: device fp64 [M].  log2(P+eps) - log2(max+eps)."""
    rt = rt or get_runtime()
    lib = rt.lib
    M = int(power.shape[0])
    per = int(np.prod(power.shape[1:]))
    out = rt.empty(power.shape, dt)
    rc = lib.qi_power_bits(rt.ptr(power), M, per, DTYPE_CODE[dt], rt.ptr(max_value), float(eps), rt.ptr(out), rt.stream())
    _lib.check(lib, rc, "qi_power_bits")
    return out


def tdr_marginal(sig, dt, rt=None):
    rt = rt or get_runtime()
    lib = rt.lib
    M, n = int(sig.shape[0]), int(sig.shape[1])
    ss = rt.empty((M,), "float64")
    sn = rt.empty((M, n), dt)
    mg = rt.empty((M, n), dt)
    rc = lib.qi_tdr_marginal(rt.ptr(sig), M, n, n, DTYPE_CODE[dt], rt.ptr(ss), rt.ptr(sn), rt.ptr(mg), rt.stream())
    _lib.check(lib, rc, "qi_tdr_marginal")
    return sn, mg, ss


def fft_c2c(buf, dt, inverse=False, rt=None):
    """qi_fft_c2c over the rows of a complex [M, 2^m] device buffer: forward = natural in, bit-reversed out; inverse =
    bit-reversed in, natural out, scaled by 1 / n."""
    rt = rt or get_runtime()
    M, n = int(buf.shape[0]), int(buf.shape[1])
    out = rt.empty((M, n), COMPLEX_OF[dt])
    rc = rt.lib.qi_fft_c2c(rt.ptr(buf), rt.ptr(out), M, n.bit_length() - 1, int(bool(inverse)), DTYPE_CODE[dt], rt.stream())
    _lib.check(rt.lib, rc, "qi_fft_c2c")
    return out


def _rfft_bluestein(sig, dt, rt):
    """One-sided DFT of records whose length n is not a power of two (scipy.fft.rfft takes any n, reference
    tfr_info.py:177): Bluestein's chirp-z identity  X[k] = c[k] * sum_m (x[m] c[m]) conj(c)[k - m],  c[m] = exp(-pi i m^2 / n),
    as one circular convolution of length 2^p >= 2n - 1 through qi_fft_c2c (both spectra in bit-reversed order, so their
    product is too).  The chirp is a host table with the phase reduced in integers (m^2 mod 2n), like the STFT windows."""
    M, n = int(sig.shape[0]), int(sig.shape[1])
    m = np.arange(n, dtype=np.int64)
    ph = ((m * m) % (2 * n)).astype(np.float64) / n
    c_host = np.cos(np.pi * ph) - 1j * np.sin(np.pi * ph)
    F = 1 << (2 * n - 2).bit_length()
    b_host = np.zeros(F, dtype=np.complex128)
    b_host[:n] = np.conj(c_host)
    b_host[F - n + 1:] = np.conj(c_host[1:][::-1])
    cdt = COMPLEX_OF[dt]
    c = rt.asarray(c_host, cdt)
    a = rt.zeros((M, F), cdt)
    a[:, :n] = sig * c
    A = fft_c2c(a, dt, rt=rt)
    B = fft_c2c(rt.asarray(b_host[None, :], cdt), dt, rt=rt)
    y = fft_c2c(A * B, dt, inverse=True, rt=rt)
    k = n // 2 + 1
    return y[:, :k] * c[:k]


def rfft(sig, dt, rt=None):
    rt = rt or get_runtime()
    lib = rt.lib
    M, n = int(sig.shape[0]), int(sig.shape[1])
    if n & (n - 1):
        return _rfft_bluestein(sig, dt, rt)
    out = rt.empty((M, n // 2 + 1), COMPLEX_OF[dt])
    nbytes = M * n * (8 if dt == "float32" else 16)
    ws = rt.workspace(nbytes)
    rc = lib.qi_rfft(rt.ptr(sig), M, n, n, DTYPE_CODE[dt], rt.ptr(out), rt.ptr(ws), nbytes, rt.stream())
    _lib.check(lib, rc, "qi_rfft")
    return out


def abs_log2(buf, dt, is_complex, eps=EPS64, square=False, rt=None, signed=False):
    """log2(|x| + eps) (utilities/rescaling.py:13-20), |x|^2 + eps when square=True (1) or |x| + eps when square=2,
    elementwise on the device."""
    rt = rt or get_runtime()
    lib = rt.lib
    n = int(np.prod(buf.shape))
    out = rt.empty(buf.shape, dt)
    rc = lib.qi_abs_log2(rt.ptr(buf), n, DTYPE_CODE[dt], 2 if signed else (1 if is_complex else 0), int(square), float(eps),
                         rt.ptr(out), rt.stream())
    _lib.check(lib, rc, "qi_abs_log2")
    return out


def cwt_multirate(sig, bands, want_power=True, want_complex=False, want_band_sum=False, rt=None, out_power=None,
                  want_info=False, out_info=None, allreduce=None, eps=EPS64):
    """Run qi_cwt_multirate (float32).  sig: device float32 [C, N]; bands: numpy MR_BAND table.

    want_info fuses the information plane -log2(P/S + eps) and the per-band entropy sums into the pass that writes
    the power plane.  S (per record) is estimated from the decimated band outputs first; with ``allreduce`` (band
    sharding) the call is split in two phases and the estimate is all-reduced in between."""
    rt = rt or get_runtime()
    lib = rt.lib
    C, N = int(sig.shape[0]), int(sig.shape[1])
    if rt.ptr(sig) % 16:
        # the kernels read the record as float4; a slice x[k:] of a device buffer can start anywhere on a 4-byte grid
        buf = rt.empty((C, N), "float32")
        buf[...] = sig
        sig = buf
    bands = np.ascontiguousarray(bands, dtype=_lib.MR_BAND)
    B = len(bands)
    nbytes = lib.qi_cwt_multirate_workspace_bytes(C, N, bands.ctypes.data, B)
    if nbytes == 0:
        raise ValueError("qi_cwt_multirate: unsupported size or band table")
    ws = rt.workspace(nbytes)
    if (want_power or want_info) and out_power is None:
        out_power = rt.empty((C, B, N), "float32")
    out_c = rt.empty((C, B, N), "complex64") if want_complex else None
    bsum = rt.empty((C, B), "float64") if (want_band_sum or want_info) else None
    ent = est = total = None
    if want_info:
        if out_info is None:
            out_info = rt.empty((C, B, N), "float32")
        ent, est, total = rt.empty((C, B), "float64"), rt.empty((C, B), "float64"), rt.empty((C,), "float64")

    def call(phase):
        rc = lib.qi_cwt_multirate(rt.ptr(sig), C, N, N, bands.ctypes.data, B, rt.ptr(out_power), rt.ptr(out_c),
                                  rt.ptr(bsum), rt.ptr(out_info) if want_info else None, rt.ptr(ent), rt.ptr(est),
                                  rt.ptr(total), float(eps), phase, rt.ptr(ws), nbytes, rt.stream())
        _lib.check(lib, rc, "qi_cwt_multirate")

    if want_info and allreduce is not None:
        call(1)                     # QI_MR_PHASE_ESTIMATE
        allreduce(total)            # the one collective of the band-sharded case
        call(2)                     # QI_MR_PHASE_EXPAND
    else:
        call(0)
    return {"complex": out_c, "power": out_power, "band_sum": bsum, "info": out_info if want_info else None,
            "entropy_sum": ent, "band_sum_est": est, "total": total}


def subsample(buf, factor, method, dt, rt=None):
    """Run qi_subsample on a device buffer [M, n] (utilities/sampling.py:13-50,87-120).  Returns [M, n_out]."""
    rt = rt or get_runtime()
    lib = rt.lib
    M, n = int(buf.shape[0]), int(buf.shape[1])
    factor = int(factor)
    n_out = -(-n // factor) if method == "nth" else n // factor
    out = rt.empty((M, n_out), dt)
    if n_out > 0 and M > 0:
        rc = lib.qi_subsample(rt.ptr(buf), M, n, n, factor, _lib.SUBSAMPLE_METHOD_CODE[method], DTYPE_CODE[dt],
                              rt.ptr(out), n_out, rt.stream())
        _lib.check(lib, rc, "qi_subsample")
    return out


def extrema(buf, dt, rt=None):
    """Run qi_extrema on a device buffer [M, n]: host float64 array [M, 4] = (nanmax, nanmin, nanmax|x|, #NaN)."""
    rt = rt or get_runtime()
    lib = rt.lib
    M, n = int(buf.shape[0]), int(buf.shape[1])
    out = rt.empty((M, 4), "float64")
    rc = lib.qi_extrema(rt.ptr(buf), M, n, n, DTYPE_CODE[dt], rt.ptr(out), rt.stream())
    _lib.check(lib, rc, "qi_extrema")
    return rt.to_numpy(out)


def local_maxima(buf, dt, height=None, rt=None, first_capacity=1 << 16):
    """Run qi_local_maxima on a device record [n]: host arrays (positions int64 ascending, x there float64) of the
    plateau-aware local maxima with x[peak] >= height (scipy.signal.find_peaks(x, height=height))."""
    rt = rt or get_runtime()
    lib = rt.lib
    n = int(buf.shape[0])
    cap = max(1, min(first_capacity, n // 2 + 1))
    count = rt.empty((1,), "int64")
    use_h = height is not None
    h = float(height) if use_h else 0.0
    while True:
        peaks = rt.empty((cap,), "int64")
        values = rt.empty((cap,), "float64")
        rc = lib.qi_local_maxima(rt.ptr(buf), n, DTYPE_CODE[dt], h, int(use_h), rt.ptr(peaks), rt.ptr(values), cap,
                                 rt.ptr(count), rt.stream())
        _lib.check(lib, rc, "qi_local_maxima")
        found = int(rt.to_numpy(count)[0])
        if found <= cap:
            pos, val = rt.to_numpy(peaks)[:found], rt.to_numpy(values)[:found]
            order = np.argsort(pos, kind="stable")
            return pos[order], val[order]
        cap = found


def divide(buf, dt, divisor, rt=None):
    """out = buf / divisor in the buffer's dtype (qi_divide; utilities/picker.py:46-53)."""
    rt = rt or get_runtime()
    lib = rt.lib
    n = int(np.prod(buf.shape))
    out = rt.empty(buf.shape, dt)
    if n:
        rc = lib.qi_divide(rt.ptr(buf), n, DTYPE_CODE[dt], float(divisor), rt.ptr(out), rt.stream())
        _lib.check(lib, rc, "qi_divide")
    return out


def filtfilt(sig, dt, padlen, tukey_alpha=None, b=None, a=None, sos=None, zi=None, rt=None):
    """Run qi_filtfilt on a device buffer [M, n]: scipy.signal.filtfilt(b, a, x) (ba form) or sosfiltfilt(sos, x) along
    the last axis, optionally after a Tukey taper.  b, a, sos, zi: host float64 (designed by the caller)."""
    rt = rt or get_runtime()
    lib = rt.lib
    M, n = int(sig.shape[0]), int(sig.shape[1])
    filt = np.zeros(1, dtype=_lib.IIR_FILTER)
    if sos is None:
        b, a = np.atleast_1d(np.asarray(b, dtype=np.float64)), np.atleast_1d(np.asarray(a, dtype=np.float64))
        ntaps = max(len(a), len(b))
        if ntaps - 1 > _lib.QI_IIR_MAX_STATE or ntaps < 2:
            raise ValueError(f"filter order must be 1..{_lib.QI_IIR_MAX_STATE}")
        filt["form"], filt["n_coef"] = _lib.QI_IIR_BA, ntaps
        filt["b"][0, :len(b)] = b / a[0]
        filt["a"][0, :len(a)] = a / a[0]
        n_state = ntaps - 1
    else:
        sos = np.asarray(sos, dtype=np.float64)
        if sos.ndim != 2 or sos.shape[1] != 6 or not 1 <= sos.shape[0] <= _lib.QI_IIR_MAX_STATE // 2:
            raise ValueError(f"sos must be [1..{_lib.QI_IIR_MAX_STATE // 2}, 6]")
        filt["form"], filt["n_coef"] = _lib.QI_IIR_SOS, sos.shape[0]
        filt["sos"][0, :sos.shape[0]] = sos
        n_state = 2 * sos.shape[0]
    zi = np.asarray(zi, dtype=np.float64).reshape(-1)
    filt["zi"][0, :n_state] = zi[:n_state]
    if n <= padlen:
        raise ValueError(f"The length of the input vector x must be greater than padlen, which is {padlen}.")
    nbytes = lib.qi_filtfilt_workspace_bytes(M, n, int(padlen), n_state)
    ws = rt.workspace(nbytes)
    out = rt.empty((M, n), dt)
    rc = lib.qi_filtfilt(rt.ptr(sig), M, n, n, filt.ctypes.data, int(padlen), -1.0 if tukey_alpha is None else float(tukey_alpha),
                         DTYPE_CODE[dt], rt.ptr(out), rt.ptr(ws), nbytes, rt.stream())
    _lib.check(lib, rc, "qi_filtfilt")
    return out


def synth_chirp(n, dt, omega, t_center=0.0, half_gamma=0.0, chirp_scale=1.0, gauss=False, want_imag=False, rt=None):
    """Run qi_synth_chirp: device buffer [1, n] (real part) or [2, n] (real, imaginary) of the Gabor chirp / tone
    (synth/benchmark_signals.py:92-101, :323-335)."""
    rt = rt or get_runtime()
    lib = rt.lib
    n = int(n)
    out = rt.empty((2 if want_imag else 1, n), dt)
    itemsize = 4 if dt == "float32" else 8
    rc = lib.qi_synth_chirp(1, n, n, 0, float(t_center), float(omega), float(half_gamma), float(chirp_scale),
                            int(bool(gauss)), DTYPE_CODE[dt], rt.ptr(out), rt.ptr(out) + n * itemsize if want_imag else None,
                            rt.stream())
    _lib.check(lib, rc, "qi_synth_chirp")
    return out
