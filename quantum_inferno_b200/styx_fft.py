"""
STFT / Gaussian-taper STFT / Welch spectra on the B200 -- drop-in for the FFT functions of
``quantum_inferno.styx_fft`` (reference styx_fft.py:14-57, :152-266).

The reference delegates to scipy.signal.stft / welch; here the frame gather, detrend, window, FFT and
scaling are one CUDA kernel (csrc/qi_stft.cu) with scipy's exact edge semantics: zero extension by
nperseg//2 on both sides, zero padding to a whole number of hops, per-frame mean removal after the
extension, DFT-even (periodic) window, scale 1/sum(window).  ``nfft`` must be a power of two (it always is
through the *_pow2 defaults).  Frames longer than one CTA's shared memory holds (float32 nfft > 8192, float64 > 4096)
take multi-pass FFTs of frame pairs through a scratch buffer instead, with the same edge semantics.  Keyword-only
extra: ``dtype``.

The Butterworth pre-filters of the reference module (styx_fft.py:60-149: Tukey taper, ``scipy.signal.butter``,
``scipy.signal.filtfilt``) run on the device too: scipy designs the (b, a) taps and the steady-state initial
conditions on the host (a few dozen numbers; ``_iir.py`` re-factors the rounded taps into second-order sections so
that the blocked evaluation stays well conditioned), and the taper, the odd extension and the two recursions over the
record are the blocked parallel scan of csrc/qi_iir.cu (fp64 arithmetic; 2-D [channels, points] input accepted).
"""
from typing import Tuple

import warnings

import numpy as np

from . import _driver, _iir, _plan
from .scales_dyadic import cycles_from_order
from ._runtime import dtype_name, finish, get_runtime
from .utilities.calculations import get_num_points
from .utilities.rescaling import is_power_of_two, to_log2_with_epsilon


def _pow2_defaults(segment_points, overlap_points, nfft_points):
    if nfft_points is None:
        nfft_points = int(2 ** np.ceil(np.log2(segment_points)))
    if overlap_points is None:
        overlap_points = int(segment_points / 2)
    return overlap_points, nfft_points


def _spectral(sig_wf, fs, window, nperseg, noverlap, nfft, dtype, welch=False):
    """scipy.signal._spectral_helper for the two call patterns the reference uses."""
    if nperseg < 1:
        raise ValueError("nperseg must be a positive integer")
    if nfft < nperseg:
        raise ValueError("nfft must be greater than or equal to nperseg.")
    if not is_power_of_two(int(nfft)):
        raise ValueError(f"the STFT kernel needs nfft = 2^m, got {nfft}")
    rt = get_runtime(sig_wf)
    dt = dtype_name(dtype)
    want_numpy = not rt.is_device_array(sig_wf)
    x = rt.asarray(sig_wf, dt)
    lead = tuple(int(s) for s in x.shape[:-1])
    n_points = int(x.shape[-1])
    if nperseg > n_points:
        # scipy.signal._spectral_py._triage_segments: warn, shorten the segment to the record, rebuild the window;
        # noverlap and nfft stay as given (reference styx_fft.py:175-187 hands them to scipy.signal.stft unchanged)
        warnings.warn(f"nperseg = {nperseg:d} is greater than input length  = {n_points:d}, using nperseg = {n_points:d}",
                      stacklevel=3)
        nperseg = n_points
        if noverlap >= nperseg:
            raise ValueError("noverlap must be less than nperseg.")
    x2 = rt.reshape(x, (int(np.prod(lead)) if lead else 1, n_points))
    win = _plan.periodic_window(window[0], window[1], nperseg)
    n_frames, pad_left, ext = _plan.stft_frames(n_points, nperseg, noverlap, boundary_zeros=not welch,
                                                padded=not welch)
    freqs = np.fft.rfftfreq(nfft, 1 / fs)
    hop = nperseg - noverlap
    if welch:
        acc = _driver.stft(x2, win, nperseg, hop, nfft, n_frames, pad_left, 1.0, dt, psd=True, rt=rt)
        return freqs, acc, win, n_frames, lead, rt, want_numpy
    z = _driver.stft(x2, win, nperseg, hop, nfft, n_frames, pad_left, 1.0 / win.sum(), dt, rt=rt)
    z = rt.reshape(z, lead + (nfft // 2 + 1, n_frames))
    return freqs, _plan.stft_time_axis(ext, nperseg, noverlap, fs), finish(rt, z, want_numpy)


def stft_complex_pow2(sig_wf, frequency_sample_rate_hz: float, segment_points: int, overlap_points: int = None,
                      nfft_points: int = None, alpha: float = 0.25, *, dtype=None):
    """Tukey-window STFT, 50 % overlap and power-of-two FFT by default (reference styx_fft.py:152-187).

    :return: frequency_stft_hz [nfft/2+1], time_stft_s [T], stft_complex [..., nfft/2+1, T]
    """
    overlap_points, nfft_points = _pow2_defaults(segment_points, overlap_points, nfft_points)
    return _spectral(sig_wf, frequency_sample_rate_hz, ("tukey", alpha), segment_points, overlap_points,
                     nfft_points, dtype)


def gtx_complex_pow2(sig_wf, frequency_sample_rate_hz: float, segment_points: int, gaussian_sigma: int = None,
                     overlap_points: int = None, nfft_points: int = None, *, dtype=None):
    """Gaussian-taper STFT (reference styx_fft.py:190-227).

    :return: frequency_stft_hz, time_stft_s, stft_complex
    """
    overlap_points, nfft_points = _pow2_defaults(segment_points, overlap_points, nfft_points)
    if gaussian_sigma is None:
        gaussian_sigma = int(segment_points / 4)
    return _spectral(sig_wf, frequency_sample_rate_hz, ("gaussian", gaussian_sigma), segment_points, overlap_points,
                     nfft_points, dtype)


def welch_power_pow2(sig_wf, frequency_sample_rate_hz: float, segment_points: int, nfft_points: int = None,
                     overlap_points: int = None, alpha: float = 0.25, *, dtype=None):
    """Welch power spectrum, scaling='spectrum', mean over segments (reference styx_fft.py:230-266).

    :return: frequency_welch_hz, welch_power [..., nfft/2+1]
    """
    overlap_points, nfft_points = _pow2_defaults(segment_points, overlap_points, nfft_points)
    freqs, acc, win, n_frames, lead, rt, want_numpy = _spectral(
        sig_wf, frequency_sample_rate_hz, ("tukey", alpha), segment_points, overlap_points, nfft_points, dtype,
        welch=True)
    # [C, K] fp64 accumulator -> mean over frames, window scaling, one-sided doubling (tiny: K values per record)
    onesided = np.full(nfft_points // 2 + 1, 2.0)
    onesided[0] = 1.0
    if nfft_points % 2 == 0:
        onesided[-1] = 1.0
    factor = onesided * (1.0 / win.sum() ** 2) / n_frames
    if want_numpy:
        p = rt.to_numpy(acc) * factor
        return freqs, p.reshape(lead + (nfft_points // 2 + 1,)).astype(np.float64)
    p = acc * rt.asarray(factor, "float64")
    return freqs, rt.reshape(p, lead + (nfft_points // 2 + 1,))


def stft_from_sig(sig_wf, frequency_sample_rate_hz: float, band_order_nth: float, center_frequency_hz: float = None,
                  octaves_below_center: int = 4, *, dtype=None) -> Tuple:
    """Hann STFT whose window holds M(N) cycles of the averaging frequency (reference styx_fft.py:14-57).

    :return: stft_complex, stft_bits, time_stft_s, frequency_stft_hz
    """
    if center_frequency_hz is None:
        center_frequency_hz = frequency_sample_rate_hz * 0.075
    frequency_averaging_hz = center_frequency_hz / octaves_below_center
    duration_fft_s = cycles_from_order(band_order_nth) / frequency_averaging_hz
    time_fft_nd: int = 2 ** get_num_points(sample_rate_hz=frequency_sample_rate_hz, duration_s=duration_fft_s,
                                           rounding_type="ceil", output_unit="log2")
    if len(sig_wf) < time_fft_nd:
        raise ValueError(f"Signal length: {len(sig_wf)} is less than time_fft_nd: {time_fft_nd}")
    stft_scaling = 2 * np.sqrt(np.pi) / time_fft_nd
    rt = get_runtime(sig_wf)
    want_numpy = not rt.is_device_array(sig_wf)
    frequency_stft_hz, time_stft_s, stft_complex = stft_complex_pow2(
        sig_wf=rt.asarray(sig_wf, dtype_name(dtype)), frequency_sample_rate_hz=frequency_sample_rate_hz,
        segment_points=time_fft_nd, alpha=1.0, dtype=dtype)                 # stays on the device
    stft_complex *= stft_scaling
    stft_bits = to_log2_with_epsilon(stft_complex)
    return finish(rt, stft_complex, want_numpy), finish(rt, stft_bits, want_numpy), time_stft_s, frequency_stft_hz


# ----------------------------------------------------------------------------- Butterworth pre-filters (styx_fft.py:60-149)
def _butter_filtfilt(sig_wf, b, a, tukey_alpha):
    """signal.filtfilt(b, a, sig * tukey(len(sig), alpha)) along the last axis (reference styx_fft.py:87-90)."""
    rt = get_runtime(sig_wf)
    want_numpy = not rt.is_device_array(sig_wf)
    name = str(sig_wf.dtype).replace("torch.", "") if not want_numpy else np.asarray(sig_wf).dtype.name
    dt = name if name in ("float32", "float64") else "float64"
    x = rt.asarray(sig_wf, dt)
    lead = tuple(int(v) for v in x.shape[:-1])
    x2 = rt.reshape(x, (int(np.prod(lead)) if lead else 1, int(x.shape[-1])))
    padlen = 3 * max(len(a), len(b))                                  # scipy.signal.filtfilt default
    sos = _iir.tf2sos_exact(b, a)                                     # same transfer function, well-conditioned form
    out = _driver.filtfilt(x2, dt, padlen, tukey_alpha=tukey_alpha, sos=sos, zi=_iir.sosfilt_zi(sos), rt=rt)
    return finish(rt, rt.reshape(out, lead + (int(x.shape[-1]),)), want_numpy)


def butter_bandpass(sig_wf: np.ndarray, frequency_sample_rate_hz: float, frequency_cut_low_hz, frequency_cut_high_hz,
                    filter_order: int = 4, tukey_alpha: float = 0.5) -> np.ndarray:
    """
    Tukey-tapered zero-phase Butterworth band-pass (reference styx_fft.py:60-90).

    :return: filtered signal waveform
    """
    from scipy import signal
    nyquist = 0.5 * frequency_sample_rate_hz
    edge_low = frequency_cut_low_hz / nyquist
    edge_high = frequency_cut_high_hz / nyquist
    if edge_high >= 1:
        print(
            f"Warning: Frequency cutoff {frequency_cut_high_hz} greater than Nyquist {nyquist} Hz, using half Nyquist"
        )
        edge_high = 0.5  # Half of nyquist
    [b, a] = signal.butter(N=filter_order, Wn=[edge_low, edge_high], btype="bandpass")
    return _butter_filtfilt(sig_wf, b, a, tukey_alpha)


def butter_highpass(sig_wf: np.ndarray, frequency_sample_rate_hz: float, frequency_cut_low_hz, filter_order: int = 4,
                    tukey_alpha: float = 0.5) -> np.ndarray:
    """
    Tukey-tapered zero-phase Butterworth high-pass (reference styx_fft.py:93-120).

    :return: filtered signal waveform
    """
    from scipy import signal
    edge_low = frequency_cut_low_hz / (0.5 * frequency_sample_rate_hz)
    if edge_low >= 1:
        raise ValueError(
            f"Frequency cutoff {frequency_cut_low_hz} is greater than Nyquist {0.5*frequency_sample_rate_hz}"
        )
    [b, a] = signal.butter(N=filter_order, Wn=[edge_low], btype="highpass")
    return _butter_filtfilt(sig_wf, b, a, tukey_alpha)


def butter_lowpass(sig_wf: np.ndarray, frequency_sample_rate_hz: float, frequency_cut_high_hz, filter_order: int = 4,
                   tukey_alpha: float = 0.5) -> np.ndarray:
    """
    Tukey-tapered zero-phase Butterworth low-pass (reference styx_fft.py:123-149).

    :return: filtered signal waveform
    """
    from scipy import signal
    edge_high = frequency_cut_high_hz / (0.5 * frequency_sample_rate_hz)
    if edge_high >= 1:
        raise ValueError(
            f"Frequency cutoff {frequency_cut_high_hz} is greater than Nyquist {0.5*frequency_sample_rate_hz}"
        )
    [b, a] = signal.butter(N=filter_order, Wn=[edge_high], btype="lowpass")
    return _butter_filtfilt(sig_wf, b, a, tukey_alpha)
