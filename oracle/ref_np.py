"""CPU oracle: NumPy/SciPy restatement of librosa's stft / istft / melspectrogram / mfcc path and of the
frame-wise features built on it (spectral centroid / bandwidth / rolloff / flatness, rms, zero-crossing rate).

TEST INFRASTRUCTURE ONLY.  Nothing under ``librosa_b200/`` imports this module; it is used by
``tests/``, by ``__graft_entry__.smoke()`` and by ``bench.py``'s CPU-baseline / ``--impl reference``
legs as the checker and as the timed CPU port.  The product path is the CUDA library and fails
loudly if it is missing.

Parity status: PINNED.  Every function below is checked against committed fixtures generated from the
unmodified reference (``tests/golden/*.npz`` written by ``tools/make_golden.py`` through
``tools/ref_shim.py``): bit for bit in ``tests/test_oracle_vs_reference.py``, within a tolerance that
absorbs SIMD / BLAS differences between hosts in ``tests/test_oracle_golden.py``.

The reference is pure Python; its arithmetic lives in third-party libraries that are not under
/root/reference and are called here exactly as the reference calls them:
``scipy.fft.rfft / irfft / dct`` (SciPy >= 1.15, ducc0 backend; this image: 1.18.1),
``numpy.einsum`` -> OpenBLAS sgemm (NumPy >= 2.1; this image: 2.3.5) and
``scipy.signal.get_window``.  ``numba`` (used by the reference to JIT a few serial loops) is not needed
here: the loops are restated with NumPy slices, and ``phasor`` (phase vocoder) calls libm's ``cosf`` /
``sinf`` through ctypes, which is what the reference's numba ufunc lowers to.

Each function cites the reference lines it restates (paths relative to /root/reference).
"""
from __future__ import annotations

import warnings

import numpy as np
import scipy.fft
import scipy.signal

MAX_MEM_BLOCK = 2 ** 8 * 2 ** 10  # librosa/util/utils.py:41 (256 KiB column-block bound)


class ParameterError(Exception):
    """librosa/util/exceptions.py:11-15."""


# --------------------------------------------------------------------------- small helpers
def tiny(x):
    """Smallest positive normal of x's dtype (librosa/util/utils.py:1935-2001)."""
    x = np.asarray(x)
    if np.issubdtype(x.dtype, np.floating) or np.issubdtype(x.dtype, np.complexfloating):
        dtype = x.dtype
    else:
        dtype = np.dtype(np.float32)
    return np.finfo(dtype).tiny


def dtype_r2c(d, default=np.complex64):
    """float32->complex64, float64->complex128 (librosa/util/utils.py:2362-2417)."""
    mapping = {np.dtype(np.float32): np.complex64, np.dtype(np.float64): np.complex128}
    dt = np.dtype(d)
    if dt.kind == "c":
        return dt
    return np.dtype(mapping.get(dt, default))


def dtype_c2r(d, default=np.float32):
    """complex64->float32, complex128->float64 (librosa/util/utils.py:2420-2476)."""
    mapping = {np.dtype(np.complex64): np.float32, np.dtype(np.complex128): np.float64}
    dt = np.dtype(d)
    if dt.kind == "f":
        return dt
    return np.dtype(mapping.get(dt, default))


def pad_center(data, size, axis=-1):
    """Zero-pad symmetrically, extra sample on the right (librosa/util/utils.py:436-458)."""
    n = data.shape[axis]
    left = int((size - n) // 2)
    if left < 0:
        raise ParameterError(f"Target size ({size}) must be at least input size ({n})")
    widths = [(0, 0)] * data.ndim
    widths[axis] = (left, int(size - n - left))
    return np.pad(data, widths, mode="constant")


def fix_length(data, size, axis=-1):
    """Trim or zero-pad on the right to ``size`` (librosa/util/utils.py:570-588)."""
    n = data.shape[axis]
    if n > size:
        sl = [slice(None)] * data.ndim
        sl[axis] = slice(0, size)
        return data[tuple(sl)]
    if n < size:
        widths = [(0, 0)] * data.ndim
        widths[axis] = (0, size - n)
        return np.pad(data, widths, mode="constant")
    return data


def frame(x, frame_length, hop_length):
    """Strided view ``xf[..., k, j] = x[..., j*hop + k]`` (librosa/util/utils.py:210-242, axis=-1)."""
    x = np.asarray(x)
    if x.shape[-1] < frame_length:
        raise ParameterError(f"Input is too short (n={x.shape[-1]}) for frame_length={frame_length}")
    if hop_length < 1:
        raise ParameterError(f"Invalid hop_length: {hop_length}")
    n_frames = 1 + (x.shape[-1] - frame_length) // hop_length
    s = x.strides[-1]
    return np.lib.stride_tricks.as_strided(
        x,
        shape=x.shape[:-1] + (frame_length, n_frames),
        strides=x.strides[:-1] + (s, s * hop_length),
        writeable=False,
    )


def valid_audio(y):
    """librosa/util/utils.py:294-308."""
    if not isinstance(y, np.ndarray):
        raise ParameterError("Audio data must be of type numpy.ndarray")
    if not np.issubdtype(y.dtype, np.floating):
        raise ParameterError("Audio data must be floating-point")
    if y.ndim == 0:
        raise ParameterError("Audio data must be at least one-dimensional")
    if not np.isfinite(y).all():
        raise ParameterError("Audio buffer is not finite everywhere")
    return True


def normalize(S, norm=np.inf, axis=0):
    """Row/column normalisation, default threshold/fill (librosa/util/utils.py:797-1026)."""
    S = np.asarray(S)
    mag = np.abs(S).astype(float)
    thresh = tiny(S)
    if norm is None:
        return S
    if norm == np.inf:
        length = mag.max(axis=axis, keepdims=True)
    elif norm == -np.inf:
        length = mag.min(axis=axis, keepdims=True)
    elif norm == 0:
        length = (mag > 0).sum(axis=axis, keepdims=True).astype(mag.dtype)
    elif np.issubdtype(type(norm), np.number) and norm > 0:
        length = (mag ** norm).sum(axis=axis, keepdims=True) ** (1.0 / norm)
    else:
        raise ParameterError(f"Unsupported norm: {norm!r}")
    small = length < thresh
    out = np.empty_like(S)
    length = np.where(small, 1.0, length)
    out[:] = S / length
    return out


# --------------------------------------------------------------------------- filters
def get_window(window, Nx, fftbins=True):
    """librosa/filters.py:961-977."""
    if callable(window):
        return window(Nx)
    if isinstance(window, (str, tuple)) or np.isscalar(window):
        return scipy.signal.get_window(window, Nx, fftbins=fftbins)
    if isinstance(window, (np.ndarray, list)):
        if len(window) == Nx:
            return np.asarray(window)
        raise ParameterError(f"Window size mismatch: {len(window)} != {Nx}")
    raise ParameterError(f"Invalid window specification: {window!r}")


def hz_to_mel(f, htk=False):
    """librosa/core/convert.py:1032-1058 (Slaney: linear below 1 kHz, log above)."""
    f = np.asanyarray(f, dtype=float)
    if htk:
        return 2595.0 * np.log10(1.0 + f / 700.0)
    f_sp = 200.0 / 3
    brk_hz = 1000.0
    brk_mel = brk_hz / f_sp
    logstep = np.log(6.4) / 27.0
    lin = f / f_sp
    with np.errstate(divide="ignore", invalid="ignore"):
        log = brk_mel + np.log(np.maximum(f, 1e-300) / brk_hz) / logstep
    return np.where(f >= brk_hz, log, lin)[()]


def mel_to_hz(m, htk=False):
    """librosa/core/convert.py:1098-1121."""
    m = np.asanyarray(m, dtype=float)
    if htk:
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
    f_sp = 200.0 / 3
    brk_hz = 1000.0
    brk_mel = brk_hz / f_sp
    logstep = np.log(6.4) / 27.0
    return np.where(m >= brk_mel, brk_hz * np.exp(logstep * (m - brk_mel)), f_sp * m)[()]


def mel_frequencies(n_mels=128, fmin=0.0, fmax=11025.0, htk=False):
    """librosa/core/convert.py:1500-1508."""
    lo = hz_to_mel(fmin, htk=htk)
    hi = hz_to_mel(fmax, htk=htk)
    return mel_to_hz(np.linspace(lo, hi, n_mels), htk=htk)


def fft_frequencies(sr=22050, n_fft=2048):
    """librosa/core/convert.py:1369 (np.fft.rfftfreq)."""
    return np.fft.rfftfreq(n=n_fft, d=1.0 / sr)


def mel(sr, n_fft, n_mels=128, fmin=0.0, fmax=None, htk=False, norm="slaney", dtype=np.float32):
    """Triangular mel filterbank (librosa/filters.py:206-251)."""
    if fmax is None:
        fmax = float(sr) / 2
    n_mels = int(n_mels)
    W = np.zeros((n_mels, 1 + n_fft // 2), dtype=dtype)
    bins = fft_frequencies(sr=sr, n_fft=n_fft)
    edges = mel_frequencies(n_mels + 2, fmin=fmin, fmax=fmax, htk=htk)
    width = np.diff(edges)
    ramps = np.subtract.outer(edges, bins)
    for i in range(n_mels):
        rising = -ramps[i] / width[i]
        falling = ramps[i + 2] / width[i + 1]
        W[i] = np.maximum(0, np.minimum(rising, falling))  # stored in `dtype` before scaling
    if isinstance(norm, str):
        if norm != "slaney":
            raise ParameterError(f"Unsupported norm={norm}")
        W *= (2.0 / (edges[2 : n_mels + 2] - edges[:n_mels]))[:, np.newaxis]
    else:
        W = normalize(W, norm=norm, axis=-1)
    if not np.all((edges[:-2] == 0) | (W.max(axis=1) > 0)):
        warnings.warn("Empty filters detected in mel frequency basis.", stacklevel=2)
    return W


def window_sumsquare(window, n_frames, hop_length=512, win_length=None, n_fft=2048,
                     dtype=np.float32, norm=None):
    """librosa/filters.py:1325-1339 with the numba fill loop of :1258-1265 restated."""
    if win_length is None:
        win_length = n_fft
    n = n_fft + hop_length * (n_frames - 1)
    x = np.zeros(n, dtype=dtype)
    wsq = get_window(window, win_length)
    wsq = normalize(wsq, norm=norm) ** 2
    wsq = pad_center(wsq, n_fft)
    for i in range(n_frames):
        s = i * hop_length
        x[s : min(n, s + n_fft)] += wsq[: max(0, min(n_fft, n - s))]
    return x


# --------------------------------------------------------------------------- stft / istft
_BAD_PAD = ("wrap", "maximum", "mean", "median", "minimum")


def stft(y, n_fft=2048, hop_length=None, win_length=None, window="hann", center=True,
         dtype=None, pad_mode="constant"):
    """Short-time Fourier transform, restating librosa/core/spectrum.py:231-391.

    The reference pads only the head and tail chunks (:273-328); SURVEY Appendix A.2 verified
    that this equals framing ``np.pad(y, n_fft//2, mode)`` — which is what is done here.  The
    float64 window product, the double-precision rfft, the rounding to ``dtype`` on store, the
    Fortran-ordered output and the MAX_MEM_BLOCK column blocking (:380-390) are kept because they
    determine both the numerics and the CPU cost.
    """
    if win_length is None:
        win_length = n_fft
    if hop_length is None:
        hop_length = int(win_length // 4)
    elif not (isinstance(hop_length, (int, np.integer)) and hop_length > 0):
        raise ParameterError(f"hop_length={hop_length} must be a positive integer")
    valid_audio(y)
    win = pad_center(get_window(window, win_length, fftbins=True), n_fft)
    win = win.reshape((1,) * (y.ndim - 1) + (n_fft, 1))
    if center:
        if pad_mode in _BAD_PAD:
            raise ParameterError(f"pad_mode='{pad_mode}' is not supported by librosa.stft")
        if n_fft > y.shape[-1]:
            warnings.warn(f"n_fft={n_fft} is too large for input signal of length={y.shape[-1]}",
                          stacklevel=2)
        widths = [(0, 0)] * (y.ndim - 1) + [(n_fft // 2, n_fft // 2)]
        y = np.pad(y, widths, mode=pad_mode)
    elif n_fft > y.shape[-1]:
        raise ParameterError(f"n_fft={n_fft} is too large for uncentered analysis of input "
                             f"signal of length={y.shape[-1]}")
    if dtype is None:
        dtype = dtype_r2c(y.dtype)
    frames = frame(y, n_fft, hop_length)
    shape = list(frames.shape)
    shape[-2] = 1 + n_fft // 2
    D = np.zeros(shape, dtype=dtype, order="F")
    cols = max(int(MAX_MEM_BLOCK // (np.prod(frames.shape[:-1]) * frames.itemsize)), 1)
    for s in range(0, frames.shape[-1], cols):
        t = min(s + cols, frames.shape[-1])
        D[..., s:t] = scipy.fft.rfft(win * frames[..., s:t], axis=-2)
    return D


def istft(D, hop_length=None, win_length=None, n_fft=None, window="hann", center=True,
          dtype=None, length=None):
    """Inverse STFT with least-squares WOLA normalisation, restating
    librosa/core/spectrum.py:506-626 and the overlap-add loop of :629-643.

    The head-block special case (:557-582) only avoids a padded copy; overlap-adding every frame
    into a buffer of the untrimmed length and slicing ``n_fft//2`` off the front gives the same
    sums in the same order per sample (frames are added in increasing frame index in both).
    """
    if n_fft is None:
        n_fft = 2 * (D.shape[-2] - 1)
    if win_length is None:
        win_length = n_fft
    if hop_length is None:
        hop_length = int(win_length // 4)
    win = pad_center(get_window(window, win_length, fftbins=True), n_fft)
    win = win.reshape((1,) * (D.ndim - 2) + (n_fft, 1))
    if length:
        padded = length + 2 * (n_fft // 2) if center else length
        n_frames = min(D.shape[-1], int(np.ceil(padded / hop_length)))
    else:
        n_frames = D.shape[-1]
    if dtype is None:
        dtype = dtype_c2r(D.dtype)
    full_len = n_fft + hop_length * (n_frames - 1)
    if length:
        out_len = length
    elif center:
        out_len = full_len - 2 * (n_fft // 2)
    else:
        out_len = full_len
    lead = list(D.shape[:-2])
    start = n_fft // 2 if center else 0
    buf = np.zeros(lead + [max(full_len, start + out_len)], dtype=dtype)
    cols = max(int(MAX_MEM_BLOCK // (np.prod(D.shape[:-1]) * D.itemsize)), 1)
    limit = start + out_len  # samples at or beyond this are never kept (:639-641 clipping)
    for s in range(0, n_frames, cols):
        t = min(s + cols, n_frames)
        ytmp = win * scipy.fft.irfft(D[..., s:t], n=n_fft, axis=-2)
        for j in range(t - s):
            a = (s + j) * hop_length
            n = min(n_fft, limit - a)
            if n > 0:
                buf[..., a : a + n] += ytmp[..., :n, j]
    y = np.ascontiguousarray(buf[..., start : start + out_len])
    wss = window_sumsquare(window, n_frames, hop_length=hop_length, win_length=win_length,
                           n_fft=n_fft, dtype=dtype)
    wss = fix_length(wss[start:], out_len)
    nz = wss > tiny(wss)
    y[..., nz] /= wss[nz]
    return y


# --------------------------------------------------------------------------- features
def spectrogram(y, n_fft=2048, hop_length=512, power=1.0, win_length=None, window="hann",
                center=True, pad_mode="constant"):
    """``|stft|**power`` (librosa/core/spectrum.py:3000-3013)."""
    return np.abs(stft(y, n_fft=n_fft, hop_length=hop_length, win_length=win_length,
                       window=window, center=center, pad_mode=pad_mode)) ** power


def power_to_db(S, ref=1.0, amin=1e-10, top_db=80.0, axes="auto"):
    """librosa/core/spectrum.py:1839-1883 for real input, scalar or callable ``ref``;
    ``axes='auto'`` reduces over the last two axes, per leading index (:1855-1861)."""
    S = np.asarray(S)
    if amin <= 0:
        raise ParameterError("amin must be strictly positive")
    mag = np.abs(S) if np.iscomplexobj(S) else S
    if isinstance(axes, str) and axes == "auto":
        axes = (-2, -1) if mag.ndim >= 2 else ((-1,) if mag.ndim == 1 else None)
    ref_value = ref(mag, axis=axes, keepdims=True) if callable(ref) else np.abs(ref)
    out = 10.0 * np.log10(np.maximum(amin, mag))
    out -= 10.0 * np.log10(np.maximum(amin, ref_value))
    if top_db is not None:
        if top_db < 0:
            raise ParameterError("top_db must be non-negative")
        out = np.maximum(out, out.max(axis=axes, keepdims=True) - top_db)
    return out[()]


def amplitude_to_db(S, ref=1.0, amin=1e-5, top_db=80.0):
    """librosa/core/spectrum.py:2000-2038 (``axes='auto'``): power_to_db of the squared magnitudes."""
    S = np.asarray(S)
    magnitude = np.abs(S)
    axes = (-2, -1) if magnitude.ndim >= 2 else ((-1,) if magnitude.ndim == 1 else None)
    ref_value = ref(magnitude, axis=axes, keepdims=True) if callable(ref) else np.abs(ref)
    power = np.square(magnitude, out=magnitude if isinstance(magnitude, np.ndarray) else None)
    return power_to_db(power, ref=ref_value ** 2, amin=amin ** 2, top_db=top_db)


def db_to_power(S_db, ref=1.0):
    """librosa/core/spectrum.py:1925."""
    return ref * np.power(10.0, S_db * 0.1)


def db_to_amplitude(S_db, ref=1.0):
    """librosa/core/spectrum.py:2081."""
    return db_to_power(S_db, ref=ref ** 2) ** 0.5


def melspectrogram(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, win_length=None,
                   window="hann", center=True, pad_mode="constant", power=2.0, **mel_kwargs):
    """librosa/feature/spectral.py:2145-2161."""
    if S is None:
        S = spectrogram(y, n_fft=n_fft, hop_length=hop_length, power=power,
                        win_length=win_length, window=window, center=center, pad_mode=pad_mode)
    else:
        if n_fft is None or n_fft // 2 + 1 != S.shape[-2]:
            n_fft = 2 * (S.shape[-2] - 1)
    basis = mel(sr=sr, n_fft=n_fft, **mel_kwargs)
    return np.einsum("...ft,mf->...mt", S, basis, optimize=True)


def mfcc(y=None, sr=22050, S=None, n_mfcc=20, dct_type=2, norm="ortho", lifter=0,
         mel_norm="slaney", **kwargs):
    """librosa/feature/spectral.py:1999-2019."""
    if S is None:
        S = power_to_db(melspectrogram(y=y, sr=sr, norm=mel_norm, **kwargs))
    M = scipy.fft.dct(S, axis=-2, type=dct_type, norm=norm)[..., :n_mfcc, :]
    if lifter > 0:
        li = np.sin(np.pi * np.arange(1, 1 + n_mfcc, dtype=M.dtype) / lifter)
        li = li.reshape((1,) * (S.ndim - 2) + (n_mfcc, 1))
        M *= 1 + (lifter / 2) * li
        return M
    if lifter == 0:
        return M
    raise ParameterError(f"MFCC lifter={lifter} must be a non-negative number")


# --------------------------------------------------------------------------- frame-wise spectral statistics
def _spec_or_S(y, S, n_fft, hop_length, power, win_length, window, center, pad_mode):
    """``_spectrogram`` (librosa/core/spectrum.py:2988-3013): pass ``S`` through (re-inferring n_fft) or
    compute ``|stft|**power``."""
    if S is not None:
        if n_fft is None or n_fft // 2 + 1 != S.shape[-2]:
            n_fft = 2 * (S.shape[-2] - 1)
        return S, n_fft
    return spectrogram(y, n_fft=n_fft, hop_length=hop_length, power=power, win_length=win_length,
                       window=window, center=center, pad_mode=pad_mode), n_fft


def _check_energy(S, what):
    if not np.isrealobj(S):
        raise ParameterError(f"{what} is only defined with real-valued input")
    if np.any(S < 0):
        raise ParameterError(f"{what} is only defined with non-negative energies")


def spectral_centroid(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, freq=None, win_length=None,
                      window="hann", center=True, pad_mode="constant"):
    """librosa/feature/spectral.py:158-191."""
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1, win_length, window, center, pad_mode)
    _check_energy(S, "Spectral centroid")
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        freq = freq.reshape((1,) * (S.ndim - 2) + (-1, 1))
    return np.sum(freq * normalize(S, norm=1, axis=-2), axis=-2, keepdims=True)


def spectral_bandwidth(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, win_length=None, window="hann",
                       center=True, pad_mode="constant", freq=None, centroid=None, norm=True, p=2):
    """librosa/feature/spectral.py:309-352."""
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1, win_length, window, center, pad_mode)
    _check_energy(S, "Spectral bandwidth")
    if centroid is None:
        centroid = spectral_centroid(y=y, sr=sr, S=S, n_fft=n_fft, hop_length=hop_length, freq=freq)
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        deviation = np.abs(np.subtract.outer(centroid[..., 0, :], freq).swapaxes(-2, -1))
    else:
        deviation = np.abs(freq - centroid)
    if norm:
        S = normalize(S, norm=1, axis=-2)
    return np.sum(S * deviation ** p, axis=-2, keepdims=True) ** (1.0 / p)


def spectral_rolloff(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, win_length=None, window="hann",
                     center=True, pad_mode="constant", freq=None, roll_percent=0.85):
    """librosa/feature/spectral.py:641-684."""
    if not 0.0 < roll_percent < 1.0:
        raise ParameterError("roll_percent must lie in the range (0, 1)")
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1, win_length, window, center, pad_mode)
    _check_energy(S, "Spectral rolloff")
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    if freq.ndim == 1:
        freq = freq.reshape((1,) * (S.ndim - 2) + (-1, 1))
    total_energy = np.cumsum(S, axis=-2)
    threshold = np.expand_dims(roll_percent * total_energy[..., -1, :], axis=-2)
    ind = np.where(total_energy < threshold, np.nan, 1)
    return np.nanmin(ind * freq, axis=-2, keepdims=True)


def spectral_flatness(y=None, S=None, n_fft=2048, hop_length=512, win_length=None, window="hann", center=True,
                      pad_mode="constant", amin=1e-10, power=2.0):
    """librosa/feature/spectral.py:772-803."""
    if amin <= 0:
        raise ParameterError("amin must be strictly positive")
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1.0, win_length, window, center, pad_mode)
    _check_energy(S, "Spectral flatness")
    S_thresh = np.maximum(amin, S ** power)
    gmean = np.exp(np.mean(np.log(S_thresh), axis=-2, keepdims=True))
    amean = np.mean(S_thresh, axis=-2, keepdims=True)
    return gmean / amean


def spectral_contrast(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, win_length=None, window="hann",
                      center=True, pad_mode="constant", freq=None, fmin=200.0, n_bands=6, quantile=0.02,
                      linear=False):
    """librosa/feature/spectral.py:447-532."""
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1, win_length, window, center, pad_mode)
    if freq is None:
        freq = fft_frequencies(sr=sr, n_fft=n_fft)
    freq = np.atleast_1d(freq)
    if freq.ndim != 1 or len(freq) != S.shape[-2]:
        raise ParameterError(f"freq.shape mismatch: expected ({S.shape[-2]:d},)")
    if n_bands < 1 or not isinstance(n_bands, (int, np.integer)):
        raise ParameterError("n_bands must be a positive integer")
    if not 0.0 < quantile < 1.0:
        raise ParameterError("quantile must lie in the range (0, 1)")
    if fmin <= 0:
        raise ParameterError("fmin must be a positive number")
    octa = np.zeros(n_bands + 2)
    octa[1:] = fmin * (2.0 ** np.arange(0, n_bands + 1))
    if np.any(octa[:-1] >= 0.5 * sr):
        raise ParameterError("Frequency band exceeds Nyquist. Reduce either fmin or n_bands.")
    shape = list(S.shape)
    shape[-2] = n_bands + 1
    valley = np.zeros(shape)
    peak = np.zeros_like(valley)
    for k, (f_low, f_high) in enumerate(zip(octa[:-1], octa[1:])):
        current_band = np.logical_and(freq >= f_low, freq <= f_high)
        idx = np.flatnonzero(current_band)
        if k > 0:
            current_band[idx[0] - 1] = True
        if k == n_bands:
            current_band[idx[-1] + 1:] = True
        sub_band = S[..., current_band, :]
        if k < n_bands:
            sub_band = sub_band[..., :-1, :]
        idx = np.rint(quantile * np.sum(current_band))
        idx = int(np.maximum(idx, 1))
        sortedr = np.sort(sub_band, axis=-2)
        valley[..., k, :] = np.mean(sortedr[..., :idx, :], axis=-2)
        peak[..., k, :] = np.mean(sortedr[..., -idx:, :], axis=-2)
    if linear:
        return peak - valley
    return power_to_db(peak) - power_to_db(valley)


def rms(y=None, S=None, frame_length=2048, hop_length=512, center=True, pad_mode="constant", dtype=np.float32):
    """librosa/feature/spectral.py:881-916 (``util.abs2`` = ``np.square`` for real input,
    ``re^2 + im^2`` for complex, librosa/util/utils.py:2479-2530)."""
    if y is not None:
        if center:
            padding = [(0, 0)] * y.ndim
            padding[-1] = (int(frame_length // 2), int(frame_length // 2))
            y = np.pad(y, padding, mode=pad_mode)
        x = frame(y, frame_length=frame_length, hop_length=hop_length)
        power = np.mean(np.square(x, dtype=dtype), axis=-2, keepdims=True)
    elif S is not None:
        if S.shape[-2] != frame_length // 2 + 1:
            raise ParameterError(
                f"Since S.shape[-2] is {S.shape[-2]}, frame_length is expected to be {S.shape[-2] * 2 - 2} or "
                f"{S.shape[-2] * 2 - 1}; found {frame_length}")
        if np.iscomplexobj(S):
            x = (S.real ** 2 + S.imag ** 2).astype(dtype)
        else:
            x = np.square(S, dtype=dtype)
        x[..., 0, :] *= 0.5
        if frame_length % 2 == 0:
            x[..., -1, :] *= 0.5
        power = 2 * np.sum(x, axis=-2, keepdims=True) / frame_length ** 2
    else:
        raise ParameterError("Either `y` or `S` must be input.")
    return np.sqrt(power)


def zero_crossings(y, threshold=1e-10, ref_magnitude=None, pad=True, zero_pos=True, axis=-1):
    """librosa/core/audio.py:1588-1602 (stencil) and :1711-1728: samples within ``threshold`` of zero count
    as 0; position i is a crossing when the sign (bit) of y[i] differs from that of y[i-1]; position 0 is
    ``pad``."""
    if callable(ref_magnitude):
        threshold = threshold * ref_magnitude(np.abs(y))
    elif ref_magnitude is not None:
        threshold = threshold * ref_magnitude
    yi = np.moveaxis(np.asarray(y), axis, -1)
    clipped = np.where((yi >= -threshold) & (yi <= threshold), 0, yi)
    sgn = np.signbit(clipped) if zero_pos else np.sign(clipped)
    z = np.empty(yi.shape, dtype=bool)
    z[..., 1:] = sgn[..., 1:] != sgn[..., :-1]
    z[..., 0] = pad
    return np.moveaxis(z, -1, axis)


def zero_crossing_rate(y, frame_length=2048, hop_length=512, center=True, **kwargs):
    """librosa/feature/spectral.py:1115-1133."""
    valid_audio(y)
    if center:
        padding = [(0, 0)] * y.ndim
        padding[-1] = (int(frame_length // 2), int(frame_length // 2))
        y = np.pad(y, padding, mode="edge")
    y_framed = frame(y, frame_length=frame_length, hop_length=hop_length)
    kwargs["axis"] = -2
    kwargs.setdefault("pad", False)
    crossings = zero_crossings(y_framed, **kwargs)
    return np.mean(crossings, axis=-2, keepdims=True)


# --------------------------------------------------------------------------- tuning / chroma
def hz_to_octs(frequencies, tuning=0.0, bins_per_octave=12):
    """librosa/core/convert.py (hz_to_octs)."""
    A440 = 440.0 * 2.0 ** (tuning / bins_per_octave)
    return np.log2(np.asanyarray(frequencies) / (float(A440) / 16))[()]


def localmax(x, axis=0):
    """librosa/util/utils.py:1029-1118: x[i] > x[i-1] and x[i] >= x[i+1]; first False, last x[-1] > x[-2]."""
    xi = np.moveaxis(np.asarray(x), axis, -1)
    out = np.zeros(xi.shape, dtype=bool)
    out[..., 1:-1] = (xi[..., 1:-1] > xi[..., :-2]) & (xi[..., 1:-1] >= xi[..., 2:])
    out[..., -1] = xi[..., -1] > xi[..., -2]
    return np.moveaxis(out, -1, axis)


def _parabolic_interpolation(x, axis=-2):
    """librosa/core/pitch.py:422-477."""
    xi = np.moveaxis(np.asarray(x), axis, -1)
    shifts = np.zeros_like(xi)
    a = xi[..., 2:] + xi[..., :-2] - 2 * xi[..., 1:-1]
    b = (xi[..., 2:] - xi[..., :-2]) / 2
    with np.errstate(divide="ignore", invalid="ignore"):
        inner = np.where(np.abs(b) >= np.abs(a), 0, -b / a)
    shifts[..., 1:-1] = inner
    return np.moveaxis(shifts, -1, axis)


def piptrack(y=None, sr=22050, S=None, n_fft=2048, hop_length=None, fmin=150.0, fmax=4000.0, threshold=0.1,
             win_length=None, window="hann", center=True, pad_mode="constant", ref=None):
    """librosa/core/pitch.py:296-366."""
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 1, win_length, window, center, pad_mode)
    if np.iscomplexobj(S) or S.min() < 0:
        S = np.abs(S)
    fmin = np.maximum(fmin, 0)
    fmax = np.minimum(fmax, float(sr) / 2)
    fft_freqs = fft_frequencies(sr=sr, n_fft=n_fft)
    avg = np.gradient(S, axis=-2)
    shift = _parabolic_interpolation(S, axis=-2)
    dskew = 0.5 * avg * shift
    pitches = np.zeros_like(S)
    mags = np.zeros_like(S)
    freq_mask = (fmin <= fft_freqs) & (fft_freqs < fmax)
    freq_mask = freq_mask.reshape((1,) * (S.ndim - 2) + (-1, 1))
    if ref is None:
        ref = np.max
    if callable(ref):
        ref_value = np.expand_dims(threshold * ref(S, axis=-2), -2)
    else:
        ref_value = np.abs(ref)
    idx = np.nonzero(freq_mask & localmax(S * (S > ref_value), axis=-2))
    pitches[idx] = (idx[-2] + shift[idx]) * float(sr) / n_fft
    mags[idx] = S[idx] + dskew[idx]
    return pitches, mags


def pitch_tuning(frequencies, resolution=0.01, bins_per_octave=12):
    """librosa/core/pitch.py:150-179."""
    frequencies = np.atleast_1d(frequencies)
    frequencies = frequencies[frequencies > 0]
    if not np.any(frequencies):
        warnings.warn("Trying to estimate tuning from empty frequency set.", stacklevel=2)
        return 0.0
    residual = np.mod(bins_per_octave * hz_to_octs(frequencies), 1.0)
    residual[residual >= 0.5] -= 1.0
    bins = np.linspace(-0.5, 0.5, int(np.ceil(1.0 / resolution)) + 1)
    counts, tuning = np.histogram(residual, bins)
    return tuning[np.argmax(counts)]


def estimate_tuning(y=None, sr=22050, S=None, n_fft=2048, resolution=0.01, bins_per_octave=12, **kwargs):
    """librosa/core/pitch.py:95-109."""
    pitch, mag = piptrack(y=y, sr=sr, S=S, n_fft=n_fft, **kwargs)
    pitch_mask = pitch > 0
    threshold = np.median(mag[pitch_mask]) if pitch_mask.any() else 0.0
    return pitch_tuning(pitch[(mag >= threshold) & pitch_mask], resolution=resolution,
                        bins_per_octave=bins_per_octave)


def chroma_filter(sr, n_fft, n_chroma=12, tuning=0.0, ctroct=5.0, octwidth=2, norm=2, base_c=True,
                  dtype=np.float32):
    """``filters.chroma`` (librosa/filters.py:254-392)."""
    wts = np.zeros((n_chroma, n_fft))
    frequencies = np.linspace(0, sr, n_fft, endpoint=False)[1:]
    frqbins = n_chroma * hz_to_octs(frequencies, tuning=tuning, bins_per_octave=n_chroma)
    frqbins = np.concatenate(([frqbins[0] - 1.5 * n_chroma], frqbins))
    binwidthbins = np.concatenate((np.maximum(frqbins[1:] - frqbins[:-1], 1.0), [1]))
    D = np.subtract.outer(frqbins, np.arange(0, n_chroma, dtype="d")).T
    n_chroma2 = np.round(float(n_chroma) / 2)
    D = np.remainder(D + n_chroma2 + 10 * n_chroma, n_chroma) - n_chroma2
    wts = np.exp(-0.5 * (2 * D / np.tile(binwidthbins, (n_chroma, 1))) ** 2)
    wts = normalize(wts, norm=norm, axis=0)
    if octwidth is not None:
        wts *= np.exp(-0.5 * (((frqbins / n_chroma - ctroct) / octwidth) ** 2))[np.newaxis, :]
    if base_c:
        wts = np.roll(wts, -3 * (n_chroma // 12), axis=0)
    return np.ascontiguousarray(wts[:, : int(1 + n_fft / 2)], dtype=dtype)


def chroma_stft(y=None, sr=22050, S=None, norm=np.inf, n_fft=2048, hop_length=512, win_length=None,
                window="hann", center=True, pad_mode="constant", tuning=None, n_chroma=12, **kwargs):
    """librosa/feature/spectral.py:1253-1293."""
    S, n_fft = _spec_or_S(y, S, n_fft, hop_length, 2, win_length, window, center, pad_mode)
    if tuning is None:
        tuning = estimate_tuning(S=S, sr=sr, bins_per_octave=n_chroma)
    chromafb = chroma_filter(sr=sr, n_fft=n_fft, tuning=tuning, n_chroma=n_chroma, **kwargs)
    raw_chroma = np.einsum("cf,...ft->...ct", chromafb, S, optimize=True)
    return normalize(raw_chroma, norm=norm, axis=-2)


def pcen(S, sr=22050, hop_length=512, gain=0.98, bias=2, power=0.5, time_constant=0.400, eps=1e-6, b=None,
         max_size=1, ref=None, axis=-1, max_axis=None, zi=None, return_zf=False):
    """librosa/core/spectrum.py:2576-2666."""
    import scipy.ndimage
    import scipy.signal

    if power < 0:
        raise ParameterError(f"power={power} must be nonnegative")
    if gain < 0:
        raise ParameterError(f"gain={gain} must be non-negative")
    if bias < 0:
        raise ParameterError(f"bias={bias} must be non-negative")
    if eps <= 0:
        raise ParameterError(f"eps={eps} must be strictly positive")
    if time_constant <= 0:
        raise ParameterError(f"time_constant={time_constant} must be strictly positive")
    if not (isinstance(max_size, (int, np.integer)) and max_size > 0):
        raise ParameterError(f"max_size={max_size} must be a positive integer")
    if b is None:
        t_frames = time_constant * sr / float(hop_length)
        b = (np.sqrt(1 + 4 * t_frames ** 2) - 1) / (2 * t_frames ** 2)
    if not 0 <= b <= 1:
        raise ParameterError(f"b={b} must be between 0 and 1")
    if np.issubdtype(S.dtype, np.complexfloating):
        S = np.abs(S)
    if ref is None:
        if max_size == 1:
            ref = S
        elif S.ndim == 1:
            raise ParameterError("Max-filtering cannot be applied to 1-dimensional input")
        else:
            if max_axis is None:
                if S.ndim != 2:
                    raise ParameterError(f"Max-filtering a {S.ndim:d}-dimensional spectrogram requires you to specify max_axis")
                max_axis = np.mod(1 - axis, 2)
            ref = scipy.ndimage.maximum_filter1d(S, max_size, axis=max_axis)
    if zi is None:
        zi = np.empty(tuple([1] * ref.ndim))
        zi[:] = scipy.signal.lfilter_zi([b], [1, b - 1])[:]
    S_smooth, zf = scipy.signal.lfilter([b], [1, b - 1], ref, zi=zi, axis=axis)
    smooth = np.exp(-gain * (np.log(eps) + np.log1p(S_smooth / eps)))
    if power == 0:
        S_out = np.log1p(S * smooth)
    elif bias == 0:
        S_out = np.exp(power * (np.log(S) + np.log(smooth)))
    else:
        S_out = (bias ** power) * np.expm1(power * np.log1p(S * smooth / bias))
    return (S_out, zf) if return_zf else S_out


# --------------------------------------------------------------------------- reassigned spectrogram
def cyclic_gradient(data, edge_order=1, axis=-1):
    """librosa/util/utils.py (cyclic_gradient)."""
    padding = [(0, 0)] * data.ndim
    padding[axis] = (edge_order, edge_order)
    data_pad = np.pad(data, padding, mode="wrap")
    grad = np.gradient(data_pad, edge_order=edge_order, axis=axis)
    slices = [slice(None)] * data.ndim
    slices[axis] = slice(edge_order, -edge_order)
    return grad[tuple(slices)]


def frames_to_time(frames, sr=22050, hop_length=512, n_fft=None):
    """librosa/core/convert.py (frames_to_time via frames_to_samples / samples_to_time)."""
    offset = int(n_fft // 2) if n_fft is not None else 0
    samples = (np.asanyarray(frames) * hop_length + offset).astype(int)
    return np.asanyarray(samples) / float(sr)


def reassigned_spectrogram(y, sr=22050, S=None, n_fft=2048, hop_length=None, win_length=None, window="hann",
                           center=True, reassign_frequencies=True, reassign_times=True, ref_power=1e-6,
                           fill_nan=False, clip=True, dtype=None, pad_mode="constant"):
    """librosa/core/spectrum.py:1185-1293 with __reassign_frequencies (:812-856) and __reassign_times (:957-1016)."""
    if not callable(ref_power) and ref_power < 0:
        raise ParameterError("ref_power must be non-negative or callable.")
    if not reassign_frequencies and not reassign_times:
        raise ParameterError("reassign_frequencies or reassign_times must be True.")
    if win_length is None:
        win_length = n_fft
    if hop_length is None:
        hop_length = int(win_length // 4)
    w = pad_center(get_window(window, win_length, fftbins=True), n_fft)
    kw = dict(n_fft=n_fft, hop_length=hop_length, center=center, dtype=dtype, pad_mode=pad_mode)
    if S is None:
        S = stft(y, window=w, **kw)
    freqs = times = None
    if reassign_frequencies:
        S_dh = stft(y, window=cyclic_gradient(w), **kw)
        with np.errstate(invalid="ignore", divide="ignore"):
            correction = -np.imag(S_dh / S)
        f = fft_frequencies(sr=sr, n_fft=n_fft)
        freqs = f.reshape((1,) * (correction.ndim - 2) + (-1, 1)) + correction * (0.5 * sr / np.pi)
    if reassign_times:
        half_width = n_fft // 2
        window_times = np.arange(-half_width, half_width + 1) if n_fft % 2 else np.arange(0.5 - half_width, half_width)
        S_th = stft(y, window=w * window_times, **kw)
        with np.errstate(invalid="ignore", divide="ignore"):
            correction = np.real(S_th / S)
        t = frames_to_time(np.arange(S.shape[-1]), sr=sr, hop_length=hop_length, n_fft=None if center else n_fft)
        times = t.reshape((1,) * (correction.ndim - 1) + (-1,)) + correction / sr
    mags = np.abs(S)
    if fill_nan or not reassign_frequencies or not reassign_times:
        bin_freqs = fft_frequencies(sr=sr, n_fft=n_fft)
        frame_times = frames_to_time(np.arange(S.shape[-1]), sr=sr, hop_length=hop_length,
                                     n_fft=None if center else n_fft)
    ref_p = ref_power(mags ** 2) if callable(ref_power) else ref_power
    mags_low = np.less(mags, ref_p ** 0.5, where=~np.isnan(mags), out=None)
    if reassign_frequencies:
        if ref_p > 0:
            freqs[mags_low] = np.nan
        if fill_nan:
            freqs = np.where(np.isnan(freqs), bin_freqs[:, np.newaxis], freqs)
        if clip:
            np.clip(freqs, 0, sr / 2.0, out=freqs)
    else:
        freqs = np.broadcast_to(bin_freqs[:, np.newaxis], S.shape)
    if reassign_times:
        if ref_p > 0:
            times[mags_low] = np.nan
        if fill_nan:
            times = np.where(np.isnan(times), frame_times[np.newaxis, :], times)
        if clip:
            np.clip(times, 0, y.shape[-1] / float(sr), out=times)
    else:
        times = np.broadcast_to(frame_times[np.newaxis, :], S.shape)
    return freqs, times, mags


# --------------------------------------------------------------------------- phase vocoder / time stretch
_LIBM = None


def phasor(angles):
    """``util.phasor`` (librosa/util/utils.py:2634-2710): cos + i sin.  The reference evaluates it through a
    numba ufunc, which for float32 input calls libm's ``cosf`` / ``sinf`` — not NumPy's SIMD float32 kernels,
    which differ in the last bit.  The same libm entry points are called here through ctypes (element by
    element: this is the checker, not a fast path)."""
    global _LIBM
    angles = np.asarray(angles)
    z = np.empty_like(angles, dtype=dtype_r2c(angles.dtype))
    if angles.dtype != np.float32:
        z.real, z.imag = np.cos(angles), np.sin(angles)
        return z
    if _LIBM is None:
        import ctypes
        import ctypes.util

        _LIBM = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
        for fn in (_LIBM.cosf, _LIBM.sinf):
            fn.restype = ctypes.c_float
            fn.argtypes = [ctypes.c_float]
    flat = angles.reshape(-1)
    re = np.fromiter((_LIBM.cosf(float(v)) for v in flat), dtype=np.float32, count=flat.size)
    im = np.fromiter((_LIBM.sinf(float(v)) for v in flat), dtype=np.float32, count=flat.size)
    z.real, z.imag = re.reshape(angles.shape), im.reshape(angles.shape)
    return z


def phase_vocoder(D, rate=None, t_out=None, kind="linear"):
    """librosa/core/spectrum.py:1476-1530."""
    import scipy.interpolate

    n_frames = D.shape[-1]
    if (rate is None) == (t_out is None):
        raise ParameterError("Must specify exactly one of `rate` or `t_out`")
    if (rate is not None) and (rate <= 0):
        raise ParameterError(f"rate={rate} must be a positive number")
    if t_out is None:
        t_out = np.arange(0.0, n_frames, rate)
    t_out = np.asarray(t_out, dtype=float)
    if np.any(t_out < 0) or np.any(t_out >= n_frames):
        raise ParameterError("t_out values must be in the range [0, D.shape[-1])")
    i0 = np.floor(t_out).astype(int)
    i1 = np.minimum(i0 + 1, n_frames - 1)
    ph = np.angle(D)
    diff = ph[..., i1] - ph[..., i0]
    phase = np.empty_like(diff)
    phase[..., 0] = np.angle(D[..., i0[0]])
    phase[..., 1:] = diff[..., :-1]
    np.cumsum(phase, axis=-1, out=phase)
    mag_interp = scipy.interpolate.interp1d(np.arange(n_frames), np.abs(D), kind=kind, axis=-1,
                                            fill_value="extrapolate", assume_sorted=True, copy=False)
    z = phasor(phase)
    z *= mag_interp(t_out)
    return z


def effects_time_stretch(y, rate, **kwargs):
    """librosa/effects.py:284-361."""
    if rate <= 0:
        raise ParameterError("rate must be a positive number")
    D = stft(y, **kwargs)
    Ds = phase_vocoder(D, rate=rate)
    return istft(Ds, dtype=y.dtype, length=round(y.shape[-1] / rate), **kwargs)


# --------------------------------------------------------------------------- harmonic / percussive separation
def softmask(X, X_ref, power=1, split_zeros=False):
    """librosa/util/utils.py (softmask)."""
    if X.shape != X_ref.shape:
        raise ParameterError(f"Shape mismatch: {X.shape}!={X_ref.shape}")
    if np.any(X < 0) or np.any(X_ref < 0):
        raise ParameterError("X and X_ref must be non-negative")
    if power <= 0:
        raise ParameterError("power must be strictly positive")
    dtype = X.dtype if np.issubdtype(X.dtype, np.floating) else np.float32
    Z = np.maximum(X, X_ref).astype(dtype)
    bad_idx = Z < np.finfo(dtype).tiny
    Z[bad_idx] = 1
    if np.isfinite(power):
        mask = (X / Z) ** power
        ref_mask = (X_ref / Z) ** power
        good_idx = ~bad_idx
        mask[good_idx] /= mask[good_idx] + ref_mask[good_idx]
        mask[bad_idx] = 0.5 if split_zeros else 0.0
    else:
        mask = X > X_ref
    return mask


def magphase(D, power=1):
    """librosa/core/spectrum.py (magphase)."""
    mag = np.abs(D)
    zeros_to_ones = mag == 0
    mag_nonzero = mag + zeros_to_ones
    phase = np.empty_like(D, dtype=dtype_r2c(D.dtype))
    phase.real = D.real / mag_nonzero + zeros_to_ones
    phase.imag = D.imag / mag_nonzero
    mag **= power
    return mag, phase


def resample(y, orig_sr, target_sr, res_type="polyphase", fix=True, scale=False, axis=-1):
    """librosa.resample (librosa/core/audio.py:1002-1179) for the resamplers whose arithmetic lives in SciPy:
    ``polyphase`` = scipy.signal.resample_poly(y, target_sr // gcd, orig_sr // gcd) (:1129-1145, integer rates only) and
    ``fft`` / ``scipy`` = scipy.signal.resample (:1125-1128); then fix_length to ceil(n * ratio) (:1172-1173), the
    optional 1 / sqrt(ratio) scale (:1175-1176) and a cast back to the input dtype (:1179).  The other resamplers
    (soxr, resampy, samplerate) are third-party libraries that are not vendored with the reference."""
    import scipy.signal

    if orig_sr == target_sr:
        return y
    ratio = float(target_sr) / orig_sr
    n_samples = int(np.ceil(y.shape[axis] * ratio))
    if res_type in ("scipy", "fft"):
        y_hat = scipy.signal.resample(y, n_samples, axis=axis)
    elif res_type == "polyphase":
        if int(orig_sr) != orig_sr or int(target_sr) != target_sr:
            raise ParameterError("polyphase resampling is only supported for integer-valued sampling rates.")
        orig_sr, target_sr = int(orig_sr), int(target_sr)
        gcd = np.gcd(orig_sr, target_sr)
        y_hat = scipy.signal.resample_poly(y, target_sr // gcd, orig_sr // gcd, axis=axis)
    else:
        raise ParameterError(f"the oracle restates only the SciPy resamplers, not res_type={res_type!r}")
    if fix:
        y_hat = fix_length(y_hat, size=n_samples, axis=axis)
    if scale:
        y_hat /= np.sqrt(ratio)
    return np.asarray(y_hat, dtype=y.dtype)


def effects_pitch_shift(y, sr, n_steps, bins_per_octave=12, res_type="polyphase", scale=False, **kwargs):
    """librosa.effects.pitch_shift (librosa/effects.py:487-574): time_stretch by 2^(-n_steps / bins_per_octave), resample
    from sr / rate back to sr, crop / pad to the input length."""
    rate = 2.0 ** (-float(n_steps) / bins_per_octave)
    y_shift = resample(effects_time_stretch(y, rate=rate, **kwargs), orig_sr=float(sr) / rate, target_sr=sr,
                       res_type=res_type, scale=scale)
    return fix_length(y_shift, size=y.shape[-1])


def decompose_hpss(S, kernel_size=31, power=2.0, mask=False, margin=1.0):
    """librosa/decompose.py:338-389."""
    from scipy.ndimage import median_filter

    if np.iscomplexobj(S):
        S, phase = magphase(S)
    else:
        phase = 1
    win_harm, win_perc = kernel_size if isinstance(kernel_size, (tuple, list)) else (kernel_size, kernel_size)
    margin_harm, margin_perc = margin if isinstance(margin, (tuple, list)) else (margin, margin)
    if margin_harm < 1 or margin_perc < 1:
        raise ParameterError("Margins must be >= 1.0. A typical range is between 1 and 10.")
    harm_shape = [1] * S.ndim
    harm_shape[-1] = int(win_harm)
    perc_shape = [1] * S.ndim
    perc_shape[-2] = int(win_perc)
    harm = np.empty_like(S)
    harm[:] = median_filter(S, size=harm_shape, mode="reflect")
    perc = np.empty_like(S)
    perc[:] = median_filter(S, size=perc_shape, mode="reflect")
    split_zeros = margin_harm == 1 and margin_perc == 1
    mask_harm = softmask(harm, perc * margin_harm, power=power, split_zeros=split_zeros)
    mask_perc = softmask(perc, harm * margin_perc, power=power, split_zeros=split_zeros)
    if mask:
        return mask_harm, mask_perc
    return ((S * mask_harm) * phase, (S * mask_perc) * phase)


def effects_hpss(y, kernel_size=31, power=2.0, mask=False, margin=1.0, n_fft=2048, hop_length=None,
                 win_length=None, window="hann", center=True, pad_mode="constant"):
    """librosa/effects.py:58-131 (``window`` is accepted but, as in the reference, not forwarded)."""
    D = stft(y, n_fft=n_fft, hop_length=hop_length, win_length=win_length, center=center, pad_mode=pad_mode)
    Dh, Dp = decompose_hpss(D, kernel_size=kernel_size, power=power, mask=mask, margin=margin)
    kw = dict(dtype=y.dtype, n_fft=n_fft, hop_length=hop_length, win_length=win_length, center=center,
              length=y.shape[-1])
    return istft(Dh, **kw), istft(Dp, **kw)


def effects_harmonic(y, **kwargs):
    """librosa/effects.py:134-206."""
    return effects_hpss(y, **kwargs)[0]


def effects_percussive(y, **kwargs):
    """librosa/effects.py:209-281."""
    return effects_hpss(y, **kwargs)[1]


# --------------------------------------------------------------------------- onset strength
def _channel_slices(channels, n_rows, pad):
    """``util.sync`` index handling (librosa/util/utils.py: sync, index_to_slice, fix_frames)."""
    if all(isinstance(c, slice) for c in channels):
        return list(channels)
    frames = np.asarray(channels)
    if np.any(frames < 0):
        raise ParameterError("Negative frame index detected")
    if pad:
        frames = np.concatenate((np.asarray([0, n_rows]), np.clip(frames, 0, n_rows)))
    frames = frames[(frames >= 0) & (frames <= n_rows)]
    edges = np.unique(frames).astype(int)
    return [slice(a, b) for a, b in zip(edges[:-1], edges[1:])]


def onset_strength_multi(y=None, sr=22050, S=None, n_fft=2048, hop_length=512, lag=1, max_size=1, ref=None,
                         detrend=False, center=True, aggregate=None, channels=None, **kwargs):
    """librosa/onset.py:566-640 with ``feature=melspectrogram``."""
    import scipy.ndimage
    import scipy.signal

    kwargs.setdefault("fmax", 0.5 * sr)
    if aggregate is None:
        aggregate = np.mean
    if not (isinstance(lag, (int, np.integer)) and lag > 0):
        raise ParameterError(f"lag={lag} must be a positive integer")
    if not (isinstance(max_size, (int, np.integer)) and max_size > 0):
        raise ParameterError(f"max_size={max_size} must be a positive integer")
    if S is None:
        S = power_to_db(np.abs(melspectrogram(y=y, sr=sr, n_fft=n_fft, hop_length=hop_length, **kwargs)))
    S = np.atleast_2d(S)
    if ref is None:
        ref = S if max_size == 1 else scipy.ndimage.maximum_filter1d(S, max_size, axis=-2)
    elif ref.shape != S.shape:
        raise ParameterError(f"Reference spectrum shape {ref.shape} must match input spectrum {S.shape}")
    onset_env = np.maximum(0.0, S[..., lag:] - ref[..., :-lag])
    pad = True
    if channels is None:
        channels = [slice(None)]
    else:
        pad = False
    if callable(aggregate):
        slices = _channel_slices(channels, onset_env.shape[-2], pad)
        agg = np.empty(onset_env.shape[:-2] + (len(slices), onset_env.shape[-1]), dtype=onset_env.dtype)
        for i, seg in enumerate(slices):
            agg[..., i, :] = aggregate(onset_env[..., seg, :], axis=-2)
        onset_env = agg
    pad_width = lag
    if center:
        pad_width += n_fft // (2 * hop_length)
    padding = [(0, 0)] * onset_env.ndim
    padding[-1] = (int(pad_width), 0)
    onset_env = np.pad(onset_env, padding, mode="constant")
    if detrend:
        onset_env = scipy.signal.lfilter([1.0, -1.0], [1.0, -0.99], onset_env, axis=-1)
    if center:
        onset_env = onset_env[..., : S.shape[-1]]
    return onset_env


def onset_strength(y=None, sr=22050, S=None, lag=1, max_size=1, ref=None, detrend=False, center=True,
                   aggregate=None, **kwargs):
    """librosa/onset.py:346-367."""
    if aggregate is False:
        raise ParameterError("aggregate parameter cannot be False when computing full-spectrum onset strength.")
    return onset_strength_multi(y=y, sr=sr, S=S, lag=lag, max_size=max_size, ref=ref, detrend=detrend, center=center,
                                aggregate=aggregate, channels=None, **kwargs)[..., 0, :]


def griffinlim(S, n_iter=32, hop_length=None, win_length=None, n_fft=None, window="hann", center=True,
               dtype=None, length=None, pad_mode="constant", momentum=0.99, init="random", rng=None):
    """Fast Griffin-Lim, restating librosa/core/spectrum.py:2819-2917 (first "next" row of SURVEY 8f)."""
    if not isinstance(rng, np.random.RandomState):
        rng = np.random.default_rng(rng)
    if momentum < 0:
        raise ParameterError(f"griffinlim() called with momentum={momentum} < 0")
    if n_fft is None:
        n_fft = 2 * (S.shape[-2] - 1)
    angles = np.empty(S.shape, dtype=dtype_r2c(S.dtype))
    eps = tiny(angles)
    if init == "random":
        ph = 2 * np.pi * rng.random(size=S.shape)
        angles[:] = np.cos(ph) + 1j * np.sin(ph)
    elif init is None:
        angles[:] = 1.0
    else:
        raise ParameterError(f"init={init} must either None or 'random'")
    angles *= S
    tprev = None
    kw_i = dict(hop_length=hop_length, win_length=win_length, n_fft=n_fft, window=window, center=center,
                dtype=dtype, length=length)
    for _ in range(n_iter):
        inverse = istft(angles, **kw_i)
        rebuilt = stft(inverse, n_fft=n_fft, hop_length=hop_length, win_length=win_length, window=window,
                       center=center, pad_mode=pad_mode)
        angles[:] = rebuilt
        if tprev is not None:
            angles -= (momentum / (1 + momentum)) * tprev
        angles /= np.abs(angles) + eps
        angles *= S
        tprev = rebuilt
    return istft(angles, **kw_i)


# ------------------------------------------------------------------ feature.inverse (SURVEY 8f rank 1)
MAX_MEM_BLOCK = 2 ** 8 * 2 ** 10   # librosa/util/utils.py:41


def _nnls_obj(x, shape, A, B):
    """librosa/util/_nnls.py:22-41: objective and gradient of the block problem."""
    x = x.reshape(shape)
    diff = np.einsum("mf,...ft->...mt", A, x, optimize=True) - B
    value = (1 / B.size) * 0.5 * np.sum(diff ** 2)
    grad = (1 / B.size) * np.einsum("mf,...mt->...ft", A, diff, optimize=True)
    return value, grad.flatten()


def _nnls_lbfgs_block(A, B, x_init=None, **kwargs):
    """librosa/util/_nnls.py:44-89: L-BFGS-B from the clipped pseudo-inverse solution."""
    import scipy.optimize

    if x_init is None:
        x_init = np.einsum("fm,...mt->...ft", np.linalg.pinv(A), B, optimize=True)
        np.clip(x_init, 0, None, out=x_init)
    kwargs.setdefault("m", A.shape[1])
    bounds = [(0, None)] * x_init.size
    shape = x_init.shape
    x, _obj, _diag = scipy.optimize.fmin_l_bfgs_b(_nnls_obj, x_init, args=(shape, A, B), bounds=bounds, **kwargs)
    return x.reshape(shape)


def nnls(A, B, **kwargs):
    """librosa/util/_nnls.py:92-175."""
    import scipy.optimize

    if B.ndim == 1:
        return scipy.optimize.nnls(A, B)[0]
    n_columns = int(MAX_MEM_BLOCK // (np.prod(B.shape[:-1]) * A.itemsize))
    n_columns = max(n_columns, 1)
    if B.shape[-1] <= n_columns:
        return _nnls_lbfgs_block(A, B, **kwargs).astype(A.dtype)
    x = np.einsum("fm,...mt->...ft", np.linalg.pinv(A), B, optimize=True)
    np.clip(x, 0, None, out=x)
    x_init = x
    for bl_s in range(0, x.shape[-1], n_columns):
        bl_t = min(bl_s + n_columns, B.shape[-1])
        x[..., bl_s:bl_t] = _nnls_lbfgs_block(A, B[..., bl_s:bl_t], x_init=x_init[..., bl_s:bl_t], **kwargs)
    return x


def mel_to_stft(M, sr=22050, n_fft=2048, power=2.0, **kwargs):
    """librosa/feature/inverse.py:104-114."""
    mel_basis = mel(sr=sr, n_fft=n_fft, n_mels=M.shape[-2], dtype=M.dtype, **kwargs)
    inverse = nnls(mel_basis, M)
    np.power(inverse, 1.0 / power, out=inverse)
    return inverse


def mfcc_to_mel(mfcc, n_mels=128, dct_type=2, norm="ortho", ref=1.0, lifter=0):
    """librosa/feature/inverse.py:265-287."""
    if lifter > 0:
        n_mfcc = mfcc.shape[-2]
        idx = np.arange(1, 1 + n_mfcc, dtype=mfcc.dtype)
        idx = idx.reshape([-1 if i == mfcc.ndim - 2 else 1 for i in range(mfcc.ndim)])
        lifter_sine = 1 + lifter * 0.5 * np.sin(np.pi * idx / lifter)
        if np.any(np.abs(lifter_sine) < np.finfo(lifter_sine.dtype).eps):
            warnings.warn(message="lifter array includes critical values that may invoke underflow.",
                          category=UserWarning, stacklevel=2)
        mfcc = mfcc / (lifter_sine + tiny(mfcc))
    elif lifter != 0:
        raise ParameterError("MFCC to mel lifter must be a non-negative number.")
    logmel = scipy.fft.idct(mfcc, axis=-2, type=dct_type, norm=norm, n=n_mels)
    return db_to_power(logmel, ref=ref)
