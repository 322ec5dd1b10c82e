"""Outputs of the reference that the oracle and the product's host-side builders must reproduce bit for bit
(tests/test_oracle_vs_reference.py).

Every group below takes a module laid out like librosa (``stft``, ``feature.mfcc``, ``filters.mel``, ...) and
returns ``{key: array}``.  tools/make_golden.py calls the groups with the unmodified reference and stores a
record of each output in tests/golden/reference_exact_v1.npz: its shape, a SHA-256 of its values and a
seeded sample of them.  The test calls the same groups with the oracle (through ``librosa_layout``) or with
the product and checks every output against that record.
"""
from __future__ import annotations

import hashlib
import types

import numpy as np

STFT_GRID = [
    (22050, 2048, 512, True, "constant"), (5000, 1024, 256, True, "reflect"), (4000, 512, None, False, "constant"),
    (1000, 2048, 512, True, "constant"), (3000, 501, 128, True, "edge"), (7000, 1025, 300, True, "symmetric"),
    (6000, 256, 64, True, "linear_ramp"), (900, 64, 7, True, "reflect"),
]
SAMPLE = 64


def librosa_layout(oracle):
    """The flat oracle module under the names the reference uses."""
    ns = types.SimpleNamespace
    return ns(stft=oracle.stft, istft=oracle.istft, griffinlim=oracle.griffinlim, power_to_db=oracle.power_to_db,
              filters=ns(mel=oracle.mel),
              feature=ns(melspectrogram=oracle.melspectrogram, mfcc=oracle.mfcc,
                         inverse=ns(mel_to_stft=oracle.mel_to_stft, mfcc_to_mel=oracle.mfcc_to_mel)))


# ------------------------------------------------------------------------------------------------ groups
def stft_istft(lib, n, n_fft, hop, center, pad_mode):
    y = (0.1 * np.random.default_rng(n).standard_normal(n)).astype(np.float32)
    tag = f"stft_{n}_{n_fft}_{hop}_{center}_{pad_mode}"
    D = lib.stft(y, n_fft=n_fft, hop_length=hop, center=center, pad_mode=pad_mode)
    out = {tag: D}
    for length in (None, n):
        out[f"{tag}/istft_{length}"] = lib.istft(D, hop_length=hop, n_fft=n_fft, center=center, length=length)
    return out


def features(lib):
    y = (0.1 * np.random.default_rng(5).standard_normal((2, 3, 8000))).astype(np.float32)
    return {"features/mel": lib.feature.melspectrogram(y=y, sr=16000, n_fft=1024, hop_length=256),
            "features/mfcc40": lib.feature.mfcc(y=y, sr=16000, n_mfcc=40, n_fft=1024, hop_length=256),
            "features/mfcc13_dct3": lib.feature.mfcc(y=y, sr=16000, n_mfcc=13, lifter=22, dct_type=3)}


CHROMA_KW = [dict(sr=22050, n_fft=2048), dict(sr=16000, n_fft=1024, tuning=0.27), dict(sr=22050, n_fft=400, n_chroma=24, octwidth=None),
             dict(sr=44100, n_fft=4096, norm=None, base_c=False, ctroct=4.0, octwidth=1.5), dict(sr=22050, n_fft=1025, tuning=-0.3)]


def chroma(lib):
    out = {f"chroma/{i}": lib.filters.chroma(**kw) for i, kw in enumerate(CHROMA_KW)}
    out["chroma/hz_to_octs"] = lib.hz_to_octs(np.array([27.5, 55.0, 440.0, 1234.5]), tuning=0.2, bins_per_octave=24)
    return out


def griffinlim(lib):
    y = (0.1 * np.random.default_rng(2).standard_normal(6000)).astype(np.float32)
    S = np.abs(lib.stft(y, n_fft=512, hop_length=128))
    kws = [dict(n_iter=4, rng=0), dict(n_iter=3, init=None, momentum=0.5), dict(n_iter=2, rng=7, length=6000)]
    return {f"griffinlim/{i}": lib.griffinlim(S, hop_length=128, **kw) for i, kw in enumerate(kws)}


MEL_KW = [dict(sr=22050, n_fft=2048), dict(sr=44100, n_fft=4096), dict(sr=16000, n_fft=1024, n_mels=40, htk=True),
          dict(sr=22050, n_fft=2048, norm=1), dict(sr=22050, n_fft=2048, norm=None, fmin=300, fmax=8000),
          dict(sr=22050, n_fft=2048, norm=np.inf), dict(sr=8000, n_fft=512, n_mels=20, dtype=np.float64)]


def host_constants(lib):
    """The host-side constant builders that feed the GPU plans (filters / convert / util)."""
    out = {f"const/mel_{i}": lib.filters.mel(**kw) for i, kw in enumerate(MEL_KW)}
    out["const/window_sumsquare"] = lib.filters.window_sumsquare(window="hann", n_frames=50)
    for i, w in enumerate(["hann", "hamming", ("kaiser", 4.0), np.ones(64)]):
        out[f"const/window_{i}"] = lib.filters.get_window(w, 64)
    f = np.array([0.0, 60.0, 999.0, 1000.0, 5000.0])
    for htk in (False, True):
        out[f"const/hz_to_mel_{htk}"] = lib.hz_to_mel(f, htk=htk)
        out[f"const/mel_to_hz_{htk}"] = lib.mel_to_hz(f / 50, htk=htk)
    out["const/hz_to_mel_60"] = lib.hz_to_mel(60.0)
    out["const/mel_to_hz_20"] = lib.mel_to_hz(20.0)
    x = np.arange(40.0).reshape(2, 20)
    for axis in (-1, 0, 1):
        if x.shape[axis] >= 5:
            out[f"const/frame_axis{axis}"] = lib.util.frame(x, frame_length=5, hop_length=2, axis=axis)
    out["const/pad_center"] = lib.util.pad_center(np.ones(5), size=12)
    out["const/fix_length"] = lib.util.fix_length(np.ones(5), size=3)
    out["const/tiny"] = lib.util.tiny(np.float32(1))
    return out


POWER_TO_DB_KW = [dict(), dict(axes=(-1,)), dict(axes=(-2,)), dict(axes=None, ref=np.max), dict(axes=(0, -1), top_db=30.0),
                  dict(axes=(-1,), ref=np.max)]


def power_to_db_and_float64(lib):
    """power_to_db with explicit reduction axes, and float64 audio through the whole path (the reference computes
    it in float64: complex128 STFT, float64 mel / MFCC)."""
    rng = np.random.default_rng(9)
    P = np.abs(rng.standard_normal((2, 3, 40, 30))) ** 2
    out = {f"db/{i}": lib.power_to_db(P, **kw) for i, kw in enumerate(POWER_TO_DB_KW)}
    y = 0.1 * rng.standard_normal((2, 9000))
    for kw in (dict(n_fft=1024, hop_length=256), dict(n_fft=1000, hop_length=250, pad_mode="reflect")):
        D = lib.stft(y, **kw)
        out[f"f64/stft_{kw['n_fft']}"] = D
        out[f"f64/istft_{kw['n_fft']}"] = lib.istft(D, hop_length=kw["hop_length"], n_fft=kw["n_fft"])
    out["f64/mel"] = lib.feature.melspectrogram(y=y, sr=16000, n_fft=1024)
    out["f64/mfcc"] = lib.feature.mfcc(y=y, sr=16000, n_fft=1024)
    return out


def feature_inverse(lib):
    """mel_to_stft (NNLS through SciPy's L-BFGS-B) and mfcc_to_mel."""
    rng = np.random.default_rng(21)
    out = {}
    for dtype in (np.float32, np.float64):
        basis = lib.filters.mel(sr=22050, n_fft=1024, n_mels=64, dtype=dtype)
        S = np.abs(rng.standard_normal((513, 6))).astype(dtype) ** 2
        out[f"inverse/mel_to_stft_{np.dtype(dtype).name}"] = lib.feature.inverse.mel_to_stft(basis.dot(S), n_fft=1024, power=2.0)
    mf = rng.standard_normal((2, 13, 20)).astype(np.float32) * 10
    for i, kw in enumerate((dict(), dict(lifter=3, dct_type=3), dict(n_mels=64, norm=None), dict(ref=2.5, lifter=22))):
        out[f"inverse/mfcc_to_mel_{i}"] = lib.feature.inverse.mfcc_to_mel(mf, **kw)
    return out


def all_groups(lib):
    """Every output the oracle must reproduce (the product's host builders are recorded by the same calls)."""
    out = {}
    for args in STFT_GRID:
        out.update(stft_istft(lib, *args))
    for group in (features, chroma, griffinlim, host_constants, power_to_db_and_float64, feature_inverse):
        out.update(group(lib))
    return out


# ------------------------------------------------------------------------------------------------ records
def _values(a):
    """The values of ``a`` as assert_array_equal sees them: -0.0 equals 0.0 and NaN equals NaN."""
    flat = np.ascontiguousarray(a).reshape(-1)
    if flat.dtype.kind == "c":
        flat = np.stack([flat.real, flat.imag], axis=-1)
    if flat.dtype.kind == "f":
        flat = flat + flat.dtype.type(0)
        flat[np.isnan(flat)] = np.nan
    return flat


def sha256(a) -> str:
    return hashlib.sha256(_values(a).tobytes()).hexdigest()


def sample_index(size: int) -> np.ndarray:
    return np.sort(np.random.default_rng(0).choice(size, min(size, SAMPLE), replace=False))


def record(outputs) -> dict:
    """npz entries for ``{key: array}``: shape, SHA-256 of the values and a seeded sample (which keeps the dtype)."""
    rec = {}
    for key, a in outputs.items():
        a = np.asarray(a)
        rec[f"{key}/shape"] = np.array(a.shape, dtype=np.int64)
        rec[f"{key}/sha256"] = np.array(sha256(a))
        rec[f"{key}/sample"] = a.reshape(-1)[sample_index(a.size)]
    return rec


def check(stored, key, got):
    """``got`` equals, element for element and in dtype and shape, the reference output recorded under ``key``."""
    got = np.asarray(got)
    sample = stored[f"{key}/sample"]
    assert got.dtype == sample.dtype, (key, got.dtype, sample.dtype)
    assert got.shape == tuple(stored[f"{key}/shape"]), (key, got.shape, tuple(stored[f"{key}/shape"]))
    np.testing.assert_array_equal(got.reshape(-1)[sample_index(got.size)], sample, err_msg=key)
    assert sha256(got) == str(stored[f"{key}/sha256"]), f"{key}: values differ from the reference outside the stored sample"
