"""Generate tests/golden/hotpath_v1.npz (tests/cases.py), tests/golden/features_v1.npz
(tests/feature_cases.py) and tests/golden/reference_exact_v1.npz (tests/reference_outputs.py) by running
the cases through the UNMODIFIED reference.

Build-container only (needs /root/reference; see tools/ref_shim.py).  The fixtures travel to the GPU box,
where /root/reference does not exist.  Also stores a handful of constant tables (mel bases, window
sum-square, mel-scale known answers) produced by the reference.

    python tools/make_golden.py            # all three fixtures
    python tools/make_golden.py exact      # only reference_exact_v1.npz
"""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ref_shim  # noqa: E402
from cases import BY_NAME, CASES  # noqa: E402
import signals  # noqa: E402


def run_case(ref, case, store):
    op, kw = case["op"], dict(case["kw"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if op == "istft":
            D = store[case["src"]]
            return ref.istft(D, **kw)
        sr = kw.get("sr", 22050)
        y = signals.make(case["mix"], case["shape"], seed=len(case["name"]), sr=sr)
        if op == "stft":
            return ref.stft(y, **kw)
        if op == "mel":
            return ref.feature.melspectrogram(y=y, **kw)
        if op == "mfcc":
            return ref.feature.mfcc(y=y, **kw)
    raise ValueError(op)


def main():
    ref = ref_shim.load_reference()
    store = {}
    for case in CASES:
        out = run_case(ref, case, store)
        store[case["name"]] = np.ascontiguousarray(out)
        print(f"{case['name']:40s} {out.shape} {out.dtype}")
    # constant tables straight from the reference
    consts = {
        "const/mel_22050_2048": ref.filters.mel(sr=22050, n_fft=2048),
        "const/mel_44100_4096": ref.filters.mel(sr=44100, n_fft=4096),
        "const/mel_16000_1024_htk40": ref.filters.mel(sr=16000, n_fft=1024, n_mels=40, htk=True),
        "const/mel_22050_2048_norm1": ref.filters.mel(sr=22050, n_fft=2048, norm=1, fmin=300.0, fmax=8000.0, n_mels=64),
        "const/wss_hann_2048_512_50": ref.filters.window_sumsquare(window="hann", n_frames=50, hop_length=512, n_fft=2048),
        "const/wss_hamming_600_1024_300_20": ref.filters.window_sumsquare(window="hamming", n_frames=20, hop_length=300, win_length=600, n_fft=1024),
        "const/hz_to_mel": ref.hz_to_mel(np.array([0.0, 60.0, 440.0, 999.0, 1000.0, 5000.0, 11025.0])),
        "const/hz_to_mel_htk": ref.hz_to_mel(np.array([0.0, 60.0, 440.0, 999.0, 1000.0, 5000.0, 11025.0]), htk=True),
        "const/mel_to_hz": ref.mel_to_hz(np.array([0.0, 3.0, 14.9, 15.0, 25.0, 40.0])),
        "const/mel_to_hz_htk": ref.mel_to_hz(np.array([0.0, 300.0, 1000.0, 2000.0, 3000.0]), htk=True),
        "const/mel_frequencies_40": ref.mel_frequencies(n_mels=40),
        "const/window_hann_2048": ref.filters.get_window("hann", 2048),
        "const/power_to_db_in": (np.abs(np.random.default_rng(7).standard_normal((2, 16, 12))) ** 2).astype(np.float32),
    }
    consts["const/power_to_db_out"] = ref.power_to_db(consts["const/power_to_db_in"])
    consts["const/power_to_db_out_refmax"] = ref.power_to_db(consts["const/power_to_db_in"], ref=np.max)
    consts["const/power_to_db_out_top40"] = ref.power_to_db(consts["const/power_to_db_in"], top_db=40.0)
    store.update(consts)
    path = os.path.join(ROOT, "tests", "golden", "hotpath_v1.npz")
    np.savez_compressed(path, **store)
    print("wrote", path, os.path.getsize(path), "bytes; reference", ref.__version__)
    # ---- frame-wise consumers (tests/feature_cases.py)
    from feature_cases import FEATURE_CASES, call, fixture_names, outputs

    feats = {}
    for case in FEATURE_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out = call(ref, case, store)
        outs = outputs(out)
        for key, arr in zip(fixture_names(case, len(outs)), outs):
            feats[key] = np.ascontiguousarray(arr) if arr.ndim else arr
            print(f"{key:40s} {arr.shape} {arr.dtype}")
    path = os.path.join(ROOT, "tests", "golden", "features_v1.npz")
    np.savez_compressed(path, **feats)
    print("wrote", path, os.path.getsize(path), "bytes")
    write_reference_exact(ref)


def write_reference_exact(ref):
    """Records (shape, SHA-256, seeded sample) of the outputs tests/test_oracle_vs_reference.py pins bit for bit."""
    import reference_outputs

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        outputs = reference_outputs.all_groups(ref)
    path = os.path.join(ROOT, "tests", "golden", "reference_exact_v1.npz")
    np.savez_compressed(path, **reference_outputs.record(outputs))
    print("wrote", path, os.path.getsize(path), "bytes;", len(outputs), "outputs")


if __name__ == "__main__":
    if sys.argv[1:] == ["exact"]:
        write_reference_exact(ref_shim.load_reference())
    else:
        main()
