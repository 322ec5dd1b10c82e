"""CPU: the oracle, and the product's host-side constant builders, reproduce the unmodified reference bit for bit.

The reference's outputs are recorded in tests/golden/reference_exact_v1.npz (tools/make_golden.py; what is
computed is defined once, in tests/reference_outputs.py) and the frame-wise features in
tests/golden/features_v1.npz, so these tests need nothing outside the repository."""
import os
import warnings

import numpy as np
import pytest

import reference_outputs as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def stored():
    with np.load(os.path.join(ROOT, "tests", "golden", "reference_exact_v1.npz")) as z:
        return {k: z[k] for k in z.files}


def check_all(stored, outputs):
    for key, got in outputs.items():
        R.check(stored, key, got)


@pytest.mark.parametrize("n,n_fft,hop,center,pad_mode", R.STFT_GRID)
def test_stft_istft_bit_exact(stored, oracle, n, n_fft, hop, center, pad_mode):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        check_all(stored, R.stft_istft(R.librosa_layout(oracle), n, n_fft, hop, center, pad_mode))


def test_features_bit_exact(stored, oracle):
    check_all(stored, R.features(R.librosa_layout(oracle)))


def test_frame_statistics_bit_exact(oracle, golden):
    from feature_cases import FEATURE_CASES, call, fixture_names, outputs

    for case in FEATURE_CASES:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            B = outputs(call(oracle, case, golden))
        stored = [k for k in golden if k == case["name"] or k.startswith(case["name"] + "#")]
        assert len(stored) == len(B), case["name"]
        for key, b in zip(fixture_names(case, len(B)), B):
            a = golden[key]
            assert a.dtype == b.dtype and a.shape == b.shape, case["name"]
            np.testing.assert_array_equal(a, b, err_msg=case["name"])


def test_product_chroma_filter_matches_reference(stored):
    import librosa_b200 as lb

    check_all(stored, R.chroma(lb))


def test_griffinlim_bit_exact(stored, oracle):
    check_all(stored, R.griffinlim(R.librosa_layout(oracle)))


def test_product_host_constants_match_reference(stored):
    """The product's own host-side constant builders (librosa_b200.filters / convert / util) against the
    reference — these feed the GPU plans, so they are pinned as tightly as the oracle."""
    import librosa_b200 as lb

    check_all(stored, R.host_constants(lb))


def test_power_to_db_axes_and_float64_bit_exact(stored, oracle):
    """power_to_db with explicit reduction axes, and the float64 behaviour of the whole path (the reference
    computes float64 audio in float64: complex128 STFT, float64 mel / MFCC)."""
    check_all(stored, R.power_to_db_and_float64(R.librosa_layout(oracle)))


def test_feature_inverse_bit_exact(stored, oracle):
    """mel_to_stft (NNLS through SciPy's L-BFGS-B) and mfcc_to_mel restated in the oracle."""
    check_all(stored, R.feature_inverse(R.librosa_layout(oracle)))
