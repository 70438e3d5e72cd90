"""Pins the oracle: the numpy/cv2 restatement of process_frame against (i) golden vectors produced
by the compiled, unmodified reference, (ii) stored outputs of the reference on the larger frames and the HSI branch
(tests/golden/process_frame_outputs.npz) and (iii) the compiled reference itself when present."""
import glob
import hashlib
import os

import numpy as np
import pytest

from oracle import color_balance_np as cb
from oracle import ref_balance, synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
STORED_OUTPUTS = os.path.join(GOLDEN, "process_frame_outputs.npz")

DEFAULT_FLAG_CASES = [((96, 160), 3), ((200, 320), 5), ((479, 641), 9), ((270, 480), 4)]
HSI_CASES = [("underwater", (480, 640), 7, {}), ("random", (480, 640), 4, dict(hsv_contrast_correct=False)),
             ("underwater", (1242, 2208), 6, dict(equalize_rgb=False, rgb_extrema_clipping=False))]


def stored_cases():
    """{key: (kind, shape, seed, process_frame flags)} of every frame in STORED_OUTPUTS."""
    cases = [("underwater", shape, seed, {}) for shape, seed in DEFAULT_FLAG_CASES]
    cases += [(kind, shape, seed, dict(hsi_contrast_correct=True, **flags)) for kind, shape, seed, flags in HSI_CASES]
    return {"%s_%dx%d_seed%d" % (kind, shape[0], shape[1], seed) + "".join("_%s%d" % (k, v) for k, v in sorted(flags.items())):
            (kind, shape, seed, flags) for kind, shape, seed, flags in cases}


def synth_frame(kind, shape, seed):
    return synth.gen_underwater(shape[0], shape[1], seed) if kind == "underwater" else synth.gen_random_bgr(shape[0], shape[1], seed)


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def check_stored_output(key, img, got):
    """`got` (process_frame of `img`) against the stored output: a few full rows first, so that a mismatch says where,
    then the SHA-256 of the whole frame."""
    z = np.load(STORED_OUTPUTS)
    assert sha256(img) == str(z[key + "__src_sha256"]), "the synthetic input of %s is not the one stored" % key
    rows = z[key + "__row_index"]
    assert np.array_equal(got[rows], z[key + "__rows"]), "%s: stored rows %s differ" % (key, rows.tolist())
    assert sha256(got) == str(z[key + "__out_sha256"]), key


def golden_balance_cases():
    return sorted(glob.glob(os.path.join(GOLDEN, "balance_*.npz")))


def load_case(path):
    z = np.load(path, allow_pickle=True)
    flags = {k: v for k, v in z["flags"]} if z["flags"].size else {}
    return z["src"], z["out"], flags


@pytest.mark.parametrize("path", golden_balance_cases(), ids=lambda p: os.path.basename(p)[8:-4])
def test_restatement_matches_golden(path):
    src, want, flags = load_case(path)
    got = cb.process_frame_np(src, sequential_mean=True, **flags)
    assert np.array_equal(got, want)
    # the exact-mean variant (what the GPU computes) must give the same bytes
    assert np.array_equal(cb.process_frame_np(src, sequential_mean=False, **flags), want)


def test_golden_set_is_complete():
    names = {os.path.basename(p) for p in golden_balance_cases()}
    assert {"balance_default_96x160.npz", "balance_default_120x161.npz", "balance_rgbcc_96x160.npz",
            "balance_adaptive_96x160.npz", "balance_nohsv_96x160.npz"} <= names


@pytest.mark.skipif(not ref_balance.available(), reason="oracle/_ref not built")
@pytest.mark.parametrize("shape,seed", DEFAULT_FLAG_CASES)
def test_restatement_matches_compiled_reference(shape, seed):
    img = synth.gen_underwater(shape[0], shape[1], seed)
    assert np.array_equal(cb.process_frame_np(img), ref_balance.balance(img))


@pytest.mark.skipif(not ref_balance.available(), reason="oracle/_ref not built")
def test_compiled_reference_reproduces_golden():
    for path in golden_balance_cases():
        src, want, flags = load_case(path)
        assert np.array_equal(ref_balance.balance(src, **flags), want), path
    for key, (kind, shape, seed, flags) in stored_cases().items():
        img = synth_frame(kind, shape, seed)
        check_stored_output(key, img, ref_balance.balance(img, **flags))


def test_percentile_bounds_follow_float32_products():
    # 0.002f * N and 0.998f * N are float32 products truncated to int (color_balance.cpp:113-114)
    n = 2208 * 1242
    ch = np.zeros(n, np.uint8)
    ch[: int(np.float32(0.002) * np.float32(n)) + 1] = 7          # just enough to pass the low bound
    lo, hi = cb.percentile_min_max(ch)
    assert (lo, hi) == (0, 0) or lo in (0, 7)
    ch = np.arange(n, dtype=np.uint32).astype(np.uint8)
    assert cb.percentile_min_max(ch) == (0, 255)


def test_degenerate_sv_range_is_reported():
    img = np.full((32, 32, 3), 90, np.uint8)
    with pytest.raises(ZeroDivisionError):
        cb.process_frame_np(img)


@pytest.mark.skipif(not ref_balance.available(), reason="oracle/_ref not built")
@pytest.mark.parametrize("kind,shape,seed,flags", HSI_CASES)
def test_hsi_branch_restatement_matches_compiled_reference(kind, shape, seed, flags):
    """color_balance.cpp:702-774 (P2): float32 HSI planes, 0.2 % / 99.8 % order statistics, sector-wise HSI -> RGB."""
    img = synth_frame(kind, shape, seed)
    want = ref_balance.balance(img, hsi_contrast_correct=True, **flags)
    got = cb.process_frame_np(img, hsi_contrast_correct=True, **flags)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("key", sorted(stored_cases()))
def test_restatement_matches_stored_reference_outputs(key):
    """The compiled-reference comparisons above (default flags on larger frames, the HSI branch) without the compiled
    reference: the same inputs against its stored outputs."""
    kind, shape, seed, flags = stored_cases()[key]
    img = synth_frame(kind, shape, seed)
    check_stored_output(key, img, cb.process_frame_np(img, **flags))
