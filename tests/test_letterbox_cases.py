"""The letterbox case matrix (oracle/letterbox_cases.py) and the arithmetic its GPU tests rely on, without a GPU.

- every case reaches the paths it was written for, and the cases together reach every path of bv_letterbox;
- the host instantiation of the resize arithmetic (csrc/pixel_math.cuh: linear_coef / linear_vblend) is identical to
  cv2.resize over a sweep of small, odd and extreme sizes and over every letterbox geometry of the matrix;
- u / 255 rounded to fp16 is the same value whether the division is done in float32 (the kernels), float64, or by
  torch on half operands (`im.half() / 255`, the Ultralytics preprocess), so the GPU tests may demand 0 differing
  values."""
import ctypes
import os
import subprocess

import cv2
import numpy as np
import pytest
import torch

from oracle import letterbox, letterbox_cases as lc

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostmath", "hostmath.cpp")
OUT = os.path.join(HERE, "hostmath", "_build", "libhostmath.so")


@pytest.fixture(scope="module")
def hm():
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    csrc = os.path.join(HERE, "..", "cuauv_vision_pipeline_b200", "csrc")
    deps = [SRC, os.path.join(csrc, "pixel_math.cuh"), os.path.join(csrc, "luv_fix.inc")]
    if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-x", "c++", SRC, "-o", OUT])
    return ctypes.CDLL(OUT)


ALL_CASES = lc.single_cases() + lc.batch_cases()


@pytest.mark.parametrize("case", ALL_CASES, ids=lambda c: c.name)
def test_case_reaches_the_paths_it_was_written_for(case):
    paths = case.paths()
    assert case.wants <= paths, (case.name, case.wants - paths)
    # the kernel choice is exclusive
    assert ("gather" in paths) != bool(paths & {"tma", "staged"})


def test_cases_cover_every_path():
    reached = set()
    for c in ALL_CASES:
        reached |= c.paths()
    assert reached == set(lc.ALL_PATHS)
    # with BV_LETTERBOX_GATHER set every case takes the gather kernel
    for c in ALL_CASES:
        p = c.paths(gather_env=True)
        assert "gather" in p and not p & {"tma", "staged", "smem_gather", "narrow_rows", "global_descs", "cross_images"}


def test_case_geometry_claims():
    """Spot checks of the geometry the matrix was built around, worked out independently of expected_paths."""
    g = letterbox.letterbox_geometry
    assert g(5, 3000) == (640, 1, 319, 320, 0, 0)
    assert g(3000, 5)[:2] == (1, 640)
    assert g(4000, 6000)[2:4] == (106, 107)
    uw, uh = g(641, 300)[:2]
    assert uw == 300 and uh == 640                    # horizontal scale exactly 1, vertical not
    assert g(640, 320)[:2] == (320, 640) and g(320, 640)[:2] == (640, 320)
    assert 3840 * 3 == lc.LB_MAX_ROW_BYTES and 3841 * 3 > lc.LB_MAX_ROW_BYTES
    # the 30000-wide output's tap table alone exceeds a block's shared memory
    assert lc.tma_smem([1920], 30000) > lc.SMEM_SURE_EXCEEDS
    assert lc.tma_smem([3840], 1280) <= lc.SMEM_SURE_FITS


def test_persistent_grid_cases_straddle_the_grid():
    full = lc.persistent_grid([64], 65535, 48, lc.B200_SMS)
    items = sorted(len(c.srcs) * c.out_h for c in lc.batch_cases() if c.name.startswith("items"))
    assert items == [1, full - 1, full, full + 1]


def test_expected_paths_rejects_too_many_images():
    assert len(lc.too_many_images()) == lc.LB_MAX_IMGS + 1
    with pytest.raises(ValueError):
        lc.expected_paths([(4, 4)] * (lc.LB_MAX_IMGS + 1), 64, 64)


# ---------------------------------------------------------------------------------------------------------------------
# resize arithmetic
# ---------------------------------------------------------------------------------------------------------------------
def hm_resize(hm, im, dh, dw):
    sh, sw, c = im.shape
    out = np.empty((dh, dw, c), np.uint8)
    hm.hm_resize(im.ctypes.data_as(ctypes.c_void_p), sh, sw, out.ctypes.data_as(ctypes.c_void_p), dh, dw, c)
    return out


def cv_resize(im, dh, dw):
    return cv2.resize(im, (dw, dh), interpolation=cv2.INTER_LINEAR).reshape(dh, dw, im.shape[2])


SWEEP_W = list(range(1, 34)) + [63, 64, 65, 127, 255, 641]


def test_resize_arithmetic_sweep(hm):
    rng = np.random.default_rng(11)
    bad = []
    for sh in (1, 2, 3, 7, 31):
        for sw in SWEEP_W:
            im = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
            for dh in (1, 2, 5, 31, 62):
                for dw in SWEEP_W:
                    if not np.array_equal(hm_resize(hm, im, dh, dw), cv_resize(im, dh, dw)):
                        bad.append((sh, sw, dh, dw))
    assert not bad, bad[:10]


@pytest.mark.parametrize("src,dst", [((1, 3840), (1, 1)), ((3840, 1), (1, 1)), ((3, 3), (3000, 3000)),
                                     ((1, 4000), (1, 3)), ((2, 2), (4096, 4096)), ((2, 2), (1, 4096))])
def test_resize_arithmetic_extreme_ratios(hm, src, dst):
    im = np.random.default_rng(12).integers(0, 256, src + (3,), dtype=np.uint8)
    assert np.array_equal(hm_resize(hm, im, *dst), cv_resize(im, *dst))


def test_resize_arithmetic_letterbox_geometries(hm):
    """Every resize the case matrix asks of the letterbox (its un-padded size), one source of each shape."""
    seen = set()
    for c in ALL_CASES:
        for (h, w) in c.shapes:
            uw, uh = letterbox.letterbox_geometry(h, w, c.out_h, c.out_w)[:2]
            if (h, w) != (uh, uw):
                seen.add((h, w, uh, uw))
    bad = []
    for h, w, uh, uw in sorted(seen):
        im = lc.random_image(h, w, h * 7 + w)
        if not np.array_equal(hm_resize(hm, im, uh, uw), cv_resize(im, uh, uw)):
            bad.append((h, w, uh, uw))
    assert len(seen) > 30 and not bad, bad


# ---------------------------------------------------------------------------------------------------------------------
# normalisation
# ---------------------------------------------------------------------------------------------------------------------
def test_fp16_normalisation_table_is_the_same_in_every_precision():
    u = np.arange(256)
    via_f32 = (u.astype(np.float32) / np.float32(255)).astype(np.float16)
    via_f64 = (u.astype(np.float64) / 255.0).astype(np.float16)
    via_torch = (torch.arange(256, dtype=torch.uint8).half() / 255).numpy()
    via_oracle = letterbox.yolo_input([np.repeat(u.astype(np.uint8), 3).reshape(1, 256, 3)], 1, 256)[0, 0, 0]
    assert np.array_equal(via_f32.view(np.uint16), via_f64.view(np.uint16))
    assert np.array_equal(via_f32.view(np.uint16), via_torch.view(np.uint16))
    assert np.array_equal(via_f32.view(np.uint16), via_oracle.view(np.uint16))
    # fp32 output: one IEEE division, the value the kernels' table holds
    assert np.array_equal(letterbox.yolo_input([np.repeat(u.astype(np.uint8), 3).reshape(1, 256, 3)], 1, 256,
                                               half=False)[0, 0, 0], u.astype(np.float32) / np.float32(255))
