"""CPU: the cases of oracle/filter_cases.py reach the blur paths they were written for, oracle/spec_np.py equals cv2 on
every case, and the cv2 4.13.0 rounding facts the warp, remap and undistortion kernels reproduce.

cvRound / saturate_cast<int> compile to cvtss2si / cvtsd2si on x86-64, which return INT_MIN for NaN, +-inf and anything
outside int32.  Other architectures round such values differently, so the tests that depend on them say so and skip
there."""
import platform
from collections import defaultdict

import cv2
import numpy as np
import pytest

from oracle import filter_cases as fc, spec_np

X86 = platform.machine().lower() in ("x86_64", "amd64")
x86_only = pytest.mark.skipif(not X86, reason="cv2 rounds NaN and out-of-range coordinates with x86-64's cvtss2si / "
                                              "cvtsd2si (INT_MIN); other CPUs round them differently")

BLUR = fc.blur_cases()
BLUR_GROUPS, WARP_GROUPS, REMAP_GROUPS = fc.by_group(BLUR), fc.by_group(fc.warp_cases()), fc.by_group(fc.remap_cases())
BORDER = {"constant": cv2.BORDER_CONSTANT, "replicate": cv2.BORDER_REPLICATE}


def first_difference(got, want):
    bad = np.argwhere(got != want)
    return "%d differing bytes, first at %s: %r vs %r" % (len(bad), tuple(bad[0]), got[tuple(bad[0])],
                                                          want[tuple(bad[0])]) if bad.size else ""


# ---------------------------------------------------------------------------------------------------------------------
# blur paths
# ---------------------------------------------------------------------------------------------------------------------
def test_every_blur_case_reaches_its_path():
    for c in BLUR:
        p = c.predicted()
        assert fc.path_label(p) == c.path, (c.name, fc.path_label(p))
        if c.smem is not None:
            assert p.kind == "tile" and p.smem == c.smem, (c.name, p)


def test_blur_cases_reach_every_reachable_path():
    reached = defaultdict(list)
    for c in BLUR:
        reached[c.path].append(c.name)
    assert set(reached) == fc.reachable_blur_paths(), sorted(set(reached) ^ fc.reachable_blur_paths())
    for path in sorted(reached):            # the listing: every reachable path and how many cases take it
        print("%-16s %4d cases, e.g. %s" % (path, len(reached[path]), reached[path][0]))
    # the families of the case list: both sides of 48 KiB and of the 200 KiB switch, batches on every family
    sizes = sorted(fc.expected_blur_path(*c.shape, *c.ksize, 0, 0).smem for c in BLUR_GROUPS["smem"]
                   if c.path.startswith("tile"))
    assert sizes[0] <= fc.SMEM_DEFAULT < sizes[-1] <= fc.BLUR_TWO_LAUNCH_SMEM
    assert {c.path.split("<")[0] for c in BLUR_GROUPS["batch"]} == {"fast", "tile", "two_launch"}
    assert {c.shape[3] for c in BLUR_GROUPS["batch"] if c.path.startswith("fast")} == {1, 3}


def test_two_launch_grey_is_unreachable():
    """blur_rows16_kernel<1> / blur_cols16_kernel<1> are not built: no grey kernel size needs more than the tile."""
    worst = max(fc.blur_tile_smem(1, kx, ky) for kx in range(1, 202, 2) for ky in range(1, 202, 2))
    assert worst == fc.blur_tile_smem(1, 201, 201) == 90944 < fc.BLUR_TWO_LAUNCH_SMEM
    for kx in range(1, 202, 2):
        for ky in (1, 101, 201):
            for w in (1, 3, 4, 4000):
                assert fc.expected_blur_path(1, 8, w, 1, kx, ky, 0, 0).kind != "two_launch"


def test_square_kernel_boundaries():
    smem = fc.blur_tile_smem
    n = fc.BGR_SQUARE_ABOVE_48K
    assert smem(3, n - 2, n - 2) == 48304 <= fc.SMEM_DEFAULT < smem(3, n, n) == 50112
    n = fc.GREY_SQUARE_ABOVE_48K
    assert smem(1, n - 2, n - 2) == 48368 <= fc.SMEM_DEFAULT < smem(1, n, n) == 49296
    n = fc.BGR_SQUARE_TWO_LAUNCH
    assert smem(3, n - 2, n - 2) == 202752 <= fc.BLUR_TWO_LAUNCH_SMEM < smem(3, n, n) == 206032
    assert smem(3, 151, 151) == 186736 and smem(3, 151, 161) < fc.BLUR_TWO_LAUNCH_SMEM < smem(3, 151, 171)


# ---------------------------------------------------------------------------------------------------------------------
# spec_np against cv2 on every case
# ---------------------------------------------------------------------------------------------------------------------
SPEC_BLUR_WORK = 5e7      # pixels x taps; the 4K cases are left to the device test, which compares with cv2 directly


@pytest.mark.parametrize("group", sorted(BLUR_GROUPS))
def test_spec_blur_matches_cv2(group):
    checked = 0
    for c in BLUR_GROUPS[group]:
        if c.pixels * sum(c.ksize) > SPEC_BLUR_WORK:
            continue
        for im in c.image():
            im = im[..., 0] if c.shape[3] == 1 else im
            want = cv2.GaussianBlur(im, c.ksize, c.sigma[0], sigmaY=c.sigma[1])
            got = spec_np.gaussian_blur_8u(im, c.ksize, *c.sigma)
            assert np.array_equal(got, want), (c.name, first_difference(got, want))
        checked += 1
    assert checked or group == "uhd"


def cv2_warp(c, im):
    return cv2.warpAffine(im, c.matrix.astype(np.float64), c.dsize, flags=cv2.INTER_LINEAR, borderMode=BORDER[c.border],
                          borderValue=c.border_value)


@x86_only
@pytest.mark.parametrize("group", sorted(WARP_GROUPS))
def test_spec_warp_affine_matches_cv2(group):
    for c in WARP_GROUPS[group]:
        for im in c.image():
            im = im[..., 0] if c.shape[3] == 1 else im
            want = cv2_warp(c, im)
            got = spec_np.warp_affine_8u(im, c.matrix, c.dsize, c.border, c.border_value[:c.shape[3]])
            assert np.array_equal(got, want), (c.name, first_difference(got, want))


def cv2_remap(c, im):
    return cv2.remap(im, c.map1, c.map2, cv2.INTER_LINEAR, borderMode=BORDER[c.border], borderValue=c.border_value)


@x86_only
@pytest.mark.parametrize("group", sorted(REMAP_GROUPS))
def test_spec_remap_matches_cv2(group):
    for c in REMAP_GROUPS[group]:
        for im in c.image():
            im = im[..., 0] if c.shape[3] == 1 else im
            want = cv2_remap(c, im)
            got = spec_np.remap_linear_8u(im, c.map1, c.map2, c.border, c.border_value[:c.shape[3]])
            assert np.array_equal(got, want), (c.name, first_difference(got, want))
        if not c.fixed:
            m1, m2 = cv2.convertMaps(c.map1, c.map2, cv2.CV_16SC2)
            s1, s2 = spec_np.fixed_point_maps(c.map1, c.map2)
            assert np.array_equal(s1, m1) and np.array_equal(s2, m2), c.name


@x86_only
@pytest.mark.parametrize("case", fc.undistort_cases(), ids=lambda c: c.name)
def test_spec_undistort_maps_match_cv2(case):
    r1, r2 = cv2.initUndistortRectifyMap(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size, cv2.CV_16SC2)
    s1, s2 = spec_np.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, case.new_k, case.size, fixed=True)
    v = case.vector_cols
    assert np.array_equal(s1[:, :v], r1[:, :v]) and np.array_equal(s2[:, :v], r2[:, :v])
    # the columns cv2 may finish with scalar code (see CV_SIMD_COLS) differ only where that code truncates to short
    tail = (s1[:, v:] != r1[:, v:]).any(-1)
    assert np.array_equal(s2[:, v:], r2[:, v:])
    assert (np.abs(s1[:, v:][tail].astype(np.int64)) >= 32767).any(-1).all()


# ---------------------------------------------------------------------------------------------------------------------
# cv2 4.13.0 facts (x86-64)
# ---------------------------------------------------------------------------------------------------------------------
@x86_only
def test_cvround_gives_int_min_for_nan_and_out_of_range():
    """convertMaps (cvRound(x * 32) of a float32 map) returns the integer part -32768 and fraction 0 for NaN, +-inf
    and every |x * 32| >= 2^31, on both sides; the largest in-range float32 below 2^26 saturates to 32767 instead."""
    vals = np.array([np.nan, np.inf, -np.inf, 1e9, -1e9, 7e7, -7e7, 2 ** 26, 2 ** 26 + 8, -(2 ** 26 + 8)], np.float32)
    ok = np.array([2 ** 26 - 4, 32768.0, -32769.0], np.float32)
    x = np.concatenate([vals, ok])[None, :]
    m1, m2 = cv2.convertMaps(x, np.zeros_like(x), cv2.CV_16SC2)
    assert list(m1[0, :vals.size, 0]) == [-32768] * vals.size
    assert list(m1[0, vals.size:, 0]) == [32767, 32767, -32768]
    assert not (m2[0] & 31).any()
    assert np.array_equal(spec_np.cv_round(np.float32([2.5, -2.5, 3.5, np.nan, 2 ** 31, -2 ** 31])),
                          [2, -2, 4, -2 ** 31, -2 ** 31, -2 ** 31])
    assert spec_np.cv_round(np.float64(2 ** 31 - 1.5)) == 2 ** 31 - 2
    assert spec_np.cv_round(np.float64(2 ** 31 - 0.5)) == -2 ** 31          # rounds to 2^31: out of range
    assert spec_np.cv_round(np.float64(-2 ** 31 - 0.5)) == -2 ** 31         # rounds (to even) to -2^31: in range
    img = fc.random_image((6, 9, 3), 7)
    for v, col in ((1e9, 0), (7e7, 0), (np.nan, 0), (2 ** 26 - 4, 8), (-7e7, 0)):
        mx, my = np.full((1, 1), v, np.float32), np.full((1, 1), 2.0, np.float32)
        got = cv2.remap(img, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)
        assert np.array_equal(got[0, 0], img[2, col]), v


@x86_only
def test_warp_affine_coordinates_saturate_like_cvround():
    """A translation of -40000 px keeps the int coordinate in range: it saturates to short and lands on the right edge.
    One of -2.2e6 px leaves int32 after x 1024: cvRound gives INT_MIN and it lands on the left edge."""
    img = fc.random_image((9, 13, 3), 8)
    for tx, col in ((-40000.0, -1), (-2.2e6, 0), (-3e6, 0), (40000.0, 0), (2.2e6, 0)):
        got = cv2.warpAffine(img, np.array([[1.0, 0, tx], [0, 1, 0]]), (13, 9), borderMode=cv2.BORDER_REPLICATE)
        assert np.array_equal(got, np.repeat(img[:, col:col + 1 if col >= 0 else None], 13, axis=1)), tx


@x86_only
def test_cv_16sc2_undistort_maps_saturate():
    """The wide new camera sends most rays far outside the frame: cv2's vector code saturates the integer part to
    int16 (the model wrapped it before); with |u * 32| beyond int32 the coordinate is INT_MIN and saturates to
    -32768.  In a 964-wide map the last 4 columns come from cv2's scalar code, which truncates instead."""
    case = fc.undistort_cases()[0]
    r1, _ = cv2.initUndistortRectifyMap(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size, cv2.CV_16SC2)
    mx, my = cv2.initUndistortRectifyMap(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size, cv2.CV_32FC1)
    assert (r1 == 32767).sum() > 1000 and (r1 == -32768).sum() > 1000
    assert np.abs(mx).max() > 2 ** 26 and np.abs(my).max() > 2 ** 26
    wrapped = ((np.trunc(mx.astype(np.float64) * 32).astype(np.int64) >> 5) + 2 ** 15) % 2 ** 16 - 2 ** 15
    assert (wrapped != r1[..., 0]).mean() > 0.5
    r1w, _ = cv2.initUndistortRectifyMap(fc.CAM_K, fc.CAM_D, None, case.new_k, (964, 724), cv2.CV_16SC2)
    s1w, _ = spec_np.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, case.new_k, (964, 724), fixed=True)
    cols = np.unique(np.argwhere((r1w != s1w).any(-1))[:, 1])
    assert cols.size and set(cols) <= {960, 961, 962, 963}, cols
