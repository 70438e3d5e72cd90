"""oracle/contour_shapes.py against cv2 4.13.0 on every border of the masks of tests/test_contour_tree_oracle.py, for
CHAIN_APPROX_NONE and SIMPLE: the definitions bv_contour_shapes computes on the device (CPU only)."""
import cv2
import numpy as np
import pytest

from oracle import contour_shapes as cs
from oracle import synth

ABS_EPS = (0.0, 0.5, 1.0, 3.0, 1e9)
REL_EPS = (0.005, 0.02, 0.1)


def _masks():
    out = []
    for seed in range(300):
        rng = np.random.default_rng(1000 + seed)
        h, w = int(rng.integers(1, 91)), int(rng.integers(1, 91))
        if seed % 3 == 0:
            m = (rng.random((h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8) * 255
        else:
            f = cv2.GaussianBlur(rng.random((h, w)).astype(np.float32), (0, 0), rng.uniform(0.7, 3.0))
            m = (f > np.quantile(f, rng.uniform(0.2, 0.8))).astype(np.uint8) * 255
        out.append(m)
    out += [synth.mask_rings(61, 70, step=3), synth.mask_diagonals(40, 50), synth.mask_random(1, 31, 3, 0.6),
            synth.mask_random(31, 1, 4, 0.6), np.full((1, 1), 255, np.uint8), np.full((20, 30), 255, np.uint8)]
    lines = np.zeros((40, 40), np.uint8)
    cv2.line(lines, (2, 3), (35, 20), 255, 1)
    cv2.line(lines, (5, 30), (30, 30), 255, 1)
    cv2.line(lines, (38, 2), (38, 37), 255, 1)
    out.append(lines)
    return out


MASKS = _masks()
GROUPS = [MASKS[k::8] for k in range(8)]


def _borders(group):
    for m in group:
        for method in (cv2.CHAIN_APPROX_NONE, cv2.CHAIN_APPROX_SIMPLE):
            yield from cv2.findContours(m, cv2.RETR_TREE, method)[0]


@pytest.mark.parametrize("g", range(len(GROUPS)))
def test_arc_length_in_any_order(g):
    rng = np.random.default_rng(g)
    for c in _borders(GROUPS[g]):
        want = cv2.arcLength(c, True)
        assert cs.arc_length(c) == want
        assert cs.arc_length(c, order=rng.permutation(len(c))) == want


@pytest.mark.parametrize("g", range(len(GROUPS)))
def test_convex_hull(g):
    repeated = differing = 0
    for c in _borders(GROUPS[g]):
        got, want = cs.convex_hull(c), cv2.convexHull(c)
        assert got.dtype == want.dtype and got.shape == want.shape
        # the same vertices in the same cyclic order, always
        k = [tuple(v) for v in want.reshape(-1, 2)].index(tuple(got[0, 0]))
        assert np.array_equal(np.roll(want, -k, axis=0), got)
        if cs.has_repeated_pixel(c):
            repeated += 1
            differing += not np.array_equal(got, want)
        else:
            assert np.array_equal(got, want)               # the same first vertex
    assert differing <= 0.25 * max(repeated, 1)            # measured: 10-15 %


def _stroke_masks(n, seed):
    """Thick open polylines (3-5 random vertices, 2-4 px wide) and hooks (a thick arc ending in a sharp turn): borders
    whose points project past the ends of the chords Douglas-Peucker draws."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        m = np.zeros((80, 80), np.uint8)
        if k % 4 == 3:
            c = tuple(int(v) for v in rng.integers(20, 60, 2))
            ax = tuple(int(v) for v in rng.integers(8, 30, 2))
            a0 = int(rng.integers(0, 360))
            cv2.ellipse(m, c, ax, 0, a0, a0 + int(rng.integers(90, 330)), 255, int(rng.integers(1, 5)))
            end = rng.integers(0, 80, 2)
            cv2.line(m, c, (int(end[0]), int(end[1])), 255, int(rng.integers(1, 4)))
        else:
            pts = rng.integers(0, 80, (int(rng.integers(3, 6)), 2)).astype(np.int32)
            cv2.polylines(m, [pts.reshape(-1, 1, 2)], False, 255, thickness=int(rng.integers(2, 5)))
        out.append(m)
    return out


STROKES = _stroke_masks(800, 0)
DP_GROUPS = GROUPS + [STROKES[k::4] for k in range(4)]


@pytest.mark.parametrize("g", range(len(DP_GROUPS)))
def test_approx_poly_dp_and_convexity(g):
    for c in _borders(DP_GROUPS[g]):
        arc = cv2.arcLength(c, True)
        for eps in ABS_EPS + (2.0,) + tuple(k * arc for k in REL_EPS + (0.05,)):
            got, want = cs.approx_poly_dp(c, eps), cv2.approxPolyDP(c, eps, True)
            assert got.dtype == want.dtype and np.array_equal(got, want), (eps, c.reshape(-1, 2).tolist())
            assert cs.is_contour_convex(got) == cv2.isContourConvex(want)


def test_approx_splits_on_the_chord_segment():
    """A point past the end of the chord counts with its distance to that end, not to the chord's line."""
    c = np.array([[[0, 0]], [[15, 1]], [[10, 0]]], np.int32)
    assert len(cv2.approxPolyDP(c, 5.0, False)) == 3 and len(cv2.approxPolyDP(c, 5.1, False)) == 2   # sqrt(26) = 5.099
    hook = np.array([[[0, 0]], [[20, 0]], [[25, 1]], [[20, 2]], [[0, 2]]], np.int32)
    for eps in (0.5, 1.0, 2.0, 5.0, 5.1, 10.0):
        assert np.array_equal(cs.approx_poly_dp(hook, eps), cv2.approxPolyDP(hook, eps, True)), eps


@pytest.mark.parametrize("g", range(len(GROUPS)))
def test_min_enclosing_circle_within_tolerance(g):
    for c in _borders(GROUPS[g]):
        (cx, cy), r = cs.enclosing_circle(c)
        (wx, wy), wr = cv2.minEnclosingCircle(c)
        assert abs(cx - wx) <= 2e-4 and abs(cy - wy) <= 2e-4 and abs(r + 1e-4 - wr) <= 2e-4
        p = c.reshape(-1, 2).astype(np.float64)
        assert (np.hypot(p[:, 0] - cx, p[:, 1] - cy) <= r + 1e-9).all()


def test_cv2_facts():
    """cv2's EPS on the radius, and that a random point set is not started at its smallest point."""
    assert cv2.minEnclosingCircle(np.array([[[3, 4]]], np.int32)) == ((3.0, 4.0), 1e-4) or \
        abs(cv2.minEnclosingCircle(np.array([[[3, 4]]], np.int32))[1] - 1e-4) < 1e-9
    sq = np.array([[[0, 0]], [[0, 10]], [[10, 10]], [[10, 0]]], np.int32)
    assert abs(cv2.minEnclosingCircle(sq)[1] - (np.sqrt(50) + 1e-4)) < 1e-5
    assert np.array_equal(cs.convex_hull(sq), cv2.convexHull(sq))
    rng = np.random.default_rng(3)
    for _ in range(50):
        p = rng.integers(0, 100, (20, 1, 2)).astype(np.int32)
        want = cv2.convexHull(p)
        got = cs.convex_hull(p)
        k = [tuple(v) for v in want.reshape(-1, 2)].index(tuple(got[0, 0]))
        assert np.array_equal(np.roll(want, -k, axis=0), got)
