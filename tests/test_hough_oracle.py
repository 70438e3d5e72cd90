"""CPU: oracle/hough_np.py (cv2.HoughLines restated in numpy) equals cv2.HoughLines and cv2.HoughLinesWithAccumulator
4.13.0 on every case of oracle/hough_cases.py, float32 bits and row order identical, with cv2's optimised code paths on
and off; rule 8 (rho of a bin) is pinned with single pixels; the cases reach the shapes they are written for."""
import contextlib

import cv2
import numpy as np
import pytest

from oracle import hough_cases as hc, hough_np as hn

CASES = hc.by_group(hc.all_cases())


@contextlib.contextmanager
def cv2_optimized(on):
    before = cv2.useOptimized()
    cv2.setUseOptimized(on)
    try:
        yield
    finally:
        cv2.setUseOptimized(before)


def cv2_lines(frame, c, votes):
    rho, theta, thr, mn, mx, ev = c.args
    if votes:
        return cv2.HoughLinesWithAccumulator(frame, rho, theta, thr, min_theta=mn, max_theta=mx, use_edgeval=ev)
    return cv2.HoughLines(frame, rho, theta, thr, min_theta=mn, max_theta=mx)


def same(got, want):
    if got is None or want is None:
        return got is None and want is None
    return got.shape == want.shape and got.dtype == want.dtype and np.array_equal(got.view(np.int32), want.view(np.int32))


@pytest.mark.parametrize("group", sorted(CASES))
def test_restatement_equals_cv2(group):
    failures = []
    for c in CASES[group]:
        for k, f in enumerate(c.frames()):
            mine = hn.hough_lines(f, *c.args, votes=True)
            for opt in (True, False):
                with cv2_optimized(opt):
                    if not same(mine, cv2_lines(f, c, True)):
                        failures.append("%s frame %d (optimized %s): with votes" % (c.name, k, opt))
                    if not c.use_edgeval and not same(None if mine is None else mine[..., :2].copy(),
                                                      cv2_lines(f, c, False)):
                        failures.append("%s frame %d (optimized %s): HoughLines" % (c.name, k, opt))
    assert not failures, "\n".join(failures)


def test_rho_of_a_bin_uses_integer_division():
    """A pixel at the origin gives rho = 0 at every angle; one at column 11, row 0 with rho = 2 gives rho = 12 at
    theta = 0 (11 / 2 = 5.5 rounds half to even to bin 6), not the 11 the half-bin (numrho - 1) * 0.5f would give."""
    origin = np.zeros((9, 9), np.uint8)
    origin[0, 0] = 255
    for rho in (1, 2, 0.7):
        got = cv2.HoughLines(origin, rho, np.pi / 180, 0)
        assert got is not None and np.all(got[:, 0, 0] == 0.0)
        assert same(hn.hough_lines(origin, rho, np.pi / 180, 0), got)
    px = np.zeros((1, 12), np.uint8)
    px[0, 11] = 255
    got = cv2.HoughLines(px, 2, np.pi / 180, 0)
    assert got[0, 0, 1] == 0.0 and got[0, 0, 0] == 12.0
    assert same(hn.hough_lines(px, 2, np.pi / 180, 0), got)


def test_cases_reach_what_they_are_written_for():
    shapes, names = set(), set()
    first_last_angle, first_last_rho, fallback, many, ties = set(), set(), False, 0, False
    for c in hc.all_cases():
        f = c.frames()
        shapes.add(f.shape[1:])
        names.add(c.name)
        for im in f:
            acc, na, nr = hn.accumulator(im, c.rho, c.theta, c.min_theta, c.max_theta, c.use_edgeval)
            fallback |= (nr + 2) * 4 > 227 * 1024
            base, v = hn.peaks(acc, c.threshold)
            many = max(many, len(base))
            ties |= bool(len(v) > 1 and (v[1:] == v[:-1]).any())
            n_i, r_i = base // (nr + 2) - 1, base % (nr + 2) - 1
            first_last_angle |= {"first" for n in n_i if n == 0} | {"last" for n in n_i if n == na - 1 and na > 1}
            first_last_rho |= {"first" for r in r_i if r == 0} | {"last" for r in r_i if r == nr - 1}
    assert {(1, 1), (1, 37), (37, 1), (2160, 3840)} <= shapes
    assert {15, 16, 17, 31, 32, 33, 47, 48, 49} <= {w for _, w in shapes}
    assert first_last_angle == {"first", "last"} and first_last_rho == {"first", "last"}
    assert fallback and many > 100_000 and ties
    assert hn.counts(1080, 1920, 1, np.pi / 180, 0, np.pi)[0] == 180          # the last angle removed
    assert hn.counts(60, 60, 1, 0.3, 0, np.pi)[0] == 10                # floor(pi / 0.3) + 1 = 11, less the last
    assert hn.counts(60, 60, 1, 0.4, 0, np.pi)[0] == 8
    assert hn.counts(10, 10, 1, 1e-4, 0, np.pi)[0] == 31416
    for part in ("all_zero", "all_255", "edgeval", "plateau", "symmetric", "batch5", "underwater", "pi_removed"):
        assert any(part in n for n in names), part
