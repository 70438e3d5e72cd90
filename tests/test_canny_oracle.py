"""CPU: oracle/canny_np.py (cv2.Canny restated in integers, without cv2.Sobel) equals cv2.Canny 4.13.0 on every case of
oracle/canny_cases.py, with one OpenCV thread and with the default; the aperture-7 rule (scale 1/16, rounded half to
even) is pinned on its own; the cases reach every (aperture, norm, channels) combination and the shapes they are
written for."""
import contextlib

import cv2
import numpy as np
import pytest
from scipy import ndimage

from oracle import canny_cases as cc, canny_np as cn

CASES = cc.by_group(cc.all_cases())


@contextlib.contextmanager
def cv2_threads(n):
    """n OpenCV threads inside the block (-1: OpenCV's default count)."""
    before = cv2.getNumThreads()
    cv2.setNumThreads(n)
    try:
        yield
    finally:
        cv2.setNumThreads(before)


def cv2_canny(frame, c):
    return cv2.Canny(frame, c.threshold1, c.threshold2, apertureSize=c.aperture, L2gradient=c.l2)


@pytest.mark.parametrize("group", sorted(CASES))
def test_restatement_equals_cv2(group):
    failures = []
    for c in CASES[group]:
        frames = c.frames()
        mine = [cn.canny(f, c.threshold1, c.threshold2, c.aperture, c.l2) for f in frames]
        for threads in (1, -1):
            with cv2_threads(threads):
                for k, f in enumerate(frames):
                    d = int((cv2_canny(f, c) != mine[k]).sum())
                    if d:
                        failures.append("%s frame %d (%s): %d bytes" % (c.name, k, "1 thread" if threads == 1 else
                                                                       "default threads", d))
    assert not failures, "\n".join(failures)


def test_cases_reach_every_combination():
    seen = set()
    for c in cc.all_cases():
        seen.add((c.aperture, c.l2, 3 if c.frames().ndim == 4 else 1))
    assert seen == {(a, l2, ch) for a in (3, 5, 7) for l2 in (False, True) for ch in (1, 3)}


def test_cases_reach_the_shapes_they_are_written_for():
    shapes = {}
    for c in cc.all_cases():
        f = c.frames()
        shapes.setdefault((f.shape[1], f.shape[2]), set()).add(f.shape[0])
    for hw in [(1, 1), (1, 77), (77, 1), (2, 2)]:
        assert hw in shapes, hw
    widths = {w for (_, w) in shapes}
    assert {31, 32, 33, 63, 64, 65} <= widths
    assert (1242, 2208) in shapes and (2160, 3840) in shapes
    assert 5 in set().union(*shapes.values())
    names = {c.name for c in cc.all_cases()}
    for part in ("reversed", "equal", "zero_low", "negative", "fractional", "l2_clamp", "ap7_ties", "nan_low",
                 "checker", "steps", "diagonals", "underwater", "serpentine"):
        assert any(part in n for n in names), part


def test_aperture7_scale_and_half_even_rounding(monkeypatch):
    """cv2.Canny's aperture-7 gradients are Sobel(CV_16S, scale=1/16): the integer sum divided by 16 and rounded half
    to even.  The restatement equals cv2.Sobel with that scale on many ties; rounding ties up, or keeping the unscaled
    sums against undivided thresholds, makes cases of the case file differ from cv2.Canny."""
    rng = np.random.default_rng(7)
    ties = half_up_differs = 0
    for _ in range(6):
        im = cv2.GaussianBlur(rng.integers(0, 256, (70, 90), dtype=np.uint8), (3, 3), 0.8)
        dx, dy = cn.sobel(im, 7)
        for (ddx, ddy), got in (((1, 0), dx), ((0, 1), dy)):
            want = cv2.Sobel(im, cv2.CV_16S, ddx, ddy, ksize=7, scale=1 / 16.0, borderType=cv2.BORDER_REPLICATE)
            assert np.array_equal(got, want)
            raw = cv2.Sobel(im, cv2.CV_32F, ddx, ddy, ksize=7, borderType=cv2.BORDER_REPLICATE).astype(np.int64)
            ties += int(((raw & 15) == 8).sum())
            half_up_differs += int((((raw + 8) >> 4) != want).sum())
    assert ties > 1000 and half_up_differs > 0
    assert cn.thresholds(3000, 9000, 7, False) == (187, 562)

    ap7 = [c for c in cc.all_cases() if c.aperture == 7 and c.group in ("combo", "thresholds", "content")]

    def differing(t_scale):
        n = 0
        for c in ap7:
            f = c.frames()
            n += any(not np.array_equal(cn.canny(x, c.threshold1 * t_scale, c.threshold2 * t_scale, 7, c.l2),
                                        cv2_canny(x, c)) for x in f)
        return n
    assert differing(1) == 0
    monkeypatch.setattr(cn, "round_half_even_div16", lambda s: (s + 8) >> 4)
    assert differing(1) > 0
    # no scale: the raw sums against the thresholds as given (the oracle divides them by 16, so hand it 16 x)
    monkeypatch.setattr(cn, "round_half_even_div16", lambda s: s)
    assert differing(16) > len(ap7) // 2


def test_thresholds_follow_cv2():
    assert cn.thresholds(100, 50, 3, False) == (50, 100)
    assert cn.thresholds(50.9, 120.2, 3, False) == (50, 120)
    assert cn.thresholds(-3.5, 10, 3, True) == (-4, 100)                  # a negative threshold is not squared
    assert cn.thresholds(40000, 50000, 3, True) == (32767 ** 2, 32767 ** 2)
    # std::min(32767, NaN) is 32767, and the swap came before: low ends above high
    assert cn.thresholds(float("nan"), 10, 3, True) == (32767 ** 2, 100)
    assert cn.thresholds(float("nan"), 10, 3, False) == (cn.INT_MIN, 10)
    assert cn.thresholds(1e10, 3e10, 3, False) == (cn.INT_MIN, cn.INT_MIN)


def test_serpentine_is_one_chain_seeded_at_its_end():
    """The long-chain case: every candidate lies on one 8-connected chain that crosses the frame, the strong pixels are
    the two beside the bump at the chain's far end, and the output keeps the whole chain."""
    for c in CASES["serpentine"]:
        f = c.frames()[0]
        cand, strong = cn.candidates(f, c.threshold1, c.threshold2, c.aperture, c.l2)
        _, n = ndimage.label(cand, structure=np.ones((3, 3), bool))
        ys, xs = np.nonzero(cand)
        assert n == 1 and ys.min() <= 2 and ys.max() >= f.shape[0] - 10 and xs.min() <= 2 and xs.max() >= f.shape[1] - 3
        assert int(strong.sum()) == 2 and np.ptp(np.nonzero(strong)[0]) <= 2
        assert np.array_equal(cn.canny(f, c.threshold1, c.threshold2, c.aperture, c.l2) > 0, cand)
