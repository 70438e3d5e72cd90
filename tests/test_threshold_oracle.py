"""CPU: oracle/threshold_np.py (cv2.threshold with THRESH_OTSU / THRESH_TRIANGLE and cv2.adaptiveThreshold restated in
numpy) equals cv2 4.13.0 on every case of oracle/threshold_cases.py, with cv2's optimised code paths on and off.
GAUSSIAN_C with k >= 11 may differ only at proven ties: pixels whose double-precision mean lies within 1e-3 of a
half-integer.  The MEAN_C rule (float32 up to k^2 = 2^23, double above) is pinned, the Gaussian taps against
cv2.getGaussianKernel, the constants of the package against cv2's, and the cases against what they are written for."""
import contextlib

import cv2
import numpy as np
import pytest

from oracle import threshold_cases as tc, threshold_np as tn

CASES = tc.by_group(tc.all_cases())


@contextlib.contextmanager
def cv2_optimized(on):
    before = cv2.useOptimized()
    cv2.setUseOptimized(on)
    try:
        yield
    finally:
        cv2.setUseOptimized(before)


def cv2_result(frame, c):
    if c.kind == "auto":
        maxval, base, method = c.args
        return cv2.threshold(frame, 0, maxval, base | method)
    mv, method, base, k, cc = c.args
    return None, cv2.adaptiveThreshold(frame, mv, method, base, k, cc)


def mine(frame, c):
    if c.kind == "auto":
        maxval, base, method = c.args
        return tn.threshold_auto(frame, maxval, base, method)
    return None, tn.adaptive(frame, *c.args)


def differences(frame, c, ref, got):
    """'' when equal, or equal but at proven ties of GAUSSIAN_C k >= 11; else what differs.  Returns (message, ties)."""
    if ref[0] != got[0]:
        return "retval %r, cv2 %r" % (got[0], ref[0]), 0
    bad = ref[1] != got[1]
    if not bad.any():
        return "", 0
    if c.kind == "adaptive" and c.args[1] == tc.GAUSSIAN_C and c.args[3] >= 11:
        ties = tn.gaussian_ties(frame, c.args[3])
        if ties[bad].all():
            return "", int(bad.sum())
    return "%d differing bytes" % int(bad.sum()), 0


@pytest.mark.parametrize("group", sorted(CASES))
def test_restatement_equals_cv2(group):
    failures, ties = [], 0
    for c in CASES[group]:
        for k, f in enumerate(c.frames()):
            got = mine(f, c)
            for opt in (True, False):
                with cv2_optimized(opt):
                    ref = cv2_result(f, c)
                if opt and c.otsu_tie:
                    # cv2's IPP Otsu may take another bin of the exact tie; the restatement is cv2's own loop
                    if ref[0] not in c.otsu_tie:
                        failures.append("%s frame %d: IPP chose %r, outside the tie" % (c.name, k, ref[0]))
                    continue
                msg, n = differences(f, c, ref, got)
                ties += n
                if msg:
                    failures.append("%s frame %d (optimized %s): %s" % (c.name, k, opt, msg))
    assert not failures, "\n".join(failures)
    print("%s: %d bytes differ at proven ties" % (group, ties))


def test_mean_c_is_float32_up_to_2_23_then_double():
    """cv2.boxFilter sums 8-bit windows in int32 and scales in float32 while k^2 <= 2^23, and in double above (k >= 2897).
    At k = 255 and 1001 the float32 product rounds some sums that exact rounding of s / k^2 rounds the other way; at
    k = 2897 and 2899 the float32 rule would part from cv2.  The restatement follows cv2 on both sides."""
    parted_small, parted_wide = 0, {}
    for c in CASES["adapt_ties"]:
        f = c.frames()[0]
        k = c.args[3]
        s = tn.box_sums(f, k)
        f32_rule = np.clip(np.rint(s.astype(np.float32) * np.float32(1.0 / (k * k))), 0, 255)
        exact = (2 * s + k * k) // (2 * k * k)
        for opt in (True, False):
            with cv2_optimized(opt):
                ref = cv2.blur(f, (k, k), borderType=cv2.BORDER_REPLICATE)
            assert np.array_equal(ref, tn.mean_c(f, k).astype(np.uint8)), (c.name, opt)
        if k * k <= 1 << 23:
            parted_small += int((exact != f32_rule).sum())
        else:
            parted_wide[k] = parted_wide.get(k, 0) + int((f32_rule != ref).sum())
    assert parted_small > 0 and parted_wide[2897] > 0 and parted_wide[2899] > 0, (parted_small, parted_wide)
    assert 2895 ** 2 <= 1 << 23 < 2897 ** 2


def test_gaussian_taps_are_cv2s():
    for k in (3, 5, 7, 9, 11, 13, 51, 255, 1001, 2901):
        want = cv2.getGaussianKernel(k, 0, cv2.CV_32F).ravel()
        assert np.array_equal(tn.gaussian_taps(k).view(np.int32), want.view(np.int32)), k


def test_constants_are_cv2s():
    from cuauv_vision_pipeline_b200 import color
    for name in ("THRESH_BINARY", "THRESH_BINARY_INV", "THRESH_TRUNC", "THRESH_TOZERO", "THRESH_TOZERO_INV",
                 "THRESH_OTSU", "THRESH_TRIANGLE", "ADAPTIVE_THRESH_MEAN_C", "ADAPTIVE_THRESH_GAUSSIAN_C"):
        assert getattr(color, name) == getattr(cv2, name), name


def test_what_cv2_rejects():
    x = np.zeros((8, 8), np.uint8)
    for call in (lambda: cv2.threshold(np.zeros((8, 8, 3), np.uint8), 0, 255, cv2.THRESH_OTSU),
                 lambda: cv2.threshold(x, 0, 255, cv2.THRESH_OTSU | cv2.THRESH_TRIANGLE),
                 lambda: cv2.adaptiveThreshold(x, 255, 0, 0, 1, 0),
                 lambda: cv2.adaptiveThreshold(x, 255, 0, 0, 4, 0),
                 lambda: cv2.adaptiveThreshold(x, 255, 0, cv2.THRESH_TRUNC, 3, 0),
                 lambda: cv2.adaptiveThreshold(x, 255, 2, 0, 3, 0),
                 lambda: cv2.adaptiveThreshold(np.zeros((8, 8, 3), np.uint8), 255, 0, 0, 3, 0)):
        with pytest.raises(cv2.error):
            call()


def test_plain_threshold_rules():
    """cv2.threshold's 8-bit reading of thresh and maxval, as color.threshold passes them to bv_threshold: cvFloor
    (INT_MIN for NaN and values past int32) and cvRound half to even."""
    from cuauv_vision_pipeline_b200.color import _cv_floor, _cvt_si32
    x = np.arange(256, dtype=np.uint8).reshape(16, 16)
    for t in (3.7, -0.5, 0, 254.5, 255, 300, float("nan"), 1e10, -1e10):
        for mv in (0.5, 1.5, 254.5, 300, -5, 1e10):
            for base in tc.BASES:
                r, d = cv2.threshold(x, t, mv, base)
                assert r == float(_cv_floor(t)), (t, r)
                ithresh = min(max(_cv_floor(t), -1), 255)
                assert np.array_equal(d, tn.apply(x, ithresh, mv, base)), (t, mv, base)
    assert [_cvt_si32(v) for v in (0.5, 1.5, 2.5, -0.5, 1e10)] == [0, 2, 2, 0, -2 ** 31]


def test_cases_reach_what_they_are_written_for():
    names = {c.name for c in tc.all_cases()}
    shapes = set()
    flipped = otsu_tie = bounds = False
    near = set()
    for c in tc.all_cases():
        f = c.frames()
        shapes.add(f.shape)
        if c.kind == "auto":
            for im in f:
                h = tn.histogram(im)
                flipped |= tn.triangle_parts(h)[3]
                bounds |= bool(h[0] and h[255])
        elif c.group == "adapt_ties":
            k = c.args[3]
            s = tn.box_sums(f[0], k)
            if (np.abs(2 * s - (2 * 100 + 1) * k * k) <= 6).any():
                near.add(k)
    for c in tc.by_group(tc.all_cases())["auto_hist"]:
        if c.name.startswith("two_0_255_equal"):
            h = tn.histogram(c.frames()[0])
            otsu_tie = True
            assert tn.otsu(h) == 0.0                    # every bin from 0 to 254 has the same sigma; the first wins
    assert flipped and otsu_tie and bounds and {255, 1001, 2897, 2899, 2901} <= near
    assert {(1, 1, 1), (1, 1, 37), (1, 37, 1), (2, 2160, 3840)} <= shapes
    assert any(s[0] == 5 for s in shapes)
    ks = {c.args[3] for c in tc.all_cases() if c.kind == "adaptive"}
    assert {3, 5, 7, 9, 11, 51, 255, 1001, 2897, 2899, 2901} <= ks
    assert any(c.kind == "adaptive" and c.args[3] > max(c.frames().shape[1:]) for c in tc.all_cases())
    mvs = {c.args[0] for c in tc.all_cases()}
    assert set(tc.MAXVALS) <= mvs
    combos = {(c.args[1], c.args[2]) for c in tc.all_cases() if c.kind == "auto"}
    assert {(b, m) for b in tc.BASES for m in (tc.OTSU, tc.TRIANGLE)} <= combos
    assert set(tc.CS) <= {c.args[4] for c in tc.all_cases() if c.kind == "adaptive"}
    assert "ties_k1001_b0" in names
