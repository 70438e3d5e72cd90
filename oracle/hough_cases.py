"""TEST INFRASTRUCTURE ONLY -- seeded cases for bv_hough_lines (csrc/hough.cu).

Every case is one batch [B, H, W] of uint8 frames with cv2.HoughLines' arguments.  Together they cover rho from 0.01
to 100, theta from 1e-4 (31 416 angles) to 4.0 (one angle), angle ranges that start below 0, end past pi or are empty;
negative, zero and high thresholds; 1x1, 1xW and Hx1 frames, widths around the 16-byte load and 3840x2160; all-zero
frames (no line) and all-255 frames (the largest votes, with use_edgeval too); symmetric patterns whose peaks tie in
votes; plateaus where neighbouring bins are equal; peaks on the first and last angle and rho bin; the angle count with
and without its pi removal; use_edgeval on grey frames; Canny maps of underwater frames; a dense map with more than
100 000 lines; rows too wide for shared memory (the global-atomic vote path); batches of 5 different frames.
tests/test_hough_oracle.py checks oracle/hough_np.py against cv2 on them; tests/test_gpu_hough.py runs them on the
device."""
import math
from dataclasses import dataclass
from typing import Callable

import cv2
import numpy as np

from oracle import canny_cases as cc

PI = math.pi


@dataclass(frozen=True)
class Case:
    name: str
    group: str
    make: Callable[[], np.ndarray]     # -> uint8 [B, H, W]
    rho: float
    theta: float
    threshold: int
    min_theta: float = 0.0
    max_theta: float = PI
    use_edgeval: bool = False

    def frames(self):
        f = self.make()
        assert f.dtype == np.uint8 and f.ndim == 3, self.name
        return np.ascontiguousarray(f)

    @property
    def args(self):
        return self.rho, self.theta, self.threshold, self.min_theta, self.max_theta, self.use_edgeval


def sparse(shape, p, seed):
    return ((np.random.default_rng(seed).random(shape) < p) * 255).astype(np.uint8)


def canny_noise(b, h, w, seed, lo=40, hi=120):
    """Canny edges of blurred noise: many short curved edges."""
    return np.stack([cv2.Canny(f, lo, hi) for f in cc.blurred_noise((b, h, w), seed)])


def canny_underwater(b, h, w, seed, lo=50, hi=150):
    return np.stack([cv2.Canny(f, lo, hi) for f in cc.underwater(b, h, w, seed)])


def lines_frame(h, w, segments, value=255):
    im = np.zeros((h, w), np.uint8)
    for (x0, y0, x1, y1) in segments:
        cv2.line(im, (x0, y0), (x1, y1), value, 1)
    return im


def param_cases():
    """Every rho, theta step, angle range and threshold shape on Canny maps and sparse masks."""
    out = []
    rhos = (0.25, 0.7, 1, 1.5, 2, 3)
    thetas = (1e-4, 0.013, PI / 360, PI / 180, PI / 90, 0.7, 4.0)
    ranges = ((0.0, PI), (0.3, 1.7), (0.0, PI / 2), (-0.5, 1.0), (0.0, 4.0), (0.2, 0.2))
    k = 0
    for rho in rhos:
        for theta in thetas:
            mn, mx = ranges[k % len(ranges)]
            h, w = (31 + 7 * k % 50, 45 + 11 * k % 70)
            make = (lambda h=h, w=w, s=k: canny_noise(1, h, w, 500 + s)) if k % 2 else \
                (lambda h=h, w=w, s=k: sparse((1, h, w), 0.04, 500 + s)[:, :, :])
            thr = (5, 0, -3, 12, 1)[k % 5] if theta > 1e-3 else 3
            out.append(Case("params_rho%g_theta%g_%g_%g_t%d" % (rho, theta, mn, mx, thr), "params", make, rho, theta,
                            thr, mn, mx))
            k += 1
    for rng_ in ranges:
        out.append(Case("range_%g_%g" % rng_, "params", lambda: canny_noise(1, 80, 120, 550), 1, PI / 180, 8, *rng_))
    for thr in (-5, 0, 1, 40, 10 ** 6):
        out.append(Case("threshold_%d" % thr, "params", lambda: canny_noise(1, 70, 90, 560), 1, PI / 180, thr))
    # the angle count: pi / 180 and 0.3 end within half a step of pi (the last angle dropped), 0.4 does not
    out.append(Case("pi_removed", "params", lambda: canny_noise(1, 60, 60, 570), 1, PI / 180, 4))
    out.append(Case("pi_removed_coarse", "params", lambda: canny_noise(1, 60, 60, 571), 1, 0.3, 2))
    out.append(Case("pi_kept", "params", lambda: canny_noise(1, 60, 60, 572), 1, 0.4, 2))
    return out


def size_cases():
    out = []
    sizes = [(1, 1), (1, 37), (37, 1), (2, 2), (5, 15), (5, 16), (5, 17), (9, 31), (9, 32), (9, 33), (7, 47), (7, 48),
             (7, 49), (3, 255), (3, 257)]
    for i, (h, w) in enumerate(sizes):
        out.append(Case("size_%dx%d" % (h, w), "sizes", (lambda h=h, w=w, s=600 + i: sparse((2, h, w), 0.3, s)),
                        (1, 0.7, 2)[i % 3], PI / 180, i % 3 - 1))
    out.append(Case("size_1x1_set", "sizes", lambda: np.full((1, 1, 1), 255, np.uint8), 1, PI / 180, 0))
    out.append(Case("4k_underwater_canny", "large", lambda: canny_underwater(1, 2160, 3840, 610), 1, PI / 180, 60))
    out.append(Case("1080p_underwater_canny", "large", lambda: canny_underwater(1, 1080, 1920, 611), 1, PI / 180, 100))
    out.append(Case("zed_underwater_canny_b2", "large", lambda: canny_underwater(2, 1242, 2208, 612), 1, PI / 180, 120))
    # a dense map: Canny of blurred noise at 1080p (685 000 edge pixels) holds 251 354 lines at rho 0.5, theta pi / 360
    out.append(Case("dense_1080p", "large", lambda: canny_noise(1, 1080, 1920, 613), 0.5, PI / 360, 20))
    return out


def content_cases():
    out = []
    out.append(Case("all_zero", "content", lambda: np.zeros((2, 40, 50), np.uint8), 1, PI / 180, -1))
    out.append(Case("all_255", "content", lambda: np.full((1, 64, 80), 255, np.uint8), 1, PI / 180, 60))
    out.append(Case("all_255_edgeval", "content", lambda: np.full((1, 64, 80), 255, np.uint8), 1, PI / 180, 10000,
                    use_edgeval=True))
    out.append(Case("all_255_edgeval_large", "content", lambda: np.full((1, 300, 500), 255, np.uint8), 2, PI / 90, 0,
                    use_edgeval=True))
    # symmetric patterns: mirrored lines and a square give peaks of equal votes, ordered by index alone
    sym = lines_frame(101, 101, [(10, 10, 90, 10), (10, 90, 90, 90), (10, 10, 10, 90), (90, 10, 90, 90),
                                 (0, 0, 100, 100), (0, 100, 100, 0)])
    out.append(Case("symmetric_ties", "content", lambda: sym[None], 1, PI / 180, 20))
    out.append(Case("symmetric_ties_fine", "content", lambda: sym[None], 0.5, PI / 720, 15))
    # plateaus: a single pixel (every angle gives it one vote at the same bin), a point on the origin, a short run
    one = np.zeros((1, 30, 40), np.uint8)
    one[0, 13, 17] = 255
    origin = np.zeros((1, 12, 12), np.uint8)
    origin[0, 0, 0] = 255
    run = lines_frame(30, 40, [(5, 20, 8, 20)])[None]
    for name, f in (("single_pixel", one), ("origin", origin), ("short_run", run)):
        out.append(Case("plateau_" + name, "content", lambda f=f: f, 1, PI / 180, 0))
        out.append(Case("plateau_%s_coarse" % name, "content", lambda f=f: f, 2.5, 0.05, -1))
    # peaks on the first and last angle: vertical lines (theta 0) and lines near theta = pi; on the first and last rho
    # bin: coarse rho on tiny frames
    vert = lines_frame(60, 80, [(20, 0, 20, 59), (60, 0, 61, 59), (0, 30, 79, 31)])[None]
    out.append(Case("first_last_angle", "content", lambda: vert, 1, PI / 180, 10))
    out.append(Case("first_last_angle_range", "content", lambda: vert, 1, 0.01, 10, -0.2, 1.6))
    for rho in (3, 7, 20, 100):
        out.append(Case("rho_edge_bins_%g" % rho, "content", (lambda s=620 + rho: sparse((2, 2, 3), 0.6, s)), rho,
                        PI / 180, -1))
    # use_edgeval on grey frames
    for k, (rho, theta, thr) in enumerate(((1, PI / 180, 2000), (1.5, 0.02, 500), (0.7, PI / 360, 800))):
        out.append(Case("edgeval_grey_%d" % k, "content", (lambda s=630 + k: cc.underwater(1, 90, 120, s, grey=True)),
                        rho, theta, thr, use_edgeval=True))
    out.append(Case("edgeval_canny", "content", lambda: canny_underwater(1, 120, 160, 640), 1, PI / 180, 30 * 255,
                    use_edgeval=True))
    return out


def fallback_cases():
    """Rows of numrho + 2 int32 bins past the opt-in shared memory (above ~58 000 bins): the global-atomic vote path."""
    return [Case("global_rho0.01_200x200", "fallback", lambda: canny_underwater(1, 200, 200, 650), 0.01, PI / 90, 2),
            Case("global_rho0.1_1080p", "fallback", lambda: canny_underwater(1, 1080, 1920, 651), 0.1, PI / 180, 8),
            Case("global_edgeval", "fallback", lambda: cc.underwater(1, 150, 200, 652, grey=True), 0.012, 0.05, 300,
                 use_edgeval=True)]


def batch_cases():
    """Five frames of different content in one call: the frames must not interact."""
    def five():
        return np.stack([canny_noise(1, 61, 83, 700)[0], sparse((61, 83), 0.05, 701), np.zeros((61, 83), np.uint8),
                         canny_underwater(1, 61, 83, 702)[0], lines_frame(61, 83, [(0, 0, 82, 60), (5, 50, 80, 3)])])
    return [Case("batch5", "batch", five, 1, PI / 180, 6),
            Case("batch5_edgeval", "batch", lambda: np.stack([cc.underwater(1, 61, 83, 710 + i, grey=True)[0]
                                                              for i in range(5)]), 2, PI / 90, 900, use_edgeval=True),
            Case("batch5_global", "batch", five, 0.004, PI / 45, 3)]


def all_cases():
    return param_cases() + size_cases() + content_cases() + fallback_cases() + batch_cases()


def by_group(cases):
    out = {}
    for c in cases:
        out.setdefault(c.group, []).append(c)
    return out
