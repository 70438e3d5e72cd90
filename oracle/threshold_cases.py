"""TEST INFRASTRUCTURE ONLY -- seeded cases for bv_threshold_auto and bv_adaptive_threshold (csrc/thresh.cu).

Every case is one batch [B, H, W] of grey frames with the arguments of one call.  Automatic thresholds: sizes from 1x1
to a 4K batch; constant, two-valued, one-sided, narrow and bimodal histograms; Triangle's flipped case and histograms
whose bounds sit at 0 and 255; Otsu ties of equal sigma (where cv2's IPP path may choose another tied bin); every base
type with OTSU and TRIANGLE; maxval 0, 0.5, 1.5, 254.5, 255, 300 and -5; batches of 5 different frames.  Adaptive
thresholds: MEAN_C and GAUSSIAN_C, BINARY and BINARY_INV, block sizes 3 to 2901 (larger than the frame too), C 0, +-2.5,
7.3 and -3; and frames of +1 pixels on a constant background whose MEAN_C window sums land within a few units of
(m + 1/2) k^2: at k = 255 and 1001, where the float32 rule and exact rounding part, and at k = 2897, 2899 and 2901, where
cv2 sums and scales in double and the float32 rule would part from it.  tests/test_threshold_oracle.py checks
oracle/threshold_np.py against cv2 on them; tests/test_gpu_threshold.py runs them on the device."""
from dataclasses import dataclass, field
from typing import Callable

import numpy as np

from oracle import canny_cases as cc

OTSU, TRIANGLE = 8, 16
MEAN_C, GAUSSIAN_C = 0, 1
BASES = (0, 1, 2, 3, 4)
MAXVALS = (0, 0.5, 1.5, 254.5, 255, 300, -5)
CS = (0, 2.5, -2.5, 7.3, -3)


@dataclass(frozen=True)
class Case:
    name: str
    group: str
    make: Callable[[], np.ndarray]     # -> uint8 [B, H, W]
    kind: str                          # "auto" or "adaptive"
    args: tuple = field(default=())    # auto: (maxval, base, method); adaptive: (max_value, method, base, k, c)
    # Otsu with two bins of equal sigma in exact arithmetic: cv2's own loop picks the one its double rounding favours,
    # cv2's IPP path (taken when optimised) may pick the other; compared with cv2's own code path
    otsu_tie: tuple = field(default=())

    def frames(self):
        f = self.make()
        assert f.dtype == np.uint8 and f.ndim == 3, self.name
        return np.ascontiguousarray(f)


def grey(b, h, w, seed):
    return cc.underwater(b, h, w, seed, grey=True)


def from_hist(h, w, values, counts, seed):
    """A frame holding each value the given number of times (the rest of the frame: values[0]), shuffled."""
    flat = np.full(h * w, values[0], np.uint8)
    pos = 0
    for v, n in zip(values, counts):
        flat[pos:pos + n] = v
        pos += n
    return np.random.default_rng(seed).permutation(flat).reshape(h, w)


def plus_one(h, w, base, p, seed):
    """Background `base` with a fraction p of pixels at base + 1: window sums near (base + 1/2) k^2 where p is 1/2."""
    return (base + (np.random.default_rng(seed).random((h, w)) < p)).astype(np.uint8)


def auto_cases():
    out = []
    k = 0
    for h, w in ((1, 1), (1, 37), (37, 1), (15, 17), (33, 47), (64, 64), (121, 250), (480, 640), (1080, 1920)):
        for m in (OTSU, TRIANGLE):
            out.append(Case("size_%dx%d_%d" % (h, w, m), "auto_sizes", lambda h=h, w=w, s=k: grey(1, h, w, 100 + s), "auto",
                            (255, BASES[k % 5], m)))
            k += 1
    hists = {
        "const0": lambda: np.zeros((20, 30), np.uint8),
        "const9": lambda: np.full((20, 30), 9, np.uint8),
        "const255": lambda: np.full((20, 30), 255, np.uint8),
        "two_0_255_equal": lambda: from_hist(16, 16, (0, 255), (128, 128), 1),          # Otsu: equal sigma, first wins
        "two_10_200": lambda: from_hist(20, 25, (10, 200), (400, 100), 2),
        "two_adjacent": lambda: from_hist(20, 25, (77, 78), (250, 250), 3),
        "one_sided_high": lambda: np.random.default_rng(4).integers(250, 256, (40, 50), dtype=np.uint8),
        "one_sided_low": lambda: np.random.default_rng(5).integers(0, 6, (40, 50), dtype=np.uint8),
        "bounds_0_255": lambda: from_hist(30, 30, (0, 255, 128, 40), (300, 200, 250, 150), 6),
        "bimodal": lambda: np.clip(np.concatenate([np.random.default_rng(7).normal(60, 10, 3000),
                                                   np.random.default_rng(8).normal(190, 25, 3000)]), 0,
                                   255).astype(np.uint8).reshape(60, 100),
        "tri_flipped": lambda: np.clip(np.random.default_rng(9).exponential(25, (80, 90)) + 20, 0, 255).astype(np.uint8),
        "tri_unflipped": lambda: np.clip(235 - np.random.default_rng(10).exponential(25, (80, 90)), 0,
                                         255).astype(np.uint8),
        "narrow": lambda: np.random.default_rng(11).integers(120, 124, (50, 70), dtype=np.uint8),
        "symmetric_three": lambda: from_hist(12, 12, (20, 120, 220), (48, 48, 48), 12),  # Otsu: two equal maxima
    }
    for name, make in hists.items():
        for m in (OTSU, TRIANGLE):
            for i, base in enumerate(BASES):
                mv = MAXVALS[(i + len(name)) % len(MAXVALS)]
                out.append(Case("%s_%d_b%d_mv%g" % (name, m, base, mv), "auto_hist", lambda mk=make: mk()[None], "auto",
                                (mv, base, m), (20.0, 120.0) if name == "symmetric_three" and m == OTSU else ()))
    for m in (OTSU, TRIANGLE):
        for mv in MAXVALS:
            out.append(Case("maxval_%g_%d" % (mv, m), "auto_maxval", lambda: grey(1, 90, 120, 20), "auto", (mv, 0, m)))
            out.append(Case("maxval_trunc_%g_%d" % (mv, m), "auto_maxval", lambda: grey(1, 90, 120, 21), "auto",
                            (mv, 2, m)))

    def five():
        fr = [grey(1, 72, 96, 30)[0], np.full((72, 96), 200, np.uint8), from_hist(72, 96, (5, 250), (3456, 3456), 31),
              np.random.default_rng(32).integers(0, 256, (72, 96), dtype=np.uint8),
              np.clip(np.random.default_rng(33).exponential(20, (72, 96)), 0, 255).astype(np.uint8)]
        return np.stack(fr)
    for m in (OTSU, TRIANGLE):
        for base in BASES:
            out.append(Case("batch5_%d_b%d" % (m, base), "auto_batch", five, "auto", (255, base, m)))
        out.append(Case("batch2_4k_%d" % m, "auto_batch", lambda: grey(2, 2160, 3840, 40), "auto", (255, 0, m)))
        out.append(Case("batch3_odd_%d" % m, "auto_batch", lambda: grey(3, 37, 53, 41), "auto", (200, 1, m)))
    return out


def adaptive_cases():
    out = []
    i = 0
    sizes = ((1, 1), (1, 40), (40, 1), (17, 33), (64, 64), (120, 160), (240, 320))
    for method in (MEAN_C, GAUSSIAN_C):
        for k in (3, 5, 7, 9, 11, 51):
            for base in (0, 1):
                for c in CS:
                    h, w = sizes[i % len(sizes)]
                    mv = (255, 100, 0.5, 300, -5, 254.5, 1.5)[i % 7]
                    out.append(Case("m%d_k%d_b%d_c%g_%dx%d" % (method, k, base, c, h, w),
                                    "adapt_mean" if method == MEAN_C else "adapt_gauss",
                                    lambda h=h, w=w, s=i: grey(1, h, w, 200 + s), "adaptive", (mv, method, base, k, c)))
                    i += 1
    for method in (MEAN_C, GAUSSIAN_C):
        for k, (h, w) in ((255, (300, 280)), (255, (100, 90)), (1001, (300, 400))):
            if method == GAUSSIAN_C and k > 255:
                continue
            for base in (0, 1):
                out.append(Case("big_m%d_k%d_b%d_%dx%d" % (method, k, base, h, w), "adapt_big",
                                lambda h=h, w=w, s=i: grey(1, h, w, 300 + s), "adaptive", (255, method, base, k, 2.5)))
                i += 1
    # +1 pixels on a constant background: MEAN_C sums within a few units of (m + 1/2) k^2
    for k, (h, w) in ((255, (400, 420)), (1001, (1100, 1150))):
        for base in (0, 1):
            out.append(Case("ties_k%d_b%d" % (k, base), "adapt_ties", lambda h=h, w=w, s=k: plus_one(h, w, 100, 0.5, s)[None],
                            "adaptive", (255, MEAN_C, base, k, 0)))
    # above k^2 = 2^23 cv2 sums and scales in double: the float32 rule of smaller windows would part from it here
    for k, seed in ((2897, 35), (2899, 18), (2901, 38)):
        for base in (0, 1):
            out.append(Case("ties_k%d_b%d" % (k, base), "adapt_ties", lambda k=k, s=seed: plus_one(300, 320, 100, 0.5, s)[None],
                            "adaptive", (255, MEAN_C, base, k, 0)))
    out.append(Case("ties_k255_c1", "adapt_ties", lambda: plus_one(400, 420, 100, 0.5, 7)[None], "adaptive",
                    (255, MEAN_C, 0, 255, 1)))

    def five():
        return np.stack([grey(1, 60, 80, 400)[0], np.full((60, 80), 30, np.uint8), plus_one(60, 80, 50, 0.5, 401),
                         np.random.default_rng(402).integers(0, 256, (60, 80), dtype=np.uint8),
                         cc.checkerboard(1, 60, 80, 7, 1)[0]])
    for method in (MEAN_C, GAUSSIAN_C):
        for k in (3, 11, 51):
            out.append(Case("batch5_m%d_k%d" % (method, k), "adapt_batch", five, "adaptive", (255, method, 0, k, 2)))
    out.append(Case("batch2_4k_mean_k51", "adapt_batch", lambda: grey(2, 2160, 3840, 410), "adaptive",
                    (255, MEAN_C, 0, 51, 5)))
    out.append(Case("batch2_4k_gauss_k11", "adapt_batch", lambda: grey(2, 2160, 3840, 411), "adaptive",
                    (255, GAUSSIAN_C, 1, 11, 3)))
    return out


def all_cases():
    return auto_cases() + adaptive_cases()


def by_group(cases):
    out = {}
    for c in cases:
        out.setdefault(c.group, []).append(c)
    return out
