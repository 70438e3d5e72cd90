"""TEST INFRASTRUCTURE ONLY -- seeded cases for bv_canny (csrc/canny.cu).

Every case is one batch [B, H, W] or [B, H, W, 3] with cv2.Canny's arguments.  Together they cover every (aperture,
L1/L2, grey/BGR) combination; 1x1, 1xN, Nx1 and 2x2 frames, widths around the 32-pixel bit word and the 64-pixel tile,
ZED and 4K BGR batches; batches of 5 different frames; thresholds in reverse order, equal, 0, negative, fractional,
NaN, past int32, past the L2 clamp and on x/16 ties at aperture 7; noise, blurred noise, underwater frames, a 0/255
checkerboard (the largest gradients), flat steps and ramps (ties between neighbours), edges of both diagonal signs, and
a serpentine whose edge is one candidate chain across the whole frame, strong only at its far end.
tests/test_canny_oracle.py checks oracle/canny_np.py against cv2 on them; tests/test_gpu_canny.py runs them on the
device."""
from dataclasses import dataclass
from typing import Callable

import cv2
import numpy as np

from oracle import synth

APERTURES = (3, 5, 7)


@dataclass(frozen=True)
class Case:
    name: str
    group: str
    make: Callable[[], np.ndarray]     # -> uint8 [B, H, W] or [B, H, W, 3]
    threshold1: float
    threshold2: float
    aperture: int = 3
    l2: bool = False

    def frames(self):
        f = self.make()
        assert f.dtype == np.uint8 and f.ndim in (3, 4) and (f.ndim == 3 or f.shape[3] == 3), self.name
        return np.ascontiguousarray(f)

    @property
    def combo(self):
        return self.aperture, self.l2


def noise(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


def blurred_noise(shape, seed, k=5, sigma=2.0):
    """Batch of noise frames, each blurred: gradients of every direction and size, few of them at the extremes."""
    f = noise(shape, seed)
    return np.stack([cv2.GaussianBlur(im, (k, k), sigma) for im in f])


def underwater(b, h, w, seed, grey=False):
    f = np.stack([synth.gen_underwater(h, w, seed + i) for i in range(b)])
    return np.stack([cv2.cvtColor(im, cv2.COLOR_BGR2GRAY) for im in f]) if grey else f


def checkerboard(b, h, w, cell, channels):
    yy, xx = np.mgrid[0:h, 0:w]
    m = (((yy // cell) + (xx // cell)) % 2 * 255).astype(np.uint8)
    m = np.repeat(m[None], b, 0)
    return np.repeat(m[..., None], 3, 3) if channels == 3 else m


def steps(h, w):
    """Flat plateaus: vertical and horizontal steps and a square, so neighbouring magnitudes tie along and across the
    edges, plus a horizontal and a vertical ramp (every magnitude equal)."""
    im = np.zeros((h, w), np.uint8)
    im[:, w // 3:] = 90
    im[h // 2:, :] += 60
    im[h // 5:h // 5 + 9, w // 6:w // 6 + 9] = 200
    ramp = np.arange(w, dtype=np.int64) * 3 % 256
    im[: h // 6, :] = ramp[None, :].astype(np.uint8)
    im[-(h // 6):, : w // 4] = (np.arange(h // 6)[:, None] * 5 % 256).astype(np.uint8)
    return im


def diagonals(h, w):
    """Edges along both diagonals (dx and dy of equal and of opposite sign), steps and thin lines."""
    yy, xx = np.mgrid[0:h, 0:w]
    im = np.where(xx + yy < (h + w) // 2, 40, 160).astype(np.int64)
    im += np.where(xx - yy > w // 4, 50, 0)
    im[(xx + 2 * yy) % 23 == 0] = 250
    im[(2 * xx - yy) % 31 == 0] = 5
    return np.clip(im, 0, 255).astype(np.uint8)


def serpentine(h, w, level=60, bump=40):
    """A 3-px band of `level` on black snaking over the whole frame: its border is one weak candidate chain.  One
    pixel at the far end of the band is `level + bump`; with thresholds between the step's magnitude and that pixel's,
    the only strong pixels are next to it."""
    im = np.zeros((h, w), np.uint8)
    ys = list(range(2, h - 4, 6))
    for k, y in enumerate(ys):
        im[y:y + 3, 2:w - 2] = level
        if k + 1 < len(ys):
            xs = slice(w - 5, w - 2) if k % 2 == 0 else slice(2, 5)
            im[y + 3:y + 6, xs] = level
    y_end = ys[-1] + 1
    x_end = 3 if len(ys) % 2 == 0 else w - 4     # the end the chain reaches last
    im[y_end, x_end] = level + bump
    return im


def combo_cases():
    """Every (aperture, L1/L2, grey/BGR) on blurred noise, with thresholds in the busy range of each combination."""
    out = []
    for ap in APERTURES:
        for l2 in (False, True):
            for ch in (1, 3):
                shape = (2, 97, 131) if ch == 1 else (2, 97, 131, 3)
                seed = ap * 10 + 2 * int(l2) + ch
                lo, hi = {3: (60, 180), 5: (500, 1500), 7: (3000, 9000)}[ap]
                if l2:
                    lo, hi = lo * 0.8, hi * 0.8
                out.append(Case("combo_ap%d_%s_c%d" % (ap, "l2" if l2 else "l1", ch), "combo",
                                (lambda s=shape, sd=seed: blurred_noise(s, sd)), lo, hi, ap, l2))
    return out


def size_cases():
    out = []
    sizes = [(1, 1), (1, 77), (77, 1), (2, 2), (3, 3), (19, 31), (19, 32), (19, 33), (17, 63), (17, 64), (17, 65),
             (33, 129), (5, 200)]
    for i, (h, w) in enumerate(sizes):
        ap = APERTURES[i % 3]
        l2 = bool(i % 2)
        ch = 3 if i % 4 >= 2 else 1
        shape = (2, h, w) if ch == 1 else (2, h, w, 3)
        lo, hi = {3: (30, 120), 5: (200, 900), 7: (1500, 6000)}[ap]
        out.append(Case("size_%dx%d_ap%d_%s_c%d" % (h, w, ap, "l2" if l2 else "l1", ch), "sizes",
                        (lambda s=shape, sd=100 + i: noise(s, sd)), lo, hi, ap, l2))
    out.append(Case("zed_2208x1242_bgr_ap3_l1", "large", lambda: underwater(3, 1242, 2208, 700), 50, 150))
    out.append(Case("4k_bgr_ap5_l2", "large", lambda: underwater(2, 2160, 3840, 710), 400, 1200, 5, True))
    return out


def batch_cases():
    """Five frames of different content in one call: the frames must not interact."""
    def grey5():
        return np.stack([noise((61, 83), 200)[:, :], blurred_noise((1, 61, 83), 201)[0], checkerboard(1, 61, 83, 4, 1)[0],
                         steps(61, 83), diagonals(61, 83)])

    def bgr5():
        return np.stack([underwater(1, 61, 83, 210)[0], noise((61, 83, 3), 211), blurred_noise((1, 61, 83, 3), 212)[0],
                         checkerboard(1, 61, 83, 3, 3)[0], np.zeros((61, 83, 3), np.uint8)])
    return [Case("batch5_grey_ap5_l2", "batch", grey5, 300, 1000, 5, True),
            Case("batch5_bgr_ap7_l1", "batch", bgr5, 2000, 7000, 7, False),
            Case("batch5_bgr_ap3_l1", "batch", bgr5, 40, 160, 3, False)]


def threshold_cases():
    out = []
    img = lambda: blurred_noise((1, 64, 96, 3), 300)      # noqa: E731
    for ap in APERTURES:
        scale = {3: 1, 5: 8, 7: 50}[ap]
        for l2 in (False, True):
            tag = "ap%d_%s" % (ap, "l2" if l2 else "l1")
            for name, (t1, t2) in {"reversed": (150 * scale, 50 * scale), "equal": (90 * scale, 90 * scale),
                                   "zero_low": (0, 100 * scale), "both_zero": (0, 0), "negative": (-40, 70 * scale),
                                   "both_negative": (-100, -5), "fractional": (50.75 * scale, 120.5 * scale),
                                   "above_all": (1e6, 2e6), "nan_low": (float("nan"), 80 * scale),
                                   "past_int32": (1e10, 3e10)}.items():
                out.append(Case("thr_%s_%s" % (name, tag), "thresholds", img, t1, t2, ap, l2))
            if l2:
                # the L2 clamp: thresholds past 32767 (at aperture 7 past 32767 * 16 after the division)
                c = 32767 * (16 if ap == 7 else 1)
                out.append(Case("thr_l2_clamp_%s" % tag, "thresholds", lambda: checkerboard(1, 40, 56, 5, 3),
                                c + 5, 3 * c, ap, True))
                out.append(Case("thr_l2_clamp_low_only_%s" % tag, "thresholds", img, 20 * scale, c * 2.5, ap, True))
    # aperture 7: thresholds on x/16 ties, and sources whose Sobel sums fall on ties of the rounding
    for k, (t1, t2) in enumerate([(16 * 200 + 8, 16 * 600 + 8), (16 * 301 + 8, 16 * 301 + 24), (8, 16 * 450 - 8)]):
        for l2 in (False, True):
            out.append(Case("thr_ap7_ties_%d_%s" % (k, "l2" if l2 else "l1"), "thresholds",
                            (lambda sd=310 + k: blurred_noise((1, 48, 72), sd, 3, 0.8)), t1, t2, 7, l2))
    return out


def content_cases():
    out = []
    for ap in APERTURES:
        for l2 in (False, True):
            tag = "ap%d_%s" % (ap, "l2" if l2 else "l1")
            # 0/255 checkerboard: the largest magnitudes each aperture reaches (int32 limits of tg67x and L2)
            big = {3: (1000, 3000), 5: (10000, 30000), 7: (7000, 25000)}[ap]
            out.append(Case("checker_c3_%s" % tag, "content", lambda: checkerboard(1, 45, 70, 1, 3), *big, ap, l2))
            out.append(Case("checker4_c1_%s" % tag, "content", lambda: checkerboard(1, 45, 70, 4, 1), *big, ap, l2))
            small = {3: (50, 150), 5: (400, 1200), 7: (3000, 9000)}[ap]
            out.append(Case("steps_%s" % tag, "content", lambda: steps(60, 90)[None], *small, ap, l2))
            out.append(Case("diagonals_%s" % tag, "content", lambda: diagonals(60, 90)[None], *small, ap, l2))
            out.append(Case("noise_c3_%s" % tag, "content", (lambda sd=400 + ap: noise((1, 40, 50, 3), sd)),
                            small[1], small[1] * 3, ap, l2))
            out.append(Case("underwater_%s" % tag, "content", (lambda sd=420 + ap: underwater(2, 90, 160, sd)),
                            *small, ap, l2))
            out.append(Case("underwater_grey_%s" % tag, "content",
                            (lambda sd=430 + ap: underwater(2, 90, 160, sd, grey=True)), *small, ap, l2))
    return out


def serpentine_cases():
    """At aperture 3 (L1) the band's border has magnitude 240, 360 at its corners; the bump pixel's edge reaches 440,
    so with thresholds 100 and 430 the only strong pixels are the two beside the bump and the rest of the border is
    kept through hysteresis alone."""
    return [Case("serpentine_256x320", "serpentine", lambda: serpentine(256, 320)[None], 100, 430),
            Case("serpentine_4k", "serpentine", lambda: serpentine(2160, 3840)[None], 100, 430)]


def all_cases():
    return combo_cases() + size_cases() + batch_cases() + threshold_cases() + content_cases() + serpentine_cases()


def by_group(cases):
    out = {}
    for c in cases:
        out.setdefault(c.group, []).append(c)
    return out
