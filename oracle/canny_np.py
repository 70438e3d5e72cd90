"""TEST INFRASTRUCTURE ONLY -- cv2.Canny (OpenCV 4.13.0) restated in integers, without cv2.Sobel.

The rules, as csrc/canny.cu implements them (DESIGN.md section 2):

1. Gradients: Sobel dx and dy of every channel with BORDER_REPLICATE.  The kernel is separable: the smoothing row is the
   binomial of the aperture, the derivative row [-1 0 1], [-1 -2 0 2 1] or [-1 -4 -5 0 5 4 1].  Aperture 7: cv2 asks for
   scale 1/16, and the sum is rounded half to even after the division; both thresholds are divided by 16 first.
2. Magnitude: |dx| + |dy| (L1) or dx^2 + dy^2 (L2), int32.  On 3 channels each pixel takes the channel with the largest
   magnitude (the first one on a tie) and that channel's dx, dy.
3. Thresholds: L2 clamps each to 32767 (std::min, so NaN becomes 32767) and squares it when positive; low > high swaps
   them; both are floored as cvFloor does on x86-64 (INT_MIN for NaN and anything outside int32).
4. Non-maximum suppression along the gradient direction, quantised with TG22 in 15-bit fixed point (magnitude outside the
   image is 0): horizontal keeps m > left and m >= right, vertical m > up and m >= down, diagonal m > both neighbours
   on the diagonal the signs of dx, dy select.  A kept pixel with m > low is a candidate; a candidate with m > high is
   strong.
5. Hysteresis: 255 on every candidate whose 8-connected component of candidates holds a strong pixel.
"""
import math

import numpy as np
from scipy import ndimage

TG22 = int(0.4142135623730950488016887242097 * (1 << 15) + 0.5)     # 13573

SMOOTH = {3: [1, 2, 1], 5: [1, 4, 6, 4, 1], 7: [1, 6, 15, 20, 15, 6, 1]}
DERIV = {3: [-1, 0, 1], 5: [-1, -2, 0, 2, 1], 7: [-1, -4, -5, 0, 5, 4, 1]}
INT_MIN = -(1 << 31)


def cv_floor(v):
    """cvFloor on x86-64: floor, or INT_MIN when the value is NaN or does not fit in int32."""
    if math.isnan(v):
        return INT_MIN
    f = math.floor(v)
    return f if -(1 << 31) <= f < (1 << 31) else INT_MIN


def thresholds(threshold1, threshold2, aperture_size, l2_gradient):
    """Rule 3 (with the aperture-7 division of rule 1): the integer (low, high) the comparisons use."""
    lo, hi = float(threshold1), float(threshold2)
    if lo > hi:
        lo, hi = hi, lo
    if aperture_size == 7:
        lo, hi = lo / 16.0, hi / 16.0
    if l2_gradient:
        lo = lo if lo < 32767.0 else 32767.0          # std::min(32767.0, t)
        hi = hi if hi < 32767.0 else 32767.0
        if lo > 0:
            lo *= lo
        if hi > 0:
            hi *= hi
    return cv_floor(lo), cv_floor(hi)


def round_half_even_div16(s):
    """s / 16 rounded half to even, in integers (s int64 array)."""
    q, r = s >> 4, s & 15
    return q + ((r > 8) | ((r == 8) & ((q & 1) == 1)))


def sobel(plane, aperture_size):
    """(dx, dy) of one uint8 plane as int64, BORDER_REPLICATE, cv2's CV_16S result (aperture 7: scale 1/16)."""
    r = aperture_size // 2
    p = np.pad(plane.astype(np.int64), r, mode="edge")
    h, w = plane.shape
    sm, de = SMOOTH[aperture_size], DERIV[aperture_size]

    def rows(k):      # filter along x with kernel k: [H + 2r, W]
        return sum(c * p[:, i:i + w] for i, c in enumerate(k) if c)

    def cols(q, k):   # filter along y
        return sum(c * q[j:j + h, :] for j, c in enumerate(k) if c)
    dx = cols(rows(de), sm)
    dy = cols(rows(sm), de)
    if aperture_size == 7:
        dx, dy = round_half_even_div16(dx), round_half_even_div16(dy)
    return dx, dy


def gradients(src, aperture_size, l2_gradient):
    """Rule 1 and 2: (dx, dy, magnitude) of the selected channel, int64 [H, W]."""
    planes = [src] if src.ndim == 2 else [src[..., c] for c in range(src.shape[2])]
    best = None
    for pl in planes:
        dx, dy = sobel(pl, aperture_size)
        m = dx * dx + dy * dy if l2_gradient else np.abs(dx) + np.abs(dy)
        if best is None:
            best = [dx, dy, m]
        else:
            take = m > best[2]                    # first channel wins a tie
            for k, v in enumerate((dx, dy, m)):
                best[k] = np.where(take, v, best[k])
    return best


def candidates(src, threshold1, threshold2, aperture_size=3, l2_gradient=False):
    """Rules 1-4: (candidate, strong) boolean images of one frame."""
    if aperture_size not in (3, 5, 7):
        raise ValueError("aperture_size must be 3, 5 or 7")
    low, high = thresholds(threshold1, threshold2, aperture_size, l2_gradient)
    dx, dy, m = gradients(src, aperture_size, l2_gradient)
    h, w = m.shape
    P = np.zeros((h + 2, w + 2), np.int64)
    P[1:-1, 1:-1] = m

    def nb(oy, ox):
        return P[1 + oy:h + 1 + oy, 1 + ox:w + 1 + ox]
    ax, ay = np.abs(dx), np.abs(dy)
    tg22x = ax * TG22
    tg67x = tg22x + (ax << 16)
    y15 = ay << 15
    horiz = y15 < tg22x
    vert = ~horiz & (y15 > tg67x)
    diag = ~(horiz | vert)
    neg = (dx ^ dy) < 0
    keep = horiz & (m > nb(0, -1)) & (m >= nb(0, 1))
    keep |= vert & (m > nb(-1, 0)) & (m >= nb(1, 0))
    keep |= diag & neg & (m > nb(-1, 1)) & (m > nb(1, -1))
    keep |= diag & ~neg & (m > nb(-1, -1)) & (m > nb(1, 1))
    cand = keep & (m > low)
    return cand, cand & (m > high)


def canny(src, threshold1, threshold2, aperture_size=3, l2_gradient=False):
    """cv2.Canny(src, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of one uint8 frame
    [H, W] or [H, W, 3]: uint8 0/255 [H, W]."""
    cand, strong = candidates(src, threshold1, threshold2, aperture_size, l2_gradient)
    lab, n = ndimage.label(cand, structure=np.ones((3, 3), bool))
    keep = np.zeros(n + 1, bool)
    keep[np.unique(lab[strong])] = True
    keep[0] = False
    return np.where(keep[lab], 255, 0).astype(np.uint8)
