"""TEST INFRASTRUCTURE ONLY -- cv2.threshold with THRESH_OTSU / THRESH_TRIANGLE and cv2.adaptiveThreshold (OpenCV
4.13.0, 8-bit) restated in numpy, rule by rule as include/b200vision.h states them for bv_threshold_auto and
bv_adaptive_threshold.  tests/test_threshold_oracle.py holds these equal to cv2; tests/test_gpu_threshold.py holds the
device equal to cv2."""
import math
from fractions import Fraction

import numpy as np

f32 = np.float32
FLT_EPSILON = float(np.finfo(np.float32).eps)
INT_MIN = -2 ** 31


def histogram(frame):
    return np.bincount(np.asarray(frame, np.uint8).ravel(), minlength=256).astype(np.int64)


def otsu(h):
    """Rule 1: getThreshVal_Otsu, double, every operation rounded on its own (python floats are IEEE doubles)."""
    scale = 1.0 / int(h.sum())
    mu = 0.0
    for i in range(256):
        mu += i * float(h[i])
    mu *= scale
    mu1 = q1 = max_sigma = 0.0
    max_val = 0
    for i in range(256):
        p = float(h[i]) * scale
        mu1 *= q1
        q1 += p
        q2 = 1.0 - q1
        if min(q1, q2) < FLT_EPSILON or max(q1, q2) > 1.0 - FLT_EPSILON:
            continue
        mu1 = (mu1 + i * p) / q1
        mu2 = (mu - q1 * mu1) / q2
        sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2)
        if sigma > max_sigma:
            max_sigma, max_val = sigma, i
    return float(max_val)


def triangle_parts(h):
    """Rule 2's integer steps: (left, right, peak, flipped) after the flip."""
    nz = np.nonzero(h)[0]
    left = int(nz[0]) if nz.size else 0
    left -= left > 0
    right = next((i for i in range(255, 0, -1) if h[i] > 0), 0)
    right += right < 255
    peak = int(np.argmax(h))
    flipped = peak - left < right - peak
    if flipped:
        left, peak = 255 - right, 255 - peak
    return left, right, peak, flipped


def triangle(h):
    """Rule 2: getThreshVal_Triangle_8u, the distance search in float32 with no FMA."""
    left, _, peak, flipped = triangle_parts(h)
    hh = h[::-1] if flipped else h
    a, b = f32(h.max()), f32(left - peak)
    dist, thresh = f32(0), left
    for i in range(left + 1, peak + 1):
        t = f32(f32(a * f32(i)) + f32(b * f32(hh[i])))
        if t > dist:
            dist, thresh = t, i
    thresh -= 1
    return float(255 - thresh if flipped else thresh)


def cv_round(v):
    """cvRound of a double on x86-64: half to even, INT_MIN where there is no int32."""
    if not math.isfinite(v):
        return INT_MIN
    r = round(v)
    return r if INT_MIN <= r < 2 ** 31 else INT_MIN


def apply(frame, thresh, maxval, base):
    """Rule 3: cv2.threshold's 8-bit rule for a threshold already found."""
    x = np.asarray(frame, np.int64)
    t = math.floor(thresh)
    m = t if base == 2 else cv_round(maxval)
    m = min(max(m, 0), 255)
    above = x > t
    if base == 0:
        out = np.where(above, m, 0)
    elif base == 1:
        out = np.where(above, 0, m)
    elif base == 2:
        out = np.where(above, min(max(t, 0), 255), x)
    elif base == 3:
        out = np.where(above, x, 0)
    else:
        out = np.where(above, 0, x)
    return out.astype(np.uint8)


def threshold_auto(frame, maxval, base, method):
    """-> (retval, dst) of cv2.threshold(frame, 0, maxval, base | method), method 8 (OTSU) or 16 (TRIANGLE)."""
    h = histogram(frame)
    t = otsu(h) if method == 8 else triangle(h)
    return t, apply(frame, t, maxval, base)


def box_sums(frame, k):
    """The integer k x k window sums with BORDER_REPLICATE (int64)."""
    r = k // 2
    xp = np.pad(np.asarray(frame, np.int64), r, mode="edge")
    c = np.zeros((xp.shape[0] + 1, xp.shape[1] + 1), np.int64)
    c[1:, 1:] = xp.cumsum(0).cumsum(1)
    hh, ww = frame.shape
    return c[k:k + hh, k:k + ww] - c[0:hh, k:k + ww] - c[k:k + hh, 0:ww] + c[0:hh, 0:ww]


def mean_c(frame, k):
    """Rule 4's mean, as cv2.boxFilter sums 8-bit pixels: up to k^2 = 2^23 an int32 sum scaled in float32,
    cvRound((float)sum * (float)(1. / (k * k))); above (k >= 2897) a double sum scaled in double,
    cvRound(sum * (1. / (k * k)))."""
    if k * k > 1 << 23:
        m = np.rint(box_sums(frame, k).astype(np.float64) * (1.0 / (k * k)))
    else:
        m = np.rint(box_sums(frame, k).astype(np.float32) * f32(1.0 / (k * k)))
    return np.clip(m, 0, 255).astype(np.int64)


def gaussian_taps(k):
    """cv2.getGaussianKernel(k, 0, CV_32F) as OpenCV 4.x builds it (getGaussianKernelBitExact): a dyadic table for
    k <= 9; above, sigma = fma(k, 0.15, 0.35) (one rounding), the half-kernel exp(x^2 * (-0.125 / sigma^2)) at doubled
    offsets x = 1 - k, 3 - k, .., the sum of the half doubled plus the centre's 1, each tap times 1 / sum."""
    small = {1: [1.0], 3: [0.25, 0.5, 0.25], 5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
             7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
             9: [v / 256 for v in (4, 13, 30, 51, 60, 51, 30, 13, 4)]}
    if k in small:
        return np.array(small[k], np.float32)
    sigma = float(Fraction(k) * Fraction(0.15) + Fraction(0.35))
    scale2 = -0.125 / (sigma * sigma)
    half = (k - 1) // 2
    v = [math.exp(float((1 - k + 2 * i) ** 2) * scale2) for i in range(half)]
    s = 0.0
    for t in v:
        s += t
    mul = 1.0 / (s * 2 + 1.0)
    out = np.empty(k, np.float32)
    for i in range(half):
        out[i] = out[k - 1 - i] = f32(v[i] * mul)
    out[half] = f32(mul)
    return out


def gaussian_f32(frame, k):
    """Rule 5's float32 blur as the device takes it: rows then columns, each sum in tap order, float32 steps."""
    taps = gaussian_taps(k)
    r = k // 2
    x = np.pad(np.asarray(frame, np.float32), r, mode="edge")
    hh, ww = frame.shape
    rows = np.zeros((hh + 2 * r, ww), np.float32)
    for j in range(k):
        rows = rows + taps[j] * x[:, j:j + ww]
    out = np.zeros((hh, ww), np.float32)
    for j in range(k):
        out = out + taps[j] * rows[j:j + hh, :]
    return out


def gaussian_f64(frame, k):
    """Rule 5's blur with the float32 taps in double: the mean the tie rule measures against half-integers."""
    taps = gaussian_taps(k).astype(np.float64)
    r = k // 2
    x = np.pad(np.asarray(frame, np.float64), r, mode="edge")
    hh, ww = frame.shape
    rows = sum(taps[j] * x[:, j:j + ww] for j in range(k))
    return sum(taps[j] * rows[j:j + hh, :] for j in range(k))


def gaussian_c(frame, k):
    return np.clip(np.rint(gaussian_f32(frame, k)), 0, 255).astype(np.int64)


def compare(frame, mean, max_value, base, c):
    """cv2's table: idelta = ceil(c) (BINARY) / floor(c) (BINARY_INV), v = saturate_cast<uchar>(max_value)."""
    if max_value < 0:
        return np.zeros(np.shape(frame), np.uint8)
    v = min(max(cv_round(max_value), 0), 255)
    d = np.asarray(frame, np.int64) - mean
    if base == 0:
        return np.where(d > -math.ceil(c), v, 0).astype(np.uint8)
    return np.where(d <= -math.floor(c), v, 0).astype(np.uint8)


def adaptive(frame, max_value, method, base, k, c):
    mean = mean_c(frame, k) if method == 0 else gaussian_c(frame, k)
    return compare(frame, mean, max_value, base, c)


def gaussian_ties(frame, k, tol=1e-3):
    """Pixels whose double-precision mean lies within tol of a half-integer: where a float32 sum in another order may
    round the other way."""
    m = gaussian_f64(frame, k)
    return np.abs(m - np.floor(m) - 0.5) < tol
