"""TEST INFRASTRUCTURE ONLY -- cv2.HoughLines / cv2.HoughLinesWithAccumulator (OpenCV 4.13.0, the standard transform,
srn = stn = 0) restated in numpy, float32 wherever cv2 computes in float.  tests/test_hough_oracle.py holds it equal to
cv2 bit for bit; csrc/hough.cu implements the same rules (include/b200vision.h, bv_hough_lines)."""
import math

import numpy as np


def counts(height, width, rho, theta, min_theta, max_theta):
    """(numangle, numrho) as HoughLinesStandard sizes its accumulator: theta and rho as float32, the angle count in
    double with the last angle dropped when it lands within half a step of pi, the rho count as cvRound of a float."""
    rho, theta = np.float32(rho), np.float32(theta)
    numangle = math.floor((max_theta - min_theta) / float(theta)) + 1
    if numangle > 1 and abs(math.pi - (numangle - 1) * float(theta)) < float(theta) / 2:
        numangle -= 1
    numrho = int(np.rint(np.float32(2 * (width + height) + 1) / rho))
    return numangle, numrho


def trig_table(numangle, rho, theta, min_theta):
    """tabSin, tabCos: sin / cos of the float32 angle in double, times float32(1 / rho), rounded to float32; the angle
    advances by float32 theta in float32, so its error accumulates as cv2's does."""
    irho = np.float32(1) / np.float32(rho)
    tsin = np.empty(numangle, np.float32)
    tcos = np.empty(numangle, np.float32)
    ang = np.float32(min_theta)
    for n in range(numangle):
        tsin[n] = np.float32(math.sin(float(ang)) * float(irho))
        tcos[n] = np.float32(math.cos(float(ang)) * float(irho))
        ang = np.float32(ang + np.float32(theta))
    return tsin, tcos


def accumulator(img, rho, theta, min_theta=0.0, max_theta=math.pi, use_edgeval=False):
    """int64 [numangle + 2, numrho + 2] with its zero border: every non-zero pixel adds 1 (its value with use_edgeval) at
    flat index (n + 1) * (numrho + 2) + r + 1, r = cvRound(x * tabCos[n] + y * tabSin[n]) + (numrho - 1) / 2 (two
    float32 products and a float32 sum, each rounded; cvRound half to even; integer division)."""
    h, w = img.shape
    numangle, numrho = counts(h, w, rho, theta, min_theta, max_theta)
    tsin, tcos = trig_table(numangle, rho, theta, min_theta)
    acc = np.zeros((numangle + 2) * (numrho + 2), np.int64)
    ys, xs = np.nonzero(img)
    val = img[ys, xs].astype(np.int64) if use_edgeval else np.ones(len(ys), np.int64)
    xf, yf = xs.astype(np.float32), ys.astype(np.float32)
    shift = int((numrho - 1) / 2)          # C division truncates toward zero
    step = max(1, (1 << 24) // max(1, len(xs)))
    for n0 in range(0, numangle, step):
        n = np.arange(n0, min(numangle, n0 + step))[:, None]
        r = np.rint(xf[None] * tcos[n] + yf[None] * tsin[n]).astype(np.int64) + shift
        idx = ((n + 1) * (numrho + 2) + r + 1).ravel()
        inside = (idx >= 0) & (idx < acc.size)      # cv2 would write past its buffer; such votes are dropped
        w = np.broadcast_to(val[None], r.shape).ravel()
        acc += np.bincount(idx[inside], w[inside], minlength=acc.size).astype(np.int64)
    return acc.reshape(numangle + 2, numrho + 2), numangle, numrho


def peaks(acc, threshold):
    """Flat indices and votes of the bins with acc > threshold, acc > left, acc >= right, acc > previous angle and
    acc >= next angle (the border zeros take part), ordered by votes descending, then index ascending."""
    c = acc[1:-1, 1:-1]
    m = ((c > threshold) & (c > acc[1:-1, :-2]) & (c >= acc[1:-1, 2:]) & (c > acc[:-2, 1:-1]) & (c >= acc[2:, 1:-1]))
    n_i, r_i = np.nonzero(m)
    base = (n_i + 1) * acc.shape[1] + r_i + 1
    v = c[n_i, r_i]
    order = np.lexsort((base, -v))
    return base[order], v[order]


def hough_lines(img, rho, theta, threshold, min_theta=0.0, max_theta=math.pi, use_edgeval=False, votes=False):
    """cv2.HoughLines(img, rho, theta, threshold, min_theta=, max_theta=) ([N,1,2] float32 rho, theta), or with
    votes=True cv2.HoughLinesWithAccumulator(..., use_edgeval=) ([N,1,3] with the votes); None when there is no line."""
    assert img.dtype == np.uint8 and img.ndim == 2
    acc, numangle, numrho = accumulator(img, rho, theta, min_theta, max_theta, use_edgeval)
    base, v = peaks(acc, threshold)
    if not len(base):
        return None
    n_i = base // (numrho + 2) - 1
    r_i = base - (n_i + 1) * (numrho + 2) - 1
    out_rho = (r_i - int((numrho - 1) / 2)).astype(np.float32) * np.float32(rho)
    out_ang = np.float32(min_theta) + n_i.astype(np.float32) * np.float32(theta)
    cols = [out_rho, out_ang] + ([v.astype(np.float32)] if votes else [])
    return np.stack(cols, -1).astype(np.float32).reshape(-1, 1, len(cols))
