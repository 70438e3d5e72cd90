"""GPU mirror of the reference's utils/color.py (same function names, arguments and return
shapes).  Citations are to /root/reference/utils/color.py."""
import math

import numpy as np

from ._host import ctx_for, to_device, like_input


def _convert_colorspace(code):
    """utils/color.py:11-23: returns (converted image, list of split channels)."""
    def _inner(mat):
        ctx = ctx_for(mat)
        src = to_device(ctx, mat)
        if code == "bgr2gray":
            conv = ctx.cvt_color(src, code)
            out = like_input(ctx, mat, conv)
            return out, [out]                      # cv2.split of a 1-channel image
        if code == "gray2bgr":
            conv = ctx.cvt_color(src, code)
            out = like_input(ctx, mat, conv)
            return out, [out[..., k] for k in range(3)]
        conv, planes = ctx.cvt_color(src, code, split=True)
        return like_input(ctx, mat, conv), [like_input(ctx, mat, p) for p in planes]
    return _inner


# utils/color.py:26-32.  bgr_to_luv: OpenCV's 33^3 trilinear table, node table rebuilt with the host libm
# (<= 1 LSB on 0.004 % of all colours, csrc/pixel_math.cuh).
bgr_to_lab = _convert_colorspace("bgr2lab")
bgr_to_hsv = _convert_colorspace("bgr2hsv")
bgr_to_hls = _convert_colorspace("bgr2hls")
bgr_to_ycrcb = _convert_colorspace("bgr2ycrcb")
bgr_to_gray = _convert_colorspace("bgr2gray")
gray_to_bgr = _convert_colorspace("gray2bgr")
hsv_to_bgr = _convert_colorspace("hsv2bgr")
lab_to_bgr = _convert_colorspace("lab2bgr")
bgr_to_luv = _convert_colorspace("bgr2luv")


def range_threshold(mat, min, max):  # noqa: A002 (reference argument names)
    """utils/color.py:105-121 == cv2.inRange(mat, min, max); scalars or per-channel sequences."""
    ctx = ctx_for(mat)
    return like_input(ctx, mat, ctx.in_range(to_device(ctx, mat), min, max))


def _percentile_from_order_statistics(n, q, dtype, kth):
    """np.percentile(a, q) (method 'linear') of a 1-d float array of n values, given a function returning its k-th
    smallest value: numpy 2.x's own steps (lib/_function_base_impl.py: percentile -> _quantile -> _lerp), so the
    virtual index, its dtype (that of `a` when q is a python number) and the interpolation round the same way."""
    qq = np.true_divide(q, dtype(100))
    virtual = np.asanyarray((n - 1) * qq)
    prev = np.floor(virtual)
    nxt = prev + 1
    if virtual >= n - 1:
        prev = nxt = -1
    if virtual < 0:
        prev = nxt = 0
    prev, nxt = int(prev), int(nxt)
    a, b = kth(prev), kth(nxt)
    t = np.asanyarray(virtual - prev, dtype=virtual.dtype)[()]
    diff = np.subtract(b, a)
    out = np.add(a, diff * t)
    if t >= 0.5:
        out = np.subtract(b, diff * (1 - t)).astype(type(out))
    return out


def thresh_color_distance(split, color, distance, auto_distance_percentile=None, ignore_channels=[],  # noqa: B006
                          weights=(1, 1, 1)):
    """utils/color.py:66-103.  Returns (mask, uint8 distance image).  With auto_distance_percentile the threshold
    is min(np.percentile(dists, p), distance**2): the two order statistics come from the device (radix select on
    the float32 distance image), numpy's interpolation between them is replayed on the host."""
    ctx = ctx_for(split[0])
    w = np.array([0.0 if i in ignore_channels else float(weights[i]) for i in range(3)], np.float64)
    w /= np.linalg.norm(weights)                      # norm of the UN-zeroed weights (utils/color.py:93)
    use = [0 if i in ignore_channels else 1 for i in range(3)]
    planes = [to_device(ctx, p) for p in split]
    if auto_distance_percentile:
        dists = ctx.color_distance_f32(planes, color, w, use)
        pct = _percentile_from_order_statistics(dists.numel(), auto_distance_percentile, np.float32,
                                                lambda k: ctx.select_kth(dists, k))
        limit = min(pct, distance ** 2)               # utils/color.py:99
    else:
        limit = float(distance) ** 2
    mask, dist = ctx.color_distance(planes, color, w, use, float(limit))
    return like_input(ctx, split[0], mask), like_input(ctx, split[0], dist)


def _thresh(kind, maxval=255):
    def fn(mat, threshold):
        ctx = ctx_for(mat)
        mv = maxval if maxval is not None else 0
        return like_input(ctx, mat, ctx.threshold(to_device(ctx, mat), threshold, mv, kind))
    return fn


# cv2's constants, so that callers of threshold / adaptive_threshold do not need OpenCV
THRESH_BINARY, THRESH_BINARY_INV, THRESH_TRUNC, THRESH_TOZERO, THRESH_TOZERO_INV = 0, 1, 2, 3, 4
THRESH_OTSU, THRESH_TRIANGLE = 8, 16
ADAPTIVE_THRESH_MEAN_C, ADAPTIVE_THRESH_GAUSSIAN_C = 0, 1
_INT_MIN = -2 ** 31


def _cvt_si32(v):
    """x86-64's double -> int32 conversion under cvRound: half to even, INT_MIN where the value has no int32."""
    if not math.isfinite(v):
        return _INT_MIN
    r = round(v)
    return r if _INT_MIN <= r < 2 ** 31 else _INT_MIN


def _cv_floor(v):
    """cvFloor as cv2.threshold reads its threshold: INT_MIN where the floor has no int32."""
    if not math.isfinite(v):
        return _INT_MIN
    f = math.floor(v)
    return f if _INT_MIN <= f < 2 ** 31 else _INT_MIN


def _is_batch(shape):
    return len(shape) == 4 or (len(shape) == 3 and shape[-1] != 3)


def _grey_only(mat, what):
    shape = tuple(mat.shape)
    if not (len(shape) == 2 or len(shape) == 3 and shape[-1] != 3 or len(shape) == 4 and shape[-1] == 1):
        raise ValueError("%s takes a grey frame [H,W] or a batch [B,H,W] / [B,H,W,1], not %r" % (what, shape))


def threshold(mat, thresh, maxval, type):  # noqa: A002 (cv2's argument names)
    """cv2.threshold(mat, thresh, maxval, type) on the GPU -> (retval, dst).  type is a base type (THRESH_BINARY ..
    THRESH_TOZERO_INV), optionally with THRESH_OTSU or THRESH_TRIANGLE, which compute each frame's threshold on the device
    (bv_threshold_auto, bit-exact; where two Otsu thresholds score exactly the same, the one cv2's own loop picks, which
    cv2's IPP path, taken with its default optimisations, may not) and ignore `thresh`.  mat: [H,W] or a BGR [H,W,3]
    (base types only), or a batch [B,H,W] / [B,H,W,1]; retval is a float for one frame and a float64 array of one value per frame for a batch.  Base
    types follow cv2's 8-bit rules: retval = cvFloor(thresh), maxval rounded half to even and saturated.  Numpy in gives
    numpy out; a CUDA tensor in gives a CUDA tensor out (the thresholds come back in one small download)."""
    base, auto = type & 7, type & (THRESH_OTSU | THRESH_TRIANGLE)
    if base > THRESH_TOZERO_INV or type & ~(7 | THRESH_OTSU | THRESH_TRIANGLE):
        raise ValueError("unknown threshold type %r" % type)
    if auto == THRESH_OTSU | THRESH_TRIANGLE:
        raise ValueError("THRESH_OTSU and THRESH_TRIANGLE cannot be combined")
    shape = tuple(mat.shape)
    ctx = ctx_for(mat)
    if auto:
        _grey_only(mat, "threshold with THRESH_OTSU / THRESH_TRIANGLE")
        dst, th = ctx.threshold_auto(to_device(ctx, mat), maxval, base, "otsu" if auto == THRESH_OTSU else "triangle")
        ret = ctx.download(th)
        retval = ret if _is_batch(shape) else float(ret)
    else:
        ithresh = _cv_floor(float(thresh))
        imax = _cvt_si32(float(maxval))
        # every uint8 compares the same against any threshold below 0 or from 255 up
        dst = ctx.threshold(to_device(ctx, mat), min(max(ithresh, -1), 255), min(max(imax, 0), 255),
                            ("binary", "binary_inv", "trunc", "tozero", "tozero_inv")[base])
        retval = np.full(shape[0], float(ithresh)) if _is_batch(shape) else float(ithresh)
    return retval, like_input(ctx, mat, dst)


def adaptive_threshold(mat, maxValue, adaptiveMethod, thresholdType, blockSize, C):  # noqa: N803 (cv2's names)
    """cv2.adaptiveThreshold(mat, maxValue, adaptiveMethod, thresholdType, blockSize, C) on the GPU
    (bv_adaptive_threshold): ADAPTIVE_THRESH_MEAN_C bit-exact, ADAPTIVE_THRESH_GAUSSIAN_C bit-exact for blockSize <= 9
    and above it different only where the mean lies within 1e-3 of a half-integer (cv2's own summation order varies).  mat: a grey frame [H,W] or a batch [B,H,W] / [B,H,W,1]; a BGR
    frame is refused as cv2 refuses it.  Numpy in gives numpy out; a CUDA tensor in gives a CUDA tensor out, so
    `feature.find_contours(adaptive_threshold(frame, ...))` runs on the device throughout."""
    _grey_only(mat, "adaptive_threshold")
    ctx = ctx_for(mat)
    return like_input(ctx, mat, ctx.adaptive_threshold(to_device(ctx, mat), maxValue, int(adaptiveMethod),
                                                       int(thresholdType), blockSize, C))


binary_threshold = _thresh("binary")            # utils/color.py:124-137
binary_threshold_inv = _thresh("binary_inv")    # utils/color.py:140-153
max_threshold = _thresh("trunc", 0)             # utils/color.py:156-169
above_threshold = _thresh("tozero", 0)          # utils/color.py:172-185
below_threshold = _thresh("tozero_inv", 0)      # utils/color.py:188-201


def white_balance_bgr(bgr_img):
    """utils/color.py:370-379: BGR -> LAB, shift the a and b planes so that their means sit at 128
    (float32, then numpy's uint8 cast), LAB -> BGR.

    The per-pixel update `lab_a -= a_avg - 128; astype(uint8)` depends on the pixel value only, so it
    is a 256-entry table per plane, built here with the very numpy expressions of the reference (same
    float32 subtraction, same cast, wrap-around included) and applied on the device between the two
    conversions.  Tolerance (stated): the reference takes `np.mean` of a float32 plane, a pairwise
    float32 sum whose last bits depend on the element order; the device mean is the exact integer sum
    / N rounded to float32, which can differ by ~1e-5.  Since every pixel's fractional part after
    the shift is the same, the table changes only if the mean lies within that distance of an integer:
    then single entries move by 1 LSB in a / b."""
    ctx = ctx_for(bgr_img)
    lab = ctx.cvt_color(to_device(ctx, bgr_img), "bgr2lab")
    means = ctx.channel_means(lab)                                  # exact sums / N, float64
    lut = np.empty((3, 256), np.uint8)
    lut[0] = np.arange(256, dtype=np.uint8)
    for k in (1, 2):
        plane = np.arange(256, dtype=np.float32)
        plane -= np.float32(means[k]) - 128                         # utils/color.py:375-376
        with np.errstate(invalid="ignore"):
            lut[k] = plane.astype(np.uint8)                         # utils/color.py:378
    return like_input(ctx, bgr_img, ctx.cvt_color(ctx.apply_lut(lab, lut), "lab2bgr"))


def white_balance_bgr_blur(bgr_img, kernel_size):
    """utils/color.py:381-391: as white_balance_bgr, with the a / b means taken over a kernel_size box around every
    pixel (cv2.blur, BORDER_REPLICATE).  Bit-exact: the box sums are integers, so the double-precision mean of
    cv2.blur, the float32 shift and numpy's uint8 cast are reproduced operation for operation on the device."""
    kernel_size //= 2
    kernel_size = 2 * kernel_size + 1                                   # utils/color.py:382-383
    ctx = ctx_for(bgr_img)
    lab = ctx.cvt_color(to_device(ctx, bgr_img), "bgr2lab")
    return like_input(ctx, bgr_img, ctx.cvt_color(ctx.lab_shift_local_mean(lab, kernel_size), "lab2bgr"))
