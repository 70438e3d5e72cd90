"""TEST INFRASTRUCTURE ONLY -- numpy restatements of OpenCV's published 8-bit algorithms.

OpenCV itself is not under /root/reference (third-party dependency, `pkg-config opencv4`,
configure.py:27-33; behaviour pinned to the installed cv2 4.13.0).  These functions restate the
algorithms of modules/imgproc/src/color_hsv.simd.hpp, color_lab.cpp, color_yuv.simd.hpp,
color_rgb.simd.hpp and resize.cpp as arithmetic on integers / float32, which is exactly what the
CUDA kernels implement.  tests/test_oracle_spec.py checks every one against cv2 (all 2^24 colours
for the conversions), so they are pinned by the reference's own call sites:
utils/color.py:26-32, modules/bins.py:13, modules/preprocessor.py:56-86,136-143.
"""
import numpy as np

# ---------------------------------------------------------------------------------------------
# BGR -> HSV (8-bit, H in [0,180))
# ---------------------------------------------------------------------------------------------
HSV_SHIFT = 12


def hsv_div_tables():
    sdiv = np.zeros(256, np.int32)
    hdiv = np.zeros(256, np.int32)
    i = np.arange(1, 256, dtype=np.float64)
    sdiv[1:] = np.rint((255 << HSV_SHIFT) / i).astype(np.int32)
    hdiv[1:] = np.rint((180 << HSV_SHIFT) / (6.0 * i)).astype(np.int32)
    return sdiv, hdiv


def bgr2hsv(img):
    sdiv, hdiv = hsv_div_tables()
    b = img[..., 0].astype(np.int32)
    g = img[..., 1].astype(np.int32)
    r = img[..., 2].astype(np.int32)
    v = np.maximum(np.maximum(b, g), r)
    vmin = np.minimum(np.minimum(b, g), r)
    diff = v - vmin
    h = np.where(v == r, g - b, np.where(v == g, b - r + 2 * diff, r - g + 4 * diff))
    s = (diff * sdiv[v] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT
    h = (h * hdiv[diff] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT      # arithmetic shift
    h = np.where(h < 0, h + 180, h)
    return np.stack([h, s, v], axis=-1).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# HSV -> BGR (8-bit), float32, truncating
# ---------------------------------------------------------------------------------------------
_SECTOR = np.array([[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]], np.int64)


def _fmaf(a, b, c):
    """float32 fused multiply-add emulated through float64 (a*b is exact in float64; the sum may
    round twice, which differs from a true fmaf only on vanishingly rare ties)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def hsv2bgr(img, vector_path=True):
    """cv2 4.13.0 as measured: the bracket is a single-rounding multiply-add on both paths; the
    vector path (whole 32-px groups of each row) truncates x*255, the scalar row tail rounds to
    nearest-even.  Use hsv2bgr_rows for the per-row mix."""
    f32 = np.float32
    h = img[..., 0].astype(f32) * f32(6.0 / 180.0)
    s = img[..., 1].astype(f32) * f32(1.0 / 255.0)
    v = img[..., 2].astype(f32) * f32(1.0 / 255.0)
    fl = np.floor(h)
    sector = fl.astype(np.int64) % 6
    f = (h - fl).astype(f32)
    one = np.ones_like(s)
    t0 = v
    t1 = (v * (one - s)).astype(f32)
    t2 = (v * _fmaf(-s, f, one)).astype(f32)
    t3 = (v * _fmaf(-s, (one - f).astype(f32), one)).astype(f32)
    tab = np.stack([t0, t1, t2, t3], axis=-1)
    out = np.empty(img.shape, f32)
    for c in range(3):
        out[..., c] = np.take_along_axis(tab, _SECTOR[sector][..., c][..., None], axis=-1)[..., 0]
    grey = s == 0
    for c in range(3):
        out[..., c] = np.where(grey, v, out[..., c])
    x = out * f32(255.0)
    return np.clip(np.trunc(x) if vector_path else np.rint(x), 0, 255).astype(np.uint8)


def hsv2bgr_rows(img):
    """Per-row vector/scalar mix of cv2: columns [0, 32*floor(W/32)) truncate, the rest round."""
    w = img.shape[1]
    ve = w - (w % 32)
    out = np.empty_like(img)
    if ve:
        out[:, :ve] = hsv2bgr(img[:, :ve], True)
    if ve < w:
        out[:, ve:] = hsv2bgr(img[:, ve:], False)
    return out


# ---------------------------------------------------------------------------------------------
# BGR -> Lab (8-bit), fixed point
# ---------------------------------------------------------------------------------------------
LAB_C = np.array([[1777, 1541, 778], [871, 2929, 296], [73, 448, 3575]], np.int64)  # rows XYZ x cols RGB


def lab_tables():
    f32 = np.float32
    x = np.arange(256, dtype=f32) / f32(255.0)
    lin = np.where(x <= f32(0.04045), x / f32(12.92),
                   np.power((x + f32(0.055)) / f32(1.055), f32(2.4)).astype(f32)).astype(f32)
    gtab = np.clip(np.rint(f32(2040.0) * lin), 0, 65535).astype(np.uint16)
    y = np.arange(3072, dtype=f32) / f32(2040.0)
    fy = np.where(y < f32(0.008856), y * f32(7.787) + f32(0.13793103448275862), np.cbrt(y).astype(f32)).astype(f32)
    ctab = np.clip(np.rint(f32(32768.0) * fy), 0, 65535).astype(np.uint16)
    return gtab, ctab


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def bgr2lab(img):
    gtab, ctab = lab_tables()
    gt = gtab.astype(np.int64)
    ct = ctab.astype(np.int64)
    B = gt[img[..., 0]]
    G = gt[img[..., 1]]
    R = gt[img[..., 2]]
    fX = ct[_descale(R * LAB_C[0, 0] + G * LAB_C[0, 1] + B * LAB_C[0, 2], 12)]
    fY = ct[_descale(R * LAB_C[1, 0] + G * LAB_C[1, 1] + B * LAB_C[1, 2], 12)]
    fZ = ct[_descale(R * LAB_C[2, 0] + G * LAB_C[2, 1] + B * LAB_C[2, 2], 12)]
    L = _descale(296 * fY - 1336934, 15)
    a = _descale(500 * (fX - fY) + (128 << 15), 15)
    b = _descale(200 * (fY - fZ) + (128 << 15), 15)
    return np.clip(np.stack([L, a, b], axis=-1), 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# BGR -> GRAY / YCrCb (8-bit)
# ---------------------------------------------------------------------------------------------
def bgr2gray(img):
    b = img[..., 0].astype(np.int32)
    g = img[..., 1].astype(np.int32)
    r = img[..., 2].astype(np.int32)
    return ((b * 3735 + g * 19235 + r * 9798 + 16384) >> 15).astype(np.uint8)


def bgr2ycrcb(img):
    b = img[..., 0].astype(np.int32)
    g = img[..., 1].astype(np.int32)
    r = img[..., 2].astype(np.int32)
    y = (b * 1868 + g * 9617 + r * 4899 + 8192) >> 14
    cr = ((r - y) * 11682 + (128 << 14) + 8192) >> 14
    cb = ((b - y) * 9241 + (128 << 14) + 8192) >> 14
    return np.clip(np.stack([y, cr, cb], axis=-1), 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# BGR -> HLS (8-bit), float32, rint.  fused=True is the vector path.
# ---------------------------------------------------------------------------------------------
def bgr2hls(img, fused=True):
    f32 = np.float32
    b = img[..., 0].astype(f32) * f32(1.0 / 255.0)
    g = img[..., 1].astype(f32) * f32(1.0 / 255.0)
    r = img[..., 2].astype(f32) * f32(1.0 / 255.0)
    vmax = np.maximum(np.maximum(b, g), r)
    vmin = np.minimum(np.minimum(b, g), r)
    diff = (vmax - vmin).astype(f32)
    sm = (vmax + vmin).astype(f32)
    l = (sm * f32(0.5)).astype(f32)
    with np.errstate(divide="ignore", invalid="ignore"):
        s = np.where(l < f32(0.5), diff / sm, diff / (f32(2.0) - sm)).astype(f32)
        k = (f32(60.0) / diff).astype(f32)
        if fused:
            hg = _fmaf((b - r).astype(f32), k, np.full_like(k, 120.0))
            hb = _fmaf((r - g).astype(f32), k, np.full_like(k, 240.0))
        else:
            hg = (((b - r).astype(f32) * k).astype(f32) + f32(120.0)).astype(f32)
            hb = (((r - g).astype(f32) * k).astype(f32) + f32(240.0)).astype(f32)
        hr = ((g - b).astype(f32) * k).astype(f32)
        if fused:   # cv2's vector path wraps a negative hue with the product still unrounded: fma(g - b, k, 360)
            hr = np.where(hr < 0, _fmaf((g - b).astype(f32), k, np.full_like(k, 360.0)), hr)
        else:
            hr = np.where(hr < 0, (hr + f32(360.0)).astype(f32), hr)
        h = np.where(vmax == r, hr, np.where(vmax == g, hg, hb)).astype(f32)
    h = np.where(h < 0, (h + f32(360.0)).astype(f32), h)
    chroma = diff > np.finfo(np.float32).eps
    h = np.where(chroma, h, f32(0))
    s = np.where(chroma, s, f32(0))
    out = np.stack([np.rint(h * f32(0.5)), np.rint(l * f32(255.0)), np.rint(s * f32(255.0))], axis=-1)
    return np.clip(out, 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# cv2.resize(..., INTER_LINEAR) on 8-bit: 11-bit fixed-point coefficients
# ---------------------------------------------------------------------------------------------
def linear_coeffs(src, dst, horizontal):
    """Returns (idx0, idx1, w0, w1) as int arrays of length dst (weights are int16, sum 2048)."""
    scale = np.float64(src) / np.float64(dst)
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if horizontal:
        neg = s < 0
        f = np.where(neg, np.float32(0), f)
        s = np.where(neg, 0, s)
        big = s >= src - 1
        f = np.where(big, np.float32(0), f)
        s = np.where(big, src - 1, s)
    w1 = np.clip(np.rint(f * np.float32(2048.0)), -32768, 32767).astype(np.int64)
    w0 = np.clip(np.rint((np.float32(1.0) - f) * np.float32(2048.0)), -32768, 32767).astype(np.int64)
    i0 = np.clip(s, 0, src - 1)
    i1 = np.clip(s + 1, 0, src - 1)
    return i0, i1, w0, w1


def resize_linear(img, dst_w, dst_h):
    squeeze = img.ndim == 2
    if squeeze:
        img = img[..., None]
    sh, sw = img.shape[:2]
    x0, x1, a0, a1 = linear_coeffs(sw, dst_w, True)
    y0, y1, b0, b1 = linear_coeffs(sh, dst_h, False)
    src = img.astype(np.int64)
    hor = src[:, x0, :] * a0[None, :, None] + src[:, x1, :] * a1[None, :, None]     # [sh, dst_w, c]
    r0 = hor[y0] >> 4
    r1 = hor[y1] >> 4
    out = (((b0[:, None, None] * r0) >> 16) + ((b1[:, None, None] * r1) >> 16) + 2) >> 2
    out = np.clip(out, 0, 255).astype(np.uint8)
    return out[..., 0] if squeeze else out


# ---------------------------------------------------------------------------------------------
# cv2.GaussianBlur on uint8 (OpenCV smooth.dispatch.cpp: getGaussianKernelBitExact +
# getGaussianKernelFixedPoint_ED, hlineSmooth / vlineSmooth with ufixedpoint16), pinned against
# cv2 4.13.0 in tests/test_oracle_spec.py.  Call site: modules/preprocessor.py:110-114.
# ---------------------------------------------------------------------------------------------
_SMALL_GAUSS = {1: [1.0], 3: [0.25, 0.5, 0.25], 5: [0.0625, 0.25, 0.375, 0.25, 0.0625],
                7: [0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125],
                9: [4 / 256, 13 / 256, 30 / 256, 51 / 256, 60 / 256, 51 / 256, 30 / 256, 13 / 256, 4 / 256]}


def gaussian_kernel_f64(n, sigma=0.0):
    if sigma <= 0 and n in _SMALL_GAUSS:
        return np.array(_SMALL_GAUSS[n], np.float64)
    s = sigma if sigma > 0 else ((n - 1) * 0.5 - 1) * 0.3 + 0.8
    x = np.arange(n) - (n - 1) * 0.5
    t = np.exp((-0.5 / (s * s)) * x * x)
    return t / t.sum()


def gaussian_kernel_fixed(n, sigma=0.0):
    """8.8 fixed-point taps: error diffusion from the outside in, the centre takes the rest of 256."""
    k = gaussian_kernel_f64(n, sigma) * 256.0
    out = np.zeros(n, np.int64)
    err, h = 0.0, n // 2
    for i in range(h):
        adj = k[i] + err
        v = int(np.rint(adj))
        err = adj - v
        out[i] = out[n - 1 - i] = v
    out[h] = 256 - 2 * out[:h].sum()
    return out


def gaussian_blur_8u(img, ksize, sigma_x=0.0, sigma_y=0.0):
    kw, kh = ksize
    fx, fy = gaussian_kernel_fixed(kw, sigma_x), gaussian_kernel_fixed(kh, sigma_y if sigma_y > 0 else sigma_x)
    rx, ry = kw // 2, kh // 2
    h, w = img.shape[:2]
    iy = np.arange(-ry, h + ry)
    ix = np.arange(-rx, w + rx)

    def reflect(p, n):
        if n == 1:
            return np.zeros_like(p)
        p = p.copy()
        while np.any((p < 0) | (p >= n)):                 # kernels larger than the image reflect more than once
            p = np.where(p < 0, -p, p)
            p = np.where(p >= n, 2 * n - 2 - p, p)
        return p
    src = img[reflect(iy, h)][:, reflect(ix, w)].astype(np.int64)
    hz = sum(fx[k] * src[:, k:k + w] for k in range(kw))
    hz = np.minimum(hz, 0xFFFF)
    v = sum(fy[k] * hz[k:k + h] for k in range(kh))
    return np.clip((v + (1 << 15)) >> 16, 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# cv2.warpAffine on uint8, INTER_LINEAR (OpenCV imgwarp.cpp: WarpAffineInvoker + remapBilinear with
# BilinearTab_i), pinned against cv2 4.13.0.  Call sites: modules/preprocessor.py:130-135, 144-149.
# ---------------------------------------------------------------------------------------------
def _bilinear_tab():
    t = np.arange(32, dtype=np.float32) * np.float32(1 / 32)
    t1 = np.stack([np.float32(1) - t, t], axis=1)                       # [32, 2]
    w = (t1[:, None, :, None] * t1[None, :, None, :]).astype(np.float32)  # [fy, fx, k1, k2]
    tab = np.rint(w * np.float32(32768)).astype(np.int64).reshape(32 * 32, 4)
    assert (tab.sum(axis=1) == 32768).all()                              # so OpenCV's fix-up never triggers
    return tab


INT_MIN = -2 ** 31


def cv_round(v):
    """cvRound / saturate_cast<int> of a float32 or float64 value as OpenCV computes it on x86-64 (cvtss2si, cvtsd2si):
    round half to even; NaN, +-inf and every value whose rounded result lies outside int32 give INT_MIN, on either side
    ("integer indefinite").  So a huge positive coordinate lands on the left / top edge, not the right / bottom one."""
    v = np.asarray(v)
    with np.errstate(invalid="ignore"):
        r = np.rint(v).astype(np.float64)              # exact: rint of a float32 is a float32 integer
        ok = (r >= -2.0 ** 31) & (r <= 2.0 ** 31 - 1)
    return np.where(ok, np.where(ok, r, 0).astype(np.int64), np.int64(INT_MIN))


def wrap_int32(v):
    """int32 arithmetic of C on two's complement: the int64 value reduced mod 2^32."""
    return ((np.asarray(v, np.int64) + 2 ** 31) & 0xFFFFFFFF) - 2 ** 31


def rotation_matrix_2d(center, angle, scale):
    a = angle * (np.pi / 180)          # cv2: angle *= CV_PI/180
    alpha, beta = np.cos(a) * scale, np.sin(a) * scale
    return np.array([[alpha, beta, (1 - alpha) * center[0] - beta * center[1]],
                     [-beta, alpha, beta * center[0] + (1 - alpha) * center[1]]], np.float64)


def warp_affine_8u(img, matrix, dsize=None, border="constant", border_value=0):
    squeeze = img.ndim == 2
    if squeeze:
        img = img[..., None]
    h, w = img.shape[:2]
    dw, dh = (w, h) if dsize is None else dsize
    m = np.asarray(matrix, np.float64).reshape(6).copy()
    with np.errstate(invalid="ignore", divide="ignore"):      # NaN / inf entries propagate as in cv2
        d = m[0] * m[4] - m[1] * m[3]
        d = 1.0 / d if d != 0 else 0.0
        a11, a22 = m[4] * d, m[0] * d
        m[0], m[1], m[3], m[4] = a11, m[1] * -d, m[3] * -d, a22
        b1 = -m[0] * m[2] - m[1] * m[5]
        b2 = -m[3] * m[2] - m[4] * m[5]
    m[2], m[5] = b1, b2
    tab = _bilinear_tab()

    rnd = cv_round                                     # saturate_cast<int>(double)
    xs = np.arange(dw, dtype=np.float64)
    with np.errstate(invalid="ignore"):                # NaN / inf matrix entries
        adelta, bdelta = rnd(m[0] * xs * 1024.0), rnd(m[3] * xs * 1024.0)
    out = np.zeros((dh, dw, img.shape[2]), np.uint8)
    src = img.astype(np.int64)
    bval = np.broadcast_to(np.asarray(border_value, np.int64), (img.shape[2],))
    for y in range(dh):
        with np.errstate(invalid="ignore"):
            x0 = int(rnd(np.float64((m[1] * y + m[2]) * 1024.0))) + 16
            y0 = int(rnd(np.float64((m[4] * y + m[5]) * 1024.0))) + 16
        X, Y = wrap_int32(x0 + adelta) >> 5, wrap_int32(y0 + bdelta) >> 5      # int additions wrap
        sx, sy = np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767)
        wt = tab[(Y & 31) * 32 + (X & 31)]                               # [dw, 4]
        acc = np.zeros((dw, img.shape[2]), np.int64)
        for q, (oy, ox) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
            yy, xx = sy + oy, sx + ox
            px = src[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)]
            if border == "constant":
                outside = (yy < 0) | (yy >= h) | (xx < 0) | (xx >= w)
                px = np.where(outside[:, None], bval[None, :], px)
            acc += px * wt[:, q:q + 1]
        out[y] = np.clip((acc + (1 << 14)) >> 15, 0, 255)
    return out[..., 0] if squeeze else out


# ---------------------------------------------------------------------------------------------
# cv2.remap(INTER_LINEAR) on uint8 and cv2.initUndistortRectifyMap (lens undistortion,
# include/camera_filters.hpp:6-11; SURVEY 8f rank 4).  OpenCV modules/imgproc/src/imgwarp.cpp (RemapInvoker,
# remapBilinear) and modules/calib3d (4.x: imgproc)/src/undistort.dispatch.cpp.
# ---------------------------------------------------------------------------------------------
def fixed_point_maps(mapx, mapy):
    """float32 maps -> (int16 xy [H,W,2], uint16 fractional index [H,W]) as RemapInvoker converts them per block:
    cvRound(float32(x) * 32) (INT_MIN for NaN, +-inf and |x * 32| >= 2^31, see cv_round), integer part saturated to
    short, 5-bit fractions combined into fy*32 + fx."""
    with np.errstate(invalid="ignore", over="ignore"):
        sx = cv_round(np.asarray(mapx, np.float32) * np.float32(32))
        sy = cv_round(np.asarray(mapy, np.float32) * np.float32(32))
    xy = np.stack([np.clip(sx >> 5, -32768, 32767), np.clip(sy >> 5, -32768, 32767)], axis=-1).astype(np.int16)
    return xy, ((sy & 31) * 32 + (sx & 31)).astype(np.uint16)


def remap_linear_8u(img, map1, map2, border="constant", border_value=0):
    """map1/map2: float32 x / y planes, or int16 [H,W,2] + uint16 [H,W] (CV_16SC2 + CV_16UC1)."""
    squeeze = img.ndim == 2
    if squeeze:
        img = img[..., None]
    if np.asarray(map1).dtype != np.int16:
        map1, map2 = fixed_point_maps(map1, map2)
    h, w = img.shape[:2]
    sx, sy = map1[..., 0].astype(np.int64), map1[..., 1].astype(np.int64)
    wt = _bilinear_tab()[np.asarray(map2, np.int64) & 1023]                 # [H, W, 4]
    src = img.astype(np.int64)
    bval = np.broadcast_to(np.asarray(border_value, np.int64), (img.shape[2],))
    acc = np.zeros(sx.shape + (img.shape[2],), np.int64)
    for q, (oy, ox) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        yy, xx = sy + oy, sx + ox
        px = src[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)]
        if border == "constant":
            outside = (yy < 0) | (yy >= h) | (xx < 0) | (xx >= w)
            px = np.where(outside[..., None], bval, px)
        acc += px * wt[..., q:q + 1]
    out = np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)
    return out[..., 0] if squeeze else out


def init_undistort_rectify_map(camera_matrix, dist_coeffs, new_camera_matrix, size, rotation=None, fixed=False):
    """cv2.initUndistortRectifyMap(K, D, R, newK, (w, h), CV_32FC1) in float64 (k1 k2 p1 p2 [k3 [k4 k5 k6]]; thin-prism
    and tilt terms not modelled): float32 x / y maps.  OpenCV evaluates the same expressions in double (with fused
    multiply-adds in its SIMD path), so single map values can differ in the last float32 bit."""
    w, h = size
    k = np.zeros(8)
    d = np.asarray(dist_coeffs, np.float64).ravel()
    k[:min(8, d.size)] = d[:8]
    k1, k2, p1, p2, k3, k4, k5, k6 = k
    A = np.asarray(camera_matrix, np.float64)
    fx, fy, cx, cy = A[0, 0], A[1, 1], A[0, 2], A[1, 2]
    R = np.eye(3) if rotation is None else np.asarray(rotation, np.float64)
    iR = np.linalg.inv(np.asarray(new_camera_matrix, np.float64)[:3, :3] @ R)
    u, v = np.meshgrid(np.arange(w, dtype=np.float64), np.arange(h, dtype=np.float64))
    X = iR[0, 0] * u + (iR[0, 1] * v + iR[0, 2])
    Y = iR[1, 0] * u + (iR[1, 1] * v + iR[1, 2])
    W = iR[2, 0] * u + (iR[2, 1] * v + iR[2, 2])
    x, y = X / W, Y / W
    x2, y2 = x * x, y * y
    r2, _2xy = x2 + y2, 2 * x * y
    kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2)
    xd = x * kr + p1 * _2xy + p2 * (r2 + 2 * x2)
    yd = y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy
    us, vs = fx * xd + cx, fy * yd + cy
    if fixed:   # the CV_16SC2 + CV_16UC1 pair, rounded straight from the doubles (what cv2.undistort builds):
        # saturate_cast<int>(u * 32) (see cv_round), then saturate_cast<short> of the integer part
        iu, iv = cv_round(us * 32), cv_round(vs * 32)
        xy = np.stack([np.clip(iu >> 5, -32768, 32767), np.clip(iv >> 5, -32768, 32767)], axis=-1).astype(np.int16)
        return xy, ((iv & 31) * 32 + (iu & 31)).astype(np.uint16)
    return us.astype(np.float32), vs.astype(np.float32)
