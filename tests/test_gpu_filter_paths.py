"""GPU: the blur, warp, remap, undistortion and local-mean steps of csrc/filter.cu on every path they take and at the
limits of their coordinate arithmetic (oracle/filter_cases.py), against cv2 with 0 differing bytes.

Each blur case names the kernel family it was written for (tests/test_filter_cases.py checks the prediction on the
host); here the profiler confirms that family ran.  Sources and destinations at byte offsets go through the C ABI, with
guard bytes around the destination.  Failures are collected per group and listed with the first differing byte."""
import cv2
import numpy as np
import pytest
import torch

from oracle import filter_cases as fc, spec_np

pytestmark = pytest.mark.gpu

BORDER = {"constant": cv2.BORDER_CONSTANT, "replicate": cv2.BORDER_REPLICATE}
GUARD = 64
FAMILY = {"fast": {"gaussian_blur_fast_kernel": 1}, "tile": {"gaussian_blur_kernel": 1},
          "two_launch": {"blur_rows16_kernel": 1, "blur_cols16_kernel": 1}}


BLUR = fc.by_group(fc.blur_cases())
WARP = fc.by_group(fc.warp_cases())
REMAP = fc.by_group(fc.remap_cases())


def lib():
    from cuauv_vision_pipeline_b200.runtime import ffi, lib as lib_
    return ffi, lib_


def profiled(ctx, fn):
    """fn() plus {kernel name: launches} of the call."""
    ctx.profile(True)
    try:
        ctx.profile_dump()
        out = fn()
        kernels = {k: v["launches"] for k, v in ctx.profile_dump().items()}
    finally:
        ctx.profile(False)
    return out, kernels


def difference(got, want):
    if got.shape != want.shape:
        return "shape %s, want %s" % (got.shape, want.shape)
    bad = np.argwhere(got != want)
    if not bad.size:
        return None
    i = tuple(int(v) for v in bad[0])
    return "%d differing bytes, first at %s: got %d, want %d" % (len(bad), i, got[i], want[i])


def report(failures):
    if failures:
        pytest.fail("%d failing cases:\n  %s" % (len(failures), "\n  ".join(failures[:20])))


def placed(ctx, nbytes, off, fill=None):
    """A flat device buffer whose byte `GUARD + off` is 16-byte aligned plus `off`; returns (buffer, start index)."""
    with torch.cuda.stream(ctx.torch_stream):
        buf = ctx.empty((GUARD + off + nbytes + GUARD,))
        if fill is not None:
            buf.fill_(fill)
    assert (buf.data_ptr() + GUARD) % 16 == 0
    return buf, GUARD + off


# ---------------------------------------------------------------------------------------------------------------------
# Gaussian blur
# ---------------------------------------------------------------------------------------------------------------------
def run_blur(ctx, c):
    ffi, L = lib()
    b, h, w, cn = c.shape
    img = c.image()
    src_buf, s0 = placed(ctx, img.size, c.src_off)
    dst_buf, d0 = placed(ctx, img.size, c.dst_off, fill=0xA5)
    with torch.cuda.stream(ctx.torch_stream):
        src_buf[s0:s0 + img.size].copy_(ctx.upload(img.reshape(-1)))
    ptr = lambda t, i: ffi.cast("uint8_t *", t.data_ptr() + i)     # noqa: E731
    assert (src_buf.data_ptr() + s0) % 16 == c.src_off and (dst_buf.data_ptr() + d0) % 16 == c.dst_off

    def call():
        return L.bv_gaussian_blur(ctx.handle, ptr(src_buf, s0), ptr(dst_buf, d0), b, h, w, cn, c.ksize[0], c.ksize[1],
                                  float(c.sigma[0]), float(c.sigma[1]))
    rc, kernels = profiled(ctx, call)
    if rc != 0:
        return "%s: status %d: %s" % (c.name, rc, ffi.string(L.bv_last_error()).decode())
    out = ctx.download(dst_buf)
    if (out[:d0] != 0xA5).any() or (out[d0 + img.size:] != 0xA5).any():
        return "%s: wrote outside the destination" % c.name
    got = out[d0:d0 + img.size].reshape(c.shape)
    for k in range(b):
        im = img[k, ..., 0] if cn == 1 else img[k]
        want = cv2.GaussianBlur(im, c.ksize, c.sigma[0], sigmaY=c.sigma[1]).reshape(h, w, cn)
        d = difference(got[k], want)
        if d:
            return "%s (%s) frame %d: %s" % (c.name, c.path, k, d)
    family = FAMILY[c.path.split("<")[0]]
    if kernels != family:
        return "%s: ran %s, want %s" % (c.name, kernels, family)
    return None


@pytest.mark.parametrize("group", sorted(BLUR))
def test_blur_paths(ctx, group):
    report([f for f in (run_blur(ctx, c) for c in BLUR[group]) if f])


def test_in_place_calls_are_rejected(ctx):
    """src == dst is refused by the C ABI of every step that reads neighbours, before anything is launched."""
    ffi, L = lib()
    buf = ctx.upload(fc.random_image((40, 60, 3), 1))
    p = ffi.cast("uint8_t *", buf.data_ptr())
    m = ffi.new("double[6]", [1, 0, 0.5, 0, 1, 0.5])
    mx, my = ctx.empty((40, 60), torch.float32), ctx.empty((40, 60), torch.float32)
    n0 = ctx.launches
    assert L.bv_gaussian_blur(ctx.handle, p, p, 1, 40, 60, 3, 5, 5, 0.0, 0.0) != 0
    assert "in-place" in ffi.string(L.bv_last_error()).decode()
    assert L.bv_warp_affine(ctx.handle, p, p, 1, 40, 60, 3, 40, 60, m, 0, ffi.NULL) != 0
    assert "in-place" in ffi.string(L.bv_last_error()).decode()
    assert L.bv_remap(ctx.handle, p, p, 1, 40, 60, 3, 40, 60, ffi.cast("void *", mx.data_ptr()),
                      ffi.cast("void *", my.data_ptr()), L.BV_MAP_F32, 0, ffi.NULL) != 0
    assert "in-place" in ffi.string(L.bv_last_error()).decode()
    assert ctx.launches == n0


# ---------------------------------------------------------------------------------------------------------------------
# warpAffine
# ---------------------------------------------------------------------------------------------------------------------
def run_warp(ctx, c):
    img = c.image()
    cn = c.shape[3]
    got, kernels = profiled(ctx, lambda: ctx.download(ctx.warp_affine(ctx.upload(img), c.matrix, c.dsize, c.border,
                                                                       c.border_value)))
    for k in range(c.shape[0]):
        im = img[k, ..., 0] if cn == 1 else img[k]
        want = cv2.warpAffine(im, c.matrix.astype(np.float64), c.dsize, flags=cv2.INTER_LINEAR,
                              borderMode=BORDER[c.border], borderValue=c.border_value).reshape(c.dsize[1], c.dsize[0], cn)
        d = difference(got[k], want)
        if d:
            return "%s frame %d: %s" % (c.name, k, d)
    if kernels != {"warp_coords_kernel": 1, "warp_affine_kernel": 1}:
        return "%s: ran %s" % (c.name, kernels)
    return None


@pytest.mark.parametrize("group", sorted(WARP))
def test_warp_affine_cases(ctx, group):
    report([f for f in (run_warp(ctx, c) for c in WARP[group]) if f])


# ---------------------------------------------------------------------------------------------------------------------
# remap
# ---------------------------------------------------------------------------------------------------------------------
def run_remap(ctx, c):
    img = c.image()
    cn = c.shape[3]
    with torch.cuda.stream(ctx.torch_stream):
        m1 = torch.from_numpy(np.ascontiguousarray(c.map1)).to(ctx.device)
        m2 = torch.from_numpy(np.ascontiguousarray(c.map2.view(np.int16) if c.fixed else c.map2)).to(ctx.device)
    got, kernels = profiled(ctx, lambda: ctx.download(ctx.remap(ctx.upload(img), m1, m2, c.border, c.border_value)))
    dh, dw = c.map1.shape[:2]
    for k in range(c.shape[0]):
        im = img[k, ..., 0] if cn == 1 else img[k]
        want = cv2.remap(im, c.map1, c.map2, cv2.INTER_LINEAR, borderMode=BORDER[c.border],
                         borderValue=c.border_value).reshape(dh, dw, cn)
        d = difference(got[k], want)
        if d:
            y, x = (int(v) for v in np.argwhere(got[k] != want)[0][:2])
            return "%s frame %d: %s; map (%r, %r)" % (c.name, k, d, c.map1[y, x], c.map2[y, x])
    if kernels != {"remap_kernel": 1}:
        return "%s: ran %s" % (c.name, kernels)
    return None


@pytest.mark.parametrize("group", sorted(REMAP))
def test_remap_cases(ctx, group):
    report([f for f in (run_remap(ctx, c) for c in REMAP[group]) if f])


# ---------------------------------------------------------------------------------------------------------------------
# undistortion maps: int16 saturation and INT_MIN; transform.undistort == cv2.undistort
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", fc.undistort_cases(), ids=lambda c: c.name)
def test_undistort_maps_saturate_like_cv2(ctx, case):
    from cuauv_vision_pipeline_b200 import transform
    v = case.vector_cols
    f1, f2 = transform.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size, fixed=True)
    f1, f2 = f1.cpu().numpy(), f2.cpu().numpy().view(np.uint16)
    r1, r2 = cv2.initUndistortRectifyMap(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size, cv2.CV_16SC2)
    s1, s2 = spec_np.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, case.new_k, case.size, fixed=True)
    assert difference(f1[:, :v], r1[:, :v]) is None and difference(f2[:, :v], r2[:, :v]) is None
    assert difference(f1, s1) is None and difference(f2, s2) is None     # cv2's scalar columns: the saturation rule
    img = fc.smooth_image((1, case.size[1], case.size[0], 3), 11)[0]
    want = cv2.undistort(img, fc.CAM_K, fc.CAM_D, None, case.new_k)
    got = transform.undistort(img, fc.CAM_K, fc.CAM_D, case.new_k)
    assert difference(got[:, :v], want[:, :v]) is None
    # the float32 maps (values up to 1.45e9) through the float remap path
    mx, my = transform.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, None, case.new_k, case.size)
    mx, my = mx.cpu().numpy(), my.cpu().numpy()
    sx, sy = spec_np.init_undistort_rectify_map(fc.CAM_K, fc.CAM_D, case.new_k, case.size)
    assert np.array_equal(mx, sx) and np.array_equal(my, sy)
    for border in ("constant", "replicate"):
        want = cv2.remap(img, mx, my, cv2.INTER_LINEAR, borderMode=BORDER[border])
        assert difference(transform.remap(img, mx, my, border=border), want) is None, border


# ---------------------------------------------------------------------------------------------------------------------
# the local mean shift of white_balance_bgr_blur (utils/color.py:381-391)
# ---------------------------------------------------------------------------------------------------------------------
def local_mean_reference(lab, k):
    lab_l, lab_a, lab_b = cv2.split(lab.astype(np.float32))
    lab_a -= cv2.blur(lab_a, (k, k), borderType=cv2.BORDER_REPLICATE) - 128
    lab_b -= cv2.blur(lab_b, (k, k), borderType=cv2.BORDER_REPLICATE) - 128
    with np.errstate(invalid="ignore"):
        return cv2.merge((lab_l, lab_a, lab_b)).astype(np.uint8)


@pytest.mark.parametrize("case", fc.local_mean_cases(), ids=lambda c: c.name)
def test_lab_shift_local_mean(ctx, case):
    lab = case.image()
    got, kernels = profiled(ctx, lambda: ctx.download(ctx.lab_shift_local_mean(ctx.upload(lab), case.ksize)))
    for k in range(case.shape[0]):
        assert difference(got[k], local_mean_reference(lab[k], case.ksize)) is None, k
    assert kernels == {"box_rows_ab_kernel": 1, "box_cols_shift_kernel": 1}, kernels


# ---------------------------------------------------------------------------------------------------------------------
# the wrappers check their source tensors before anything reaches the device
# ---------------------------------------------------------------------------------------------------------------------
def test_wrappers_reject_bad_sources(ctx):
    from cuauv_vision_pipeline_b200 import BVError
    host = fc.random_image((48, 96, 3), 3)
    frame = ctx.upload(host)
    maps = (ctx.empty((48, 40), torch.float32).zero_(), ctx.empty((48, 40), torch.float32).zero_())
    calls = {
        "gaussian_blur": lambda s: ctx.gaussian_blur(s, (5, 5)),
        "warp_affine": lambda s: ctx.warp_affine(s, np.array([[1.0, 0, 1], [0, 1, 1]])),
        "remap": lambda s: ctx.remap(s, *maps),
        "lab_shift_local_mean": lambda s: ctx.lab_shift_local_mean(s, 5),
        "morph": lambda s: ctx.morph(s, "erode", np.ones((3, 3))),
        "add_gaussian_noise": lambda s: ctx.add_gaussian_noise(s, 3.0, np.random.RandomState(1)),
    }
    bad = {"crop": frame[:, 20:60], "strided": frame[::2], "float": frame.float(), "int16": frame.to(torch.int16),
           "host": torch.from_numpy(host)}
    n0 = ctx.launches
    for name, fn in calls.items():
        for what, src in bad.items():
            with pytest.raises(BVError):
                fn(src)
                pytest.fail("%s accepted a %s source" % (name, what))
    for m in ((maps[0].cpu(), maps[1]), (maps[0], maps[1].cpu()), (maps[0][:, :20], maps[1][:, :20])):
        with pytest.raises(BVError):
            ctx.remap(frame, *m)
    assert ctx.launches == n0
    for name, fn in calls.items():                  # and the packed frame itself is accepted
        fn(frame)
