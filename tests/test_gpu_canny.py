"""GPU: bv_canny against cv2.Canny with 0 differing bytes on every case of oracle/canny_cases.py (each batch in one call,
guard bytes around the destination, the launch list checked by the profiler), the arguments it rejects, the wrappers'
checks, stream ordering of the device-in / device-out mirror, and the device chain find_contours(canny(...))."""
import cv2
import numpy as np
import pytest
import torch

from cuauv_vision_pipeline_b200 import BVError, feature
from oracle import canny_cases as cc
from oracle import contour_tree as ct

pytestmark = pytest.mark.gpu

CASES = cc.by_group(cc.all_cases())
GUARD = 64
# the NMS kernel, the two union-find kernels of ccl.cu, the seed and write kernels: no count, scan, rank or final pass
LAUNCHES = {"canny_nms_kernel": 1, "ccl_init_kernel": 1, "ccl_merge_kernel": 1, "canny_seed_kernel": 1,
            "canny_write_kernel": 1}


def lib():
    from cuauv_vision_pipeline_b200.runtime import ffi, lib as lib_
    return ffi, lib_


def cv2_canny(frame, c):
    return cv2.Canny(frame, c.threshold1, c.threshold2, apertureSize=c.aperture, L2gradient=c.l2)


def difference(got, want):
    bad = np.argwhere(got != want)
    if not bad.size:
        return None
    i = tuple(int(v) for v in bad[0])
    return "%d differing bytes, first at %s: got %d, want %d" % (len(bad), i, got[i], want[i])


def run_case(ctx, c):
    """One C-ABI call for the whole batch into a destination with guard bytes on both sides."""
    ffi, L = lib()
    frames = c.frames()
    b, h, w = frames.shape[:3]
    ch = 3 if frames.ndim == 4 else 1
    src = ctx.upload(frames)
    with torch.cuda.stream(ctx.torch_stream):
        buf = ctx.empty((GUARD + b * h * w + GUARD,))
        buf.fill_(0xA5)
    ctx.profile(True)
    try:
        ctx.profile_dump()
        rc = L.bv_canny(ctx.handle, ffi.cast("uint8_t *", src.data_ptr()), ffi.cast("uint8_t *", buf.data_ptr() + GUARD),
                        b, h, w, ch, float(c.threshold1), float(c.threshold2), c.aperture, 1 if c.l2 else 0)
        kernels = {k: v["launches"] for k, v in ctx.profile_dump().items()}
    finally:
        ctx.profile(False)
    if rc != 0:
        return "%s: status %d: %s" % (c.name, rc, ffi.string(L.bv_last_error()).decode())
    out = ctx.download(buf)
    if (out[:GUARD] != 0xA5).any() or (out[GUARD + b * h * w:] != 0xA5).any():
        return "%s: wrote outside the destination" % c.name
    got = out[GUARD:GUARD + b * h * w].reshape(b, h, w)
    for k in range(b):
        d = difference(got[k], cv2_canny(frames[k], c))
        if d:
            return "%s frame %d: %s" % (c.name, k, d)
    if kernels != LAUNCHES:
        return "%s: ran %s" % (c.name, kernels)
    return None


@pytest.mark.parametrize("group", sorted(CASES))
def test_cases_match_cv2(ctx, group):
    failures = [f for f in (run_case(ctx, c) for c in CASES[group]) if f]
    assert not failures, "%d failing cases:\n  %s" % (len(failures), "\n  ".join(failures[:20]))


def test_context_canny_shapes(ctx):
    """[H,W], [H,W,3], [B,H,W] and [B,H,W,3] in; [H,W] or [B,H,W] out; the same bytes as the batched C call."""
    grey = cc.blurred_noise((3, 45, 67), 5)
    bgr = cc.blurred_noise((3, 45, 67, 3), 6)
    for src, lead in ((grey[0], ()), (bgr[0], ()), (grey, (3,)), (bgr, (3,))):
        out = ctx.download(ctx.canny(ctx.upload(src), 40, 120, 5, True))
        assert out.shape == lead + (45, 67) and out.dtype == np.uint8
        frames = src if lead else src[None]
        for k in range(frames.shape[0]):
            want = cv2.Canny(frames[k], 40, 120, apertureSize=5, L2gradient=True)
            assert difference(out[k] if lead else out, want) is None


def test_rejects_in_place_overlap_and_invalid_apertures(ctx):
    """cv2 raises for apertures 1, 4 and 9 (and Scharr's -1 is out of scope); src == dst and overlapping ranges are
    refused too.  Nothing is launched."""
    ffi, L = lib()
    buf = ctx.upload(cc.noise((2 * 40 * 60 * 3,), 1))
    p = lambda off: ffi.cast("uint8_t *", buf.data_ptr() + off)      # noqa: E731
    other = ctx.empty((40 * 60,))
    q = ffi.cast("uint8_t *", other.data_ptr())
    n0 = ctx.launches
    for ap in (1, 2, 4, 6, 8, 9, -1, 0):
        assert L.bv_canny(ctx.handle, p(0), q, 1, 40, 60, 1, 10.0, 30.0, ap, 0) == L.BV_ERR_INVALID, ap
        assert "aperture" in ffi.string(L.bv_last_error()).decode()
    assert L.bv_canny(ctx.handle, p(0), p(0), 1, 40, 60, 1, 10.0, 30.0, 3, 0) == L.BV_ERR_INVALID
    assert "in-place" in ffi.string(L.bv_last_error()).decode()
    for off in (1, 40 * 60 * 3 - 1, -(40 * 60) + 1):       # dst overlapping the source from inside, the end and before
        base = 40 * 60 if off < 0 else 0
        assert L.bv_canny(ctx.handle, p(base), p(base + off), 1, 40, 60, 3, 10.0, 30.0, 3, 0) == L.BV_ERR_INVALID, off
    # touching ranges are fine: the destination right after / right before the source
    assert L.bv_canny(ctx.handle, p(0), p(40 * 60 * 3), 1, 40, 60, 3, 10.0, 30.0, 3, 0) == 0
    n1 = ctx.launches
    assert L.bv_canny(ctx.handle, p(40 * 60), p(0), 1, 40, 60, 1, 10.0, 30.0, 3, 0) == 0
    for bad in ((0, 40, 60, 1), (1, 0, 60, 1), (1, 40, 0, 1), (1, 40, 60, 2), (1, 40, 60, 4)):
        b, h, w, ch = bad
        assert L.bv_canny(ctx.handle, p(0), q, b, h, w, ch, 10.0, 30.0, 3, 0) == L.BV_ERR_INVALID, bad
    assert L.bv_canny(ctx.handle, ffi.NULL, q, 1, 40, 60, 1, 10.0, 30.0, 3, 0) == L.BV_ERR_INVALID
    assert n1 - n0 == len(LAUNCHES) and ctx.launches - n1 == len(LAUNCHES)
    with pytest.raises(BVError):
        ctx.canny(ctx.upload(cc.noise((40, 60), 2)), 10, 30, aperture_size=4)


def test_wrapper_rejects_bad_sources(ctx):
    host = cc.noise((48, 96, 3), 3)
    frame = ctx.upload(host)
    bad = {"crop": frame[:, 20:60], "strided": frame[::2], "float": frame.float(), "int16": frame.to(torch.int16),
           "host": torch.from_numpy(host), "rank5": frame[None, None], "channels2": frame[..., :2].contiguous()[None]}
    n0 = ctx.launches
    for what, src in bad.items():
        with pytest.raises(BVError):
            ctx.canny(src, 50, 150)
            pytest.fail("canny accepted a %s source" % what)
    assert ctx.launches == n0
    assert ctx.download(ctx.canny(frame, 50, 150)).shape == (48, 96)
    with pytest.raises(TypeError):
        feature.canny(host.astype(np.float32), 50, 150)


def test_feature_canny_numpy_and_device_on_a_side_stream():
    """numpy in -> numpy out; a CUDA tensor produced on the caller's side stream -> a CUDA tensor the caller can consume
    on that stream with no synchronisation of its own."""
    frames = cc.underwater(2, 270, 480, 40)
    want = [cv2.Canny(f, 60, 180, apertureSize=3) for f in frames]
    got = feature.canny(frames[0], 60, 180)
    assert isinstance(got, np.ndarray) and difference(got, want[0]) is None
    side = torch.cuda.Stream()
    pinned = torch.from_numpy(frames).pin_memory()
    for rep in range(3):
        with torch.cuda.stream(side):
            # a long producer on the caller's stream: the frames are only correct after 80 passes of arithmetic
            acc = pinned.to("cuda", non_blocking=True).to(torch.int32)
            for _ in range(40):
                acc = acc + 3
            for _ in range(40):
                acc = acc - 3
            out = feature.canny(acc.to(torch.uint8), 60, 180)             # the context's stream
            assert out.is_cuda and out.dtype == torch.uint8 and tuple(out.shape) == (2, 270, 480)
            host = (out.to(torch.int32) + 0).to(torch.uint8).cpu()      # the caller's stream again
        side.synchronize()
        for k in range(2):
            assert difference(host.numpy()[k], want[k]) is None, (rep, k)


@pytest.mark.parametrize("mode", ["external", "list", "ccomp", "tree"])
def test_find_contours_of_device_edges_matches_cv2(ctx, mode):
    """find_contours(canny(device frame)) never leaves the device between the two steps and gives cv2's borders of
    cv2.findContours(cv2.Canny(...)), compared as tests/test_gpu_find_contours.py compares them."""
    frame = cc.underwater(1, 240, 320, 50)[0]
    edges = feature.canny(ctx.upload(frame), 50, 150, 3, False)
    assert edges.is_cuda
    got, hier = feature.find_contours(edges, mode, "simple")
    ref_edges = cv2.Canny(frame, 50, 150)
    assert np.array_equal(edges.cpu().numpy(), ref_edges)           # on the caller's stream, as the mirror ordered it
    cv_mode = cv2.RETR_EXTERNAL if mode == "external" else ct.MODES[mode]
    ref, ref_h = cv2.findContours(ref_edges, cv_mode, cv2.CHAIN_APPROX_SIMPLE)
    assert len(ref) > 20 and hier.shape == (1, len(ref), 4) == ref_h.shape
    key = lambda c: (int(c[0, 0, 0]), int(c[0, 0, 1]), len(c))      # noqa: E731
    assert sorted(key(c["points"]) for c in got) == sorted(key(c) for c in ref)
    by_key = {key(c): c for c in ref}
    for c in got:
        r = by_key[key(c["points"])]
        assert np.array_equal(c["points"], r)
        assert feature.contour_area(c) == cv2.contourArea(r)
