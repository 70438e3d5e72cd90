"""GPU: bv_threshold_auto and bv_adaptive_threshold against cv2 on every case of oracle/threshold_cases.py, each batch
in one call: 0 differing bytes and identical thresholds (GAUSSIAN_C with k >= 11: differences only at proven ties, whose
count is reported), guard bytes around dst and thresh_dev, the launch list; then in-place Otsu, the rejected arguments,
the wrappers' shapes and types, ordering from a side stream, and find_contours(adaptive_threshold(...)) on the device."""
import cv2
import numpy as np
import pytest
import torch

from cuauv_vision_pipeline_b200 import BVError, color, feature
from oracle import threshold_cases as tc
from oracle import threshold_np as tn

pytestmark = pytest.mark.gpu

CASES = tc.by_group(tc.all_cases())
GUARD = 64
POISON = 0xA5
DPOISON = -12345.0


def lib():
    from cuauv_vision_pipeline_b200.runtime import ffi, lib as lib_
    return ffi, lib_


def cv2_result(frame, c):
    """cv2's (retval, dst); on an exact Otsu tie, cv2's own code path (its IPP path may pick another tied bin)."""
    if c.kind == "auto":
        maxval, base, method = c.args
        before = cv2.useOptimized()
        cv2.setUseOptimized(not c.otsu_tie)
        try:
            return cv2.threshold(frame, 0, maxval, base | method)
        finally:
            cv2.setUseOptimized(before)
    mv, method, base, k, cc = c.args
    return None, cv2.adaptiveThreshold(frame, mv, method, base, k, cc)


def expected_launches(c):
    if c.kind == "auto":
        return {"thresh_hist_kernel": 1, "thresh_search_kernel": 1, "thresh_apply_kernel": 1}
    if c.args[1] == tc.MEAN_C:
        return {"adapt_prefix_kernel": 1, "adapt_mean_cols_kernel": 1}
    return {"adapt_gauss_rows_kernel": 1, "adapt_gauss_cols_kernel": 1}


def call(ctx, frames, c, profile=True, in_place=False):
    """One C-ABI call for the whole batch into buffers with guard bytes -> (status, dst, thresholds, launches)."""
    ffi, L = lib()
    b, h, w = frames.shape
    n = frames.size
    with torch.cuda.stream(ctx.torch_stream):
        buf = torch.full((GUARD + n + GUARD,), POISON, dtype=torch.uint8, device=ctx.device)
        th = torch.full((GUARD + b + GUARD,), DPOISON, dtype=torch.float64, device=ctx.device)
    src = ctx.upload(frames)
    if in_place:
        buf[GUARD:GUARD + n].copy_(src.view(-1))
        src_ptr = ffi.cast("uint8_t *", buf.data_ptr() + GUARD)
    else:
        src_ptr = ffi.cast("uint8_t *", src.data_ptr())
    dst_ptr = ffi.cast("uint8_t *", buf.data_ptr() + GUARD)
    if profile:
        ctx.profile(True)
        ctx.profile_dump()
    try:
        if c.kind == "auto":
            maxval, base, method = c.args
            rc = L.bv_threshold_auto(ctx.handle, src_ptr, dst_ptr, b, h, w, float(maxval), base, method,
                                     ffi.cast("double *", th.data_ptr() + 8 * GUARD))
        else:
            mv, method, base, k, cc = c.args
            rc = L.bv_adaptive_threshold(ctx.handle, src_ptr, dst_ptr, b, h, w, float(mv), method, base, k, float(cc))
        kernels = {k_.split("<")[0].replace("(", ""): v["launches"] for k_, v in ctx.profile_dump().items()} \
            if profile else None
    finally:
        if profile:
            ctx.profile(False)
    host, hth = ctx.download(buf), ctx.download(th)
    assert (host[:GUARD] == POISON).all() and (host[GUARD + n:] == POISON).all(), "wrote outside dst"
    assert (hth[:GUARD] == DPOISON).all() and (hth[GUARD + b:] == DPOISON).all(), "wrote outside thresh_dev"
    return rc, host[GUARD:GUARD + n].reshape(b, h, w), hth[GUARD:GUARD + b], kernels


def run_case(ctx, c):
    """-> (failure message or None, bytes that differ at proven ties)."""
    frames = c.frames()
    rc, dst, th, kernels = call(ctx, frames, c)
    if rc != 0:
        ffi, L = lib()
        return "%s: status %d: %s" % (c.name, rc, ffi.string(L.bv_last_error()).decode()), 0
    ties = 0
    for k, f in enumerate(frames):
        ret, want = cv2_result(f, c)
        if c.kind == "auto" and th[k] != ret:
            return "%s frame %d: threshold %r, cv2 %r" % (c.name, k, th[k], ret), 0
        bad = dst[k] != want
        if bad.any():
            if c.kind == "adaptive" and c.args[1] == tc.GAUSSIAN_C and c.args[3] >= 11 and \
                    tn.gaussian_ties(f, c.args[3])[bad].all():
                ties += int(bad.sum())
            else:
                y, x = np.argwhere(bad)[0]
                return "%s frame %d: %d differing bytes, first (%d, %d): %d, cv2 %d" % (
                    c.name, k, int(bad.sum()), y, x, dst[k][y, x], want[y, x]), 0
    if kernels != expected_launches(c):
        return "%s: ran %s" % (c.name, kernels), 0
    return None, ties


@pytest.mark.parametrize("group", sorted(CASES))
def test_cases_match_cv2(ctx, group):
    results = [run_case(ctx, c) for c in CASES[group]]
    failures = [f for f, _ in results if f]
    print("%s: %d bytes differ from cv2 at proven GAUSSIAN_C ties" % (group, sum(t for _, t in results)))
    assert not failures, "%d failing cases:\n  %s" % (len(failures), "\n  ".join(failures[:20]))


def test_in_place_otsu_and_triangle(ctx):
    """dst == src: every frame's histogram is complete before a byte of it is written."""
    frames = tc.grey(3, 240, 320, 700)
    for method in (tc.OTSU, tc.TRIANGLE):
        c = tc.Case("in_place", "x", lambda: frames, "auto", (255, 0, method))
        rc, dst, th, _ = call(ctx, frames, c, profile=False, in_place=True)
        assert rc == 0
        for k in range(3):
            ret, want = cv2.threshold(frames[k], 0, 255, method)
            assert th[k] == ret and np.array_equal(dst[k], want)


def test_rejects_what_cv2_rejects_and_past_the_limits(ctx):
    ffi, L = lib()
    buf = ctx.upload(np.zeros(3 * 64 * 64, np.uint8))
    out = ctx.empty((3 * 64 * 64,))
    thb = ctx.empty((8,), torch.float64)
    src = ffi.cast("uint8_t *", buf.data_ptr())
    dst = ffi.cast("uint8_t *", out.data_ptr())
    th = ffi.cast("double *", thb.data_ptr())

    def auto(b=1, h=64, w=64, mv=255.0, typ=0, m=tc.OTSU, s=src, d=dst, t=th):
        return L.bv_threshold_auto(ctx.handle, s, d, b, h, w, mv, typ, m, t)

    def adapt(b=1, h=64, w=64, mv=255.0, m=0, typ=0, k=3, c=0.0, s=src, d=dst):
        return L.bv_adaptive_threshold(ctx.handle, s, d, b, h, w, mv, m, typ, k, c)
    n0 = ctx.launches
    bad_auto = [dict(m=0), dict(m=tc.OTSU | tc.TRIANGLE), dict(m=7), dict(typ=5), dict(typ=-1),
                dict(mv=float("nan")), dict(mv=float("inf")), dict(b=0), dict(h=0), dict(w=-3), dict(b=65536),
                dict(h=65536, w=32768), dict(s=ffi.NULL), dict(d=ffi.NULL), dict(t=ffi.NULL),
                dict(d=ffi.cast("uint8_t *", buf.data_ptr() + 1)),                  # partial overlap
                dict(t=ffi.cast("double *", buf.data_ptr() + 64)),                  # thresholds inside the source
                dict(t=ffi.cast("double *", out.data_ptr() + 4096 - 4))]            # inside the destination
    for kw in bad_auto:
        assert auto(**kw) == L.BV_ERR_INVALID, kw
    bad_adapt = [dict(k=1), dict(k=4), dict(k=0), dict(k=-3), dict(k=2903), dict(m=2), dict(m=-1), dict(typ=2),
                 dict(typ=3), dict(typ=4), dict(typ=8), dict(mv=float("nan")), dict(c=float("inf")),
                 dict(c=float("nan")), dict(c=2.0 ** 31), dict(c=-(2.0 ** 31)), dict(b=0), dict(h=-1),
                 dict(h=65536, w=32768), dict(s=ffi.NULL), dict(d=ffi.NULL), dict(d=src),
                 dict(d=ffi.cast("uint8_t *", buf.data_ptr() + 4095))]
    for kw in bad_adapt:
        assert adapt(**kw) == L.BV_ERR_INVALID, kw
    assert ctx.launches == n0
    # accepted at the edges: the largest block, on a frame smaller than it, in both methods
    assert adapt(k=2901) == 0 and adapt(k=2901, m=1, h=8, w=8) == 0 and adapt(c=2.0 ** 31 - 2) == 0
    assert auto(d=src) == 0 and auto(mv=1e300) == 0
    ctx.sync()


def test_wrapper_shapes_and_types(ctx):
    frame = tc.grey(1, 120, 160, 710)[0]
    batch = tc.grey(3, 120, 160, 711)
    for typ in (color.THRESH_BINARY | color.THRESH_OTSU, color.THRESH_TOZERO | color.THRESH_TRIANGLE):
        r, d = color.threshold(frame, 0, 255, typ)
        rr, dd = cv2.threshold(frame, 0, 255, typ)
        assert isinstance(r, float) and r == rr and isinstance(d, np.ndarray) and np.array_equal(d, dd)
        r, d = color.threshold(batch, 0, 255, typ)
        assert isinstance(r, np.ndarray) and r.dtype == np.float64 and r.shape == (3,) and d.shape == batch.shape
        for k in range(3):
            rr, dd = cv2.threshold(batch[k], 0, 255, typ)
            assert r[k] == rr and np.array_equal(d[k], dd)
        r, d = color.threshold(batch[..., None], 0, 255, typ)
        assert d.shape == batch.shape + (1,) and r.shape == (3,)
        r, d = color.threshold(ctx.upload(frame), 0, 255, typ)
        assert isinstance(r, float) and d.is_cuda and np.array_equal(d.cpu().numpy(), cv2.threshold(frame, 0, 255, typ)[1])
    dev, th = ctx.threshold_auto(ctx.upload(batch), 255, "binary", "otsu")
    assert th.is_cuda and th.dtype == torch.float64 and tuple(th.shape) == (3,) and dev.is_cuda
    # base types: cv2's floor / round rules, retval the floored threshold, BGR frames served
    bgr = np.random.default_rng(712).integers(0, 256, (50, 60, 3), dtype=np.uint8)
    for t, mv, typ in ((100.7, 254.5, 0), (-0.5, 1.5, 1), (300, 0.5, 2), (float("nan"), 255, 3), (1e10, 300, 4)):
        for x in (frame, bgr):
            r, d = color.threshold(x, t, mv, typ)
            rr, dd = cv2.threshold(x, t, mv, typ)
            assert r == rr and np.array_equal(d, dd), (t, mv, typ)
    r, d = color.threshold(batch, 99.5, 255, 0)
    assert np.array_equal(r, np.full(3, 99.0)) and np.array_equal(d, np.stack([cv2.threshold(f, 99.5, 255, 0)[1]
                                                                               for f in batch]))
    # adaptive
    for m in (color.ADAPTIVE_THRESH_MEAN_C, color.ADAPTIVE_THRESH_GAUSSIAN_C):
        got = color.adaptive_threshold(frame, 255, m, color.THRESH_BINARY_INV, 7, 2)
        assert isinstance(got, np.ndarray) and np.array_equal(got, cv2.adaptiveThreshold(frame, 255, m, 1, 7, 2))
        got = color.adaptive_threshold(batch[..., None], 255, m, color.THRESH_BINARY, 5, -1)
        assert got.shape == batch.shape + (1,)
        for k in range(3):
            assert np.array_equal(got[k, ..., 0], cv2.adaptiveThreshold(batch[k], 255, m, 0, 5, -1))
        dev = color.adaptive_threshold(ctx.upload(frame), 255, m, 0, 9, 0)
        assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), cv2.adaptiveThreshold(frame, 255, m, 0, 9, 0))
    # refused as cv2 refuses them
    for call_ in (lambda: color.threshold(bgr, 0, 255, color.THRESH_OTSU),
                  lambda: color.threshold(frame, 0, 255, color.THRESH_OTSU | color.THRESH_TRIANGLE),
                  lambda: color.threshold(frame, 0, 255, 5),
                  lambda: color.adaptive_threshold(bgr, 255, 0, 0, 3, 0)):
        with pytest.raises(ValueError):
            call_()
    for call_ in (lambda: color.adaptive_threshold(frame, 255, 0, 0, 4, 0),
                  lambda: color.adaptive_threshold(frame, 255, 0, color.THRESH_TRUNC, 3, 0),
                  lambda: color.adaptive_threshold(frame, 255, 3, 0, 3, 0)):
        with pytest.raises(BVError):
            call_()
    with pytest.raises(TypeError):
        color.adaptive_threshold(frame.astype(np.float32), 255, 0, 0, 3, 0)
    for bad in (ctx.upload(frame)[:, 10:50], ctx.upload(frame).float(), ctx.upload(bgr)[None]):
        with pytest.raises(BVError):
            ctx.adaptive_threshold(bad, 255, "mean", "binary", 3, 0)


def test_adaptive_threshold_on_a_side_stream():
    """A CUDA tensor produced on the caller's side stream -> a CUDA tensor the caller can consume on that stream with no
    synchronisation of its own."""
    frames = tc.grey(2, 540, 960, 720)
    want = [cv2.adaptiveThreshold(f, 255, 0, 0, 31, 3) for f in frames]
    want_otsu = [cv2.threshold(f, 0, 255, cv2.THRESH_OTSU) for f in frames]
    side = torch.cuda.Stream()
    pinned = torch.from_numpy(frames).pin_memory()
    for rep in range(3):
        with torch.cuda.stream(side):
            acc = pinned.to("cuda", non_blocking=True).to(torch.int32)
            for _ in range(40):
                acc = acc + 3
            for _ in range(40):
                acc = acc - 3
            x = acc.to(torch.uint8)
            out = color.adaptive_threshold(x, 255, 0, 0, 31, 3)
            ret, otsu = color.threshold(x, 0, 255, cv2.THRESH_OTSU)
            host, host_otsu = (out + 0).cpu(), (otsu + 0).cpu()
        side.synchronize()
        for k in range(2):
            assert np.array_equal(host[k].numpy(), want[k]), (rep, k)
            assert ret[k] == want_otsu[k][0] and np.array_equal(host_otsu[k].numpy(), want_otsu[k][1]), (rep, k)


def test_find_contours_of_device_adaptive_threshold_matches_cv2(ctx):
    """find_contours(adaptive_threshold(device frame)) stays on the device and finds cv2's borders."""
    frame = tc.grey(1, 480, 640, 730)[0]
    mask = color.adaptive_threshold(ctx.upload(frame), 255, color.ADAPTIVE_THRESH_MEAN_C, color.THRESH_BINARY_INV, 31, 5)
    assert mask.is_cuda
    ref_mask = cv2.adaptiveThreshold(frame, 255, 0, 1, 31, 5)
    assert np.array_equal(mask.cpu().numpy(), ref_mask)
    got, _ = feature.find_contours(mask, "external", "simple")
    ref, _ = cv2.findContours(ref_mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    key = lambda c: (int(c[0, 0, 0]), int(c[0, 0, 1]), len(c))      # noqa: E731
    assert len(ref) > 20 and sorted(key(c["points"]) for c in got) == sorted(key(c) for c in ref)
    by_key = {key(c): c for c in ref}
    for c in got:
        assert np.array_equal(c["points"], by_key[key(c["points"])])
