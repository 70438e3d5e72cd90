"""GPU: the YOLO input transform (bv_letterbox) on every path it takes, and bv_resize_linear on batches, single pixels
and extreme ratios, against cv2.resize + cv2.copyMakeBorder (oracle/letterbox.py).

The arithmetic is OpenCV's fixed-point bilinear scheme and one float32 division per value, rounded once to fp16;
tests/test_letterbox_cases.py shows both identical to the oracle on the host.  What can go wrong on the device is data
movement -- staging, alignment, padding, image boundaries inside a block, the tap cache -- so every comparison here
demands 0 differing values (fp16 compared as uint16, fp32 as uint32), and names the kernel that ran."""
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest
import torch

from oracle import letterbox, letterbox_cases as lc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GATHER_ENV = os.environ.get("BV_LETTERBOX_GATHER") is not None
SINGLE = lc.single_cases()
BATCH = lc.batch_cases()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def device_sources(ctx, case, imgs):
    """The case's sources on the device, at the byte offsets past a 16-byte boundary it asks for."""
    with torch.cuda.stream(ctx.torch_stream):
        if case.stacked:
            batch = ctx.upload(np.stack(imgs))
            srcs = [batch[k] for k in range(len(imgs))]
        else:
            srcs = []
            for im, off in zip(imgs, case.offsets):
                flat = ctx.empty((off + im.size,))
                flat[off:].copy_(ctx.upload(im).view(-1))
                srcs.append(flat[off:].view(im.shape))
    assert [s.data_ptr() % 16 for s in srcs] == list(case.offsets)
    return srcs


def device_out(ctx, case):
    if not case.out_offset:
        return None
    n = len(case.srcs)
    numel = n * 3 * case.out_h * case.out_w
    flat = ctx.empty((numel + case.out_offset,), torch.float16 if case.half else torch.float32)
    out = flat[case.out_offset:].view(n, 3, case.out_h, case.out_w)
    assert out.data_ptr() % 16 == case.out_offset_bytes()
    return out


def letterbox_profiled(ctx, srcs, out_h, out_w, pad=114, half=True, out=None):
    """ctx.letterbox plus {kernel name: launches} of the call."""
    ctx.profile(True)
    try:
        ctx.profile_dump()
        got = ctx.letterbox(srcs, out_h, out_w, pad, half, out=out)
        kernels = {k: v["launches"] for k, v in ctx.profile_dump().items()}
    finally:
        ctx.profile(False)
    return got, kernels


def assert_same(got, want, what=""):
    """0 differing values; on a mismatch, the image, plane and (y, x) of the first one."""
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, got.dtype, want.shape, want.dtype)
    bits = np.uint16 if got.dtype == np.float16 else np.uint32
    diff = got.view(bits) != want.view(bits)
    if diff.any():
        idx = tuple(int(v) for v in np.argwhere(diff)[0])
        loc = "image %d, plane %d, (y, x) = (%d, %d)" % idx if got.ndim == 4 else "index %s" % (idx,)
        pytest.fail("%d differing values; first at %s: got %r, want %r; %s" % (int(diff.sum()), loc, got[idx],
                                                                             want[idx], what))


def check_kernels(kernels, paths):
    if "gather" in paths:
        assert kernels.get("letterbox_kernel") == 1 and "letterbox_tma_kernel" not in kernels, kernels
    else:
        assert kernels.get("letterbox_tma_kernel") == 1 and "letterbox_kernel" not in kernels, kernels


def run_case(ctx, case):
    paths = case.paths(GATHER_ENV, sm_count())
    imgs = case.images()
    srcs = device_sources(ctx, case, imgs)
    out = device_out(ctx, case)
    got, kernels = letterbox_profiled(ctx, srcs, case.out_h, case.out_w, case.pad, case.half, out=out)
    if out is not None:
        assert got.data_ptr() == out.data_ptr()
    want = letterbox.yolo_input(imgs, case.out_h, case.out_w, case.pad, case.half)
    assert_same(ctx.download(got), want, "case %s, paths %s" % (case.name, sorted(paths)))
    check_kernels(kernels, paths)


@pytest.mark.parametrize("i", range(len(SINGLE)), ids=[c.name for c in SINGLE])
def test_letterbox_single_case(ctx, i):
    run_case(ctx, SINGLE[i])


@pytest.mark.parametrize("i", range(len(BATCH)), ids=[c.name for c in BATCH])
def test_letterbox_batch_case(ctx, i):
    run_case(ctx, lc.batch_cases(sm_count())[i])


@pytest.mark.skipif(GATHER_ENV, reason="this process already runs the gather kernel")
def test_letterbox_gather_kernel_everywhere():
    """BV_LETTERBOX_GATHER is read once per process: the single-image matrix again, in a child that has it set."""
    env = dict(os.environ, BV_LETTERBOX_GATHER="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", "-q", "-m", "gpu", "-p", "no:cacheprovider", "-k", "test_letterbox_single_case",
        os.path.join("tests", os.path.basename(__file__))]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "%d passed" % len(SINGLE) in r.stdout, r.stdout[-2000:]


def test_letterbox_rejects_257_images(ctx):
    imgs = lc.too_many_images()
    srcs = [ctx.upload(im) for im in imgs]
    n0 = ctx.launches
    from cuauv_vision_pipeline_b200 import BVError
    with pytest.raises(BVError, match="256 images"):
        ctx.letterbox(srcs, 64, 64)
    assert ctx.launches == n0


# ---------------------------------------------------------------------------------------------------------------------
# the tap cache: descriptors and horizontal taps stay on the device while the same cameras come back
# ---------------------------------------------------------------------------------------------------------------------
def cached_call(ctx, srcs, imgs, out_h=640, out_w=640, pad=114, half=True):
    """One checked call; returns whether it rebuilt the tap table (a cache miss)."""
    got, kernels = letterbox_profiled(ctx, srcs, out_h, out_w, pad, half)
    assert_same(ctx.download(got), letterbox.yolo_input(imgs, out_h, out_w, pad, half),
                "%d images -> %dx%d pad %d half %s" % (len(imgs), out_h, out_w, pad, half))
    return "letterbox_coef_kernel" in kernels


def camera_set(shapes, seed):
    return [lc.random_image(h, w, seed + k) for k, (h, w) in enumerate(shapes)]


SET_SHAPES = [(1080, 1920), (479, 641), (641, 479)]


def test_cache_hit_reads_new_contents(ctx):
    imgs = camera_set(SET_SHAPES, 1000)
    srcs = [ctx.upload(im) for im in imgs]
    cached_call(ctx, srcs, imgs)
    for k in range(2):
        imgs = camera_set(SET_SHAPES, 1100 + 10 * k)
        with torch.cuda.stream(ctx.torch_stream):
            for s, im in zip(srcs, imgs):
                s.copy_(ctx.upload(im))
        assert not cached_call(ctx, srcs, imgs), "same tensors and sizes: the taps must be reused"


def test_cache_same_storage_other_shape(ctx):
    a = lc.random_image(480, 640, 1200)
    src = ctx.upload(a)
    cached_call(ctx, [src], [a])
    assert not cached_call(ctx, [src], [a])
    b = a.reshape(640, 480, 3)             # same bytes, same pointer, portrait
    assert cached_call(ctx, [src.view(640, 480, 3)], [b])
    c = a.reshape(240, 1280, 3)
    assert cached_call(ctx, [src.view(240, 1280, 3)], [c])


def test_cache_camera_sets_x_y_x(ctx):
    x_imgs, y_imgs = camera_set(SET_SHAPES, 1300), camera_set(SET_SHAPES, 1400)
    x, y = [ctx.upload(im) for im in x_imgs], [ctx.upload(im) for im in y_imgs]   # both sets stay alive
    cached_call(ctx, x, x_imgs)
    assert not cached_call(ctx, x, x_imgs)
    assert cached_call(ctx, y, y_imgs), "other source pointers: the descriptors must be re-uploaded"
    assert cached_call(ctx, x, x_imgs)
    assert not cached_call(ctx, x, x_imgs)


def test_cache_output_size_changes(ctx):
    imgs = camera_set(SET_SHAPES, 1500)
    srcs = [ctx.upload(im) for im in imgs]
    cached_call(ctx, srcs, imgs, 640, 640)
    assert cached_call(ctx, srcs, imgs, 320, 320)
    assert cached_call(ctx, srcs, imgs, 640, 640)
    assert cached_call(ctx, srcs, imgs, 640, 320)
    assert cached_call(ctx, srcs, imgs, 320, 640)


def test_cache_type_and_pad_change_between_hits(ctx):
    imgs = camera_set(SET_SHAPES, 1600)
    srcs = [ctx.upload(im) for im in imgs]
    cached_call(ctx, srcs, imgs)
    for pad, half in ((114, False), (0, True), (255, False), (300, True), (-5, False), (114, True)):
        assert not cached_call(ctx, srcs, imgs, pad=pad, half=half)


def test_cache_gather_call_between_staged_calls(ctx):
    imgs = camera_set(SET_SHAPES, 1700)
    srcs = [ctx.upload(im) for im in imgs]
    wide = camera_set([(2160, 4096)] + SET_SHAPES[1:], 1800)
    wide_srcs = [ctx.upload(im) for im in wide]
    cached_call(ctx, srcs, imgs)
    assert not cached_call(ctx, srcs, imgs)
    got, kernels = letterbox_profiled(ctx, wide_srcs, 640, 640)
    assert "letterbox_kernel" in kernels
    assert_same(ctx.download(got), letterbox.yolo_input(wide))
    cached_call(ctx, srcs, imgs)
    assert not cached_call(ctx, srcs, imgs)
    # the gather kernel over the cached set's own sources (the tap table is out of the way, not stale)
    got, kernels = letterbox_profiled(ctx, srcs, 8, 30000)
    assert "letterbox_kernel" in kernels
    assert_same(ctx.download(got), letterbox.yolo_input(imgs, 8, 30000))
    cached_call(ctx, srcs, imgs)


def test_cache_batch_grows_past_scratch(ctx):
    shapes = [(120, 160), (97, 131), (131, 97)]
    for n in (2, 40, 256, 3, 256):
        imgs = camera_set([shapes[k % 3] for k in range(n)], 1900 + n)
        srcs = [ctx.upload(im) for im in imgs]
        assert cached_call(ctx, srcs, imgs, 64, 1280)
        assert not cached_call(ctx, srcs, imgs, 64, 1280)


# ---------------------------------------------------------------------------------------------------------------------
# the wrappers check their tensors before anything reaches the device
# ---------------------------------------------------------------------------------------------------------------------
def test_letterbox_wrapper_rejects_bad_tensors(ctx):
    from cuauv_vision_pipeline_b200 import BVError
    frame = ctx.upload(lc.random_image(480, 1280, 2000))
    ok = ctx.upload(lc.random_image(480, 640, 2001))
    n0 = ctx.launches
    with pytest.raises(BVError):
        ctx.letterbox([frame[:, 100:740]])                          # a crop: rows are not packed
    with pytest.raises(BVError):
        ctx.letterbox([ok, frame[::2]])
    good = ctx.empty((1, 3, 640, 640), torch.float16)
    for bad, kw in ((ctx.empty((1, 3, 640, 639), torch.float16), {}),             # short
                    (ctx.empty((2, 3, 640, 640), torch.float16), {}),
                    (ctx.empty((1, 3, 640, 640), torch.float32), {}),             # dtype against half
                    (good, dict(half=False)),
                    (ctx.empty((1, 3, 640, 1280), torch.float16)[..., ::2], {}),  # not contiguous
                    (torch.empty((1, 3, 640, 640), dtype=torch.float16), {})):    # host memory
        with pytest.raises(BVError):
            ctx.letterbox([ok], out=bad, **kw)
    assert ctx.launches == n0
    got = ctx.letterbox([ok], out=good)
    assert got.data_ptr() == good.data_ptr()


def test_resize_wrapper_rejects_bad_tensors(ctx):
    from cuauv_vision_pipeline_b200 import BVError
    frame = ctx.upload(lc.random_image(480, 1280, 2100))
    n0 = ctx.launches
    for bad in (frame[:, 100:740], frame[::2], frame.float(), torch.from_numpy(lc.random_image(8, 8, 1))):
        with pytest.raises(BVError):
            ctx.resize(bad, 320, 240)
    assert ctx.launches == n0


# ---------------------------------------------------------------------------------------------------------------------
# bv_resize_linear
# ---------------------------------------------------------------------------------------------------------------------
RESIZE_SHAPES = [(1, 1, 1, 1), (1, 1, 5, 7), (7, 5, 1, 1), (1, 3840, 1, 1), (3840, 1, 1, 1), (1, 3840, 3, 1),
                 (3, 3, 3000, 3000), (480, 640, 480, 640), (480, 640, 240, 320), (1080, 1920, 540, 960),
                 (479, 641, 62, 641), (31, 641, 62, 641), (641, 641, 31, 33), (2, 641, 641, 2)]


@pytest.mark.parametrize("channels", [1, 3])
@pytest.mark.parametrize("batch", [1, 4])
@pytest.mark.parametrize("shape", RESIZE_SHAPES, ids=lambda s: "%dx%d_to_%dx%d" % s)
def test_resize_linear_batched(ctx, shape, batch, channels):
    sh, sw, dh, dw = shape
    ims = np.random.default_rng(sum(shape) + batch + channels).integers(0, 256, (batch, sh, sw, channels), np.uint8)
    want = np.stack([cv2.resize(im, (dw, dh), interpolation=cv2.INTER_LINEAR).reshape(dh, dw, channels) for im in ims])
    if batch == 1:
        src = ims[0] if channels == 3 else ims[0, ..., 0]
        got = ctx.download(ctx.resize(ctx.upload(src), dw, dh))
        assert got.shape == ((dh, dw, 3) if channels == 3 else (dh, dw))
        got = got.reshape(1, dh, dw, channels)
    else:
        got = ctx.download(ctx.resize(ctx.upload(ims), dw, dh))
        assert got.shape == (batch, dh, dw, channels)
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%d differing bytes, first at (image, y, x, c) = %s" % (len(bad), tuple(bad[0]))
