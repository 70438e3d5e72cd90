"""GPU parity of the colour balance at the edges of its per-frame statistics (oracle/edge_frames.py): cumulative
counts exactly on the percentile bounds, equal channel means, zero-width S / V ranges, zero channel means, tiny and
> 2^24-pixel frames, every BGR colour at once.  The oracle is the numpy restatement with the device's definition of a
zero-width stretch (`zero_width_stretch="zero"`, equal to the reference wherever the reference is defined:
tests/test_balance_edge_frames.py); 0 differing bytes and the per-frame statistics are asserted on every path --
vector and scalar passes 2 / 3, the tiled kernels, the fused stage for each conversion, the mask-only hue-interval
table, the tuning knobs and a chunked batch on side streams."""
import functools

import cv2
import numpy as np
import pytest
import torch

from oracle import color_balance_np as cb
from oracle import edge_frames as ef
from oracle import synth

pytestmark = pytest.mark.gpu

CVT = {"bgr2hsv": cv2.COLOR_BGR2HSV, "bgr2lab": cv2.COLOR_BGR2LAB, "bgr2gray": cv2.COLOR_BGR2GRAY,
       "bgr2ycrcb": cv2.COLOR_BGR2YCrCb, "bgr2hls": cv2.COLOR_BGR2HLS}
MASK_BOUNDS = [((0, 0, 60), (179, 255, 255)), ((0, 0, 0), (179, 30, 255)), ((10, 20, 60), (30, 100, 255)),
               ((0, 0, 0), (179, 255, 0))]


def restate(img, **flags):
    return cb.process_frame_np(img, return_stats=True, zero_width_stretch="zero", **flags)


@functools.lru_cache(maxsize=None)
def cached(name):
    """Frames whose restatement takes seconds (> 2^24 pixels): built and restated once per session."""
    if name == "all_colours":
        img = synth.all_colors_image()
        return img, restate(img)
    if name == "glare":
        img = ef.glare_frame(*ef.GLARE_SHAPE, seed=7)[0]
        return img, restate(img)
    raise KeyError(name)


def assert_same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    d = got != want
    assert not d.any(), "%s: %d differing bytes, first at %s" % (what, int(d.sum()), np.argwhere(d)[0].tolist())


def check_stats(s, st, flags, what):
    assert s["bgr_min"] == tuple(st["bgr_min"]) and s["bgr_max"] == tuple(st["bgr_max"]), what
    assert s["bgr_avg"] == tuple(st["bgr_avg"]), what
    if flags.get("equalize_rgb", True):
        assert "bgr"[s["dominant"]] == st["tiles"][0]["dom"], what
    if flags.get("hsv_contrast_correct", True):
        assert (s["s_min"], s["s_max"], s["v_min"], s["v_max"]) == (st["s_min"], st["s_max"], st["v_min"], st["v_max"]), what
        assert s["degenerate"] == int(st["s_min"] == st["s_max"] or st["v_min"] == st["v_max"]), what


def misaligned(ctx, frames):
    """The same bytes at an odd device address: every balance pass takes its scalar (byte-wise) path."""
    flat = ctx.upload(np.ascontiguousarray(frames).reshape(-1))
    buf = ctx.empty((flat.numel() + 1,))
    with torch.cuda.stream(ctx.torch_stream):
        buf[1:].copy_(flat)
    view = buf[1:].view(frames.shape)
    assert view.data_ptr() % 2 == 1 and view.is_contiguous()
    return view


def balance_and_check(ctx, frames, wants, flags, what, path="vector"):
    """color_balance of a batch (vector path, or the scalar path through a misaligned view) against the restatements
    `wants` = [(out, stats)] frame by frame."""
    src = ctx.upload(frames) if path == "vector" else misaligned(ctx, frames)
    got, stats = ctx.color_balance(src, want_stats=True, **flags)
    got = ctx.download(got)
    for i, (want, st) in enumerate(wants):
        assert_same(got[i], want, "%s frame %d (%s path)" % (what, i, path))
        check_stats(stats[i], st, flags, "%s frame %d (%s path)" % (what, i, path))


def stage_and_check(ctx, frames, wants, flags, what, codes=tuple(CVT), lo=(0, 40, 60), hi=(179, 255, 255)):
    """The fused stage with balanced + converted + mask outputs for each conversion, then the mask-only HSV call
    (hue-interval table where the shape allows it)."""
    dev = ctx.upload(frames)
    for code in codes:
        desc = ctx.make_stage(balance=flags, cvt=code, lo=lo, hi=hi)
        out = ctx.stage(desc, dev, want=("balanced", "converted", "mask"))
        bal, conv, mask = (ctx.download(out[k]) for k in ("balanced", "converted", "mask"))
        for i, (want, _) in enumerate(wants):
            c_ref = cv2.cvtColor(want, CVT[code])
            m_ref = cv2.inRange(c_ref, lo[0], hi[0]) if code == "bgr2gray" else cv2.inRange(c_ref, np.array(lo), np.array(hi))
            assert_same(bal[i], want, "%s %s balanced %d" % (what, code, i))
            assert_same(conv[i], c_ref, "%s %s converted %d" % (what, code, i))
            assert_same(mask[i], m_ref, "%s %s mask %d" % (what, code, i))
    for blo, bhi in MASK_BOUNDS:
        desc = ctx.make_stage(balance=flags, cvt="bgr2hsv", lo=blo, hi=bhi)
        mask = ctx.download(ctx.stage(desc, dev, want=("mask",))["mask"])
        for i, (want, _) in enumerate(wants):
            m_ref = cv2.inRange(cv2.cvtColor(want, cv2.COLOR_BGR2HSV), np.array(blo), np.array(bhi))
            assert_same(mask[i], m_ref, "%s mask-only %s..%s %d" % (what, blo, bhi, i))


# ---------------------------------------------------------------------------------------------------------------------
# cumulative counts on the percentile bounds
# ---------------------------------------------------------------------------------------------------------------------
BOUND_SHAPES = [(214, 2208), (281, 1920), (203, 601), (4097, 4099), (1, 500), (1, 501), (480, 640)]


@functools.lru_cache(maxsize=None)
def exact_bound_case(shape, rgbcc):
    frames = np.stack([ef.exact_bound_frame(shape[0], shape[1], seed=s)[0] for s in (1, 2)])
    flags = dict(rgb_contrast_correct=True) if rgbcc else {}
    return frames, [restate(f, **flags) for f in frames], flags


@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("rgbcc", [False, True], ids=["default", "rgbcc"])
@pytest.mark.parametrize("shape", BOUND_SHAPES, ids=lambda s: "%dx%d" % s)
def test_exact_bound_frames(ctx, shape, rgbcc, path):
    frames, wants, flags = exact_bound_case(shape, rgbcc)
    balance_and_check(ctx, frames, wants, flags, "exact bounds", path)


@pytest.mark.parametrize("path", ["vector", "scalar"])
@pytest.mark.parametrize("shape", [(214, 2208), (203, 601), (480, 640)], ids=lambda s: "%dx%d" % s)
def test_exact_bound_sv_frames(ctx, shape, path):
    frames = np.stack([ef.exact_bound_sv_frame(shape[0], shape[1], seed=s, offsets=o)[0]
                       for s, o in ((2, ((0, 1), (1, -1))), (3, ((1, 0), (-1, 0))))])
    wants = [restate(f, **ef.SV_FLAGS) for f in frames]
    balance_and_check(ctx, frames, wants, ef.SV_FLAGS, "S/V bounds", path)
    if path == "vector":
        stage_and_check(ctx, frames, wants, ef.SV_FLAGS, "S/V bounds", codes=("bgr2hsv", "bgr2lab"))


# ---------------------------------------------------------------------------------------------------------------------
# equal channel means
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [{}, dict(rgb_contrast_correct=True), dict(horizontal_blocks=2, vertical_blocks=2),
                                   dict(horizontal_blocks=2, vertical_blocks=2, rgb_contrast_correct=True)],
                         ids=["default", "rgbcc", "tiles2x2", "tiles2x2_rgbcc"])
@pytest.mark.parametrize("pattern", ef.TIE_PATTERNS)
def test_tie_frames(ctx, pattern, flags):
    frames = np.stack([ef.tie_frame(240, 320, s, pattern)[0] for s in (5, 6)])
    wants = [restate(f, **flags) for f in frames]
    balance_and_check(ctx, frames, wants, flags, "tie " + pattern)
    if not flags.get("horizontal_blocks"):
        balance_and_check(ctx, frames, wants, flags, "tie " + pattern, "scalar")
    stage_and_check(ctx, frames, wants, flags, "tie " + pattern, codes=("bgr2hsv",))


# ---------------------------------------------------------------------------------------------------------------------
# zero-width S / V ranges and zero channel means
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ef.ZERO_WIDTH_KINDS)
def test_zero_width_frames(ctx, kind):
    frames, claims = zip(*(ef.zero_width_frame(240, 320, s, kind) for s in (5, 6)))
    frames, flags = np.stack(frames), claims[0]["flags"]
    wants = [restate(f, **flags) for f in frames]
    for _, st in wants:
        assert st["s_min"] == st["s_max"] or st["v_min"] == st["v_max"]
    balance_and_check(ctx, frames, wants, flags, kind)
    balance_and_check(ctx, frames, wants, flags, kind, "scalar")
    stage_and_check(ctx, frames, wants, flags, kind)
    # with the RGB contrast stretch a zero-width or zero-mean channel gives an infinite or NaN ratio
    flags_cc = dict(flags, rgb_contrast_correct=True)
    balance_and_check(ctx, frames, [restate(f, **flags_cc) for f in frames], flags_cc, kind + " rgbcc")


@pytest.mark.parametrize("kind", ["random", "grey", "red_free"])
@pytest.mark.parametrize("shape", [(1, 2), (2, 3), (3, 5), (1, 499), (1, 500), (1, 501), (15, 1)], ids=lambda s: "%dx%d" % s)
def test_tiny_frames(ctx, shape, kind):
    if kind == "random":
        frames = np.stack([synth.gen_random_bgr(shape[0], shape[1], s) for s in (1, 2)])
    else:
        frames = np.stack([ef.zero_width_frame(shape[0], shape[1], s, kind)[0] for s in (1, 2)])
    for flags in ({}, dict(rgb_contrast_correct=True), dict(hsv_contrast_correct=False)):
        wants = [restate(f, **flags) for f in frames]
        balance_and_check(ctx, frames, wants, flags, "%s %dx%d" % ((kind,) + shape))
    wants = [restate(f) for f in frames]
    balance_and_check(ctx, frames, wants, {}, "%s %dx%d" % ((kind,) + shape), "scalar")
    stage_and_check(ctx, frames, wants, {}, "%s %dx%d" % ((kind,) + shape))


def test_one_pixel_frame_is_defined(ctx):
    """1x1: the reference reads an uninitialised maximum there (its high bound, 1, is never crossed); only the call has
    to succeed."""
    img = np.array([[[10, 200, 30]]], np.uint8)
    out, stats = ctx.color_balance(ctx.upload(img), want_stats=True)
    assert ctx.download(out).shape == img.shape and len(stats) == 1
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255))
    assert ctx.download(ctx.stage(desc, ctx.upload(img), want=("mask",))["mask"]).shape == (1, 1)


def test_glare_frame_above_two_to_the_24_pixels(ctx):
    """96 % white glare on 17.4 M pixels: channel sums above 2^32, one histogram bin holding almost the whole frame."""
    img, want = cached("glare")
    balance_and_check(ctx, img[None], [want], {}, "glare")
    out = ctx.stage(ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 0, 200), hi=(179, 40, 255)), ctx.upload(img), want=("mask",))
    assert_same(ctx.download(out["mask"]), cv2.inRange(cv2.cvtColor(want[0], cv2.COLOR_BGR2HSV), np.array([0, 0, 200]),
                                                       np.array([179, 40, 255])), "glare mask-only")


# ---------------------------------------------------------------------------------------------------------------------
# every BGR colour through passes 2 and 3
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def all_colours_ref(code):
    return cv2.cvtColor(cached("all_colours")[1][0], CVT[code])


@pytest.mark.parametrize("option,value", [(None, 0), ("no_hue_table", 1)], ids=lambda x: str(x))
def test_all_colours_frame(ctx, option, value):
    """synth.all_colors_image(): identity pass-1 tables (uniform histograms, three equal means of 127.5, a tie), a
    non-identity S / V stretch, a float32 bound (33 554 against 33 555 in double): every (B, G, R) through pass 2's HSV,
    the H,S,V scratch and pass 3's HSV -> BGR -> conversion, under each tuning knob."""
    img, (want, st) = cached("all_colours")
    assert (st["s_min"], st["s_max"], st["v_min"], st["v_max"]) != (0, 255, 0, 255)
    dev = ctx.upload(img)
    try:
        if option:
            ctx.set_option(option, value)
        got, stats = ctx.color_balance(dev, want_stats=True)
        assert_same(ctx.download(got), want, "all colours")
        check_stats(stats[0], st, {}, "all colours")
        balance_and_check(ctx, img[None], [(want, st)], {}, "all colours", "scalar")
        for code in CVT:
            out = ctx.stage(ctx.make_stage(balance={}, cvt=code), dev, want=("converted",))
            assert_same(ctx.download(out["converted"]), all_colours_ref(code), "all colours " + code)
        out = ctx.stage(ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255)), dev,
                        want=("balanced", "converted", "mask"))
        assert_same(ctx.download(out["balanced"]), want, "all colours stage balanced")
        assert_same(ctx.download(out["converted"]), all_colours_ref("bgr2hsv"), "all colours stage converted")
        for lo, hi in MASK_BOUNDS:
            mask = ctx.download(ctx.stage(ctx.make_stage(balance={}, cvt="bgr2hsv", lo=lo, hi=hi), dev, want=("mask",))["mask"])
            assert_same(mask, cv2.inRange(all_colours_ref("bgr2hsv"), np.array(lo), np.array(hi)), "all colours mask %s..%s" % (lo, hi))
    finally:
        if option:
            ctx.set_option(option, 0)


# ---------------------------------------------------------------------------------------------------------------------
# nothing leaks between the frames and chunks of a batch
# ---------------------------------------------------------------------------------------------------------------------
def test_mixed_batch_on_chunks_and_side_streams(ctx):
    """Normal, degenerate, red-free, saturated and tie frames of one shape in one batch, cut into 1 MB chunks over four
    side streams: every frame's bytes, statistics and `degenerate` flag are its own."""
    h, w = 240, 320
    glare = synth.gen_underwater(h, w, 31)
    glare.reshape(-1, 3)[np.random.default_rng(31).permutation(h * w)[:int(0.95 * h * w)]] = 255
    frames = np.stack([synth.gen_underwater(h, w, 30), ef.zero_width_frame(h, w, 5, "constant")[0],
                       ef.zero_width_frame(h, w, 6, "red_free")[0], glare, ef.tie_frame(h, w, 7, "b=g=r")[0],
                       ef.zero_width_frame(h, w, 8, "grey")[0], ef.tie_frame(h, w, 9, "g=r>b")[0],
                       ef.zero_width_frame(h, w, 10, "sparse_red")[0], synth.gen_underwater(h, w, 11),
                       ef.zero_width_frame(h, w, 12, "black")[0], ef.exact_bound_frame(h, w, seed=13)[0]])
    wants = [restate(f) for f in frames]
    assert len({st["s_min"] == st["s_max"] or st["v_min"] == st["v_max"] for _, st in wants}) == 2
    try:
        ctx.set_option("l2_chunk_mb", 1)
        ctx.set_option("side_streams", 4)
        balance_and_check(ctx, frames, wants, {}, "mixed batch")
        stage_and_check(ctx, frames, wants, {}, "mixed batch", codes=("bgr2hsv", "bgr2lab"))
    finally:
        ctx.set_option("l2_chunk_mb", 0)
        ctx.set_option("side_streams", 0)


# ---------------------------------------------------------------------------------------------------------------------
# HSI branch on grey, black and primary pixels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", [dict(equalize_rgb=False, rgb_extrema_clipping=False), {}], ids=["identity_pass1", "default"])
def test_hsi_branch_on_grey_black_and_primary_pixels(ctx, flags):
    """Grey pixels (0/0 hue), black pixels (I = 0) and pure primaries / secondaries (hue on a sector boundary).  Stated
    tolerance of the HSI branch (tests/test_gpu_balance_stage.py::test_balance_hsi_branch): <= 1 LSB on <= 8 pixels."""
    flags = dict(flags, hsi_contrast_correct=True, hsv_contrast_correct=False)
    img = ef.hsi_edge_frame(384, 512, 3)[0]
    want = cb.process_frame_np(img, **flags)
    got = ctx.download(ctx.color_balance(ctx.upload(img), **flags))
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16))
    assert int(diff.max()) <= 1 and int((diff != 0).sum()) <= 8, (int(diff.max()), int((diff != 0).sum()))
