"""GPU parity: colour balance against the compiled, unmodified reference (oracle/_ref) and its
golden vectors; the fused stage against the reference's module pipelines (modules/bins.py,
modules/red_buoy.py) expressed as cv2 calls; resize / YOLO input; drop-in modules.

Colour balance tolerance (stated): the device computes the channel means as exact integer sums / N
where the reference uses a sequential running mean (color_balance.cpp:459-470, equal to <= 1.2e-12);
a differing gain could move a table entry by 1 LSB, so the stated bound is max |diff| <= 1 LSB --
and 0 differing bytes is what is asserted on every case here."""
import glob
import os

import cv2
import numpy as np
import pytest

from oracle import ccl, color_balance_np as cb, cv_ops, letterbox, ref_balance, synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_cases():
    return sorted(glob.glob(os.path.join(GOLDEN, "balance_*.npz")))


@pytest.mark.parametrize("path", golden_cases(), ids=lambda p: os.path.basename(p)[8:-4])
def test_balance_golden_vectors_from_the_reference(ctx, path):
    z = np.load(path, allow_pickle=True)
    flags = {k: v for k, v in z["flags"]} if z["flags"].size else {}
    got = ctx.download(ctx.color_balance(ctx.upload(z["src"]), **flags))
    assert np.array_equal(got, z["out"])


def oracle_balance(img, **flags):
    """compiled reference when it travelled to this box, else its pinned restatement"""
    if ref_balance.available():
        return ref_balance.balance(img, **flags)
    return cb.process_frame_np(img, **flags)


@pytest.mark.parametrize("shape,seed", [((480, 640), 1), ((479, 641), 2), ((1080, 1920), 3), ((1242, 2208), 7),
                                        ((1243, 2209), 8), ((2160, 3840), 9)])
def test_balance_default_flags_vs_reference(ctx, shape, seed):
    img = synth.gen_underwater(shape[0], shape[1], seed)
    want = oracle_balance(img)
    got, stats = ctx.color_balance(ctx.upload(img), want_stats=True)
    got = ctx.download(got)
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16))
    assert int(diff.max()) <= 1, "stated tolerance: 1 LSB"
    assert int((diff != 0).sum()) == 0, "expected: identical bytes"
    _, st = cb.process_frame_np(img, return_stats=True)
    s = stats[0]
    assert s["bgr_min"] == tuple(st["bgr_min"]) and s["bgr_max"] == tuple(st["bgr_max"])
    assert s["bgr_avg"] == pytest.approx(st["bgr_avg"], rel=0, abs=0)
    assert (s["s_min"], s["s_max"], s["v_min"], s["v_max"]) == (st["s_min"], st["s_max"], st["v_min"], st["v_max"])
    assert "bgr"[s["dominant"]] == st["tiles"][0]["dom"]


@pytest.mark.parametrize("flags", [dict(hsv_contrast_correct=False), dict(rgb_extrema_clipping=False),
                                   dict(rgb_contrast_correct=True), dict(adaptive_cast_correction=True),
                                   dict(equalize_rgb=False), dict(equalize_rgb=False, hsv_contrast_correct=False),
                                   dict(rgb_contrast_correct=True, hsv_contrast_correct=False,
                                        adaptive_cast_correction=True)],
                         ids=lambda f: ",".join(sorted(f)))
def test_balance_flag_combinations(ctx, flags):
    img = synth.gen_underwater(360, 640, 21)
    got = ctx.download(ctx.color_balance(ctx.upload(img), **flags))
    assert np.array_equal(got, oracle_balance(img, **flags))


@pytest.mark.parametrize("hb,vb,flags", [(2, 2, {}), (4, 2, {}), (1, 3, {}), (8, 5, {}), (4, 4, dict(adaptive_cast_correction=True)),
                                         (2, 2, dict(rgb_contrast_correct=True)), (5, 2, dict(hsv_contrast_correct=False)),
                                         (16, 12, {})])
def test_balance_tiled_equalisation(ctx, hb, vb, flags):
    """horizontal/vertical_blocks > 1 (P1, color_balance.cpp:441-544): per-tile gains with the
    fall-back-to-global rule of line 474."""
    img = synth.gen_underwater(240, 320, 5)
    img[:120, :160] = np.clip(img[:120, :160].astype(int) + np.array([25, 5, 0]), 0, 255).astype(np.uint8)
    got = ctx.download(ctx.color_balance(ctx.upload(img), horizontal_blocks=hb, vertical_blocks=vb, **flags))
    want = oracle_balance(img, horizontal_blocks=hb, vertical_blocks=vb, **flags)
    assert np.array_equal(got, want)


def test_balance_tiled_batch_and_stage(ctx):
    frames = np.stack([synth.gen_underwater(240, 320, 60 + s) for s in range(3)])
    frames[1, :120, :160] = np.clip(frames[1, :120, :160].astype(int) + np.array([30, 0, 0]), 0, 255).astype(np.uint8)
    desc = ctx.make_stage(balance=dict(horizontal_blocks=4, vertical_blocks=2), cvt="bgr2hsv", lo=(0, 40, 60),
                          hi=(179, 255, 255), morph=[("open", 5, 5, 1)])
    out = ctx.stage(desc, ctx.upload(frames), want=("balanced", "mask"))
    for i in range(3):
        b_ref = oracle_balance(frames[i], horizontal_blocks=4, vertical_blocks=2)
        assert np.array_equal(ctx.download(out["balanced"])[i], b_ref)
        m_ref = cv2.morphologyEx(cv2.inRange(cv2.cvtColor(b_ref, cv2.COLOR_BGR2HSV), np.array([0, 40, 60]),
                                             np.array([179, 255, 255])), cv2.MORPH_OPEN, cv_ops.rect_kernel(5))
        assert np.array_equal(ctx.download(out["mask"])[i], m_ref)


def test_balance_batch_of_distinct_frames_and_in_place(ctx):
    frames = np.stack([synth.gen_underwater(242, 368, 40 + s) for s in range(11)])
    d = ctx.upload(frames)
    got = ctx.download(ctx.color_balance(d))
    for i in range(frames.shape[0]):
        assert np.array_equal(got[i], oracle_balance(frames[i])), i
    from cuauv_vision_pipeline_b200.runtime import ffi, lib, check, _u8ptr
    prm = ffi.new("bv_balance_params *")
    lib.bv_balance_default(prm)
    check(lib.bv_color_balance(ctx.handle, _u8ptr(d), _u8ptr(d), frames.shape[0], 242, 368, prm, ffi.NULL))
    assert np.array_equal(ctx.download(d), got)


def test_balance_red_and_green_dominant(ctx):
    for perm in ((2, 1, 0), (1, 0, 2)):
        img = np.ascontiguousarray(synth.gen_underwater(240, 320, 5)[..., list(perm)])
        assert np.array_equal(ctx.download(ctx.color_balance(ctx.upload(img))), oracle_balance(img))


def test_balance_unsupported_flags_fail_loudly(ctx):
    import cuauv_vision_pipeline_b200 as bv
    d = ctx.upload(synth.gen_underwater(64, 64, 1))
    with pytest.raises(bv.BVError):
        ctx.color_balance(d, horizontal_blocks=3)       # 64 % 3 != 0: the reference walks off the row here


def test_balance_degenerate_frame_is_defined(ctx):
    """Constant frame: the reference dies with an integer division by zero (color_balance.cpp:684).
    Here the stretch of a zero-width range is defined as 0 and flagged; nothing crashes."""
    img = np.full((48, 64, 3), 90, np.uint8)
    out, stats = ctx.color_balance(ctx.upload(img), want_stats=True)
    assert stats[0]["degenerate"] == 1
    assert ctx.download(out).shape == img.shape


def test_legacy_process_frame_symbol_is_a_drop_in(ctx):
    """modules/color_balance.py:93-110 verbatim against the CUDA-backed libauv-color-balance.so."""
    from cuauv_vision_pipeline_b200.color_balance import balance, balance_legacy
    img = synth.gen_underwater(479, 641, 17)
    want = oracle_balance(img)
    assert np.array_equal(balance_legacy(img), want)
    assert np.array_equal(balance(img), want)
    assert np.array_equal(balance_legacy(img, hsv_contrast_correct=False), oracle_balance(img, hsv_contrast_correct=False))


# ----------------------------------------------------------------------------------------------
# fused stage
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1080, 1920), (480, 640), (479, 641), (270, 496)])
def test_stage_bins_pipeline(ctx, shape):
    """modules/bins.py:13-27: BGR2HSV -> inRange -> OPEN 5x5 -> blobs."""
    img = synth.gen_underwater(shape[0], shape[1], 30)
    mask_ref, cleaned_ref = cv_ops.bins_mask(img)
    desc = ctx.make_stage(cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)], label=True)
    out = ctx.stage(desc, ctx.upload(img), want=("converted", "mask", "labels", "blobs"), max_blobs=4096)
    assert np.array_equal(ctx.download(out["converted"]), cv2.cvtColor(img, cv2.COLOR_BGR2HSV))
    assert np.array_equal(ctx.download(out["mask"]), cleaned_ref)
    n_ref, lab_ref, tab = ccl.label_and_moments(cleaned_ref)
    n, tables = ctx.blobs_to_numpy(out["blobs"], out["n_blobs"])
    assert int(n[0]) == n_ref and np.array_equal(ctx.download(out["labels"]), lab_ref)
    for key in ccl.MOMENT_KEYS:
        assert np.array_equal(tables[0][key].astype(np.int64), tab[key]), key
    # threshold only (no morphology): the raw mask
    desc0 = ctx.make_stage(cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255))
    assert np.array_equal(ctx.download(ctx.stage(desc0, ctx.upload(img), want=("mask",))["mask"]), mask_ref)


@pytest.mark.parametrize("shape", [(480, 640), (1242, 2208), (479, 641)])
def test_stage_buoy_pipeline(ctx, shape):
    """modules/red_buoy.py:21-34: LAB a-channel inRange -> OPEN -> CLOSE."""
    img = synth.gen_underwater(shape[0], shape[1], 31)
    th_ref, cl_ref = cv_ops.buoy_mask(img, 150, 255)
    desc = ctx.make_stage(cvt="bgr2lab", lo=(0, 150, 0), hi=(255, 255, 255), morph=[("open", 5, 5, 1), ("close", 5, 5, 1)])
    assert np.array_equal(ctx.download(ctx.stage(desc, ctx.upload(img), want=("mask",))["mask"]), cl_ref)
    desc0 = ctx.make_stage(cvt="bgr2lab", lo=(0, 150, 0), hi=(255, 255, 255))
    assert np.array_equal(ctx.download(ctx.stage(desc0, ctx.upload(img), want=("mask",))["mask"]), th_ref)


@pytest.mark.parametrize("shape", [(1242, 2208), (479, 641)])
def test_stage_balance_convert_threshold_morph(ctx, shape):
    """The north-star stage: balance -> LAB / HSV -> inRange -> OPEN, every output checked."""
    frames = np.stack([synth.gen_underwater(shape[0], shape[1], 50 + s) for s in range(3)])
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[("open", 5, 5, 1)], label=True)
    out = ctx.stage(desc, ctx.upload(frames), want=("balanced", "converted", "mask", "labels", "blobs"), max_blobs=8192)
    bal = ctx.download(out["balanced"])
    cvt = ctx.download(out["converted"])
    mask = ctx.download(out["mask"])
    lab = ctx.download(out["labels"])
    n, tables = ctx.blobs_to_numpy(out["blobs"], out["n_blobs"])
    for i in range(frames.shape[0]):
        b_ref = oracle_balance(frames[i])
        assert np.array_equal(bal[i], b_ref)
        hsv_ref = cv2.cvtColor(b_ref, cv2.COLOR_BGR2HSV)
        assert np.array_equal(cvt[i], hsv_ref)
        m_ref = cv2.morphologyEx(cv2.inRange(hsv_ref, np.array([0, 40, 60]), np.array([179, 255, 255])), cv2.MORPH_OPEN,
                                 cv_ops.rect_kernel(5))
        assert np.array_equal(mask[i], m_ref)
        n_ref, lab_ref, tab = ccl.label_and_moments(m_ref)
        assert int(n[i]) == n_ref and np.array_equal(lab[i], lab_ref)
        k = min(n_ref, 8192)
        assert np.array_equal(tables[i]["m10"].astype(np.int64), tab["m10"][:k])
    # config 2 of BASELINE.json: balance -> LAB image
    desc2 = ctx.make_stage(balance={}, cvt="bgr2lab")
    lab_img = ctx.download(ctx.stage(desc2, ctx.upload(frames), want=("converted",))["converted"])
    for i in range(frames.shape[0]):
        assert np.array_equal(lab_img[i], cv2.cvtColor(oracle_balance(frames[i]), cv2.COLOR_BGR2LAB))


def test_stage_host_equals_device_stage(ctx):
    frames = np.stack([synth.gen_underwater(360, 640, 70 + s) for s in range(9)])
    desc = ctx.make_stage(balance={}, cvt="bgr2lab", lo=(0, 130, 0), hi=(255, 255, 255), morph=[("open", 5, 5, 1)], label=True)
    want = ("balanced", "converted", "mask", "labels", "blobs")
    dev = ctx.stage(desc, ctx.upload(frames), want=want, max_blobs=512)
    host = ctx.stage_host(desc, frames, want=want, max_blobs=512)
    for k in ("balanced", "converted", "mask", "labels"):
        assert np.array_equal(host[k], ctx.download(dev[k])), k
    assert np.array_equal(host["n_blobs"], ctx.download(dev["n_blobs"]))
    n, tables = ctx.blobs_to_numpy(dev["blobs"], dev["n_blobs"])
    for i in range(frames.shape[0]):
        assert np.array_equal(host["blobs"][i][:int(n[i])], tables[i])
    # pinned buffers take the same path
    import cuauv_vision_pipeline_b200 as bv
    pin = bv.PinnedArray(frames.shape)
    pin.array[...] = frames
    out = bv.PinnedArray(frames.shape)
    res = ctx.stage_host(desc, pin.array, want=("converted",), out={"converted": out.array})
    assert np.array_equal(res["converted"], host["converted"])


def test_stage_host_submit_wait_two_batches_in_flight(ctx):
    """bv_stage_host_submit / _wait: two calls in flight on the two staging slots deliver what the blocking call delivers,
    for different batch sizes and stages per slot, over several rounds (a slot is re-used while the other is in flight)."""
    import cuauv_vision_pipeline_b200 as bv
    shapes = [(9, 360, 640), (5, 480, 656)]
    descs = [ctx.make_stage(balance={}, cvt="bgr2lab"),
             ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)], label=True)]
    wants = [("converted",), ("mask", "blobs")]
    rounds = 4
    src = [[bv.PinnedArray(shapes[k] + (3,)) for _ in range(rounds)] for k in range(2)]
    expect = [[None] * rounds for _ in range(2)]
    for k in range(2):
        for r in range(rounds):
            b, h, w = shapes[k]
            src[k][r].array[...] = np.stack([synth.gen_underwater(h, w, 1000 * k + 10 * r + i) for i in range(b)])
            expect[k][r] = {n: np.array(v, copy=True)
                            for n, v in ctx.stage_host(descs[k], src[k][r].array, want=wants[k], max_blobs=256).items()}
    pins = [bv.PinnedArray(shapes[0] + (3,)), bv.PinnedArray(shapes[1]), bv.PinnedArray((shapes[1][0], 256), bv.BLOB_DTYPE),
            bv.PinnedArray((shapes[1][0],), np.int32)]   # the PinnedArray objects own the memory: keep them
    outs = [{"converted": pins[0].array}, {"mask": pins[1].array, "blobs": pins[2].array, "n_blobs": pins[3].array}]
    for r in range(rounds):
        for k in range(2):     # both slots in flight before either is waited for
            ctx.stage_host(descs[k], src[k][r].array, want=wants[k], max_blobs=256, out=outs[k], slot=k)
        for k in (1, 0):
            ctx.stage_host_wait(k)
            for n in wants[k]:
                if n == "blobs":
                    for i in range(shapes[k][0]):
                        nb = int(expect[k][r]["n_blobs"][i])
                        assert int(outs[k]["n_blobs"][i]) == nb
                        assert np.array_equal(outs[k]["blobs"][i][:nb], expect[k][r]["blobs"][i][:nb]), (r, k, i)
                else:
                    assert np.array_equal(outs[k][n], expect[k][r][n]), (r, k, n)
    # back-to-back submits on ONE slot: the second waits for the first by itself
    ctx.stage_host(descs[0], src[0][0].array, want=wants[0], out=outs[0], slot=0)
    ctx.stage_host(descs[0], src[0][1].array, want=wants[0], out=outs[0], slot=0)
    ctx.stage_host_wait(0)
    assert np.array_equal(outs[0]["converted"], expect[0][1]["converted"])
    ctx.stage_host_wait(1)   # nothing in flight: returns at once
    with pytest.raises(Exception):
        ctx.stage_host(descs[0], src[0][0].array, want=wants[0], out=outs[0], slot=2)


def test_stage_gradient_and_threshold_on_bgr(ctx):
    img = synth.gen_underwater(200, 320, 33)
    desc = ctx.make_stage(cvt=None, lo=(60, 40, 0), hi=(255, 200, 120), morph=[("gradient", 3, 3, 1)])
    m_ref = cv2.morphologyEx(cv2.inRange(img, np.array([60, 40, 0]), np.array([255, 200, 120])), cv2.MORPH_GRADIENT,
                             cv_ops.rect_kernel(3))
    assert np.array_equal(ctx.download(ctx.stage(desc, ctx.upload(img), want=("mask",))["mask"]), m_ref)


# ----------------------------------------------------------------------------------------------
# resize / YOLO input / preprocessor / modules
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1242, 2208, 360, 640, 3), (479, 641, 777, 333, 3), (480, 640, 960, 1280, 1),
                                   (2160, 3840, 459, 816, 3), (100, 100, 37, 53, 3)])
def test_resize_linear(ctx, shape):
    sh, sw, dh, dw, c = shape
    im = np.random.default_rng(3).integers(0, 256, (sh, sw, c), dtype=np.uint8)
    if c == 1:
        im = im[..., 0]
    assert np.array_equal(ctx.download(ctx.resize(ctx.upload(im), dw, dh)), cv2.resize(im, (dw, dh)))


def test_yolo_input_batch_of_mixed_cameras(ctx):
    """config 4: 16 frames of mixed sizes -> [16,3,640,640] fp16.  The uint8 letterbox is exact
    (cv2.resize + copyMakeBorder) and so is the normalised tensor: u/255 rounds to the same fp16 in
    every precision (tests/test_letterbox_cases.py), so 0 differing values are asserted.  Parity of
    the Ultralytics side itself is unpinned (not installed)."""
    from cuauv_vision_pipeline_b200.yolo_input import yolo_input
    sizes = [(1242, 2208), (1080, 1920), (720, 1280), (480, 640)] * 4
    imgs = [synth.gen_underwater(h, w, 90 + i) for i, (h, w) in enumerate(sizes)]
    got = yolo_input(imgs)
    want = letterbox.yolo_input(imgs)
    assert got.shape == (16, 3, 640, 640) and got.dtype == np.float16
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))
    got32 = yolo_input(imgs[:2], half=False)
    assert np.array_equal(got32, letterbox.yolo_input(imgs[:2], half=False))
    # scale-up and identity geometry
    small = [synth.gen_underwater(90, 160, 5), synth.gen_underwater(64, 64, 6)]
    assert np.array_equal(yolo_input(small, (64, 64)).view(np.uint16), letterbox.yolo_input(small, 64, 64).view(np.uint16))


def test_letterbox_golden(ctx):
    from cuauv_vision_pipeline_b200.yolo_input import yolo_input
    z = np.load(os.path.join(GOLDEN, "letterbox_90x160_to_64.npz"))
    assert np.array_equal(yolo_input([z["src"]], (64, 64)).view(np.uint16), z["f16"].view(np.uint16))


def test_cv_call_site_golden(ctx):
    z = np.load(os.path.join(GOLDEN, "cv_calls_72x128.npz"))
    d = ctx.upload(z["src"])
    for code in ("bgr2lab", "bgr2hsv", "bgr2ycrcb", "bgr2gray"):
        assert np.array_equal(ctx.download(ctx.cvt_color(d, code)), z[code]), code
    assert np.array_equal(ctx.download(ctx.cvt_color(ctx.upload(z["bgr2hsv"]), "hsv2bgr")), z["hsv2bgr"])
    desc = ctx.make_stage(cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)])
    assert np.array_equal(ctx.download(ctx.stage(desc, d, want=("mask",))["mask"]), z["bins_cleaned"])
    assert np.array_equal(ctx.download(ctx.resize(d, 50, 37)), z["resize_50x37"])
    from cuauv_vision_pipeline_b200 import transform
    assert np.array_equal(ctx.download(ctx.morph(d, "erode", transform.elliptic_kernel(5))), z["ellipse_erode_2"])
    assert np.array_equal(ctx.download(ctx.morph(d, "dilate", transform.elliptic_kernel(7))), z["ellipse_dilate_3"])


def test_preprocessor_mirror(ctx):
    from cuauv_vision_pipeline_b200.preprocessor import Preprocessor

    class Mod:
        def __init__(self):
            self.posted = {}

        def post(self, name, img):
            self.posted[name] = np.asarray(img)
    mod = Mod()
    pp = Preprocessor(mod)
    img = synth.gen_underwater(242, 368, 12)
    for k, v in dict(PPX_lab=True, PPX_hsv_split=True, PPX_grayscale=True, PPX_color_correction=True, PPX_r_bias=20,
                     PPX_contrast=1.3, PPX_brightness=-15, PPX_erode=True, PPX_erode_kernel=2, PPX_dilate=True,
                     PPX_dilate_kernel=1, PPX_resize_ratio=0.37).items():
        pp.options_dict[k].value = v
    out = pp.process(img)[0]
    assert np.array_equal(mod.posted["PPX_lab"], cv2.cvtColor(img, cv2.COLOR_BGR2LAB))
    assert np.array_equal(mod.posted["PPX_hsv_s_channel"], cv2.cvtColor(img, cv2.COLOR_BGR2HSV)[..., 1])
    assert np.array_equal(mod.posted["PPX_grayscale"], cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    ref = oracle_balance(img)
    ref = cv_ops.channel_bias(ref, 2, 20)
    ref = cv_ops.contrast(ref, 1.3)
    ref = cv_ops.brightness(ref, -15)
    ref = cv_ops.ellipse_erode(ref, 2)
    ref = cv_ops.ellipse_dilate(ref, 1)
    ref = cv_ops.resize_ratio(ref, 0.37)
    assert np.array_equal(out, ref)
    # the remaining tuner-gated steps, in the reference's order: blur (110-114) ... rotate (130-135) ... translate (144-149)
    pp2 = Preprocessor(None)
    for k, v in (("PPX_gaussian_blur", True), ("PPX_gaussian_blur_kernel", 2), ("PPX_rotate", 10), ("PPX_resize", True),
                 ("PPX_resize_width", 320), ("PPX_resize_height", 200), ("PPX_translate_x", 12), ("PPX_translate_y", -7)):
        pp2.options_dict[k].value = v
    ref2 = cv2.GaussianBlur(img, (5, 5), 0)
    ref2 = cv2.warpAffine(ref2, cv2.getRotationMatrix2D((ref2.shape[1] / 2, ref2.shape[0] / 2), 10, 1), (ref2.shape[1], ref2.shape[0]),
                          borderMode=cv2.BORDER_REPLICATE)
    ref2 = cv2.resize(ref2, (320, 200))
    ref2 = cv2.warpAffine(ref2, np.float32([[1, 0, 12], [0, 1, -7]]), (ref2.shape[1], ref2.shape[0]))
    assert np.array_equal(pp2.process(img)[0], ref2)
    # Gaussian noise (115-119) sits between blur and erode; numpy's global generator, seeded, is replayed on the device
    pp2.options_dict["PPX_gaussian_noise"].value = 3
    np.random.seed(2024)
    got3 = pp2.process(img)[0]
    after_ours = np.random.get_state()
    np.random.seed(2024)
    ref3 = cv2.GaussianBlur(img, (5, 5), 0)
    noise = np.random.randn(*ref3.shape) * 3
    ref3 = np.clip(ref3 + noise, 0., 255.).astype(np.uint8)
    after_ref = np.random.get_state()
    ref3 = cv2.warpAffine(ref3, cv2.getRotationMatrix2D((ref3.shape[1] / 2, ref3.shape[0] / 2), 10, 1), (ref3.shape[1], ref3.shape[0]),
                          borderMode=cv2.BORDER_REPLICATE)
    ref3 = cv2.resize(ref3, (320, 200))
    ref3 = cv2.warpAffine(ref3, np.float32([[1, 0, 12], [0, 1, -7]]), (ref3.shape[1], ref3.shape[0]))
    assert np.array_equal(got3, ref3)
    assert np.array_equal(after_ours[1], after_ref[1]) and after_ours[2:4] == after_ref[2:4]


def _noise_reference(img, sigma):
    """modules/preprocessor.py:115-119, verbatim."""
    noise = np.random.randn(*img.shape) * sigma
    return np.clip(img + noise, 0., 255.).astype(np.uint8)


@pytest.mark.parametrize("shape,sigma,pre", [((37, 53, 3), 12.5, 0), ((37, 53, 3), 4, 1), ((480, 640, 3), 7, 311),
                                             ((1242, 2208, 3), 20, 0), ((1, 1, 1), 50, 1), ((1, 1, 1), 50, 0),
                                             ((5, 7), 30, 2), ((1080, 1920, 3), 1, 623)])
def test_gaussian_noise_replays_numpy_global_generator(ctx, shape, sigma, pre):
    """Values: stated tolerance <= 1 LSB on at most 2 pixels (device log vs libm log, include/b200vision.h); the
    generator state after the call (key, position, cached flag) is identical, the cached value to 1 ulp, and the
    next draws of numpy agree."""
    img = np.random.default_rng(5).integers(0, 256, shape, dtype=np.uint8)
    np.random.seed(99)
    if pre:
        np.random.randn(pre)
    start = np.random.get_state()
    ref = _noise_reference(img, sigma)
    after_ref = np.random.get_state()
    next_ref = np.random.randn(4)
    np.random.set_state(start)
    got = ctx.download(ctx.add_gaussian_noise(ctx.upload(img), sigma))
    after = np.random.get_state()
    next_got = np.random.randn(4)
    d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
    assert int(d.max()) <= 1 and int((d != 0).sum()) <= 2
    assert np.array_equal(after[1], after_ref[1]) and after[2:4] == after_ref[2:4]
    assert after[4] == pytest.approx(after_ref[4], rel=4e-16, abs=0)
    assert np.allclose(next_got, next_ref, rtol=4e-16, atol=0)
    # an own RandomState instead of the global one; two consecutive calls continue the same stream
    rs_ref, rs = np.random.RandomState(7), np.random.RandomState(7)
    a = np.clip(img + rs_ref.randn(*img.shape) * sigma, 0., 255.).astype(np.uint8)
    b = np.clip(a + rs_ref.randn(*img.shape) * sigma, 0., 255.).astype(np.uint8)
    ga = ctx.add_gaussian_noise(ctx.upload(img), sigma, random_state=rs)
    gb = ctx.download(ctx.add_gaussian_noise(ga, sigma, random_state=rs))
    assert int((gb != b).sum()) <= 2
    assert rs.get_state()[2:4] == rs_ref.get_state()[2:4] and np.array_equal(rs.get_state()[1], rs_ref.get_state()[1])


def reference_bins_post(img):
    """modules/bins.py:11-81 literally (np.int0 spelled np.intp: numpy 2 removed the alias)."""
    hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
    mask = cv2.inRange(hsv, np.array([10, 20, 60]), np.array([30, 100, 255]))
    overlayed = cv2.addWeighted(img, 0.7, cv2.cvtColor(mask, cv2.COLOR_GRAY2BGR), 0.3, 0)
    cleaned = cv_ops.morph_remove_noise(mask, cv_ops.rect_kernel(5))
    valid_rects = []
    for contour in cv_ops.outer_contours(cleaned):
        rect = cv2.minAreaRect(contour)
        (center, (w, h), angle) = rect
        if w * h < 500:
            continue
        if 1.0 <= max(w, h) / min(w, h) <= 3.0:
            valid_rects.append(rect)
    for rect in valid_rects:
        cv2.drawContours(overlayed, [cv2.boxPoints(rect).astype(np.intp)], 0, (0, 255, 0), 4)
    return overlayed, valid_rects, cleaned


def test_drop_in_modules(ctx):
    from cuauv_vision_pipeline_b200.modules import BinDetectorGPU, BuoyLABGPU, ColorBalanceGPU
    img = synth.gen_c5_frame(77, 480, 640)                    # contains one large bin-coloured target
    img[60:200, 60:330] = (131, 164, 180)                    # and a beige box (HSV 20,70,180) that passes bins.py's threshold unbalanced
    mod = BinDetectorGPU(video_sources=["forward"], tuners=[])
    rects = mod.process("forward", img.copy())
    post_ref, rects_ref, cleaned = reference_bins_post(img)
    assert len(rects_ref) >= 1, "the fixture must exercise the rectangle drawing of bins.py:71-74"
    # same accepted rectangles (bins.py:58-69) to the stated minAreaRect tolerance, same posted image
    assert len(rects) == len(rects_ref)
    for got, want in zip(sorted(rects), sorted(rects_ref)):
        assert got[0] == pytest.approx(want[0], abs=1e-3)
        assert sorted(got[1]) == pytest.approx(sorted(want[1]), rel=1e-4, abs=1e-3)
    assert np.array_equal(mod.posted["bins"], post_ref)
    assert mod.pixels.uploads == 1 and mod.pixels.h2d_bytes == img.nbytes, "one H2D per process() call"
    # the vertex arrays handed to minAreaRect are cv2's own (bins.py:27)
    ref_sets = sorted(sorted(map(tuple, c.reshape(-1, 2).tolist())) for c in cv_ops.outer_contours(cleaned))
    got_sets = sorted(sorted(map(tuple, c["points"].reshape(-1, 2).tolist())) for c in mod.contours)
    assert got_sets == ref_sets
    n_ref, _, tab = ccl.label_and_moments(cleaned)
    assert len(mod.blobs) == n_ref and [b["m00"] for b in mod.blobs] == tab["m00"].tolist()

    buoy = BuoyLABGPU(["zed"], thresh_min=150, thresh_max=255)
    img2 = synth.gen_underwater(480, 640, 77)
    res = buoy.process("zed", img2)
    th, cl = cv_ops.buoy_mask(img2, 150, 255)
    assert np.array_equal(buoy.posted["threshed"], th) and np.array_equal(buoy.posted["threshed_cleaned"], cl)
    assert buoy.posted_color_space["threshed"] == "GRAY"
    assert buoy.pixels.uploads == 1, "one upload, one LAB conversion (red_buoy.py:21-34)"
    n_ref, _, tab = ccl.label_and_moments(cl)
    if n_ref:
        i = int(np.argmax(tab["m00"]))
        assert buoy.blob_result["pixel"] == (int(tab["m10"][i] / tab["m00"][i]), int(tab["m01"][i] / tab["m00"][i]))
        assert buoy.blob_result["area"] == float(tab["m00"][i])
    ref_contours = cv_ops.outer_contours(th)                      # red_buoy.py:38 (un-cleaned mask)
    if ref_contours:
        best = max(ref_contours, key=cv_ops.contour_area)
        assert res["pixel"] == cv_ops.contour_centroid(best)      # red_buoy.py:43-45
        assert res["area"] == cv_ops.contour_area(best)
    else:
        assert res is None
    cbm = ColorBalanceGPU(["forward"])
    assert np.array_equal(cbm.process("forward", img2), oracle_balance(img2))
    assert np.array_equal(cbm.posted["orig"], img2) and np.array_equal(cbm.posted["balanced"], oracle_balance(img2))


HUE_TABLE_BOUNDS = [((10, 20, 60), (30, 100, 255)),      # modules/bins.py:14-15
                    ((0, 40, 60), (179, 255, 255)),
                    ((0, 0, 0), (5, 255, 255)),           # hue interval touching 0
                    ((170, 0, 0), (179, 255, 255)),       # ... and 179 (round trip may wrap)
                    ((0, 0, 0), (179, 30, 40)),           # dark / grey pixels: hue is unstable there
                    ((50, 0, 0), (40, 255, 255)),         # empty range
                    ((0, 0, 0), (255, 255, 255)),
                    ((90, 100, 100), (90, 200, 200))]


@pytest.mark.parametrize("lo,hi", HUE_TABLE_BOUNDS)
def test_stage_mask_only_hue_interval_table(ctx, lo, hi):
    """Mask-only HSV threshold of a balanced frame (the shared-memory hue-interval table instead of the
    HSV -> BGR -> HSV round trip) == balance() -> cv2.cvtColor(BGR2HSV) -> cv2.inRange -> OPEN."""
    frames = np.stack([synth.gen_underwater(480, 640, 90 + s) for s in range(3)] + [synth.gen_random_bgr(480, 640, 5)])
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=lo, hi=hi)
    mask = ctx.download(ctx.stage(desc, ctx.upload(frames), want=("mask",))["mask"])
    desc_m = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=lo, hi=hi, morph=[("open", 5, 5, 1)], label=True)
    out = ctx.stage(desc_m, ctx.upload(frames), want=("mask", "labels", "blobs"), max_blobs=4096)
    opened, lab = ctx.download(out["mask"]), ctx.download(out["labels"])
    for i in range(frames.shape[0]):
        hsv_ref = cv2.cvtColor(oracle_balance(frames[i]), cv2.COLOR_BGR2HSV)
        m_ref = cv2.inRange(hsv_ref, np.array(lo), np.array(hi))
        assert np.array_equal(mask[i], m_ref)
        o_ref = cv2.morphologyEx(m_ref, cv2.MORPH_OPEN, cv_ops.rect_kernel(5))
        assert np.array_equal(opened[i], o_ref)
        assert np.array_equal(lab[i], ccl.label_and_moments(o_ref)[1])


def test_stage_mask_only_many_bounds_reuse_and_evict_tables(ctx):
    """More distinct bounds than table slots, revisited: cached, evicted and rebuilt tables all agree
    with the full-output pass (which does the round trip arithmetically)."""
    frames = np.stack([synth.gen_underwater(352, 640, 120 + s) for s in range(2)])
    dev = ctx.upload(frames)
    rng = np.random.default_rng(11)
    bounds = []
    for _ in range(6):
        a, b = rng.integers(0, 180, 2), rng.integers(0, 256, (2, 2))
        bounds.append(((int(min(a)), int(b[:, 0].min()), int(b[:, 1].min())), (int(max(a)), int(b[:, 0].max()), int(b[:, 1].max()))))
    for lo, hi in bounds + bounds[:3]:
        desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=lo, hi=hi)
        fast = ctx.download(ctx.stage(desc, dev, want=("mask",))["mask"])
        full = ctx.download(ctx.stage(desc, dev, want=("mask", "converted"))["mask"])
        assert np.array_equal(fast, full), (lo, hi)


@pytest.mark.parametrize("kind,shape,seed,flags", [("underwater", (480, 640), 7, {}), ("random", (480, 640), 4, dict(hsv_contrast_correct=False)),
                                                   ("underwater", (1242, 2208), 6, dict(equalize_rgb=False, rgb_extrema_clipping=False)),
                                                   ("underwater", (479, 641), 9, dict(rgb_contrast_correct=True)),
                                                   ("underwater", (480, 640), 11, dict(horizontal_blocks=4, vertical_blocks=2))])
def test_balance_hsi_branch(ctx, kind, shape, seed, flags):
    """color_balance.cpp:702-774 (P2).  Stated tolerance <= 1 LSB (CUDA's double-precision acos / cos vs glibc's);
    frames of >= 128 k pixels, where the reference's quickselect is deterministic.  The oracle warms the reference's
    racy memo table first (oracle/ref_balance.py, DESIGN.md finding 9b); a mismatch reports which side moved."""
    img = synth.gen_underwater(shape[0], shape[1], seed) if kind == "underwater" else synth.gen_random_bgr(shape[0], shape[1], seed)
    want = oracle_balance(img, hsi_contrast_correct=True, **flags)
    got = ctx.download(ctx.color_balance(ctx.upload(img), hsi_contrast_correct=True, **flags))
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16))
    if int(diff.max()) > 1:   # say which side moved: both are recomputed
        d = np.argwhere(np.any(diff > 1, axis=2))
        want2 = oracle_balance(img, hsi_contrast_correct=True, **flags)
        got2 = ctx.download(ctx.color_balance(ctx.upload(img), hsi_contrast_correct=True, **flags))
        raise AssertionError("HSI branch: %d pixels off by more than 1 (max %d), rows %d..%d, cols %d..%d; oracle repeatable: %s, "
                             "device repeatable: %s, repeated device vs repeated oracle max diff %d"
                             % (len(d), int(diff.max()), d[:, 0].min(), d[:, 0].max(), d[:, 1].min(), d[:, 1].max(),
                                np.array_equal(want, want2), np.array_equal(got, got2),
                                int(np.abs(got2.astype(np.int16) - want2.astype(np.int16)).max())))
    assert int(diff.max()) <= 1
    assert int((diff != 0).sum()) <= 8, int((diff != 0).sum())
    # the same through the fused stage with a conversion behind it
    desc = ctx.make_stage(balance=dict(hsi_contrast_correct=True, **flags), cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255))
    out = ctx.stage(desc, ctx.upload(img[None]), want=("balanced", "mask"))
    assert np.array_equal(ctx.download(out["balanced"])[0], got)
    assert np.array_equal(ctx.download(out["mask"])[0], cv2.inRange(cv2.cvtColor(got, cv2.COLOR_BGR2HSV), np.array([0, 40, 60]), np.array([179, 255, 255])))


def test_two_module_threads_with_their_own_contexts(ctx):
    """core/base.py:701-703: every module runs process() on its own worker thread, never the main thread; two modules
    in one process (or two processes on one GPU) each own a context.  Both threads hammer the fused stage at once
    (different descriptions, different frame sizes) and every result must equal the single-threaded one."""
    import threading
    import cuauv_vision_pipeline_b200 as bv
    jobs = [(synth.gen_underwater(480, 640, 301), dict(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[("open", 5, 5, 1)], label=True)),
            (synth.gen_underwater(360, 512, 302), dict(balance={}, cvt="bgr2lab", lo=(0, 130, 0), hi=(255, 255, 255), morph=[("close", 3, 3, 1)], label=True))]
    want = []
    for img, kw in jobs:
        out = ctx.stage_host(ctx.make_stage(**kw), img[None], want=("converted", "mask", "labels"))
        want.append({k: out[k].copy() for k in ("converted", "mask", "labels")})
    errors = []

    def worker(i):
        try:
            c = bv.Context(0)
            img, kw = jobs[i]
            desc = c.make_stage(**kw)
            for _ in range(25):
                out = c.stage_host(desc, img[None], want=("converted", "mask", "labels"))
                for k in ("converted", "mask", "labels"):
                    if not np.array_equal(out[k], want[i][k]):
                        errors.append((i, k))
                        return
            c.close()
        except Exception as e:  # noqa: BLE001
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in (0, 1, 0, 1)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


@pytest.mark.parametrize("batch,chunk_mb,side", [(7, 1, 3), (9, 1, 4), (5, 2, 2)])
def test_stage_many_chunks_on_side_streams(ctx, batch, chunk_mb, side):
    """Batches are cut into L2-sized chunks that run on side streams, with the morphology chain launched per chunk on the
    chunk's stream: uneven chunk counts / sizes must give exactly the per-frame results (mask-only fast path and the
    full-output path)."""
    frames = np.stack([synth.gen_underwater(352, 512, 700 + i) for i in range(batch)])      # 0.54 MB per frame
    dev = ctx.upload(frames)
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[("open", 5, 5, 1)], label=True)
    try:
        ctx.set_option("l2_chunk_mb", chunk_mb)
        ctx.set_option("side_streams", side)
        fast = ctx.stage(desc, dev, want=("mask", "labels", "blobs"), max_blobs=2048)
        full = ctx.stage(desc, dev, want=("balanced", "converted", "mask", "labels"), max_blobs=2048)
        fast_mask, fast_lab = ctx.download(fast["mask"]), ctx.download(fast["labels"])
        bal, full_mask, full_lab = ctx.download(full["balanced"]), ctx.download(full["mask"]), ctx.download(full["labels"])
    finally:
        ctx.set_option("l2_chunk_mb", 0)
        ctx.set_option("side_streams", 0)
    for i in range(batch):
        b_ref = oracle_balance(frames[i])
        assert np.array_equal(bal[i], b_ref), i
        m_ref = cv2.morphologyEx(cv2.inRange(cv2.cvtColor(b_ref, cv2.COLOR_BGR2HSV), np.array([0, 40, 60]), np.array([179, 255, 255])),
                                 cv2.MORPH_OPEN, cv_ops.rect_kernel(5))
        assert np.array_equal(fast_mask[i], m_ref) and np.array_equal(full_mask[i], m_ref), i
        lab_ref = ccl.label_and_moments(m_ref)[1]
        assert np.array_equal(fast_lab[i], lab_ref) and np.array_equal(full_lab[i], lab_ref), i


@pytest.mark.parametrize("shape", [(270, 496), (479, 641), (64, 32), (33, 64)])
def test_stage_mask_only_shapes_outside_the_hue_table_path(ctx, shape):
    """Widths that are not a multiple of 32 (cv2's scalar HSV2BGR row tail rounds differently) or odd sizes take the
    arithmetic pass; tiny frames take the table path with a single group per row: all equal the cv2 pipeline."""
    frames = np.stack([synth.gen_underwater(shape[0], shape[1], 40 + s) for s in range(2)])
    lo, hi = (10, 20, 60), (30, 100, 255)
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=lo, hi=hi, morph=[("open", 3, 3, 1)], label=True)
    out = ctx.stage(desc, ctx.upload(frames), want=("mask", "labels", "blobs"), max_blobs=1024)
    mask, lab = ctx.download(out["mask"]), ctx.download(out["labels"])
    for i in range(2):
        hsv_ref = cv2.cvtColor(oracle_balance(frames[i]), cv2.COLOR_BGR2HSV)
        m_ref = cv2.morphologyEx(cv2.inRange(hsv_ref, np.array(lo), np.array(hi)), cv2.MORPH_OPEN, cv_ops.rect_kernel(3))
        assert np.array_equal(mask[i], m_ref)
        assert np.array_equal(lab[i], ccl.label_and_moments(m_ref)[1])


@pytest.mark.parametrize("option,values", [("final_sv_tables", (1, 2)), ("morph_warps", (1, 3)), ("no_rcp_tables", (1,)),
                                           ("fast_tables", (1,)), ("morph_variant", (1, 2)), ("no_hue_table", (1,))])
def test_tuning_options_do_not_change_results(ctx, option, values):
    """Every A-B knob of the library (bv_set_option / BV_* environment variables) selects another implementation of the
    same arithmetic: outputs are identical to the default's, on the stages the knobs act on."""
    frames = np.stack([synth.gen_underwater(416, 672, 900 + i) for i in range(6)])
    dev = ctx.upload(frames)
    stages = [(ctx.make_stage(balance={}, cvt="bgr2lab"), ("converted",)),
              (ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[("open", 5, 5, 1)], label=True),
               ("mask", "labels")),
              (ctx.make_stage(cvt="bgr2lab", lo=(0, 120, 0), hi=(255, 255, 255), morph=[("open", 3, 3, 1), ("close", 5, 5, 1)]),
               ("mask",))]

    def run():
        res = []
        for desc, want in stages:
            out = ctx.stage(desc, dev, want=want, max_blobs=2048)
            res.extend(ctx.download(out[k]).copy() for k in want)
        return res
    ref = run()
    try:
        for v in values:
            ctx.set_option(option, v)
            got = run()
            for a, b in zip(got, ref):
                assert np.array_equal(a, b), (option, v)
    finally:
        ctx.set_option(option, 0)
