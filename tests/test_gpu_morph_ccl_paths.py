"""GPU: binary morphology of the fused stage, grey morphology (bv_morph) and the labelling behind them on every path
they take (oracle/morph_cases.py), against cv2 with 0 differing bytes and against oracle/ccl.py exactly.

Each stage case names the kernel family it was written for (tests/test_morph_cases.py checks the prediction on the
host); here the profiler confirms that family ran.  BV_LAUNCH names a kernel by its source token, so the profiler tells
the roll, chain and step families apart but not the roll instances: those are covered by the case table.  Outputs go
through the C ABI with guard bytes around them.  Failures are collected per group and listed with the first differing
byte."""
import cv2
import numpy as np
import pytest
import torch

from oracle import ccl, morph_cases as mc

pytestmark = pytest.mark.gpu

GUARD = 64
FAMILIES = ("morph_roll_kernel", "morph_chain_kernel", "morph_bits_kernel")


def by_group(cases):
    out = {}
    for c in cases:
        out.setdefault(c.group, []).append(c)
    return out


STAGE = by_group(mc.stage_cases())
GREY = by_group(mc.grey_cases())
LABEL = mc.label_cases()


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


def launches_of(kernels, family):
    return sum(n for k, n in kernels.items() if family in k)


def difference(got, want):
    if got.shape != want.shape:
        return "shape %s, want %s" % (got.shape, want.shape)
    bad = np.argwhere(got != want)
    if not bad.size:
        return None
    i = tuple(int(v) for v in bad[0])
    return "%d differing values, first at %s: got %d, want %d" % (len(bad), i, got[i], want[i])


def report(failures):
    if failures:
        pytest.fail("%d failing cases:\n  %s" % (len(failures), "\n  ".join(failures[:20])))


def placed(ctx, nbytes, off, fill=0xA5):
    """A flat device buffer whose byte `GUARD + off` lies `off` bytes past a 16-byte boundary; (buffer, start)."""
    with torch.cuda.stream(ctx.torch_stream):
        buf = ctx.empty((GUARD + off + nbytes + GUARD,))
        buf.fill_(fill)
    assert (buf.data_ptr() + GUARD) % 16 == 0
    return buf, GUARD + off


def guards_intact(buf, start, nbytes, fill=0xA5):
    out = buf.cpu().numpy()
    return not (out[:start] != fill).any() and not (out[start + nbytes:] != fill).any()


def check_blobs(tab, n, want_n, want_tab, cap):
    """First differing moment / box of a downloaded blob table against the oracle's."""
    if n != want_n:
        return "n_blobs %d, want %d" % (n, want_n)
    k = min(n, cap)
    for key in ccl.MOMENT_KEYS + ("x0", "y0", "x1", "y1"):
        got = tab[key][:k].astype(np.int64)
        if not np.array_equal(got, np.asarray(want_tab[key][:k], np.int64)):
            i = int(np.argwhere(got != want_tab[key][:k])[0][0])
            return "%s of blob %d: got %d, want %d" % (key, i + 1, got[i], want_tab[key][i])
    return None


# ---------------------------------------------------------------------------------------------------------------------
# the fused stage: threshold -> bits -> morphology -> mask / labels / table
# ---------------------------------------------------------------------------------------------------------------------
OUTPUTS = (("mask",), ("labels", "blobs"), ("mask", "labels", "blobs"))


def run_stage_case(ctx, c, outputs, sm_count):
    ffi, L = lib()
    b, h, w = c.shape
    masks = c.masks()
    frames = np.repeat(masks[..., None], 3, axis=3)
    desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=c.steps, label="labels" in outputs)
    src = ctx.upload(frames)
    npx = b * h * w
    mbuf, m0 = placed(ctx, npx, c.mask_off)
    labels = ctx.empty((b, h, w), torch.int32) if "labels" in outputs else None
    cap = 4096 if b <= 16 else 256
    blobs = ctx.empty((b, cap, ccl_dtype().itemsize)) if "blobs" in outputs else None
    nb = ctx.empty((b,), torch.int32)
    ctx.set_option("morph_variant", c.variant)
    ctx.set_option("morph_warps", c.warps)
    try:
        rc, kernels = profiled(ctx, lambda: L.bv_stage(
            ctx.handle, desc, ffi.cast("uint8_t *", src.data_ptr()), b, h, w, ffi.NULL, ffi.NULL,
            ffi.cast("uint8_t *", mbuf.data_ptr() + m0) if "mask" in outputs else ffi.NULL,
            ffi.cast("int32_t *", labels.data_ptr()) if labels is not None else ffi.NULL,
            ffi.cast("bv_blob *", blobs.data_ptr()) if blobs is not None else ffi.NULL, cap if blobs is not None else 0,
            ffi.cast("int32_t *", nb.data_ptr())))
    finally:
        ctx.set_option("morph_variant", 0)
        ctx.set_option("morph_warps", 0)
    tag = "%s (%s, %s)" % (c.name, c.path, "+".join(outputs))
    if rc != 0:
        return "%s: status %d: %s" % (tag, rc, ffi.string(L.bv_last_error()).decode())
    if not guards_intact(mbuf, m0, npx):
        return "%s: wrote outside the mask" % tag
    got_mask = mbuf[m0:m0 + npx].cpu().numpy().reshape(b, h, w)
    lab = ctx.download(labels) if labels is not None else None
    n_dev = ctx.download(nb)
    tables = ctx.download(blobs) if blobs is not None else None
    for f in range(b):
        want = mc.cv2_steps(masks[f], c.steps)
        if "mask" in outputs:
            d = difference(got_mask[f], want)
            if d:
                return "%s frame %d: %s" % (tag, f, d)
        if "labels" in outputs:
            n_ref, lab_ref, tab = ccl.label_and_moments(want)
            d = difference(lab[f], lab_ref)
            if d:
                return "%s frame %d labels: %s" % (tag, f, d)
            t = tables[f, :min(n_ref, cap)].copy().view(ccl_dtype()).reshape(-1)
            d = check_blobs(t, int(n_dev[f]), n_ref, tab, cap)
            if d:
                return "%s frame %d: %s" % (tag, f, d)
    family = c.predicted(sm_count).family
    ran = {fam for fam in FAMILIES if launches_of(kernels, fam)}
    if ran != ({family} if family else set()):
        return "%s: ran %s, want %s" % (tag, sorted(ran), family)
    return None


def ccl_dtype():
    from cuauv_vision_pipeline_b200.runtime import BLOB_DTYPE
    return BLOB_DTYPE


@pytest.mark.parametrize("group", sorted(STAGE))
def test_stage_morphology_paths(ctx, group):
    """0 differing bytes against cv2.morphologyEx for every case; labels, moments and boxes exact when the morphed bits
    feed the labelling; the predicted family ran.  The output set rotates over mask only, labels + table only, both."""
    sm = torch.cuda.get_device_properties(ctx.device).multi_processor_count
    failures = []
    for i, c in enumerate(STAGE[group]):
        for outputs in (OUTPUTS[i % 3],) if c.shape[0] * c.shape[1] * c.shape[2] > 1 << 21 else OUTPUTS:
            f = run_stage_case(ctx, c, outputs, sm)
            if f:
                failures.append(f)
    report(failures)


@pytest.mark.parametrize("shape", [(2, 131, 173), (1, 75, 2208), (3, 40, 4096), (1, 3, 65)])
def test_every_variant_and_warp_count_gives_the_default_bytes(ctx, shape):
    """BV_OPT_MORPH_VARIANT x BV_OPT_MORPH_WARPS: the same mask bytes as the default for the chains the modules use."""
    b, h, w = shape
    masks = mc.edge_pixels(mc.make_mask("random0.6", shape, h + w))
    src = ctx.upload(np.repeat(masks[..., None], 3, axis=3))
    for steps in ([("open", 5, 5, 1)], [("open", 5, 5, 1), ("close", 5, 5, 1)], [("erode", 3, 3, 1)], [("close", 3, 3, 1)]):
        desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=steps)
        default = ctx.download(ctx.stage(desc, src)["mask"])
        for f in range(b):
            assert difference(default[f], mc.cv2_steps(masks[f], steps)) is None, (steps, f)
        try:
            for variant in (0, 1):
                for warps in (0, 1, 2, 3, 8, 64):
                    ctx.set_option("morph_variant", variant)
                    ctx.set_option("morph_warps", warps)
                    got = ctx.download(ctx.stage(desc, src)["mask"])
                    assert difference(got, default) is None, (steps, variant, warps)
        finally:
            ctx.set_option("morph_variant", 0)
            ctx.set_option("morph_warps", 0)


def test_chain_shared_memory_opt_in_across_calls_and_contexts(ctx):
    """The chain's opt-in above 48 KiB is an attribute of the kernel, shared by every context of the process: a smaller
    call after a larger one, and a second context's smaller call between two larger calls of the first, all run."""
    import cuauv_vision_pipeline_b200 as bv
    big, small = (1, 40, 12800), (1, 70, 6145)
    data = {s: mc.make_mask("blobs", s, s[2]) for s in (big, small)}
    steps = [("open", 5, 5, 1)]

    def run(c, s):
        desc = c.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=steps)
        got = c.download(c.stage(desc, c.upload(np.repeat(data[s][..., None], 3, axis=3)))["mask"])
        assert difference(got[0], mc.cv2_steps(data[s][0], steps)) is None, s
    other = bv.Context(0)
    try:
        for c in (ctx, other):
            c.set_option("morph_variant", 1)
        run(ctx, big)
        run(ctx, small)
        run(other, small)
        run(ctx, big)
        run(other, big)
    finally:
        ctx.set_option("morph_variant", 0)
        other.close()


def test_gradient_with_large_extents_runs_through_the_stage(ctx):
    """A binary GRADIENT whose extent passes 31 px (64 x 3; 3 x 3 at 32 iterations) used to be refused at run time."""
    m = mc.make_mask("bars", (1, 120, 300), 5)
    src = ctx.upload(np.repeat(m[..., None], 3, axis=3))
    for step in (("gradient", 64, 3, 1), ("gradient", 3, 3, 32)):
        desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=[step])
        got = ctx.download(ctx.stage(desc, src)["mask"])
        assert difference(got[0], mc.cv2_steps(m[0], [step])) is None, step


def test_gradient_with_zero_iterations_is_empty_through_the_stage(ctx):
    m = mc.make_mask("random0.5", (2, 50, 96), 6)
    src = ctx.upload(np.repeat(m[..., None], 3, axis=3))
    desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=[("gradient", 5, 5, 0)], label=True)
    out = ctx.stage(desc, src, want=("mask", "labels"))
    assert not ctx.download(out["mask"]).any() and not ctx.download(out["labels"]).any()
    assert not ctx.download(out["n_blobs"]).any()


# ---------------------------------------------------------------------------------------------------------------------
# grey morphology: bv_morph
# ---------------------------------------------------------------------------------------------------------------------
def run_grey_case(ctx, c):
    ffi, L = lib()
    b, h, w, cn = c.shape
    img = c.image()
    n = img.size
    kernel = np.ascontiguousarray(c.se != 0, dtype=np.uint8)
    kh, kw = kernel.shape
    op = {"erode": L.BV_MORPH_ERODE, "dilate": L.BV_MORPH_DILATE, "open": L.BV_MORPH_OPEN, "close": L.BV_MORPH_CLOSE,
          "gradient": L.BV_MORPH_GRADIENT}[c.op]
    src_buf, s0 = placed(ctx, n, 0)
    with torch.cuda.stream(ctx.torch_stream):
        src_buf[s0:s0 + n].copy_(ctx.upload(img.reshape(-1)))
    if c.in_place:
        dst_buf, d0 = src_buf, s0
    else:
        dst_buf, d0 = placed(ctx, n, c.dst_off)
    ptr = lambda t, i: ffi.cast("uint8_t *", t.data_ptr() + i)     # noqa: E731
    rc, kernels = profiled(ctx, lambda: L.bv_morph(ctx.handle, ptr(src_buf, s0), ptr(dst_buf, d0), b, h, w, cn, op,
                                                   ffi.from_buffer("uint8_t[]", kernel), kw, kh, c.iterations))
    p = c.predicted()
    tag = "%s (%s)" % (c.name, p)
    if rc != 0:
        return "%s: status %d: %s" % (tag, rc, ffi.string(L.bv_last_error()).decode())
    if not guards_intact(dst_buf, d0, n):
        return "%s: wrote outside the destination" % tag
    got = dst_buf[d0:d0 + n].cpu().numpy().reshape(c.shape)
    want = c.want(img)
    for f in range(b):
        d = difference(got[f], want[f])
        if d:
            return "%s frame %d: %s" % (tag, f, d)
    if p.kind in ("rect", "runs") and launches_of(kernels, "morph_grey_kernel") != p.launches:
        return "%s: %d grey launches, want %d (%s)" % (tag, launches_of(kernels, "morph_grey_kernel"), p.launches, kernels)
    if p.kind in ("copy", "zero") and kernels:
        return "%s: ran %s" % (tag, kernels)
    return None


@pytest.mark.parametrize("group", sorted(GREY))
def test_grey_morphology_paths(ctx, group):
    report([f for f in (run_grey_case(ctx, c) for c in GREY[group]) if f])


def test_grey_morphology_limits(ctx):
    """257 runs are refused before anything is launched; the wrapper takes 4-D batches."""
    from cuauv_vision_pipeline_b200 import BVError
    img = ctx.upload(mc.make_mask("random0.5", (1, 30, 80), 1)[0])
    se = np.zeros((16, 32), np.uint8)
    se[:, ::2] = 1                                  # 16 rows of 16 runs: 256
    ctx.morph(img, "dilate", se)
    se2 = np.zeros((17, 32), np.uint8)
    se2[:, ::2] = 1                                 # 272
    n0 = ctx.launches
    with pytest.raises(BVError):
        ctx.morph(img, "dilate", se2)
    assert ctx.launches == n0
    batch = mc.make_mask("random0.5", (3, 20, 30), 2)[..., None]
    got = ctx.download(ctx.morph(ctx.upload(batch), "close", np.ones((3, 5), np.uint8), iterations=2))
    for f in range(3):
        assert difference(got[f, ..., 0], cv2.morphologyEx(batch[f, ..., 0], cv2.MORPH_CLOSE, np.ones((3, 5), np.uint8),
                                                           iterations=2)) is None


# ---------------------------------------------------------------------------------------------------------------------
# labelling
# ---------------------------------------------------------------------------------------------------------------------
def check_label_case(ctx, masks, cap, want_labels=True, want_table=True):
    b = masks.shape[0]
    labels, blobs, nb = ctx.label(ctx.upload(masks), max_blobs=cap if want_table else 0, want_labels=want_labels)
    n = ctx.download(nb)
    lab = ctx.download(labels) if want_labels else None
    raw = ctx.download(blobs) if want_table and cap else None
    for f in range(b):
        n_ref, lab_ref, tab = ccl.label_and_moments(masks[f])
        if int(n[f]) != n_ref:
            return "frame %d: n_blobs %d, want %d" % (f, n[f], n_ref)
        if want_labels:
            d = difference(lab[f], lab_ref)
            if d:
                return "frame %d labels: %s" % (f, d)
        if raw is not None:
            t = raw[f, :min(n_ref, cap)].copy().view(ccl_dtype()).reshape(-1)
            d = check_blobs(t, int(n[f]), n_ref, tab, cap)
            if d:
                return "frame %d: %s" % (f, d)
    return None


@pytest.mark.parametrize("case", LABEL, ids=lambda c: c.name)
def test_labelling_paths(ctx, case):
    """Labels, n_blobs and all ten moments plus boxes exact for every frame; labels without a table and a table without
    labels as well."""
    cap = case.max_blobs if case.max_blobs is not None else 1 << 15
    for want_labels, want_table in ((True, True), (True, False), (False, True)):
        d = check_label_case(ctx, case.masks, cap, want_labels, want_table)
        assert d is None, (want_labels, want_table, d)


def test_labels_and_table_separately_through_the_stage(ctx):
    masks = np.stack([mc.make_mask("random0.3", (1, 90, 161), s)[0] for s in (1, 2, 3)])
    masks[1] = 0
    src = ctx.upload(np.repeat(masks[..., None], 3, axis=3))
    steps = [("close", 3, 3, 1)]
    desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=steps, label=True)
    for want, cap in ((("labels",), 0), (("blobs",), 40), (("blobs",), 1), (("labels", "blobs"), 0)):
        out = ctx.stage(desc, src, want=want, max_blobs=cap)
        n = ctx.download(out["n_blobs"])
        for f in range(3):
            n_ref, lab_ref, tab = ccl.label_and_moments(mc.cv2_steps(masks[f], steps))
            assert int(n[f]) == n_ref, (want, cap, f)
            if "labels" in want:
                assert difference(ctx.download(out["labels"])[f], lab_ref) is None
            if "blobs" in want and cap:
                t = ctx.download(out["blobs"])[f, :min(n_ref, cap)].copy().view(ccl_dtype()).reshape(-1)
                assert check_blobs(t, int(n[f]), n_ref, tab, cap) is None, (want, cap, f)


@pytest.mark.parametrize("transpose", [False, True], ids=["row", "column"])
def test_moments_at_the_int64_limit(ctx, transpose):
    """The widest fully set row (m30 = (W (W - 1) / 2)^2 <= 2^63 - 1) and the tallest fully set column (m03): every
    moment equals the Python-int closed form, one more pixel would overflow."""
    w = mc.m30_limit_width()
    m = np.full((1, 1, w), 255, np.uint8)
    if transpose:
        m = np.ascontiguousarray(m.transpose(0, 2, 1))
    labels, blobs, nb = ctx.label(ctx.upload(m), max_blobs=2)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    assert int(n[0]) == 1
    t = tables[0][0]
    want = mc.run_moment_sums(0, w - 1, 0)
    if transpose:     # swap the roles of x and y
        want = {k[0] + k[2] + k[1]: v for k, v in want.items()}
    for key in ccl.MOMENT_KEYS:
        assert int(t[key]) == want[key], key
    assert (int(t["x0"]), int(t["y0"]), int(t["x1"]), int(t["y1"])) == ((0, 0, 0, w - 1) if transpose else (0, 0, w - 1, 0))
    lab = ctx.download(labels)
    assert lab.min() == 1 and lab.max() == 1
