"""bv_contour_shapes against cv2 4.13.0 and oracle/contour_shapes.py, on the masks of tests/test_gpu_find_contours.py:
records are matched to cv2's borders by vertex list (oracle/contour_tree.py).  Exact: arc_length, hull, approx,
approx_convex; rectangles within _same_rectangle_or_proven_tie; circles within 2e-3 px of cv2."""
import cv2
import numpy as np
import pytest
import torch

import cuauv_vision_pipeline_b200 as bv
from cuauv_vision_pipeline_b200 import feature
from cuauv_vision_pipeline_b200.runtime import CONTOUR_DTYPE, SHAPE_DTYPE, RRECT_DTYPE
from oracle import contour_shapes as cs
from oracle import contour_tree as ct
from oracle import synth
from test_contour_shapes_oracle import STROKES
from test_gpu_find_contours import GENERATORS, SPECIAL
from test_gpu_morph_ccl import _same_rectangle_or_proven_tie

pytestmark = pytest.mark.gpu

EPS = [(0.0, 0.0), (0.5, 0.0), (1.0, 0.0), (3.0, 0.0), (1e9, 0.0), (0.0, 0.005), (0.0, 0.02), (0.0, 0.1)]


def _shapes(ctx, masks, mode, method, eps=(0.0, 0.02), max_contours=None, max_points=None):
    masks = np.ascontiguousarray(masks)
    b, h, w = masks.shape
    if max_contours is None:
        max_contours = 64 + max(len(ct.regions(m)["outer_start"]) + len(ct.regions(m)["hole_start"]) for m in masks)
    max_points = max_points or 64 + 4 * h * w
    table, hier, nc, pts, npts = ctx.find_contours(ctx.upload(masks), mode, method, max_contours, max_points)
    shapes, hull, approx = ctx.contour_shapes(table, nc, pts, method, *eps)
    return (ctx.download(table).view(CONTOUR_DTYPE).reshape(b, -1), ctx.download(nc), ctx.download(pts),
            ctx.download(shapes).view(SHAPE_DTYPE).reshape(b, -1), ctx.download(hull), ctx.download(approx))


def _check_record(c, s, hull, approx, eps, outer_rect=None):
    assert s["valid"] == 1
    arc = cv2.arcLength(c, True)
    assert s["arc_length"] == arc
    assert np.array_equal(hull, cs.convex_hull(c))
    want_hull = cv2.convexHull(c)
    k = [tuple(v) for v in want_hull.reshape(-1, 2)].index(tuple(hull[0, 0]))
    assert np.array_equal(np.roll(want_hull, -k, axis=0), hull)
    e = eps[0] + eps[1] * arc
    assert np.array_equal(approx, cs.approx_poly_dp(c, e))
    assert np.array_equal(approx, cv2.approxPolyDP(c, e, True))
    assert bool(s["approx_convex"]) == cv2.isContourConvex(approx)
    (wx, wy), wr = cv2.minEnclosingCircle(c)
    assert abs(s["circle_cx"] - wx) <= 2e-3 and abs(s["circle_cy"] - wy) <= 2e-3 and abs(s["circle_r"] - wr) <= 2e-3
    p = c.reshape(-1, 2).astype(np.float64)
    assert (np.hypot(p[:, 0] - s["circle_cx"], p[:, 1] - s["circle_cy"]) <= float(s["circle_r"])).all()
    r = s["rect"]
    mine = ((float(r["cx"]), float(r["cy"])), (float(r["width"]), float(r["height"])), float(r["angle"]))
    assert r["valid"] == 1 and _same_rectangle_or_proven_tie(c.reshape(-1, 2), cv2.minAreaRect(c), mine, 1e-3)


def _check_all(ctx, masks, modes=("list", "ccomp", "tree"), methods=("none", "simple"), eps_set=EPS[:1] + EPS[6:7]):
    masks = np.ascontiguousarray(masks)
    for mode in modes:
        for method in methods:
            for eps in eps_set:
                table, nc, pts, shapes, hull, approx = _shapes(ctx, masks, mode, method, eps)
                for f, m in enumerate(masks):
                    canon = ct.canonical(m, mode, method)
                    n = canon["n_outer"] + canon["n_holes"]
                    assert int(nc[f].sum()) == n
                    for r in range(n):
                        rec, s = table[f, r], shapes[f, r]
                        off = int(rec["point_offset"])
                        cnt = int(rec["n_points"] if method == "none" else rec["n_simple"])
                        c = canon["contours"][r]
                        assert np.array_equal(pts[f, off:off + cnt].reshape(-1, 1, 2), c)
                        _check_record(c, s, hull[f, off:off + int(s["n_hull"])].reshape(-1, 1, 2),
                                      approx[f, off:off + int(s["n_approx"])].reshape(-1, 1, 2), eps)
                    assert (shapes[f, n:]["valid"] == 0).all()


@pytest.mark.parametrize("name,gen", GENERATORS + SPECIAL, ids=[n for n, _ in GENERATORS + SPECIAL])
def test_masks_of_find_contours(ctx, name, gen):
    _check_all(ctx, gen()[None])


def test_every_epsilon(ctx):
    m = synth.mask_rings(101, 131, step=4) | synth.mask_random(101, 131, 15, 0.05)
    _check_all(ctx, m[None], modes=("tree",), eps_set=EPS)


def test_pixels_lines_and_two_point_contours(ctx):
    m = np.zeros((40, 60), np.uint8)
    m[3, 3] = m[3, 10] = m[20, 50] = 255                                    # single pixels
    m[10, 20:22] = 255                                                      # two-pixel contours
    m[30, 5] = m[31, 6] = 255
    cv2.line(m, (30, 2), (55, 15), 255, 1)                                  # 1-px lines
    cv2.line(m, (5, 38), (40, 38), 255, 1)
    cv2.line(m, (58, 5), (58, 36), 255, 1)
    _check_all(ctx, m[None], eps_set=EPS)


def test_thick_strokes_and_hooks(ctx):
    """Borders whose points project past the ends of the Douglas-Peucker chords, in one batch."""
    _check_all(ctx, np.stack(STROKES[:96]), modes=("tree",), eps_set=EPS)


def test_outer_table_takes_simple_only(ctx):
    m = np.ascontiguousarray(synth.mask_random(40, 50, 3, 0.5))
    table, nb, pts, _ = ctx.outer_contours(ctx.upload(m), max_contours=256, max_points=4096)
    with pytest.raises(bv.BVError):
        ctx.contour_shapes(table, nb, pts, "none")


def test_feature_external_shapes_grow_the_buffers(ctx):
    m = np.ascontiguousarray(synth.mask_rings(101, 131, step=4) | synth.mask_random(101, 131, 15, 0.05))
    got, _ = feature.find_contours(m, "external", "simple", max_contours=2, max_points=8, shapes=True)
    ref, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    assert len(got) == len(ref) > 2
    for c in got:
        assert c["points"] is not None and np.array_equal(c["hull"], cs.convex_hull(c["points"]))
        assert np.array_equal(c["approx"], cv2.approxPolyDP(c["points"], 0.0, True))


def test_4k_border_takes_the_fallback(ctx):
    m = np.zeros((2160, 3840), np.uint8)
    cv2.circle(m, (1920, 1080), 1000, 255, -1)
    cv2.circle(m, (1920, 1080), 700, 0, -1)
    rng = np.random.default_rng(4)
    m[rng.random(m.shape) < 0.002] = 0
    table, nc, pts, shapes, hull, approx = _shapes(ctx, m[None], "ccomp", "none", max_points=400000)
    canon = ct.canonical(m, "ccomp", "none")
    assert max(len(c) for c in canon["contours"]) > 512 * 4
    hull_sizes = []
    for r in range(int(nc[0].sum())):
        s, off = shapes[0, r], int(table[0, r]["point_offset"])
        c = canon["contours"][r]
        if len(c) > 512:
            hull_sizes.append(int(s["n_hull"]))
            _check_record(c, s, hull[0, off:off + int(s["n_hull"])].reshape(-1, 1, 2),
                          approx[0, off:off + int(s["n_approx"])].reshape(-1, 1, 2), (0.0, 0.02))
    assert hull_sizes


def test_outer_contours_table_and_bit_equal_rectangles(ctx):
    masks = np.stack([synth.mask_rings(151, 203, step=3) | synth.mask_random(151, 203, 14, 0.1),
                      np.zeros((151, 203), np.uint8), synth.mask_blobs(151, 203, 4, sigma=2.0, pct=40)])
    dev = ctx.upload(masks)
    table, nb, pts, npts = ctx.outer_contours(dev, max_contours=4096, max_points=100000)
    shapes, hull, approx = ctx.contour_shapes(table, nb, pts, "simple", 0.0, 0.02)
    sh = ctx.download(shapes).view(SHAPE_DTYPE).reshape(3, -1)
    rects = ctx.min_area_rects(table, nb, pts)
    recs = ctx.download(table).view(CONTOUR_DTYPE).reshape(3, -1)
    p, hl, ap = ctx.download(pts), ctx.download(hull), ctx.download(approx)
    for f, m in enumerate(masks):
        ref, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
        n = int(ctx.download(nb)[f])
        seen = 0
        for i in range(n):
            rec, s = recs[f, i], sh[f, i]
            if not rec["external"] or rec["point_offset"] < 0:
                assert s["valid"] == 0
                continue
            seen += 1
            off, cnt = int(rec["point_offset"]), int(rec["n_simple"])
            c = p[f, off:off + cnt].reshape(-1, 1, 2)
            assert s["rect"].tobytes() == rects[f, i].tobytes()
            _check_record(c, s, hl[f, off:off + int(s["n_hull"])].reshape(-1, 1, 2),
                          ap[f, off:off + int(s["n_approx"])].reshape(-1, 1, 2), (0.0, 0.02))
        assert seen == len(ref)
    # rectangles of every outer record of a find_contours table are bit-equal to bv_min_area_rects as well
    t2, _, nc2, p2, _ = ctx.find_contours(dev, "tree", "simple", 4096, 100000)
    s2 = ctx.download(ctx.contour_shapes(t2, nc2, p2, "simple")[0]).view(SHAPE_DTYPE).reshape(3, -1)
    for f in range(3):
        n_outer = int(ctx.download(nc2)[f, 0])
        for i in range(n_outer):
            if recs[f, i]["external"]:
                assert s2[f, i]["rect"].tobytes() == rects[f, i].tobytes()


def test_mixed_batch(ctx):
    h, w = 70, 95
    masks = np.stack([synth.mask_random(h, w, 11, 0.5), np.zeros((h, w), np.uint8), synth.mask_rings(h, w, step=3),
                      np.full((h, w), 255, np.uint8), synth.mask_blobs(h, w, 4, sigma=2.0, pct=40)])
    _check_all(ctx, masks, modes=("tree", "list"))


def test_overflow_and_null_outputs(ctx):
    m = synth.mask_random(60, 70, 13, 0.5)
    reg = ct.regions(m)
    n = len(reg["outer_start"]) + len(reg["hole_start"])
    canon = ct.canonical(m, "tree", "simple", reg)
    max_contours = n // 2
    max_points = sum(len(c) for c in canon["contours"][:max_contours]) // 2
    guard = 64
    dev = ctx.upload(m)
    table, _, nc, pts, _ = ctx.find_contours(dev, "tree", "simple", max_contours, max_points)
    size = SHAPE_DTYPE.itemsize
    shapes = torch.full(((max_contours + guard) * size,), 0x5A, dtype=torch.uint8, device=ctx.device)
    hull = torch.full(((max_points + guard) * 2,), 0x5A5A5A5A, dtype=torch.int32, device=ctx.device)
    approx = torch.full(((max_points + guard) * 2,), 0x5A5A5A5A, dtype=torch.int32, device=ctx.device)
    torch.cuda.synchronize()
    lib, ffi = bv.runtime.lib, bv.runtime.ffi
    ptr = lambda t, ty: ffi.cast(ty, t.data_ptr())
    for h_on, a_on in ((True, True), (False, True), (True, False), (False, False)):
        bv.runtime.check(lib.bv_contour_shapes(ctx.handle, ptr(table, "bv_contour *"), ptr(nc, "int32_t *"), 2,
                                               ptr(pts, "int32_t *"), 1, max_contours, max_points,
                                               lib.BV_CHAIN_APPROX_SIMPLE, 0.0, 0.02, ptr(shapes, "bv_shape *"),
                                               ptr(hull, "int32_t *") if h_on else ffi.NULL,
                                               ptr(approx, "int32_t *") if a_on else ffi.NULL))
        ctx.sync()
        assert (ctx.download(shapes)[max_contours * size:] == 0x5A).all()
        assert (ctx.download(hull)[max_points * 2:] == 0x5A5A5A5A).all()
        assert (ctx.download(approx)[max_points * 2:] == 0x5A5A5A5A).all()
        sh = ctx.download(shapes)[:max_contours * size].view(SHAPE_DTYPE)
        recs = ctx.download(table).view(CONTOUR_DTYPE).reshape(-1)
        P, H, A = ctx.download(pts), ctx.download(hull).reshape(-1, 2), ctx.download(approx).reshape(-1, 2)
        n_valid = 0
        for r in range(max_contours):
            off = int(recs[r]["point_offset"])
            if off < 0:
                assert sh[r]["valid"] == 0
                continue
            n_valid += 1
            c = canon["contours"][r]
            s = sh[r]
            assert s["arc_length"] == cv2.arcLength(c, True)
            if h_on:
                assert np.array_equal(H[off:off + int(s["n_hull"])].reshape(-1, 1, 2), cs.convex_hull(c))
            if a_on:
                assert np.array_equal(A[off:off + int(s["n_approx"])].reshape(-1, 1, 2),
                                      cs.approx_poly_dp(c, 0.02 * cv2.arcLength(c, True)))
            else:
                assert s["n_approx"] == 0
        assert 0 < n_valid < max_contours


@pytest.mark.parametrize("mode", ["external", "list", "ccomp", "tree"])
@pytest.mark.parametrize("method", ["none", "simple"])
def test_feature_find_contours_shapes(ctx, mode, method):
    m = np.ascontiguousarray(synth.mask_rings(101, 131, step=4) | synth.mask_random(101, 131, 15, 0.05))
    if mode == "external" and method == "none":
        return
    plain, plain_h = feature.find_contours(m, mode, method)
    got, hier = feature.find_contours(m, mode, method, shapes=True, approx_relative=0.02)
    assert np.array_equal(hier, plain_h) and len(got) == len(plain)
    for c, p in zip(got, plain):
        assert {k: v for k, v in c.items() if k in p and k != "points"} == {k: v for k, v in p.items() if k != "points"}
        pts = c["points"]
        assert c["arc_length"] == cv2.arcLength(pts, True)
        assert c["hull"].dtype == np.int32 and np.array_equal(c["hull"], cs.convex_hull(pts))
        assert np.array_equal(c["approx"], cv2.approxPolyDP(pts, 0.02 * c["arc_length"], True))
        assert c["approx_convex"] == cv2.isContourConvex(c["approx"])
        (wx, wy), wr = cv2.minEnclosingCircle(pts)
        (cx, cy), r = c["min_enclosing_circle"]
        assert abs(cx - wx) <= 2e-3 and abs(cy - wy) <= 2e-3 and abs(r - wr) <= 2e-3
        assert _same_rectangle_or_proven_tie(pts.reshape(-1, 2), cv2.minAreaRect(pts), c["min_area_rect"], 1e-3)
