"""bv_find_contours (RETR_LIST / CCOMP / TREE, CHAIN_APPROX_NONE / SIMPLE) against cv2.findContours, re-ordered into the
library's record order by oracle/contour_tree.py: every vertex, every parent, the sibling links and the moment sums."""
import cv2
import numpy as np
import pytest

import cuauv_vision_pipeline_b200 as bv
from cuauv_vision_pipeline_b200 import feature
from cuauv_vision_pipeline_b200.runtime import CONTOUR_DTYPE
from oracle import contour_tree as ct
from oracle import synth

pytestmark = pytest.mark.gpu

MODES = ("list", "ccomp", "tree")


@pytest.fixture(scope="module")
def ctx():
    c = bv.Context(0)
    yield c
    c.close()


def _device(ctx, masks, mode, method, max_contours=None, max_points=None):
    """Runs one batch; returns per frame (records, hierarchy [N,4], n_outer, n_holes, vertex lists)."""
    masks = np.ascontiguousarray(masks)
    b, h, w = masks.shape
    if max_contours is None:
        max_contours = 64 + max(len(ct.regions(m)["outer_start"]) + len(ct.regions(m)["hole_start"]) for m in masks)
    if max_points is None:
        max_points = 64 + 4 * h * w
    table, hier, nc, pts, npts = ctx.find_contours(ctx.upload(masks), mode, method, max_contours, max_points)
    table, hier, nc = ctx.download(table), ctx.download(hier), ctx.download(nc)
    pts, npts = ctx.download(pts), ctx.download(npts)
    out = []
    for f in range(b):
        n_outer, n_holes = int(nc[f, 0]), int(nc[f, 1])
        n = n_outer + n_holes
        assert n <= max_contours and int(npts[f]) <= max_points
        recs = table[f, :n].copy().view(CONTOUR_DTYPE).reshape(-1)
        lists = []
        for r in recs:
            cnt = int(r["n_points"] if method == "none" else r["n_simple"])
            off = int(r["point_offset"])
            assert off >= 0 and r["reserved"] == 0
            lists.append(pts[f, off:off + cnt].reshape(-1, 1, 2))
        out.append((recs, hier[f, :n], n_outer, n_holes, lists))
    return out


def _check(mask, got, mode, method):
    reg = ct.regions(mask)
    canon = ct.canonical(mask, mode, method, reg)
    recs, hier, n_outer, n_holes, lists = got
    assert (n_outer, n_holes) == (canon["n_outer"], canon["n_holes"])
    differing = sum(not np.array_equal(a, b) for a, b in zip(lists, canon["contours"]))
    assert differing == 0, "%d of %d contours differ (%s, %s)" % (differing, len(lists), mode, method)
    assert hier[:, 3].tolist() == canon["parent"].tolist(), mode
    assert np.array_equal(hier[:, :3], ct.record_links(canon["parent"].tolist())), mode
    for r, rec in enumerate(recs):
        c = canon["none"][r]
        assert bool(rec["external"]) == (r < n_outer and reg["parent_tree"][r] < 0)
        assert (int(rec["start_x"]), int(rec["start_y"])) == tuple(int(v) for v in c[0, 0])
        assert int(rec["n_points"]) == len(c) and int(rec["n_simple"]) == len(ct.simple_from_none(c))
        m00, m10, m01 = feature._contour_moments(rec)
        mo = cv2.moments(c)
        assert (m00, m10, m01) == (mo["m00"], mo["m10"], mo["m01"]), r
        assert float(rec["a00"]) * 0.5 == cv2.contourArea(c, oriented=True), r
        xs, ys = c[:, 0, 0], c[:, 0, 1]
        assert (rec["x0"], rec["y0"], rec["x1"], rec["y1"]) == (xs.min(), ys.min(), xs.max(), ys.max())
        if r >= n_outer:
            x, y = int(rec["start_x"]), int(rec["start_y"])
            assert int(rec["label"]) == int(reg["fg"][y, x]) and rec["external"] == 0


def _check_all(ctx, masks, modes=MODES, methods=("none", "simple")):
    masks = np.ascontiguousarray(masks)
    for mode in modes:
        for method in methods:
            for m, got in zip(masks, _device(ctx, masks, mode, method)):
                _check(m, got, mode, method)


GENERATORS = [
    ("blobs", lambda: synth.mask_blobs(120, 161, 3, sigma=3.0, pct=50)),
    ("lattice", lambda: synth.mask_lattice(33, 47)),
    ("serpentine", lambda: synth.mask_serpentine(41, 53)),
    ("rings", lambda: synth.mask_rings(151, 203, step=3)),
    ("random", lambda: synth.mask_random(90, 117, 5, 0.45)),
    ("random_dense", lambda: synth.mask_random(64, 64, 6, 0.7)),
    ("diagonals", lambda: synth.mask_diagonals(60, 90)),
]


@pytest.mark.parametrize("name,gen", GENERATORS, ids=[n for n, _ in GENERATORS])
def test_synth_generators(ctx, name, gen):
    _check_all(ctx, gen()[None])


def _one_hole():
    m = np.full((20, 30), 255, np.uint8)
    m[9, 13] = 0
    return m


def _edge_regions():
    m = np.full((40, 50), 255, np.uint8)
    m[10:15, 0:8] = 0
    m[0:6, 20:23] = 0
    m[30:40, 44:46] = 0
    m[20:25, 20:25] = 0                                          # the only hole
    return m


SPECIAL = [("1x1_on", lambda: np.full((1, 1), 255, np.uint8)), ("1x1_off", lambda: np.zeros((1, 1), np.uint8)),
           ("1xN", lambda: synth.mask_random(1, 77, 1, 0.6)), ("Nx1", lambda: synth.mask_random(77, 1, 2, 0.6)),
           ("all0", lambda: np.zeros((30, 40), np.uint8)), ("all255", lambda: np.full((30, 40), 255, np.uint8)),
           ("one_hole", _one_hole), ("edge_regions", _edge_regions)]


@pytest.mark.parametrize("name,gen", SPECIAL, ids=[n for n, _ in SPECIAL])
def test_special_masks(ctx, name, gen):
    _check_all(ctx, gen()[None])


def test_edge_regions_give_no_hole_border(ctx):
    (recs, hier, n_outer, n_holes, _), = _device(ctx, _edge_regions()[None], "tree", "simple")
    assert (n_outer, n_holes) == (1, 1)


@pytest.mark.parametrize("width", [29, 30, 31, 32, 33, 61, 62, 2209])
def test_widths_around_the_walk_words(ctx, width):
    h = 23 if width > 100 else 37
    m = synth.mask_random(h, width, width, 0.55)
    _check_all(ctx, m[None])
    full = np.full((h, width), 255, np.uint8)
    full[1:-1:3, 1:-1:4] = 0
    _check_all(ctx, full[None])


def test_mixed_batch(ctx):
    h, w = 70, 95
    masks = np.stack([synth.mask_random(h, w, 11, 0.5), np.zeros((h, w), np.uint8), synth.mask_rings(h, w, step=3),
                      np.full((h, w), 255, np.uint8), synth.mask_blobs(h, w, 4, sigma=2.0, pct=40)])
    _check_all(ctx, masks)


def test_c3_frame_1080p(ctx):
    frame = synth.gen_underwater(1080, 1920, 31)
    hsv = cv2.cvtColor(frame, cv2.COLOR_BGR2HSV)
    m = cv2.inRange(hsv, np.array([0, 40, 60]), np.array([179, 255, 255]))
    _check_all(ctx, m[None], methods=("simple",))
    _check_all(ctx, m[None], modes=("tree",), methods=("none",))


def test_4k_with_thousands_of_holes(ctx):
    m = np.full((2160, 3840), 255, np.uint8)
    rng = np.random.default_rng(9)
    m[rng.random((2160, 3840)) < 0.02] = 0
    m[::97, :] = 0
    reg = ct.regions(m)
    assert len(reg["hole_start"]) > 2000
    got, = _device(ctx, m[None], "tree", "simple")
    _check(m, got, "tree", "simple")


def test_vertex_pool_overflow(ctx):
    m = synth.mask_random(120, 150, 12, 0.5)
    want = _device(ctx, m[None], "tree", "none")
    for chunks in (1, 7, 40):
        try:
            ctx.set_option("contour_pool_chunks", chunks)
            for method in ("none", "simple"):
                got, = _device(ctx, m[None], "tree", method)
                _check(m, got, "tree", method)
        finally:
            ctx.set_option("contour_pool_chunks", 0)
    again, = _device(ctx, m[None], "tree", "none")
    assert all(np.array_equal(a, b) for a, b in zip(again[4], want[0][4]))


def test_capacity_overflow_reports_counts_and_writes_nothing_past_the_buffers(ctx):
    import torch
    m = synth.mask_random(60, 70, 13, 0.5)
    reg = ct.regions(m)
    n_outer, n_holes = len(reg["outer_start"]), len(reg["hole_start"])
    canon = ct.canonical(m, "tree", "simple", reg)
    max_contours, guard = n_outer + n_holes // 2, 64
    need = sum(len(c) for c in canon["contours"][:max_contours])     # vertices of the records that are written
    max_points = need // 2
    size = CONTOUR_DTYPE.itemsize
    table = torch.full(((max_contours + guard) * size,), 0x5A, dtype=torch.uint8, device=ctx.device)
    hier = torch.full(((max_contours + guard) * 4,), 0x5A5A5A5A, dtype=torch.int32, device=ctx.device)
    pts = torch.full(((max_points + guard) * 2,), 0x5A5A5A5A, dtype=torch.int32, device=ctx.device)
    nc = torch.zeros(2, dtype=torch.int32, device=ctx.device)
    npts = torch.zeros(1, dtype=torch.int32, device=ctx.device)
    mask = ctx.upload(m)
    torch.cuda.synchronize()
    lib, ffi = bv.runtime.lib, bv.runtime.ffi
    bv.runtime.check(lib.bv_find_contours(ctx.handle, ffi.cast("uint8_t *", mask.data_ptr()), 1, 60, 70, lib.BV_RETR_TREE,
                                          lib.BV_CHAIN_APPROX_SIMPLE, ffi.cast("bv_contour *", table.data_ptr()),
                                          ffi.cast("int32_t *", hier.data_ptr()), max_contours,
                                          ffi.cast("int32_t *", nc.data_ptr()), ffi.cast("int32_t *", pts.data_ptr()),
                                          max_points, ffi.cast("int32_t *", npts.data_ptr())))
    ctx.sync()
    assert ctx.download(nc).tolist() == [n_outer, n_holes]
    assert int(ctx.download(npts)[0]) == need
    assert (ctx.download(table)[max_contours * size:] == 0x5A).all()
    assert (ctx.download(hier)[max_contours * 4:] == 0x5A5A5A5A).all()
    assert (ctx.download(pts)[max_points * 2:] == 0x5A5A5A5A).all()
    # the records that were written are the leading records of the complete result
    recs = ctx.download(table)[:max_contours * size].view(CONTOUR_DTYPE)
    full, = _device(ctx, m[None], "tree", "simple")
    for k in ("a00", "a10", "a01", "start_x", "start_y", "n_points", "n_simple", "label", "external"):
        assert np.array_equal(recs[k], full[0][k][:max_contours]), k


def test_outer_records_equal_outer_contours(ctx):
    m = synth.mask_rings(151, 203, step=3) | synth.mask_random(151, 203, 14, 0.1)
    m = np.ascontiguousarray(m)
    dev = ctx.upload(m)

    def outer():
        t, nb, pts, npts = ctx.outer_contours(dev, max_contours=4096, max_points=50000)
        n = int(ctx.download(nb)[0])
        return n, ctx.download(t)[0, :n].copy(), ctx.download(pts)[0, :int(ctx.download(npts)[0])].copy()

    before = outer()
    for mode in MODES:
        table, hier, nc, pts, npts = ctx.find_contours(dev, mode, "simple", 4096, 50000)
        n_outer = int(ctx.download(nc)[0, 0])
        assert n_outer == before[0]
        recs = ctx.download(table)[0, :n_outer].copy().view(CONTOUR_DTYPE).reshape(-1)
        want = before[1].view(CONTOUR_DTYPE).reshape(-1)
        for k in ("a00", "a10", "a01", "x0", "y0", "x1", "y1", "start_x", "start_y", "n_points", "n_simple", "label",
                  "external"):
            assert np.array_equal(recs[k], want[k]), k
    after = outer()
    assert after[0] == before[0] and np.array_equal(after[1], before[1]) and np.array_equal(after[2], before[2])


@pytest.mark.parametrize("mode", ["external", "list", "ccomp", "tree"])
@pytest.mark.parametrize("method", ["none", "simple"])
def test_feature_find_contours_matches_cv2_shapes(ctx, mode, method):
    m = synth.mask_rings(101, 131, step=4) | synth.mask_random(101, 131, 15, 0.05)
    m = np.ascontiguousarray(m)
    if mode == "external" and method == "none":
        with pytest.raises(ValueError):
            feature.find_contours(m, mode, method)
        return
    # tiny first guesses: the wrapper grows the buffers once
    got, hier = feature.find_contours(m, mode, method, max_contours=4, max_points=16)
    cv_mode = cv2.RETR_EXTERNAL if mode == "external" else ct.MODES[mode]
    ref, ref_h = cv2.findContours(m, cv_mode, ct.METHODS[method])
    assert hier.dtype == np.int32 and hier.shape == (1, len(ref), 4) == ref_h.shape
    key = lambda c: (int(c[0, 0, 0]), int(c[0, 0, 1]), len(c))
    assert sorted(key(c["points"]) for c in got) == sorted(key(c) for c in ref)
    by_key = {key(c): c for c in ref}
    for c in got:
        r = by_key[key(c["points"])]
        assert c["points"].dtype == np.int32 and c["points"].shape == r.shape and np.array_equal(c["points"], r)
        assert feature.contour_area(c) == cv2.contourArea(r)
        mo = cv2.moments(r)
        if mo["m00"] > 0:
            assert feature.contour_centroid(c) == (int(mo["m10"] / mo["m00"]), int(mo["m01"] / mo["m00"]))
    assert sum(c["is_hole"] for c in got) == (0 if mode == "external" else len(ct.regions(m)["hole_start"]))
