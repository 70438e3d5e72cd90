"""GPU parity: morphology against cv2 (reference call sites utils/transform.py:80-164,
modules/preprocessor.py:120-129) and labelling + raster moments against the declared oracle
(oracle/ccl.py).  All bit-exact."""
import cv2
import numpy as np
import pytest

from oracle import ccl, cv_ops, synth

pytestmark = pytest.mark.gpu

CV_OP = {"erode": cv2.MORPH_ERODE, "dilate": cv2.MORPH_DILATE, "open": cv2.MORPH_OPEN, "close": cv2.MORPH_CLOSE,
         "gradient": cv2.MORPH_GRADIENT}


@pytest.mark.parametrize("op", list(CV_OP))
@pytest.mark.parametrize("shape", [(270, 480), (479, 641), (33, 31)])
def test_rect5_on_masks(ctx, op, shape):
    m = synth.mask_random(shape[0], shape[1], 5, 0.55)
    k = cv_ops.rect_kernel(5)
    got = ctx.download(ctx.morph(ctx.upload(m), op, k))
    assert np.array_equal(got, cv2.morphologyEx(m, CV_OP[op], k))


@pytest.mark.parametrize("kw,kh", [(3, 3), (5, 5), (7, 3), (1, 9), (4, 4), (2, 5), (6, 1), (15, 15)])
@pytest.mark.parametrize("op", ["erode", "dilate", "open", "close"])
def test_rect_sizes_incl_even(ctx, kw, kh, op):
    m = synth.mask_blobs(131, 173, 7, sigma=3.0, pct=55)
    k = np.ones((kh, kw), np.uint8)
    got = ctx.download(ctx.morph(ctx.upload(m), op, k))
    assert np.array_equal(got, cv2.morphologyEx(m, CV_OP[op], k))


@pytest.mark.parametrize("iters", [1, 2, 3])
@pytest.mark.parametrize("op", list(CV_OP))
def test_iterations(ctx, iters, op):
    m = synth.mask_blobs(150, 210, 9, sigma=5.0, pct=60)
    k = cv_ops.rect_kernel(3)
    got = ctx.download(ctx.morph(ctx.upload(m), op, k, iterations=iters))
    assert np.array_equal(got, cv2.morphologyEx(m, CV_OP[op], k, iterations=iters))
    e = cv_ops.elliptic_kernel(5)
    got = ctx.download(ctx.morph(ctx.upload(m), op, e, iterations=iters))
    assert np.array_equal(got, cv2.morphologyEx(m, CV_OP[op], e, iterations=iters))


@pytest.mark.parametrize("k", [1, 2, 5, 12])
def test_ellipse_on_three_channel_grey(ctx, k):
    """modules/preprocessor.py:120-129: MORPH_ELLIPSE (2k+1)^2 on the BGR frame."""
    img = synth.gen_underwater(96, 150, 3)
    d = ctx.upload(img)
    se = cv_ops.elliptic_kernel(2 * k + 1)
    assert np.array_equal(ctx.download(ctx.morph(d, "erode", se)), cv_ops.ellipse_erode(img, k))
    assert np.array_equal(ctx.download(ctx.morph(d, "dilate", se)), cv_ops.ellipse_dilate(img, k))


def test_ellipse_101(ctx):
    img = synth.gen_underwater(130, 170, 4)
    se = cv_ops.elliptic_kernel(101)
    assert np.array_equal(ctx.download(ctx.morph(ctx.upload(img), "erode", se)), cv2.erode(img, se))


def test_asymmetric_structuring_elements(ctx):
    """cv2 applies the SE taps unmirrored for erosion and dilation alike."""
    m = synth.mask_blobs(90, 130, 4, sigma=3.0, pct=55)
    img = synth.gen_underwater(60, 90, 2)
    for se in (np.array([[1, 1, 0]], np.uint8), np.array([[1, 0, 0], [1, 0, 0], [1, 1, 1]], np.uint8),
               np.array([[0, 1], [1, 1], [0, 0], [1, 0]], np.uint8)):
        for op in ("erode", "dilate", "open", "close", "gradient"):
            assert np.array_equal(ctx.download(ctx.morph(ctx.upload(m), op, se)), cv2.morphologyEx(m, CV_OP[op], se)), (se, op)
        assert np.array_equal(ctx.download(ctx.morph(ctx.upload(img), "dilate", se, iterations=2)), cv2.dilate(img, se, iterations=2))


@pytest.mark.parametrize("kw,kh", [(4, 4), (2, 5), (6, 1), (5, 5), (3, 7), (40, 3), (1, 1)])
@pytest.mark.parametrize("op", list(CV_OP))
@pytest.mark.parametrize("width", [160, 173])
def test_bit_packed_morphology_through_the_stage(ctx, kw, kh, op, width):
    """The fused stage runs morphology on bit-packed masks (32 px per word); same semantics."""
    img = synth.gen_underwater(131, width, 7)
    desc = ctx.make_stage(cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[(op, kw, kh, 1)])
    hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
    raw = cv2.inRange(hsv, np.array([0, 40, 60]), np.array([179, 255, 255]))
    want = cv2.morphologyEx(raw, CV_OP[op], np.ones((kh, kw), np.uint8))
    assert np.array_equal(ctx.download(ctx.stage(desc, ctx.upload(img), want=("mask",))["mask"]), want)
    desc2 = ctx.make_stage(cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[(op, 3, 3, 2), ("dilate", kw, kh, 1)])
    want2 = cv2.dilate(cv2.morphologyEx(raw, CV_OP[op], np.ones((3, 3), np.uint8), iterations=2), np.ones((kh, kw), np.uint8))
    assert np.array_equal(ctx.download(ctx.stage(desc2, ctx.upload(img), want=("mask",))["mask"]), want2)


def test_transform_mirrors(ctx):
    from cuauv_vision_pipeline_b200 import transform
    m = synth.mask_blobs(120, 160, 1, sigma=4.0)
    k = transform.rect_kernel(5)
    assert np.array_equal(transform.morph_remove_noise(m, k), cv_ops.morph_remove_noise(m, cv_ops.rect_kernel(5)))
    assert np.array_equal(transform.morph_close_holes(m, k), cv_ops.morph_close_holes(m, cv_ops.rect_kernel(5)))
    assert np.array_equal(transform.morph_borders(m, k), cv_ops.morph_borders(m, cv_ops.rect_kernel(5)))
    assert np.array_equal(transform.erode(m, k, 2), cv_ops.erode(m, cv_ops.rect_kernel(5), 2))
    assert np.array_equal(transform.dilate(m, transform.elliptic_kernel(7)), cv_ops.dilate(m, cv_ops.elliptic_kernel(7)))
    img = synth.gen_underwater(120, 160, 2)
    assert np.array_equal(transform.resize(img, 77, 45), cv_ops.resize(img, 77, 45))


# ----------------------------------------------------------------------------------------------
# labelling + moments
# ----------------------------------------------------------------------------------------------
def check_labels(ctx, mask, max_blobs=None):
    n_ref, lab_ref, tab = ccl.label_and_moments(mask)
    cap = max_blobs if max_blobs is not None else max(n_ref, 1)
    labels, blobs, nb = ctx.label(ctx.upload(mask), max_blobs=cap)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    assert int(n[0]) == n_ref
    assert np.array_equal(ctx.download(labels), lab_ref)
    t = tables[0]
    k = min(n_ref, cap)
    for key in ccl.MOMENT_KEYS + ("x0", "y0", "x1", "y1"):
        assert np.array_equal(t[key].astype(np.int64), tab[key][:k]), key
    return n_ref


@pytest.mark.parametrize("shape", [(270, 480), (479, 641), (64, 32), (65, 33), (100, 31)])
def test_ccl_blobs(ctx, shape):
    assert check_labels(ctx, synth.mask_blobs(shape[0], shape[1], 3, sigma=4.0)) > 0


@pytest.mark.parametrize("density", [0.1, 0.4, 0.5, 0.6, 0.9])
def test_ccl_random_noise(ctx, density):
    check_labels(ctx, synth.mask_random(211, 307, 13, density))


def test_ccl_lattice_of_isolated_pixels(ctx):
    m = synth.mask_lattice(270, 480)
    assert check_labels(ctx, m) == 135 * 240


def test_ccl_serpentine_single_component(ctx):
    assert check_labels(ctx, synth.mask_serpentine(241, 333)) == 1


def test_ccl_nested_rings(ctx):
    assert check_labels(ctx, synth.mask_rings(301, 403)) > 10


def test_ccl_diagonals_are_8_connected(ctx):
    m = synth.mask_diagonals(200, 260)
    n4 = cv2.connectedComponents((m != 0).astype(np.uint8), connectivity=4)[0] - 1
    n8 = check_labels(ctx, m)
    assert n8 < n4


@pytest.mark.parametrize("kind", ["empty", "full", "single", "corners"])
def test_ccl_trivial_masks(ctx, kind):
    m = np.zeros((67, 97), np.uint8)
    if kind == "full":
        m[:] = 255
    elif kind == "single":
        m[31, 64] = 1            # any non-zero value counts
    elif kind == "corners":
        m[0, 0] = m[0, -1] = m[-1, 0] = m[-1, -1] = 255
    check_labels(ctx, m)


def test_ccl_word_boundary_cases(ctx):
    """Runs that end / start exactly at 32-px word boundaries, and diagonal contacts across them."""
    m = np.zeros((12, 130), np.uint8)
    m[0, 0:32] = 255            # full word
    m[1, 32:64] = 255           # next word, diagonal contact at (0,31)-(1,32)
    m[3, 31] = 255
    m[4, 32] = 255              # single-pixel diagonal across the boundary
    m[6, 63:65] = 255           # run straddling a boundary
    m[7, 95] = 255
    m[8, 96] = 255
    m[8, 94] = 255
    m[10, 100:130] = 255        # run reaching the (partial) last word's end
    m[11, 129] = 255
    check_labels(ctx, m)


def test_ccl_batch_frames_are_independent(ctx):
    masks = np.stack([synth.mask_blobs(90, 160, s, sigma=4.0) for s in (1, 2, 3)])
    labels, blobs, nb = ctx.label(ctx.upload(masks), max_blobs=512)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    lab = ctx.download(labels)
    for i in range(3):
        n_ref, lab_ref, tab = ccl.label_and_moments(masks[i])
        assert int(n[i]) == n_ref and np.array_equal(lab[i], lab_ref)
        assert np.array_equal(tables[i]["m11"].astype(np.int64), tab["m11"])


def test_ccl_capacity_smaller_than_blob_count(ctx):
    m = synth.mask_lattice(40, 64)
    check_labels(ctx, m, max_blobs=100)


def test_golden_ccl_fixture(ctx):
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "ccl_90x160.npz"))
    labels, blobs, nb = ctx.label(ctx.upload(z["mask"]), max_blobs=int(z["n"]))
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    assert int(n[0]) == int(z["n"]) and np.array_equal(ctx.download(labels), z["labels"])
    for key in ccl.MOMENT_KEYS:
        assert np.array_equal(tables[0][key].astype(np.int64), z[key])


def test_feature_mirror_centroids(ctx):
    from cuauv_vision_pipeline_b200 import feature
    m = synth.mask_blobs(200, 300, 8, sigma=6.0)
    labels, blobs, n = feature.label_blobs(m)
    n_ref, lab_ref, tab = ccl.label_and_moments(m)
    assert n == n_ref and np.array_equal(labels, lab_ref)
    for b in blobs:
        i = b["label"] - 1
        assert feature.blob_centroid(b) == (int(tab["m10"][i] / tab["m00"][i]), int(tab["m01"][i] / tab["m00"][i]))
        assert feature.blob_area(b) == float(tab["m00"][i])


@pytest.mark.parametrize("shape", [(2160, 3840), (1080, 1920)])
def test_full_size_properties(ctx, shape):
    """At BASELINE sizes: properties that need no oracle pass over the frame.  Sum of m00 equals the
    mask popcount; full-frame blob moments are the closed forms (m30 exceeds 2^53 at 4K); opening is
    idempotent; lattice gives exactly W*H/4 blobs."""
    h, w = shape
    full = np.full((h, w), 255, np.uint8)
    labels, blobs, nb = ctx.label(ctx.upload(full), max_blobs=4)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    assert int(n[0]) == 1
    b = tables[0][0]
    xs = np.arange(w, dtype=object)
    ys = np.arange(h, dtype=object)
    assert int(b["m00"]) == h * w and int(b["m30"]) == int((xs ** 3).sum()) * h and int(b["m03"]) == int((ys ** 3).sum()) * w
    assert int(b["m21"]) == int((xs ** 2).sum()) * int(ys.sum()) and int(b["m12"]) == int(xs.sum()) * int((ys ** 2).sum())
    m = synth.mask_blobs(h, w, 3, sigma=6.0)
    d = ctx.upload(m)
    k = cv_ops.rect_kernel(5)
    opened = ctx.morph(d, "open", k)
    assert np.array_equal(ctx.download(ctx.morph(opened, "open", k)), ctx.download(opened))
    labels, blobs, nb = ctx.label(opened, max_blobs=8192)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    assert int(tables[0]["m00"].sum()) == int((ctx.download(opened) != 0).sum())
    lab = ctx.download(labels)
    assert int(lab.max()) == int(n[0]) and np.array_equal(lab != 0, ctx.download(opened) != 0)
    lat = synth.mask_lattice(h, w)
    _, _, nb = ctx.label(ctx.upload(lat), max_blobs=0, want_labels=False)
    assert int(ctx.download(nb)[0]) == (h // 2) * (w // 2)


# ----------------------------------------------------------------------------------------------
# the literal reference path: outer contours + polygon centroid / area (SURVEY.md 8f rank 1)
# ----------------------------------------------------------------------------------------------
def check_contours(mask):
    from cuauv_vision_pipeline_b200 import feature
    ref = {}
    for c in cv_ops.outer_contours(np.ascontiguousarray(mask)):
        ref[(int(c[0, 0, 0]), int(c[0, 0, 1]))] = (cv_ops.contour_centroid(c), cv_ops.contour_area(c),
                                                   cv2.boundingRect(c))
    ref_pts = {(int(c[0, 0, 0]), int(c[0, 0, 1])): c for c in cv_ops.outer_contours(np.ascontiguousarray(mask))}
    got = feature.outer_contours(mask, max_contours=max(16, 4 * len(ref) + 64), points=True)
    assert len(got) == len(ref)
    for g in got:   # the vertex lists are the arrays cv2.findContours(RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) returns
        want = ref_pts[(g["start_x"], g["start_y"])]
        assert g["points"] is not None and g["points"].shape == want.shape and np.array_equal(g["points"], want)
        assert cv2.minAreaRect(g["points"]) == cv2.minAreaRect(want)       # modules/bins.py:60
    for g in got:
        key = (g["start_x"], g["start_y"])
        assert key in ref, key
        centroid, area, (bx, by, bw, bh) = ref[key]
        assert feature.contour_centroid(g) == centroid, key
        assert feature.contour_area(g) == area, key
        assert (g["x0"], g["y0"], g["x1"] - g["x0"] + 1, g["y1"] - g["y0"] + 1) == (bx, by, bw, bh), key
    return len(ref)


@pytest.mark.parametrize("shape,seed", [((270, 480), 3), ((479, 641), 4), ((1080, 1920), 5), ((65, 33), 6)])
def test_outer_contours_match_findcontours(ctx, shape, seed):
    assert check_contours(synth.mask_blobs(shape[0], shape[1], seed, sigma=5.0)) > 0


def test_outer_contours_nested_rings_report_only_the_outermost(ctx):
    assert check_contours(synth.mask_rings(301, 403)) == 1


@pytest.mark.parametrize("density", [0.2, 0.5, 0.7])
def test_outer_contours_noise(ctx, density):
    check_contours(synth.mask_random(150, 211, 21, density))


@pytest.mark.parametrize("width", [1, 2, 29, 30, 31, 59, 60, 61, 64, 90, 91])
@pytest.mark.parametrize("height", [1, 2, 33])
def test_outer_contours_around_the_walk_word_edges(ctx, height, width):
    """The border walk reads its own copy of the mask in words of 30 pixels + 1 neighbour on either side
    (csrc/ccl.cu walk_bits_kernel): widths around the multiples of 30 and 32, one- and two-row frames, dense
    noise (borders crossing every word edge) and a full frame."""
    check_contours(synth.mask_random(height, width, 7 * width + height, 0.55))
    check_contours(np.full((height, width), 255, np.uint8))


def test_outer_contours_when_the_vertex_pool_runs_dry(ctx):
    """The first walk keeps the vertices in chunks drawn from a pool; borders the pool cannot hold are walked a second
    time (csrc/ccl.cu).  A pool of 5 / 40 chunks forces that path for most / some borders; results are unchanged,
    and the records' reserved field is back to 0 either way."""
    from cuauv_vision_pipeline_b200 import feature
    from cuauv_vision_pipeline_b200._host import default_context
    mask = synth.mask_blobs(270, 480, 3, sigma=5.0)
    want = feature.outer_contours(mask, points=True)
    contexts = (ctx, default_context(0))
    try:
        for chunks in (5, 40):
            for c in contexts:
                c.set_option("contour_pool_chunks", chunks)
            got = feature.outer_contours(mask, points=True)
            assert len(got) == len(want)
            for a, b in zip(got, want):
                assert np.array_equal(a["points"], b["points"]) and a["start_x"] == b["start_x"] and a["n_simple"] == b["n_simple"]
            check_contours(mask)
            t, nb, pts, npts = ctx.outer_contours(ctx.upload(mask), max_contours=1024, max_points=50000)
            n = int(ctx.download(nb)[0])
            recs = np.ascontiguousarray(ctx.download(t)[0, :n]).view(np.int32).reshape(n, 18)
            assert n == len(cv_ops.outer_contours(mask)) or n > 0
            assert not recs[:, 17].any()                                        # bv_contour.reserved
            assert (recs[recs[:, 15] == 1][:, 16] >= 0).all()                   # every external border got its slice
    finally:
        for c in contexts:
            c.set_option("contour_pool_chunks", 0)


def test_outer_contours_special_shapes(ctx):
    m = np.zeros((40, 70), np.uint8)
    m[3, 5] = 255                               # single pixel
    m[8, 10:30] = 255                           # 1-px horizontal line
    m[12:30, 40] = 255                          # 1-px vertical line
    for k in range(10):
        m[15 + k, 5 + k] = 255                  # diagonal
    m[32:38, 50:60] = 255
    m[34:36, 53:57] = 0                         # a hole
    m[0, 0] = m[39, 69] = m[0, 69] = 255        # frame corners
    m[20:26, 60:70] = 255                       # touches the right edge
    m[22:24, 62:66] = 0
    m[22, 63] = 255                             # island inside the hole: must not be reported
    check_contours(m)
    check_contours(synth.mask_serpentine(41, 53))
    check_contours(synth.mask_diagonals(60, 90))
    check_contours(np.full((30, 40), 255, np.uint8))
    assert check_contours(np.zeros((30, 40), np.uint8)) == 0


def test_bins_module_pipeline_with_reference_contours(ctx):
    """modules/bins.py:13-27 end to end: threshold -> OPEN -> outer contours, centroid and area of every contour."""
    img = synth.gen_underwater(480, 640, 77)
    _, cleaned = cv_ops.bins_mask(img)
    desc = ctx.make_stage(cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)])
    mask = ctx.stage(desc, ctx.upload(img), want=("mask",))["mask"]
    assert np.array_equal(ctx.download(mask), cleaned)
    check_contours(cleaned)


@pytest.mark.parametrize("shape", [(301, 333), (270, 496), (64, 2208)])
def test_morphology_chain_of_four_steps_with_labels(ctx, shape):
    """Four steps (8 elementary erosions / dilations, halo 13 rows) in the single shared-memory chain launch,
    batch of 3, final bits feeding the labelling."""
    frames = np.stack([synth.gen_underwater(shape[0], shape[1], 40 + i) for i in range(3)])
    steps = [("open", 5, 5, 1), ("close", 7, 3, 1), ("dilate", 3, 3, 2), ("erode", 9, 1, 1)]
    desc = ctx.make_stage(cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=steps, label=True)
    out = ctx.stage(desc, ctx.upload(frames), want=("mask", "labels", "blobs"), max_blobs=4096)
    mask, lab = ctx.download(out["mask"]), ctx.download(out["labels"])
    for i in range(3):
        m = cv2.inRange(cv2.cvtColor(frames[i], cv2.COLOR_BGR2HSV), np.array([0, 40, 60]), np.array([179, 255, 255]))
        m = cv2.morphologyEx(m, cv2.MORPH_OPEN, np.ones((5, 5), np.uint8))
        m = cv2.morphologyEx(m, cv2.MORPH_CLOSE, np.ones((3, 7), np.uint8))
        m = cv2.dilate(m, np.ones((3, 3), np.uint8), iterations=2)
        m = cv2.erode(m, np.ones((1, 9), np.uint8))
        assert np.array_equal(mask[i], m)
        assert np.array_equal(lab[i], ccl.label_and_moments(m)[1])


def _sorted_corners(corners):
    """Corners in a canonical order that rounding noise around 0 (-4e-16 vs 4e-16) cannot permute."""
    return np.array(sorted(corners, key=lambda p: (round(float(p[0]), 4), round(float(p[1]), 4))), dtype=np.float64)


def _rect_corners(rect):
    (cx, cy), (w, h), a = rect
    a = np.deg2rad(a)
    c, s = np.cos(a), np.sin(a)
    return _sorted_corners([(cx + sx * w * c - sy * h * s, cy + sx * w * s + sy * h * c)
                            for sx, sy in ((-.5, -.5), (.5, -.5), (.5, .5), (-.5, .5))])


def _edge_rectangles_f64(points):
    """Every rectangle that has one side on an edge of the convex hull, in float64: [(area, sorted corners)].
    The minimum-area enclosing rectangle is one of them (Freeman / Shapira); cv2.minAreaRect and the device both
    search this set with float32 rotating calipers."""
    hull = cv2.convexHull(points.reshape(-1, 1, 2).astype(np.int32)).reshape(-1, 2).astype(np.float64)
    out = []
    n = len(hull)
    for i in range(n):
        e = hull[(i + 1) % n] - hull[i]
        ln = np.hypot(*e)
        if ln == 0:
            continue
        u = e / ln
        v = np.array([-u[1], u[0]])
        pu, pv = hull @ u, hull @ v
        w, h = pu.max() - pu.min(), pv.max() - pv.min()
        corners = [a * u + b * v for a in (pu.min(), pu.max()) for b in (pv.min(), pv.max())]
        out.append((w * h, _sorted_corners(corners)))
    return out


def _same_rectangle_or_proven_tie(points, ref, rect, tol):
    """True when the two rectangles coincide (corner by corner, to tol), or when BOTH are (to tol) rectangles of the
    float64 edge set whose areas tie with the exact minimum to within float32 rounding (relative 5e-6): several hull
    edges give rectangles of the same area and the two searches stopped at different ones."""
    if np.abs(_rect_corners(ref) - _rect_corners(rect)).max() <= tol:
        return True
    cands = _edge_rectangles_f64(points)
    if not cands:
        return False
    amin = min(a for a, _ in cands)
    near = [c for a, c in cands if a <= amin * (1 + 5e-6) + 1e-9]

    def among(r):
        rc = _rect_corners(r)
        return any(np.abs(rc - c).max() <= 10 * tol for c in near)
    return len(near) >= 2 and among(ref) and among(rect)


@pytest.mark.parametrize("shape,seed", [((480, 640), 3), ((1080, 1920), 4), ((301, 333), 5)])
def test_min_area_rect_of_outer_contours_vs_cv2(ctx, shape, seed):
    """modules/bins.py:60-69: cv2.minAreaRect(contour) for every outer contour, computed on the device from the
    device-side vertex lists.  Stated tolerance: area 1e-4 relative; centre / size / angle 1e-3 (absolute, px / degrees)
    for EVERY contour whose minimum-area rectangle is unique; where several hull edges tie to within float32 rounding, both
    cv2's and the device's rectangle must be members of the float64 set of minimal rectangles (_same_rectangle_or_proven_tie)."""
    from cuauv_vision_pipeline_b200 import feature
    mask = synth.mask_blobs(shape[0], shape[1], seed, sigma=5.0, pct=72)
    got = feature.outer_contours(mask, points=True, rects=True)
    ref_contours, _ = cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    by_start = {}
    for c in ref_contours:
        pts = c.reshape(-1, 2)
        i = np.lexsort((pts[:, 0], pts[:, 1]))[0]
        by_start[(int(pts[i, 0]), int(pts[i, 1]))] = c
    assert len(got) == len(ref_contours) and len(got) > 20
    exact_params = 0
    for g in got:
        ref = cv2.minAreaRect(by_start[(g["start_x"], g["start_y"])])
        rect = feature.min_area_rect(g)
        assert np.array_equal(g["points"], by_start[(g["start_x"], g["start_y"])])
        ra, ga = ref[1][0] * ref[1][1], rect[1][0] * rect[1][1]
        assert abs(ra - ga) <= 1e-4 * max(1.0, ra), (ref, rect)
        assert -90.0 <= rect[2] < 0.0
        # every vertex lies inside the rectangle
        p = g["points"].reshape(-1, 2).astype(np.float64) - np.array(rect[0])
        a = np.deg2rad(rect[2])
        u, v = p @ np.array([np.cos(a), np.sin(a)]), p @ np.array([-np.sin(a), np.cos(a)])
        assert np.abs(u).max() <= rect[1][0] / 2 + 1e-2 and np.abs(v).max() <= rect[1][1] / 2 + 1e-2
        tol = 1e-3 * max(1.0, max(ref[1]))
        if np.abs(_rect_corners(ref) - _rect_corners(rect)).max() <= tol:
            exact_params += 1
        # EVERY contour: the same rectangle, or a proven tie between hull edges (both rectangles are exact minima)
        assert _same_rectangle_or_proven_tie(g["points"], ref, rect, tol), (ref, rect)
        # what modules/bins.py:60-69 consumes (w * h, max / min) agrees in either case
        assert sorted(rect[1]) == pytest.approx(sorted(ref[1]), rel=2e-4, abs=2e-3) or abs(ra - ga) <= 5e-6 * max(1.0, ra)
    assert exact_params >= 0.9 * len(got), (exact_params, len(got))


def test_min_area_rect_of_contours_larger_than_the_shared_memory_buffer(ctx):
    """A warp sorts up to 512 candidate hull vertices in shared memory (csrc/rects.cu); rough discs of radius 330 and 120 have
    ~2000 and ~700 contour vertices outside the extreme-point quadrilateral and take the single-thread fallback, the
    small blobs around them the warp path.  Same tolerance as above."""
    from cuauv_vision_pipeline_b200 import feature
    yy, xx = np.mgrid[0:800, 0:1100]
    rng = np.random.default_rng(3)
    m = ((xx - 400) ** 2 + (yy - 400) ** 2 <= 330 ** 2) | ((xx - 930) ** 2 + (yy - 200) ** 2 <= 120 ** 2)
    m ^= (rng.random(m.shape) < 0.35) & ((np.abs(np.hypot(xx - 400, yy - 400) - 330) < 3) | (np.abs(np.hypot(xx - 930, yy - 200) - 120) < 3))
    m[600:640, 850:1000] = True
    m = m.astype(np.uint8) * 255
    got = feature.outer_contours(m, points=True, rects=True, max_points=20000)
    ref_contours, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    assert len(got) == len(ref_contours) and max(len(c) for c in ref_contours) > 1000
    by_start = {}
    for c in ref_contours:
        pts = c.reshape(-1, 2)
        i = np.lexsort((pts[:, 0], pts[:, 1]))[0]
        by_start[(int(pts[i, 0]), int(pts[i, 1]))] = c
    for g in got:
        ref = cv2.minAreaRect(by_start[(g["start_x"], g["start_y"])])
        rect = feature.min_area_rect(g)
        ra, ga = ref[1][0] * ref[1][1], rect[1][0] * rect[1][1]
        assert abs(ra - ga) <= 1e-4 * max(1.0, ra), (ref, rect)
        if len(g["points"]) > 500:      # the discs: a unique minimum, so centre, sides and angle agree as well
            assert np.abs(_rect_corners(ref) - _rect_corners(rect)).max() <= 2e-3 * max(ref[1]), (ref, rect)


def test_min_area_rect_degenerate_contours(ctx):
    from cuauv_vision_pipeline_b200 import feature
    m = np.zeros((64, 96), np.uint8)
    m[5, 7] = 255                       # single pixel
    m[20, 10:31] = 255                  # horizontal segment
    m[30:50, 60] = 255                  # vertical segment
    for k in range(12):                 # diagonal 1-px line
        m[40 + k, 10 + k] = 255
    m[8:16, 70:90] = 255                # axis-aligned rectangle
    got = feature.outer_contours(m, points=True, rects=True)
    ref_contours, _ = cv2.findContours(m, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    assert len(got) == len(ref_contours) == 5
    for g in got:
        ref = [cv2.minAreaRect(c) for c in ref_contours if (c.reshape(-1, 2) == [g["start_x"], g["start_y"]]).all(axis=1).any()][0]
        rect = feature.min_area_rect(g)
        assert np.allclose([*rect[0], *rect[1], rect[2]], [*ref[0], *ref[1], ref[2]], rtol=0, atol=1e-3), (ref, rect)


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("shape", [(270, 480), (479, 641), (33, 31), (1242, 2208), (96, 4096), (5, 1024)])
def test_chain_variants_agree_with_cv2(ctx, variant, shape):
    """Both implementations of the binary chain (register-rolling warps / shared-memory tile) against cv2 for the chains the modules use: OPEN 5x5 (bins.py:23-24), OPEN+CLOSE 5x5 (red_buoy.py:31-34), 3x3."""
    ctx.set_option("morph_variant", variant)
    try:
        m = synth.mask_random(shape[0], shape[1], 11, 0.6)
        m[:, -3:] = 255                                     # set pixels at the right edge (tail word handling)
        m[0, :] = 255
        d = ctx.upload(m)
        for steps in ([("open", 5, 5, 1)], [("open", 5, 5, 1), ("close", 5, 5, 1)], [("erode", 3, 3, 1)], [("dilate", 5, 5, 1)],
                      [("close", 3, 3, 1)], [("open", 3, 3, 2)], [("open", 7, 7, 1)]):
            desc = ctx.make_stage(cvt=None, lo=(128, 0, 0), hi=(255, 255, 255), morph=steps)
            bgr = np.repeat(m[..., None], 3, axis=2)
            got = ctx.download(ctx.stage(desc, ctx.upload(bgr), want=("mask",))["mask"])
            want = m
            for op, kw, kh, it in steps:
                want = cv2.morphologyEx(want, CV_OP[op], np.ones((kh, kw), np.uint8), iterations=it)
            assert np.array_equal(got, want), steps
        assert np.array_equal(ctx.download(ctx.morph(d, "open", cv_ops.rect_kernel(5))), cv2.morphologyEx(m, cv2.MORPH_OPEN, cv_ops.rect_kernel(5)))
    finally:
        ctx.set_option("morph_variant", 0)
