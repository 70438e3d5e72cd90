"""Blob extraction: the role of the reference's outer_contours / contour_centroid / contour_area
(utils/feature.py:5-21,240-265) as connected-component labelling with exact raster moments; every border with its
hierarchy and shape descriptors; and cv2.Canny edges that feed them without leaving the device."""
import numpy as np

from ._host import ctx_for, to_device, is_device, release_to_caller, like_input


class Blob(dict):
    """One labelled component: label, integer raster moments m00..m03 and bbox x0,y0,x1,y1."""

    @property
    def area(self):
        return int(self["m00"])


def label_blobs(mat, max_blobs=4096, want_labels=True):
    """8-connected labelling of `mat != 0`.  Returns (labels int32[H,W] or None, [Blob...]) with
    labels 1..n in raster order of each blob's first pixel."""
    ctx = ctx_for(mat)
    labels, blobs, nb = ctx.label(to_device(ctx, mat), max_blobs=max_blobs, want_labels=want_labels)
    n, tables = ctx.blobs_to_numpy(blobs, nb)
    out = []
    for i, row in enumerate(tables[0]):
        b = Blob({k: int(row[k]) for k in row.dtype.names})
        b["label"] = i + 1
        out.append(b)
    if labels is not None:
        labels = release_to_caller(ctx, labels) if is_device(mat) else ctx.download(labels)
    return labels, out, int(n[0])


class Contour(dict):
    """One border of cv2.findContours reduced to its Green's-theorem sums (the fields of bv_contour), with its vertices
    where they were asked for."""


def outer_contours(mat, max_contours=4096, points=False, max_points=None, rects=False):
    """utils/feature.py:5-21 on the GPU: the outermost 8-connected borders of `mat != 0`, in raster
    order of their first pixel (cv2 returns the same set, in its own order).  Each record carries
    what the reference consumes next (contour_centroid / contour_area below); with `points=True`
    also the CHAIN_APPROX_SIMPLE vertices as an int32 [n,1,2] array, exactly the array cv2 returns
    (ready for cv2.minAreaRect as in modules/bins.py:60); with `rects=True` also
    `c["min_area_rect"] = ((cx, cy), (w, h), angle)`, cv2.minAreaRect of those vertices computed on
    the device (min_area_rect below)."""
    from .runtime import CONTOUR_DTYPE
    ctx = ctx_for(mat)
    h, w = mat.shape[-2], mat.shape[-1]
    points = points or rects
    if points and max_points is None:
        max_points = 4 * (h + w) + h * w // 4        # generous: borders of a very ragged mask
    table, nb, pts, npts = ctx.outer_contours(to_device(ctx, mat), max_contours=max_contours,
                                              max_points=max_points if points else 0)
    n = int(ctx.download(nb)[0])
    raw = ctx.download(table)[0, :min(n, max_contours)].copy().view(CONTOUR_DTYPE).reshape(-1)
    keep = [i for i, row in enumerate(raw) if row["external"]]
    out = [Contour({k: int(raw[i][k]) for k in CONTOUR_DTYPE.names}) for i in keep]
    if rects:
        rr = ctx.min_area_rects(table, nb, pts)[0]
        for c, i in zip(out, keep):
            q = rr[i]
            c["min_area_rect"] = ((float(q["cx"]), float(q["cy"])), (float(q["width"]), float(q["height"])),
                                  float(q["angle"])) if q["valid"] else None
    if points:
        needed = int(ctx.download(npts)[0])
        host = ctx.download(pts)[0, :min(needed, max_points)]
        for c in out:
            off = c["point_offset"]
            c["points"] = host[off:off + c["n_simple"]].reshape(-1, 1, 2).copy() if off >= 0 else None
    return out


def find_contours(mat, mode="tree", method="simple", max_contours=4096, max_points=None, shapes=False, approx_epsilon=0.0,
                  approx_relative=0.0):
    """cv2.findContours(mat, RETR_<mode>, CHAIN_APPROX_<method>) on the GPU for one mask: (contours, hierarchy) in cv2's
    shapes.  Every Contour carries `points` (int32 [n,1,2], the array cv2 returns for that border), `is_hole` and the
    Green's-theorem sums, so contour_centroid / contour_area apply to it; hierarchy is int32 [1,N,4] (next, prev,
    first_child, parent), or None when there is no border, as cv2 returns it.
    mode: "external", "list", "ccomp" or "tree"; method: "none" or "simple".  The borders are the ones cv2 finds, each
    with cv2's vertex list, ordered outer borders first (raster order of their first pixel), then hole borders (raster
    order of the hole); cv2 orders them its own way.  "external" is outer_contours(points=True) with cv2's flat
    hierarchy.  max_contours / max_points are first guesses: when a frame needs more, the call is repeated with room for
    everything it reported.
    With `shapes=True` every Contour also carries its shape descriptors, computed on the device (bv_contour_shapes):
    `arc_length` (cv2.arcLength(points, True)), `hull` (cv2.convexHull(points), int32 [k,1,2]), `approx`
    (cv2.approxPolyDP(points, approx_epsilon + approx_relative * arc_length, True), int32 [k,1,2]), `approx_convex`
    (cv2.isContourConvex(approx)), `min_enclosing_circle` ((cx, cy), r) and `min_area_rect` ((cx, cy), (w, h), angle),
    hole borders included."""
    from .runtime import CONTOUR_DTYPE
    if mode == "external":
        if method != "simple":
            raise ValueError("mode 'external' is served with CHAIN_APPROX_SIMPLE only")
        ctx = ctx_for(mat)
        dev = to_device(ctx, mat)
        h, w = mat.shape[-2], mat.shape[-1]
        _, nb, _, _ = ctx.outer_contours(dev, max_contours=max_contours)
        max_contours = max(max_contours, int(ctx.download(nb)[0]))
        max_points = max(max_points or 0, 4 * (h + w) + h * w // 4)
        if shapes:
            out = _outer_with_shapes(ctx, dev, max_contours, max_points, approx_epsilon, approx_relative)
        else:
            out = outer_contours(dev, max_contours=max_contours, points=True, max_points=max_points)
        for c in out:
            c["is_hole"] = False
        n = len(out)
        hier = np.array([[[i + 1 if i + 1 < n else -1, i - 1, -1, -1] for i in range(n)]], np.int32).reshape(1, n, 4)
        return out, (hier if n else None)
    ctx = ctx_for(mat)
    h, w = mat.shape[-2], mat.shape[-1]
    dev = to_device(ctx, mat)
    if max_points is None:
        max_points = 4 * (h + w) + h * w // 4
    # at most three calls: the vertex count covers the written records only, so it is complete once the records fit
    for _ in range(3):
        table, hier, nc, pts, npts = ctx.find_contours(dev, mode, method, max_contours=max_contours,
                                                       max_points=max_points)
        n_outer, n_holes = (int(v) for v in ctx.download(nc)[0])
        needed = int(ctx.download(npts)[0])
        if n_outer + n_holes <= max_contours and needed <= max_points:
            break
        max_contours, max_points = max(max_contours, n_outer + n_holes), max(max_points, needed)
    n = n_outer + n_holes
    raw = ctx.download(table)[0, :n].copy().view(CONTOUR_DTYPE).reshape(-1)
    host = ctx.download(pts)[0, :needed]
    none = method in ("none", ctx.CHAIN["none"])
    out = []
    for i in range(n):
        c = Contour({k: int(raw[i][k]) for k in CONTOUR_DTYPE.names})
        c["is_hole"] = i >= n_outer
        off, cnt = c["point_offset"], c["n_points"] if none else c["n_simple"]
        c["points"] = host[off:off + cnt].reshape(-1, 1, 2).copy()
        out.append(c)
    if shapes:
        _attach_shapes(ctx, out, range(n), table, nc, pts, method, approx_epsilon, approx_relative)
    return out, (ctx.download(hier)[:1, :n].copy() if n else None)


def _outer_with_shapes(ctx, dev, max_contours, max_points, approx_epsilon, approx_relative):
    """The external borders with their vertices and shape descriptors, all from one bv_outer_contours table that is
    grown until every border and every vertex fits."""
    from .runtime import CONTOUR_DTYPE
    for _ in range(3):
        table, nb, pts, npts = ctx.outer_contours(dev, max_contours=max_contours, max_points=max_points)
        n, needed = int(ctx.download(nb)[0]), int(ctx.download(npts)[0])
        if n <= max_contours and needed <= max_points:
            break
        max_contours, max_points = max(max_contours, n), max(max_points, needed)
    raw = ctx.download(table)[0, :n].copy().view(CONTOUR_DTYPE).reshape(-1)
    keep = [i for i, row in enumerate(raw) if row["external"]]
    out = [Contour({k: int(raw[i][k]) for k in CONTOUR_DTYPE.names}) for i in keep]
    host = ctx.download(pts)[0, :needed]
    for c in out:
        off = c["point_offset"]
        c["points"] = host[off:off + c["n_simple"]].reshape(-1, 1, 2).copy()
    _attach_shapes(ctx, out, keep, table, nb, pts, "simple", approx_epsilon, approx_relative)
    return out


def _attach_shapes(ctx, out, records, table, counts, pts, method, approx_epsilon, approx_relative):
    """Adds the bv_contour_shapes descriptors of record records[k] to out[k]."""
    from .runtime import SHAPE_DTYPE
    shapes, hull, approx = ctx.contour_shapes(table, counts, pts, method, approx_epsilon, approx_relative)
    sh = ctx.download(shapes)[0].copy().view(SHAPE_DTYPE).reshape(-1)
    hull, approx = ctx.download(hull)[0], ctx.download(approx)[0]
    for c, i in zip(out, records):
        s, off = sh[i], c["point_offset"]
        if not s["valid"]:
            raise RuntimeError("contour record %d has no shape descriptors" % i)
        r = s["rect"]
        c["arc_length"] = float(s["arc_length"])
        c["hull"] = hull[off:off + int(s["n_hull"])].reshape(-1, 1, 2).copy()
        c["approx"] = approx[off:off + int(s["n_approx"])].reshape(-1, 1, 2).copy()
        c["approx_convex"] = bool(s["approx_convex"])
        c["min_enclosing_circle"] = ((float(s["circle_cx"]), float(s["circle_cy"])), float(s["circle_r"]))
        c["min_area_rect"] = ((float(r["cx"]), float(r["cy"])), (float(r["width"]), float(r["height"])), float(r["angle"]))


def canny(image, threshold1, threshold2, apertureSize=3, L2gradient=False):
    """cv2.Canny(image, threshold1, threshold2, apertureSize=apertureSize, L2gradient=L2gradient) on the GPU, bit-exact:
    uint8 0/255 edges of a grey [H,W] or BGR [H,W,3] image (or a batch [B,H,W] / [B,H,W,3] of them).  Numpy in gives
    numpy out; a CUDA tensor in gives a CUDA tensor out without leaving the device, so
    `find_contours(canny(frame, ...))` runs on the device throughout."""
    ctx = ctx_for(image)
    return like_input(ctx, image, ctx.canny(to_device(ctx, image), threshold1, threshold2, apertureSize, L2gradient))


def _contour_moments(c):
    """m00, m10, m01 exactly as cv2.moments(contour) scales its sums (contourMoments: multiply by
    +-0.5 and +-1/6 in double)."""
    a00, a10, a01 = float(c["a00"]), float(c["a10"]), float(c["a01"])
    if abs(a00) <= 1.1920928955078125e-07:      # FLT_EPSILON: degenerate border, all moments 0
        return 0.0, 0.0, 0.0
    db1_2, db1_6 = (0.5, 0.16666666666666666666666666666667) if a00 > 0 else (-0.5, -0.16666666666666666666666666666667)
    return a00 * db1_2, a10 * db1_6, a01 * db1_6


def contour_centroid(contour):
    """utils/feature.py:240-252."""
    m00, m10, m01 = _contour_moments(contour)
    m00 = max(1e-10, m00)
    return int(m10 / m00), int(m01 / m00)


def contour_area(contour):
    """utils/feature.py:255-265 (cv2.contourArea, oriented=False)."""
    return abs(float(contour["a00"]) * 0.5)


def blob_centroid(blob):
    """Same rounding rule as contour_centroid (utils/feature.py:250-252): int(m10/m00), int(m01/m00)."""
    m00 = max(1e-10, float(blob["m00"]))
    return int(blob["m10"] / m00), int(blob["m01"] / m00)


def blob_area(blob):
    """Raster area in pixels (contour_area, utils/feature.py:255-265, is the polygon area)."""
    return float(blob["m00"])


def min_area_rect(contour):
    """cv2.minAreaRect(contour) (modules/bins.py:60) for a contour returned by
    `outer_contours(..., rects=True)`: ((cx, cy), (w, h), angle), angle in [-90, 0) degrees."""
    r = contour.get("min_area_rect")
    if r is None:
        raise ValueError("contour carries no rectangle: call outer_contours(..., rects=True)")
    return r


def min_enclosing_rect(contour):
    """utils/feature.py:301-312."""
    return min_area_rect(contour)
