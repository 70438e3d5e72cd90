"""TEST INFRASTRUCTURE ONLY -- cv2.findContours(RETR_LIST / CCOMP / TREE) restated in the record order of
bv_find_contours.

cv2 lists the borders of RETR_LIST / CCOMP / TREE in an order that follows no raster rule.  The library orders them
outer borders first (raster order of the component's first pixel), then hole borders (raster order of the hole's first
pixel).  `canonical` re-orders cv2's output into that order and remaps the hierarchy; the borders are matched through
their CHAIN_APPROX_NONE start pixels, which are (checked by tests/test_contour_tree_oracle.py against cv2 4.13.0):
  * outer border: the component's first pixel in raster order;
  * hole border: the pixel immediately left of the hole's first pixel (it belongs to the enclosing component).
`regions` derives, from scipy labellings alone, which borders exist, where they start and what encloses them; the
CPU test pins cv2 against it.
"""
import numpy as np
import cv2
from scipy import ndimage

MODES = {"list": cv2.RETR_LIST, "ccomp": cv2.RETR_CCOMP, "tree": cv2.RETR_TREE}
METHODS = {"none": cv2.CHAIN_APPROX_NONE, "simple": cv2.CHAIN_APPROX_SIMPLE}


def _raster_labels(labels, n):
    """Renumbers labels 1..n by raster order of their first pixel; returns (labels, first flat index per label)."""
    flat = labels.ravel()
    first = np.full(n + 1, flat.size, np.int64)
    np.minimum.at(first, flat, np.arange(flat.size, dtype=np.int64))
    order = np.argsort(first[1:], kind="stable")
    remap = np.zeros(n + 1, np.int32)
    remap[order + 1] = np.arange(1, n + 1, dtype=np.int32)
    return remap[labels], first[1:][order]


def regions(mask):
    """What the borders of `mask != 0` must be, from scipy labellings:
      fg: int32 [H,W] 8-connected component labels 1..n_outer in raster order of first pixel (0: background)
      hole: int32 [H,W] 1 + hole index of every background pixel in a hole (0: foreground or a region touching the edge)
      outer_start: [(x, y)] first pixel of every component; hole_start: [(x, y)] pixel left of every hole's first pixel
      parent_tree: the RETR_TREE parent of every record (outer records, then hole records)."""
    m = np.asarray(mask) != 0
    h, w = m.shape
    fg, n_fg = ndimage.label(m, structure=np.ones((3, 3), bool))
    fg, fg_first = _raster_labels(fg, n_fg)
    bg, n_bg = ndimage.label(~m)                                  # 4-connected
    edge = np.unique(np.concatenate([bg[0], bg[-1], bg[:, 0], bg[:, -1]]))
    is_hole = np.ones(n_bg + 1, bool)
    is_hole[edge] = False
    is_hole[0] = False
    hole_ids = np.zeros(n_bg + 1, np.int32)
    hole_ids[is_hole] = np.arange(1, int(is_hole.sum()) + 1, dtype=np.int32)
    hole, hole_first = _raster_labels(hole_ids[bg], int(is_hole.sum()))
    outer_start = [(int(i % w), int(i // w)) for i in fg_first]
    hole_start = [(int(i % w) - 1, int(i // w)) for i in hole_first]
    n_outer = len(outer_start)
    parent = []
    for x, y in outer_start:
        k = int(hole[y, x - 1]) if x > 0 else 0
        parent.append(n_outer + k - 1 if k else -1)
    for x, y in hole_start:
        parent.append(int(fg[y, x]) - 1)
    return dict(fg=fg, hole=hole, outer_start=outer_start, hole_start=hole_start, parent_tree=parent)


def simple_from_none(points):
    """CHAIN_APPROX_SIMPLE as a function of the CHAIN_APPROX_NONE list: drop every point where the step direction does
    not change, cyclically, keeping NONE's order."""
    p = np.asarray(points).reshape(-1, 2)
    if len(p) < 2:
        return p.reshape(-1, 1, 2).copy()
    step = np.roll(p, -1, axis=0) - p                             # step i: p[i] -> p[i+1]
    keep = np.any(step != np.roll(step, 1, axis=0), axis=1)       # step i differs from step i-1
    return p[keep].reshape(-1, 1, 2).copy()


def record_order(mask, cv_none, reg=None):
    """perm[r] = index in cv2's list of the border that is record r, from cv2's CHAIN_APPROX_NONE contours."""
    reg = regions(mask) if reg is None else reg
    where = {s: r for r, s in enumerate(reg["outer_start"])}
    n_outer = len(reg["outer_start"])
    where.update({s: n_outer + r for r, s in enumerate(reg["hole_start"])})
    perm = [None] * len(where)
    for i, c in enumerate(cv_none):
        start = (int(c[0, 0, 0]), int(c[0, 0, 1]))
        r = where[start]
        assert perm[r] is None, "two cv2 contours start at %s" % (start,)
        perm[r] = i
    assert len(cv_none) == len(perm) and all(i is not None for i in perm), "cv2's borders are not the expected set"
    return perm


def remap_hierarchy(hierarchy, perm):
    """cv2's hierarchy [1,N,4] re-indexed into record order: row r is cv2's row perm[r] with every index remapped."""
    n = len(perm)
    if n == 0:
        return np.zeros((0, 4), np.int32)
    inv = np.empty(n + 1, np.int64)
    inv[np.asarray(perm)] = np.arange(n)
    inv[n] = -1                                                    # index -1 -> -1
    rows = np.asarray(hierarchy).reshape(-1, 4)[np.asarray(perm)]
    return inv[np.where(rows < 0, n, rows)].astype(np.int32)


def canonical(mask, mode="tree", method="simple", reg=None):
    """cv2.findContours(mask, mode, method) in the library's record order:
      contours: list of int32 [n,1,2] arrays; hierarchy: int32 [N,4] remapped (cv2's sibling order, not the library's);
      parent: hierarchy[:, 3]; perm: record -> cv2 index; n_outer, n_holes; none: the CHAIN_APPROX_NONE contours."""
    mask = np.ascontiguousarray(mask)
    reg = regions(mask) if reg is None else reg
    cv_none, h_none = cv2.findContours(mask, MODES[mode], cv2.CHAIN_APPROX_NONE)
    cv_out, h_out = (cv_none, h_none) if method == "none" else cv2.findContours(mask, MODES[mode], METHODS[method])
    perm = record_order(mask, cv_none, reg)
    hier = remap_hierarchy(h_out, perm) if h_out is not None else np.zeros((0, 4), np.int32)
    return dict(contours=[cv_out[i] for i in perm], none=[cv_none[i] for i in perm], hierarchy=hier,
                parent=hier[:, 3].copy(), perm=perm, n_outer=len(reg["outer_start"]), n_holes=len(reg["hole_start"]),
                cv_contours=cv_out, cv_hierarchy=h_out)


def restore(canon):
    """Inverse of `canonical`: cv2's own list and hierarchy back from the record order."""
    perm = canon["perm"]
    n = len(perm)
    contours = [None] * n
    rows = np.zeros((n, 4), np.int32)
    for r, i in enumerate(perm):
        contours[i] = canon["contours"][r]
        rows[i] = [perm[v] if v >= 0 else -1 for v in canon["hierarchy"][r]]
    return contours, (rows.reshape(1, n, 4) if n else None)


def record_links(parent):
    """(next, prev, first_child) of the library's rule: siblings (records with the same parent) linked in increasing
    record order; first_child is the smallest child."""
    n = len(parent)
    nxt, prv, first = [-1] * n, [-1] * n, [-1] * n
    last = {}
    for r, p in enumerate(parent):
        if p in last:
            nxt[last[p]] = r
            prv[r] = last[p]
        elif p >= 0:
            first[p] = r
        last[p] = r
    return np.array([nxt, prv, first], np.int32).T.reshape(n, 3)


def expected_parent(reg, mode):
    """Parents of the records for a mode from the scipy regions (facts of RETR_TREE; CCOMP and LIST derived)."""
    n_outer = len(reg["outer_start"])
    tree = reg["parent_tree"]
    if mode == "tree":
        return list(tree)
    if mode == "ccomp":
        return [-1] * n_outer + tree[n_outer:]
    return [-1] * len(tree)
