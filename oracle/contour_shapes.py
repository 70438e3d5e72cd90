"""TEST INFRASTRUCTURE ONLY -- the shape descriptors of bv_contour_shapes restated on the host, step for step as the
kernels compute them (csrc/rects.cu), so that tests/test_contour_shapes_oracle.py can pin them against cv2 4.13.0 on the
CPU and tests/test_gpu_contour_shapes.py can hold the device to them.

  arc_length       cv2.arcLength(c, True): float32 steps sqrt(dx^2 + dy^2), summed in double (any order: exact)
  convex_hull      cv2.convexHull(c): Andrew's monotone chain (counter-clockwise in y-up axes, collinear points dropped),
                   started where cv2 starts it (`hull_start`)
  approx_poly_dp   cv2.approxPolyDP(c, eps, True): OpenCV 4.13's approxPolyDP_ for a closed int curve (splits on the
                   distance to the chord segment)
  is_contour_convex cv2.isContourConvex on int points
  enclosing_circle the exact minimum enclosing circle of the hull in double (cv2.minEnclosingCircle is within a
                   stated tolerance of it, plus its EPS = 1e-4 on the radius)
"""
import numpy as np


def _pts(c):
    return [(int(x), int(y)) for x, y in np.asarray(c).reshape(-1, 2)]


def arc_length(c, order=None):
    p = np.asarray(c).reshape(-1, 2).astype(np.float32)
    if len(p) == 0:
        return 0.0
    d = p - np.roll(p, 1, axis=0)
    steps = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1], dtype=np.float32)
    if order is not None:
        steps = steps[order]
    total = 0.0
    for s in steps:
        total += float(s)
    return total


def _cross(o, a, b):
    return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])


def monotone_chain(points):
    """Convex hull of the distinct points, counter-clockwise in y-up axes, from the smallest (x, y); collinear dropped."""
    pts = sorted(set(points))
    if len(pts) <= 2:
        return pts
    lower, upper = [], []
    for q in pts:
        while len(lower) >= 2 and _cross(lower[-2], lower[-1], q) <= 0:
            lower.pop()
        lower.append(q)
    for q in reversed(pts):
        while len(upper) >= 2 and _cross(upper[-2], upper[-1], q) <= 0:
            upper.pop()
        upper.append(q)
    return lower[:-1] + upper[:-1]


def hull_start(points, hull):
    """Index into `hull` of cv2.convexHull's first vertex.  Each hull vertex is given the index of its first visit in
    the contour; where those indices run cyclically upwards cv2 starts at the smallest, where they run downwards at the
    largest, and otherwise (and for hulls of 1 or 2 vertices) at the largest (x, y)."""
    top = hull.index(max(hull)) if hull else 0
    m = len(hull)
    if m < 3:
        return top
    first = {}
    for i, q in enumerate(points):
        first.setdefault(q, i)
    idx = [first[q] for q in hull]
    ups = sum(idx[(k + 1) % m] > idx[k] for k in range(m))
    if ups == m - 1:
        return idx.index(min(idx))
    if ups == 1:
        return idx.index(max(idx))
    return top


def convex_hull(c):
    points = _pts(c)
    hull = monotone_chain(points)
    s = hull_start(points, hull)
    return np.array(hull[s:] + hull[:s], np.int32).reshape(-1, 1, 2)


def has_repeated_pixel(c):
    points = _pts(c)
    return len(set(points)) != len(points)


def _segment_dist2(p, sp, ep, dx, dy):
    """Squared distance of p to the segment sp -> ep (dx, dy = ep - sp), as cv2 4.13 measures it when it splits a
    slice: to the nearer end where p projects outside the segment, else cross^2 / length^2 (one rounding)."""
    px, py = float(p[0] - sp[0]), float(p[1] - sp[1])
    dot = px * dx + py * dy
    l2 = dx * dx + dy * dy
    if dot <= 0:
        return px * px + py * py
    if dot >= l2:
        qx, qy = float(p[0] - ep[0]), float(p[1] - ep[1])
        return qx * qx + qy * qy
    cr = py * dx - px * dy
    return cr * cr / l2


def approx_poly_dp(c, eps):
    """OpenCV 4.13's approxPolyDP_ (closed curve, int points): farthest-point initialisation over 3 passes, the slice
    stack split at the point farthest from the slice's chord SEGMENT (first maximum; the slice is kept whole when that
    squared distance is <= eps^2), the final clean-up.  Integer coordinates make every step exact in double except
    the one division of the squared cross product."""
    src = _pts(c)
    n = len(src)
    if n == 0:
        return np.zeros((0, 1, 2), np.int32)
    eps = float(eps) * float(eps)
    dst = []
    stack = []
    pos, rs, le_eps = 0, 0, False
    start = src[0]
    for _ in range(3):
        pos = (pos + rs) % n
        start = src[pos]
        max_dist = 0.0
        for j in range(1, n):
            p = src[(pos + j) % n]
            dx, dy = float(p[0] - start[0]), float(p[1] - start[1])
            d = dx * dx + dy * dy
            if d > max_dist:
                max_dist, rs = d, j
        le_eps = max_dist <= eps
    if not le_eps:
        s0, e0 = pos, (rs + pos) % n
        stack.append((e0, s0))
        stack.append((s0, e0))
    else:
        dst.append(start)
    while stack:
        s0, e0 = stack.pop()
        sp, ep = src[s0], src[e0]
        if (s0 + 1) % n != e0:
            dx, dy = float(ep[0] - sp[0]), float(ep[1] - sp[1])
            max_dist, split = 0.0, None
            k = (s0 + 1) % n
            while k != e0:
                p = src[k]
                d = _segment_dist2(p, sp, ep, dx, dy)
                if d > max_dist:
                    max_dist, split = d, k
                k = (k + 1) % n
            le_eps = max_dist <= eps
        else:
            le_eps = True
        if le_eps:
            dst.append(sp)
        else:
            stack.append((split, e0))
            stack.append((s0, split))
    # clean-up of the points on [almost] straight lines
    count = new_count = len(dst)
    rp = count - 1
    st = dst[rp]
    rp = (rp + 1) % count
    wpos = rp
    pt = dst[rp]
    rp = (rp + 1) % count
    i = 0
    while i < count and new_count > 2:
        en = dst[rp]
        rp = (rp + 1) % count
        dx, dy = float(en[0] - st[0]), float(en[1] - st[1])
        dist = abs(float(pt[0] - st[0]) * dy - float(pt[1] - st[1]) * dx)
        sip = float((pt[0] - st[0]) * (en[0] - pt[0]) + (pt[1] - st[1]) * (en[1] - pt[1]))
        if dist * dist <= 0.5 * eps * (dx * dx + dy * dy) and dx != 0 and dy != 0 and sip >= 0:
            new_count -= 1
            dst[wpos] = st = en
            wpos = (wpos + 1) % count
            pt = dst[rp]
            rp = (rp + 1) % count
            i += 2
            continue
        dst[wpos] = st = pt
        wpos = (wpos + 1) % count
        pt = en
        i += 1
    return np.array(dst[:new_count], np.int32).reshape(-1, 1, 2)


def is_contour_convex(c):
    p = _pts(c)
    n = len(p)
    if n < 3:
        return False
    prev, cur = p[n - 2], p[n - 1]
    dx0, dy0 = cur[0] - prev[0], cur[1] - prev[1]
    orientation = 0
    for i in range(n):
        prev, cur = cur, p[i]
        dx, dy = cur[0] - prev[0], cur[1] - prev[1]
        a, b = dx * dy0, dy * dx0
        orientation |= 1 if b > a else (2 if b < a else 3)
        if orientation == 3:
            return False
        dx0, dy0 = dx, dy
    return True


def _circle2(a, b):
    cx, cy = (a[0] + b[0]) / 2.0, (a[1] + b[1]) / 2.0
    return cx, cy, ((a[0] - b[0]) ** 2 + (a[1] - b[1]) ** 2) / 4.0


def _circle3(a, b, c):
    bx, by, cx, cy = b[0] - a[0], b[1] - a[1], c[0] - a[0], c[1] - a[1]
    d = 2.0 * (bx * cy - by * cx)
    b2, c2 = bx * bx + by * by, cx * cx + cy * cy
    ux, uy = (cy * b2 - by * c2) / d, (bx * c2 - cx * b2) / d
    return a[0] + ux, a[1] + uy, ux * ux + uy * uy


def enclosing_circle(c):
    """((cx, cy), r) of the exact minimum enclosing circle of the contour's hull, in double (no EPS)."""
    h = monotone_chain(_pts(c))
    out = lambda cc, p: (p[0] - cc[0]) ** 2 + (p[1] - cc[1]) ** 2 > cc[2] * (1 + 1e-12)
    cc = (float(h[0][0]), float(h[0][1]), 0.0)
    for i in range(1, len(h)):
        if not out(cc, h[i]):
            continue
        cc = (float(h[i][0]), float(h[i][1]), 0.0)
        for j in range(i):
            if not out(cc, h[j]):
                continue
            cc = _circle2(h[i], h[j])
            for k in range(j):
                if out(cc, h[k]):
                    cc = _circle3(h[i], h[j], h[k])
    return (cc[0], cc[1]), float(np.sqrt(cc[2]))
