"""TEST INFRASTRUCTURE ONLY -- seeded frames at the edges of the colour balance's per-frame statistics.

`synth.gen_underwater` and random bytes give broad histograms whose cumulative counts never land on a percentile
bound, channel means that are never equal and S / V ranges that are never empty, so they cannot tell a right
statistic from a subtly wrong one.  Every generator here returns `(frame, claim)`: the uint8 BGR frame and a dict
stating the property it was built to have, which tests/test_balance_edge_frames.py checks independently.
"""
import numpy as np
import cv2

from . import synth

F32 = np.float32


def f32_bounds(n):
    """Percentile bounds of color_balance.cpp:113-114: float32 products (of a float32-rounded n) truncated to int."""
    return int(F32(0.002) * F32(n)), n - int(F32(0.998) * F32(n))


def f64_bounds(n):
    """The same bounds computed in double: what a kernel that skipped the float32 rounding would use."""
    return int(0.002 * n), n - int(0.998 * n)


# ---------------------------------------------------------------------------------------------------------------------
# exact-bound frames
# ---------------------------------------------------------------------------------------------------------------------
# per channel (B, G, R): value of the low-tail pixels, value range of the bulk (inclusive), value of the high-tail pixels
BGR_LEVELS = ((12, (40, 230), 250), (7, (30, 200), 236), (3, (16, 150), 201))
BGR_OFFSETS = ((-1, 1), (0, 0), (1, -1))   # (low, high) count offsets from the bounds, per channel


def exact_bound_frame(height, width, seed, offsets=BGR_OFFSETS):
    """Channel c has exactly lb + offsets[c][0] pixels at a low value and hb + offsets[c][1] at a high value (lb, hb:
    the float32 bounds), every other pixel strictly in between.  A cumulative count then lands on, just below or just
    above each bound, which decides whether the tail value or the first bulk value is the clipping limit.
    claim: lb, hb, per-channel low / high counts and the (lo, hi) limits that the reference's rule gives."""
    n = height * width
    lb, hb = f32_bounds(n)
    rng = np.random.default_rng(seed)
    img = np.empty((n, 3), np.uint8)
    claim = dict(lb=lb, hb=hb, n_low=[], n_high=[], limits=[], low=[], high=[])
    for c, (low, (b0, b1), high) in enumerate(BGR_LEVELS):
        k_lo, k_hi = lb + offsets[c][0], hb + offsets[c][1]
        if k_lo < 0 or k_hi < 0 or k_lo + k_hi > n:
            raise ValueError("offsets %s do not fit a %dx%d frame (lb %d, hb %d)" % (offsets[c], height, width, lb, hb))
        ch = rng.integers(b0, b1 + 1, n).astype(np.uint8)
        where = rng.permutation(n)
        # the bulk's extremes at least twice each: a tail one short of its bound is then crossed by the next value
        ch[where[n - 4:n - 2]], ch[where[n - 2:]] = b0, b1
        ch[where[:k_lo]] = low
        ch[where[k_lo:k_lo + k_hi]] = high
        img[:, c] = ch
        bulk = ch[where[k_lo + k_hi:]]
        # percentile_min_max: the first value whose inclusive prefix count exceeds lb, the last whose suffix exceeds hb
        lo = low if k_lo > lb else int(bulk.min()) if bulk.size else high
        hi = high if k_hi > hb else int(bulk.max()) if bulk.size else low
        claim["n_low"].append(k_lo)
        claim["n_high"].append(k_hi)
        claim["limits"].append((lo, hi))
        claim["low"].append(low)
        claim["high"].append(high)
    return img.reshape(height, width, 3), claim


# A palette whose cv2 S and V are fixed: the two S-tail colours sit in the middle of the V range and the two V-tail
# colours in the middle of the S range, so each tail decides one bound only.  Under equalize_rgb=False,
# rgb_extrema_clipping=False the pass-1 tables are the identity and these are the S / V histograms of pass 2.
SV_TAILS = dict(s_low=(140, 140, 134), s_high=(140, 16, 20), v_low=(40, 24, 30), v_high=(250, 150, 200))
SV_BULK = dict(s=(30, 200), v=(60, 230))     # S and V of every bulk colour lie in these ranges (inclusive)
SV_FLAGS = dict(equalize_rgb=False, rgb_extrema_clipping=False)


def bgr_to_sv(colors):
    """cv2's S and V of an (n, 3) uint8 array of BGR colours."""
    hsv = cv2.cvtColor(np.ascontiguousarray(colors, np.uint8).reshape(-1, 1, 3), cv2.COLOR_BGR2HSV).reshape(-1, 3)
    return hsv[:, 1], hsv[:, 2]


def exact_bound_sv_frame(height, width, seed, offsets=((0, 1), (1, -1))):
    """S / V counterpart of exact_bound_frame: exactly lb + offsets[0][0] pixels at the lowest S, hb + offsets[0][1] at
    the highest S, and likewise (offsets[1]) at the lowest / highest V; the bulk colours lie strictly inside both
    ranges.  Meant for SV_FLAGS.  claim: lb, hb, the tail S / V values and counts, the expected (s_min, s_max),
    (v_min, v_max)."""
    n = height * width
    lb, hb = f32_bounds(n)
    rng = np.random.default_rng(seed)
    tails = {k: np.array(v, np.uint8) for k, v in SV_TAILS.items()}
    tail_s, tail_v = bgr_to_sv(np.stack(list(tails.values())))
    tsv = {k: (int(s), int(v)) for k, s, v in zip(tails, tail_s, tail_v)}
    counts = dict(s_low=lb + offsets[0][0], s_high=hb + offsets[0][1], v_low=lb + offsets[1][0], v_high=hb + offsets[1][1])
    if min(counts.values()) < 0 or sum(counts.values()) > n:
        raise ValueError("offsets %s do not fit a %dx%d frame (lb %d, hb %d)" % (offsets, height, width, lb, hb))
    n_bulk = n - sum(counts.values())
    bulk = np.empty((0, 3), np.uint8)
    while bulk.shape[0] < n_bulk:
        cand = rng.integers(0, 256, (max(4 * n_bulk, 1024), 3)).astype(np.uint8)
        s, v = bgr_to_sv(cand)
        keep = (s >= SV_BULK["s"][0]) & (s <= SV_BULK["s"][1]) & (v >= SV_BULK["v"][0]) & (v <= SV_BULK["v"][1])
        bulk = np.concatenate([bulk, cand[keep]])
    pix = np.concatenate([bulk[:n_bulk]] + [np.repeat(tails[k][None], counts[k], 0) for k in tails])
    pix = pix[rng.permutation(n)]
    bs, bv = bgr_to_sv(bulk[:n_bulk])

    def limits(lo_key, hi_key, bulk_ch, idx):
        lo = tsv[lo_key][idx] if counts[lo_key] > lb else int(bulk_ch.min())
        hi = tsv[hi_key][idx] if counts[hi_key] > hb else int(bulk_ch.max())
        return lo, hi
    claim = dict(lb=lb, hb=hb, counts=counts, tail_sv=tsv, s_limits=limits("s_low", "s_high", bs, 0),
                 v_limits=limits("v_low", "v_high", bv, 1))
    return pix.reshape(height, width, 3), claim


# ---------------------------------------------------------------------------------------------------------------------
# tie frames
# ---------------------------------------------------------------------------------------------------------------------
TIE_PATTERNS = ("b=g>r", "b=r>g", "g=r>b", "b=g=r", "b>g=r", "g>b=r", "r>b=g")


def _swap_cols(p):
    """x -> x ^ 1: a permutation of the pixels inside every tile whose columns start and end on even indices."""
    q = p.copy()
    w = p.shape[1] - p.shape[1] % 2
    q[:, 0:w:2], q[:, 1:w:2] = p[:, 1:w:2], p[:, 0:w:2]
    return q


def _swap_rows(p):
    q = p.copy()
    h = p.shape[0] - p.shape[0] % 2
    q[0:h:2], q[1:h:2] = p[1:h:2], p[0:h:2]
    return q


def tie_frame(height, width, seed, pattern):
    """The channels named equal in `pattern` carry the same pixels in a different order (adjacent columns / rows
    swapped), so their histograms -- hence their clipped sums and means -- are exactly equal, globally and in every
    tile of even width and height; the other channel is a darker copy with a strictly lower clipped mean.
    claim: pattern, the equal channels and the strict order of the means."""
    if pattern not in TIE_PATTERNS:
        raise ValueError(pattern)
    base = synth.gen_underwater(height, width, seed)[..., 0]                   # the broad blue plane
    low = (base.astype(np.int32) * 5 // 8 + 3).astype(np.uint8)
    hi_side, lo_side = pattern.split(">") if ">" in pattern else (pattern, "")
    top = hi_side.split("=")
    bottom = lo_side.split("=") if lo_side else []
    img = np.empty((height, width, 3), np.uint8)
    perms = [lambda p: p, _swap_cols, _swap_rows]
    for k, name in enumerate(top):
        img[..., "bgr".index(name)] = perms[k](base)
    for k, name in enumerate(bottom):
        img[..., "bgr".index(name)] = perms[k](low)
    equal = top if len(top) > 1 else bottom
    return img, dict(pattern=pattern, equal=equal, higher=top, lower=bottom)


# ---------------------------------------------------------------------------------------------------------------------
# zero-width frames: an S or V range of zero width after the percentile clipping (the reference divides by zero there)
# ---------------------------------------------------------------------------------------------------------------------
ZERO_WIDTH_KINDS = ("constant", "black", "white", "grey", "red_free", "sparse_red", "v_constant")


def zero_width_frame(height, width, seed, kind):
    """claim: kind, which of S / V the frame makes zero-width ("s", "v" or "sv") and the process_frame flags it is
    meant for.  `v_constant` (V fixed at 200, S varying) needs the identity pass-1 tables of SV_FLAGS; the others hold
    under the default flags.  `sparse_red` carries red on fewer pixels than the low bound (< 0.2 %), so the
    percentile clipping removes it and the frame balances like `red_free`."""
    rng = np.random.default_rng(seed)
    flags = {}
    if kind == "constant":
        img, zero = np.empty((height, width, 3), np.uint8), "sv"
        img[...] = (90, 120, 60)
    elif kind == "black":
        img, zero = np.zeros((height, width, 3), np.uint8), "sv"
    elif kind == "white":
        img, zero = np.full((height, width, 3), 255, np.uint8), "sv"
    elif kind == "grey":
        img, zero = np.repeat(rng.integers(0, 256, (height, width, 1), dtype=np.uint8), 3, axis=2), "s"
    elif kind in ("red_free", "sparse_red"):
        img, zero = synth.gen_underwater(height, width, seed), "s"
        img[..., 2] = 0
        if kind == "sparse_red":
            n = height * width
            k = max(f32_bounds(n)[0], 1) - 1 if n >= 1000 else 0
            where = rng.permutation(n)[:k]
            img.reshape(-1, 3)[where, 2] = rng.integers(60, 256, k).astype(np.uint8)
    elif kind == "v_constant":
        img = rng.integers(0, 201, (height, width, 3)).astype(np.uint8)
        img[..., 0] = 200
        zero, flags = "v", dict(SV_FLAGS)
    else:
        raise ValueError(kind)
    return img, dict(kind=kind, zero=zero, flags=flags)


# ---------------------------------------------------------------------------------------------------------------------
# saturation
# ---------------------------------------------------------------------------------------------------------------------
GLARE_SHAPE = (4128, 4224)   # 17.4 M pixels: a full-white channel sums to more than 2^32


def glare_frame(height, width, seed, white=0.96):
    """A fraction `white` of the pixels is (255, 255, 255) glare, the rest an underwater frame: one hot histogram bin
    per channel.  claim: the white count and the three channel sums."""
    img = synth.gen_underwater(height, width, seed)
    n = height * width
    k = int(round(white * n))
    img.reshape(-1, 3)[np.random.default_rng(seed).permutation(n)[:k]] = 255
    sums = tuple(int(img[..., c].sum(dtype=np.int64)) for c in range(3))
    return img, dict(n_white=k, sums=sums)


# ---------------------------------------------------------------------------------------------------------------------
# HSI branch edges
# ---------------------------------------------------------------------------------------------------------------------
PRIMARIES = ((255, 0, 0), (0, 255, 0), (0, 0, 255), (255, 255, 0), (0, 255, 255), (255, 0, 255))


def hsi_edge_frame(height, width, seed):
    """An underwater frame with bands of grey pixels (hue 0/0), black pixels (I = 0) and pure primaries and
    secondaries (hue on a sector boundary).  claim: the pixel count of each band."""
    img = synth.gen_underwater(height, width, seed)
    rng = np.random.default_rng(seed)
    band = height // 8
    img[:band] = np.repeat(rng.integers(0, 256, (band, width, 1), dtype=np.uint8), 3, axis=2)   # grey
    img[band:band + band // 2] = 0                                                                # black
    prim = np.array(PRIMARIES, np.uint8)
    img[2 * band:3 * band] = prim[rng.integers(0, len(prim), (band, width))]
    return img, dict(grey=band * width, black=(band // 2) * width, primaries=band * width)
