"""TEST INFRASTRUCTURE ONLY -- seeded cases for binary and grey morphology (csrc/morph.cu) and the labelling behind them
(csrc/ccl.cu).

The fused stage (bv_stage) runs its morphology steps on bit-packed masks, and `morph_bits_chain` picks one of three
families for the whole list of steps:

  roll<R,N,K>   morph_roll_kernel: every elementary step a square (2R+1)^2 element, R = 1 or 2, N = 1, 2 or 4 steps,
                rows of at most 128 words (K = words per lane); one warp walks down a strip of rows
  chain<T>      morph_chain_kernel: a tile of T shared-memory rows (32..256, a multiple of 32) holding the output rows plus
                the halo of every step; "+48k" when the launch opts in to more than 48 KiB; the TMA variant stages a
                tile by bulk copy only when the tile's byte range is 16-byte aligned
  step          morph_bits_kernel, one launch per pass of every erosion / dilation, when the chain does not qualify: a
                GRADIENT step, a horizontal extent over 31, more than 256 tile rows or more than 200 KiB

`expected_morph_path` restates that choice, `expected_grey_path` restates bv_morph's (separable rectangle or run list).
Every case carries the path it was written for; tests/test_morph_cases.py checks that it still reaches that path and
that together the cases reach every reachable one; tests/test_gpu_morph_ccl_paths.py runs them on the device against
cv2 and oracle/ccl.py.
"""
from dataclasses import dataclass, field

import cv2
import numpy as np

OPS = ("erode", "dilate", "open", "close", "gradient")
CV_OP = {"erode": cv2.MORPH_ERODE, "dilate": cv2.MORPH_DILATE, "open": cv2.MORPH_OPEN, "close": cv2.MORPH_CLOSE,
         "gradient": cv2.MORPH_GRADIENT}

# csrc/morph.cu
CHAIN_MAX_ROWS = 256                 # a tile holds at most 256 shared-memory rows
CHAIN_MAX_SMEM = 200 * 1024          # and at most 200 KiB (A and B images)
SMEM_DEFAULT = 48 * 1024             # above this the launch opts in with cudaFuncSetAttribute
BITS_PASS_MAX = 31                   # morph_bits_kernel: extents of at most 31 px per pass
GREY_MAX_RUNS = 256                  # kMaxRuns: runs of one grey launch, and rows of one vertical pass
SM_COUNT = 148                       # B200


def words_per_row(width):
    return (width + 31) // 32


# ---------------------------------------------------------------------------------------------------------------------
# the binary path choice
# ---------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class MorphPath:
    kind: str                        # "roll", "chain" or "step"
    r: int = 0                       # roll: radius, steps, words per lane
    n: int = 0
    k: int = 0
    strips: int = 0                  # roll: strips per frame, rows per strip
    strip_rows: int = 0
    rows: int = 0                    # chain: shared-memory rows, output rows per tile, tiles per frame, bytes
    tile_rows: int = 0
    tiles: int = 0
    smem: int = 0
    passes: tuple = ()               # step: per step (op, passes its horizontal / vertical extent needs), "zero" (a
                                     # GRADIENT that clears the mask) or () (identity); a basic takes max(h, v) passes

    def __str__(self):
        if self.kind == "roll":
            return "roll<%d,%d,%d>" % (self.r, self.n, self.k)
        if self.kind == "chain":
            return "chain<%d>%s" % (self.rows, "+48k" if self.smem > SMEM_DEFAULT else "")
        return "step"

    @property
    def family(self):
        """The kernel the profiler sees (BV_LAUNCH names a kernel by its source token); None for a step path whose steps
        are all identities or cleared gradients (a memset, no morphology kernel)."""
        if self.kind == "step" and not any(isinstance(e, tuple) and e for e in self.passes):
            return None
        return {"roll": "morph_roll_kernel", "chain": "morph_chain_kernel", "step": "morph_bits_kernel"}[self.kind]


def elementary_steps(steps):
    """morph_bits_chain's list of elementary (erode, L, R, U, D), or None when the chain does not qualify."""
    out = []
    for op, kw, kh, it in steps:
        if op == "gradient":
            return None
        if it < 1 or (kw == 1 and kh == 1):
            continue
        ax, ay = kw // 2, kh // 2
        L, R, U, D = ax * it, (kw - 1 - ax) * it, ay * it, (kh - 1 - ay) * it
        if L > 31 or R > 31 or U > 256 or D > 256:
            return None
        first_erode = op in ("erode", "open")
        for e in range(2 if op in ("open", "close") else 1):
            out.append((first_erode if e == 0 else not first_erode, L, R, U, D))
    return out


def roll_strips(batch, height, sm_count=SM_COUNT, warps=0):
    """launch_roll: (strips per frame, rows per strip)."""
    wps = warps if warps > 0 else 8
    strips = (sm_count * wps + batch - 1) // batch
    strips = max(1, min(strips, (height + 3) // 4))
    strip_rows = (height + strips - 1) // strips
    return (height + strip_rows - 1) // strip_rows, strip_rows


def rect_extents(kw, kh, it, height, width):
    """Taps x-L .. x+R, y-U .. y+D of a kw x kh rectangle applied `it` times, clipped to the frame."""
    ax, ay = kw // 2, kh // 2
    return (min(ax * it, width - 1), min((kw - 1 - ax) * it, width - 1), min(ay * it, height - 1),
            min((kh - 1 - ay) * it, height - 1))


def bits_passes(extents):
    m = max(extents)
    return 1 if m <= BITS_PASS_MAX else (m + 30) // 31


def expected_morph_path(steps, batch, h, w, variant=0, sm_count=SM_COUNT, warps=0):
    """What morph_bits_chain / morph_bits_rect launch for `steps` [(op, kw, kh, iterations)] on a [batch, h, w] mask
    with BV_OPT_MORPH_VARIANT = variant and BV_OPT_MORPH_WARPS = warps."""
    el = elementary_steps(steps)
    wpr = words_per_row(w)
    if el is not None:
        if el and wpr <= 128 and variant == 0:
            r = el[0][1]
            if 1 <= r <= 2 and all(e[1:] == (r, r, r, r) for e in el) and len(el) in (1, 2, 4):
                strips, strip_rows = roll_strips(batch, h, sm_count, warps)
                return MorphPath("roll", r=r, n=len(el), k=(wpr + 31) // 32, strips=strips, strip_rows=strip_rows)
        halo = sum(e[3] + e[4] for e in el)
        rows = 32
        while rows - halo < rows // 2:
            rows += 32
        smem = 2 * rows * wpr * 4
        if rows <= CHAIN_MAX_ROWS and smem <= CHAIN_MAX_SMEM:
            tile_rows = rows - halo
            return MorphPath("chain", rows=rows, tile_rows=tile_rows, tiles=(h + tile_rows - 1) // tile_rows, smem=smem)
    passes = []
    for op, kw, kh, it in steps:
        if it < 1 or (kw == 1 and kh == 1):
            passes.append("zero" if op == "gradient" else ())
            continue
        L, R, U, D = rect_extents(kw, kh, it, h, w)
        passes.append((op, bits_passes((L, R)), bits_passes((U, D))))
    return MorphPath("step", passes=tuple(passes))


def tma_staged_tiles(path, batch, h, w, halo_up):
    """morph_chain_kernel<true>: {(frame, tile): staged by bulk copy} for a chain path; `frame` counts from the start of
    the bits scratch (the stage's chunks all index one scratch image, which cudaMalloc aligns)."""
    wpr = words_per_row(w)
    out = {}
    for f in range(batch):
        for t in range(path.tiles):
            ybase = t * path.tile_rows - halo_up
            ya, yb = max(ybase, 0), min(ybase + path.rows, h)
            g = ((f * h + ya) * wpr) * 4
            d = (ya - ybase) * wpr * 4
            nbytes = (yb - ya) * wpr * 4
            out[(f, t)] = yb > ya and (g | d | nbytes) % 16 == 0
    return out


def halo_up(steps):
    el = elementary_steps(steps) or []
    return sum(e[3] for e in el)


def reachable_morph_paths():
    """Every binary path label some input reaches."""
    out = {"roll<%d,%d,%d>" % (r, n, k) for r in (1, 2) for n in (1, 2, 4) for k in (1, 2, 3, 4)}
    out |= {"chain<%d>" % rows for rows in range(32, 257, 32)}
    out |= {"chain<%d>+48k" % rows for rows in range(32, 257, 32)}
    out.add("step")
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the grey path choice (bv_morph)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class GreyPath:
    kind: str                        # "copy", "zero", "rect", "runs", "unsupported"
    vpasses: int = 0                 # rect: vertical launches per basic
    launches: int = 0                # morph_grey_kernel launches of the whole call

    def __str__(self):
        return "rect/%d" % self.vpasses if self.kind == "rect" else self.kind


def horizontal_runs(se):
    n = 0
    for row in np.asarray(se) != 0:
        n += int(np.count_nonzero(row[1:] & ~row[:-1]) + row[0])
    return n


def expected_grey_path(op, se, iterations, h, w):
    """What bv_morph launches for `op` with the element `se` (kh x kw, non-zero = member) on [*, h, w, *] frames."""
    se = np.asarray(se) != 0
    kh, kw = se.shape
    if iterations < 0:
        iterations = 1
    if iterations == 0:
        return GreyPath("zero" if op == "gradient" else "copy")
    if horizontal_runs(se) > GREY_MAX_RUNS:
        return GreyPath("unsupported")
    basics = 1 if op in ("erode", "dilate") else 2
    if se.all():
        if kw == 1 and kh == 1:
            return GreyPath("copy" if op != "gradient" else "zero-by-difference")
        L, R, U, D = rect_extents(kw, kh, iterations, h, w)
        p = 1 if U + D == 0 else (U + D + GREY_MAX_RUNS - 2) // (GREY_MAX_RUNS - 1)
        return GreyPath("rect", vpasses=p, launches=basics * (1 + p))
    return GreyPath("runs", launches=basics * iterations)


# ---------------------------------------------------------------------------------------------------------------------
# masks
# ---------------------------------------------------------------------------------------------------------------------
def edge_pixels(m):
    """Set pixels on every border and on both sides of every 32-px word edge (in place)."""
    h, w = m.shape[-2:]
    m[..., 0, ::3] = 255
    m[..., h - 1, 1::3] = 255
    m[..., ::3, 0] = 255
    m[..., 1::3, w - 1] = 255
    for x in range(31, w, 32):
        m[..., 2::5, x] = 255
        if x + 1 < w:
            m[..., 4::5, x + 1] = 255
    return m


def make_mask(kind, shape, seed):
    """[b, h, w] uint8 0/255 masks.  random<d>: density d; blobs: smooth blobs about half the frame; bars: a central block
    of 60 % of each side and random rectangles (survive big erosions); points: two pixels (big dilations do not fill the
    frame); rows / cols: full rows (columns) and rows (columns) with a few holes; full / empty."""
    rng = np.random.default_rng(seed)
    b, h, w = shape
    if kind == "full":
        return np.full(shape, 255, np.uint8)
    if kind == "empty":
        return np.zeros(shape, np.uint8)
    if kind.startswith("random"):
        d = float(kind[6:] or 0.5)
        return ((rng.random(shape) < d) * 255).astype(np.uint8)
    if kind == "points":
        m = np.zeros(shape, np.uint8)
        for f in range(b):
            m[f, rng.integers(0, h, 2), rng.integers(0, w, 2)] = 255
        return m
    if kind in ("rows", "cols"):
        t = (b, h, w) if kind == "rows" else (b, w, h)
        m = np.full(t, 255, np.uint8)
        for f in range(b):
            for y in range(t[1]):
                if rng.random() < 0.5:
                    m[f, y, rng.integers(0, t[2], rng.integers(1, 4))] = 0
        return m if kind == "rows" else np.ascontiguousarray(m.transpose(0, 2, 1))
    if kind == "bars":
        m = np.zeros(shape, np.uint8)
        for f in range(b):
            m[f, h // 5:h - h // 5, w // 5:w - w // 5] = 255
            for _ in range(6):
                y0, x0 = rng.integers(0, h), rng.integers(0, w)
                m[f, y0:y0 + rng.integers(h // 8 + 1, h // 2 + 2), x0:x0 + rng.integers(w // 8 + 1, w // 2 + 2)] = 255
        return m
    if kind == "blobs":
        out = np.zeros(shape, np.uint8)
        for f in range(b):
            noise = rng.random((h, w)).astype(np.float32)
            s = max(1.0, min(h, w) / 12.0)
            sm = cv2.GaussianBlur(noise, (0, 0), s) if min(h, w) > 2 else noise
            out[f] = (sm > np.median(sm)) * 255
        return out
    raise ValueError(kind)


def cv2_steps(mask, steps):
    """cv2.morphologyEx of one frame through every step (rectangular elements)."""
    for op, kw, kh, it in steps:
        mask = cv2.morphologyEx(mask, CV_OP[op], np.ones((kh, kw), np.uint8), iterations=it)
    return mask


# ---------------------------------------------------------------------------------------------------------------------
# stage cases
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class StageCase:
    name: str
    shape: tuple                     # (b, h, w)
    steps: list                      # [(op, kw, kh, iterations)]
    path: str                        # str(expected_morph_path(...)) it was written for
    mask: str = "random0.5"          # make_mask kind
    variant: int = 0                 # BV_OPT_MORPH_VARIANT
    warps: int = 0                   # BV_OPT_MORPH_WARPS
    mask_off: int = 0                # byte offset of the mask output (non-zero: the stage enters the bits through bytes)
    edges: bool = True               # edge_pixels on top of the mask
    nontrivial: bool = False         # cv2's result must be neither empty nor full in every frame
    seed: int = 0
    group: str = ""

    def masks(self):
        m = make_mask(self.mask, self.shape, self.seed)
        return edge_pixels(m) if self.edges else m

    def predicted(self, sm_count=SM_COUNT):
        b, h, w = self.shape
        return expected_morph_path(self.steps, b, h, w, self.variant, sm_count, self.warps)

    def bits_direct(self):
        """The stage packs the threshold straight into bits (otherwise through a uint8 mask and mask_to_bits)."""
        return self.shape[2] % 16 == 0 and self.mask_off % 16 == 0


def _roll_cases():
    out = []
    widths = {1: (31, 32, 33, 63, 64, 65, 1, 1024), 2: (1025, 2048), 3: (2049, 3000), 4: (3073, 4096)}
    steps_of = {(1, 1): [("erode", 3, 3, 1)], (1, 2): [("open", 3, 3, 1)], (1, 4): [("open", 3, 3, 1), ("close", 3, 3, 1)],
                (2, 1): [("dilate", 5, 5, 1)], (2, 2): [("close", 5, 5, 1)], (2, 4): [("close", 5, 5, 1), ("open", 5, 5, 1)]}
    i = 0
    for idx, ((r, n), steps) in enumerate(steps_of.items()):
        for k, ws in widths.items():
            for w in ws if (r, n) == (1, 1) else (ws[idx % len(ws)],):
                b, h = (1, 1, 2, 3)[i % 4], (37, 1, 2, 3, 4, 61)[i % 6]
                out.append(StageCase("roll_r%d_n%d_w%d_h%d_b%d" % (r, n, w, h, b), (b, h, w), steps,
                                     "roll<%d,%d,%d>" % (r, n, k), mask="random0.6", seed=100 + i, group="roll_k%d" % k))
                i += 1
    # the strip split at its edges: one strip per frame (batch >= sm_count * 8), frames of 1..4 rows, other warp counts
    out.append(StageCase("roll_one_strip_per_frame", (1200, 9, 40), [("open", 3, 3, 1)], "roll<1,2,1>", seed=3,
                         group="roll_strips"))
    for h in (1, 2, 3, 4):
        out.append(StageCase("roll_height%d" % h, (3, h, 70), [("close", 5, 5, 1), ("open", 5, 5, 1)], "roll<2,4,1>",
                             seed=10 + h, group="roll_strips"))
    for warps in (1, 3, 64):
        out.append(StageCase("roll_warps%d" % warps, (2, 300, 500), [("open", 5, 5, 1)], "roll<2,2,1>", warps=warps,
                             seed=20 + warps, group="roll_strips"))
    out.append(StageCase("roll_tall_1025", (1, 1025, 100), [("erode", 3, 3, 1)], "roll<1,1,1>", seed=5, group="roll_strips"))
    return out


def _chain_cases():
    out = []
    # every tile size: T rows hold a halo of at most T / 2 (here exactly T / 2, from one dilation or a closing), on
    # narrow rows and on the narrowest rows that take the tile past 48 KiB
    for i, rows in enumerate(range(32, 257, 32)):
        steps = [("dilate", 3, rows // 2 + 1, 1)] if i % 2 else [("close", 5, rows // 4 + 1, 1)]
        wide = 32 * (SMEM_DEFAULT // (8 * rows) + 1) - 5
        for variant, w in ((1, 160), (2, 173), (1 + i % 2, wide)):
            p = "chain<%d>%s" % (rows, "+48k" if w == wide else "")
            out.append(StageCase("chain%d_v%d_w%d" % (rows, variant, w), (2, rows * 2 + 11, w), steps, p, mask="blobs",
                                 variant=variant, seed=30 + i, group="chain_tiles"))
    # non-square steps stay on the chain under the default variant; mixed identity and real steps
    out.append(StageCase("chain_default_nonsquare", (3, 131, 173), [("close", 7, 3, 1), ("erode", 9, 1, 1)], "chain<32>",
                         mask="blobs", seed=40, group="chain_mixed"))
    out.append(StageCase("chain_identity_steps", (2, 97, 100), [("erode", 1, 1, 3), ("dilate", 5, 3, 0), ("close", 3, 5, 1),
                                                                ("open", 1, 1, 1)], "chain<32>", mask="blobs", seed=41,
                         group="chain_mixed"))
    out.append(StageCase("roll_between_identities", (2, 97, 100), [("erode", 1, 1, 3), ("open", 3, 3, 1), ("dilate", 7, 7, 0)],
                         "roll<1,2,1>", seed=42, group="chain_mixed"))
    out.append(StageCase("chain_no_steps_left", (2, 50, 77), [("erode", 1, 1, 1), ("dilate", 3, 3, 0)], "chain<32>", seed=43,
                         group="chain_mixed"))
    # shared memory: above 48 KiB (width > 6144 at 32 rows), the widest tile under 200 KiB, above 200 KiB -> step
    for variant in (0, 1, 2):
        out.append(StageCase("chain_6145_v%d" % variant, (1, 70, 6145), [("open", 5, 5, 1)], "chain<32>+48k", variant=variant,
                             mask="blobs", seed=50 + variant, group="chain_smem"))
        out.append(StageCase("chain_12800_v%d" % variant, (1, 40, 12800), [("close", 3, 3, 1)], "chain<32>+48k",
                             variant=variant, mask="blobs", seed=53 + variant, group="chain_smem"))
    out.append(StageCase("chain_256rows_3072", (1, 300, 3072), [("close", 1, 65, 1)], "chain<256>+48k", variant=1, mask="blobs",
                         seed=56, group="chain_smem"))
    out.append(StageCase("step_over_200k_rows256", (1, 300, 3232), [("close", 1, 65, 1)], "step", variant=1, mask="blobs",
                         seed=57, group="chain_smem"))
    out.append(StageCase("step_over_200k_26000", (1, 24, 26000), [("open", 3, 3, 1)], "step", mask="blobs", seed=58,
                         group="chain_smem"))
    out.append(StageCase("step_over_256_rows", (1, 400, 64), [("dilate", 1, 131, 1)], "step", mask="points", seed=59,
                         group="chain_smem", edges=False, nontrivial=True))
    # TMA: wpr % 4 decides per tile whether the bulk copy or the plain loads stage it
    for w in (128, 160, 161, 200, 2208, 2209, 4097):
        out.append(StageCase("tma_w%d" % w, (3, 75, w), [("open", 5, 5, 1)], "chain<32>" + ("+48k" if 2 * 32 * words_per_row(w) * 4 > SMEM_DEFAULT else ""),
                             variant=2, mask="blobs", seed=60 + w % 97, group="chain_tma"))
    return out


def _step_cases():
    out = []
    # P = 2 and 3 passes, horizontal and vertical, erosion and dilation; bars survive erosions, points dilations.  A lone
    # vertical element reaches the step path only above 128 halo rows (P >= 3); P = 2 comes behind a step that does.
    for op, mk in (("erode", "bars"), ("dilate", "points"), ("open", "bars"), ("close", "points")):
        lists = [[(op, 64, 1, 1)], [(op, 127, 1, 1)], [(op, 3, 3, 32)], [(op, 3, 3, 63)]]
        if op in ("erode", "dilate"):
            lists += [[(op, 1, 141, 1)], [("dilate", 64, 1, 1), (op, 1, 101, 1)]]
        else:
            lists += [[(op, 1, 101, 1)], [(op, 3, 141, 1)]]
        for j, steps in enumerate(lists):
            name = "step_" + "_".join("%s_%dx%d_i%d" % s_ for s_ in steps)
            out.append(StageCase(name, (2, 300, 333), steps, "step", mask=mk, seed=70 + 7 * j, group="step_passes",
                                 edges=op not in ("erode", "dilate"), nontrivial=op in ("erode", "dilate")))
    # the largest elements: 255 x 1 twice (horizontal extent 254 each side, 9 passes), 1 x 255 twice
    out.append(StageCase("step_erode_255x1_i2", (1, 120, 1500), [("erode", 255, 1, 2)], "step", mask="bars", seed=80,
                         group="step_large", edges=False, nontrivial=True))
    out.append(StageCase("step_dilate_1x255_i2", (1, 1100, 90), [("dilate", 1, 255, 2)], "step", mask="points", seed=81,
                         group="step_large", edges=False, nontrivial=True))
    out.append(StageCase("step_open_255x255", (1, 700, 900), [("open", 255, 255, 1)], "step", mask="bars", seed=82,
                         group="step_large", edges=False, nontrivial=True))
    # GRADIENT: single and multi pass (the case that used to be refused), 1x1, 0 iterations, beside chain-able steps
    for kw, kh, it in ((3, 3, 1), (5, 5, 2), (64, 3, 1), (3, 3, 32), (3, 70, 1), (255, 1, 1)):
        out.append(StageCase("gradient_%dx%d_i%d" % (kw, kh, it), (2, 150, 400), [("gradient", kw, kh, it)], "step",
                             mask="bars", seed=90 + kw + it, group="step_gradient", nontrivial=True))
    for op in OPS:
        out.append(StageCase("%s_1x1" % op, (2, 40, 100), [(op, 1, 1, 1)], "chain<32>" if op != "gradient" else "step",
                             seed=95, group="identity"))
        out.append(StageCase("%s_iter0" % op, (2, 40, 100), [(op, 5, 5, 0)], "chain<32>" if op != "gradient" else "step",
                             seed=96, group="identity"))
    out.append(StageCase("gradient_iter0_then_dilate", (1, 60, 96), [("gradient", 3, 3, 0), ("dilate", 3, 3, 1)], "step",
                         seed=97, group="identity"))
    out.append(StageCase("identities_then_gradient", (2, 60, 96), [("erode", 1, 1, 2), ("close", 5, 5, 0), ("gradient", 64, 1, 1)],
                         "step", seed=99, group="identity"))
    out.append(StageCase("dilate_then_gradient_1x1", (1, 60, 96), [("dilate", 3, 3, 1), ("gradient", 1, 1, 4)], "step",
                         seed=98, group="identity"))
    return out


def _width_cases():
    """Widths and heights at the word and strip edges, batches of 1 and 3, through bytes and straight into bits."""
    out = []
    for i, w in enumerate((1, 31, 32, 33, 63, 64, 65, 1025, 2048, 2049, 4096, 4097)):
        for off in (0, 1):
            h = (1, 2, 3, 4, 1025, 45)[(i + off) % 6]
            steps = [("close", 5, 5, 1)] if i % 2 else [("open", 3, 5, 1), ("dilate", 3, 3, 1)]
            b = 3 if (i + off) % 2 else 1
            if h == 1025:
                b = 1
            p = str(expected_morph_path(steps, b, h, w))
            out.append(StageCase("w%d_h%d_b%d_off%d" % (w, h, b, off), (b, h, w), steps, p, mask_off=off, seed=200 + i,
                                 group="widths"))
    return out


def stage_cases():
    return _roll_cases() + _chain_cases() + _step_cases() + _width_cases()


# ---------------------------------------------------------------------------------------------------------------------
# grey cases (bv_morph)
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class GreyCase:
    name: str
    shape: tuple                     # (b, h, w, c)
    op: str
    se: np.ndarray = field(repr=False)
    iterations: int
    path: str                        # str(expected_grey_path(...))
    in_place: bool = False
    dst_off: int = 0
    image_kind: str = "blobs"        # make_mask kind for masks, "grey" for random bytes with structure
    seed: int = 0
    group: str = ""

    def image(self):
        b, h, w, c = self.shape
        if self.image_kind == "grey":
            rng = np.random.default_rng(self.seed)
            yy, xx = np.mgrid[0:h, 0:w]
            base = 128 + 90 * np.sin(xx[None, ..., None] * 0.05 + yy[None, ..., None] * 0.031 + rng.random((b, 1, 1, c)) * 6)
            return np.clip(base + rng.normal(0, 30, (b, h, w, c)), 0, 255).astype(np.uint8)
        m = make_mask(self.image_kind, (b * c, h, w), self.seed)
        return np.ascontiguousarray(m.reshape(b, c, h, w).transpose(0, 2, 3, 1))

    def predicted(self):
        return expected_grey_path(self.op, self.se, self.iterations, self.shape[1], self.shape[2])

    def want(self, img):
        """cv2 of every frame; cv2 treats a negative count as 1."""
        out = np.empty_like(img)
        for f in range(img.shape[0]):
            im = img[f, ..., 0] if img.shape[3] == 1 else img[f]
            out[f] = cv2.morphologyEx(im, CV_OP[self.op], self.se, iterations=self.iterations).reshape(out.shape[1:])
        return out


def _ellipse(k):
    return cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (k, k))


def grey_cases():
    out = []
    rect = lambda kw, kh: np.ones((kh, kw), np.uint8)     # noqa: E731
    i = 0
    # every op, 1..4 channels, batches, in place, offsets, rectangles and run lists over 1..3 iterations
    for op in OPS:
        for c in (1, 2, 3, 4):
            for se, it in ((rect(5, 3), 1), (_ellipse(7), 3), (rect(4, 6), 2), (np.array([[0, 1, 0], [1, 0, 1]], np.uint8), 2)):
                shape = (1 + (i % 3), 37 + i % 5, 61 + 3 * (i % 4), c)
                in_place = i % 3 == 0
                off = 0 if in_place else (1, 2, 3, 0)[i % 4]
                case = GreyCase("%s_c%d_%dx%d_i%d" % (op, c, se.shape[1], se.shape[0], it), shape, op, se, it, "",
                                in_place=in_place, dst_off=off, image_kind="grey" if c != 1 else "random0.6", seed=300 + i,
                                group="grey_%s" % op)
                case.path = str(case.predicted())
                out.append(case)
                i += 1
    # iteration counts: 0 (copy / zeros for GRADIENT) and negative (read as 1)
    for op in OPS:
        for it in (0, -1, -7):
            for se in (rect(3, 3), _ellipse(5)):
                case = GreyCase("%s_%s_i%d" % (op, "rect" if se.all() else "ellipse", it), (2, 40, 50, 3), op, se, it, "",
                                in_place=it == -1, image_kind="grey", seed=400 + i, group="grey_iterations")
                case.path = str(case.predicted())
                out.append(case)
                i += 1
    # large rectangles: horizontal extents past int16 (127 * 259 = 32 893), vertical passes past 256 rows
    for op, kw, kh, it, kind, shape in (("erode", 255, 1, 259, "rows", (1, 20, 40000, 1)),
                                        ("dilate", 255, 1, 300, "points", (1, 8, 40000, 1)),
                                        ("close", 255, 1, 260, "points", (1, 6, 36000, 1)),
                                        ("erode", 1, 255, 2, "cols", (1, 700, 30, 1)),
                                        ("dilate", 1, 255, 2, "points", (1, 700, 30, 1)),
                                        ("dilate", 3, 255, 3, "points", (1, 1000, 40, 2)),
                                        ("open", 1, 255, 3, "cols", (1, 900, 20, 1)),
                                        ("close", 5, 200, 2, "points", (1, 600, 50, 1)),
                                        ("gradient", 1, 255, 2, "cols", (1, 600, 40, 1)),
                                        ("erode", 255, 255, 2, "bars", (1, 1200, 1300, 1)),
                                        ("dilate", 3, 3, 200, "points", (1, 500, 500, 1))):
        case = GreyCase("large_%s_%dx%d_i%d" % (op, kw, kh, it), shape, op, rect(kw, kh), it, "", image_kind=kind,
                        seed=500 + i, group="grey_large")
        case.path = str(case.predicted())
        out.append(case)
        i += 1
    # an element of exactly 256 runs (the limit), and a 1x1 element
    checker = np.zeros((16, 32), np.uint8)
    checker[:, ::2] = 1
    out.append(GreyCase("runs_256", (1, 50, 70, 1), "dilate", checker, 1, "runs", image_kind="points", seed=600,
                        group="grey_limits"))
    out.append(GreyCase("one_by_one_gradient", (2, 30, 40, 3), "gradient", rect(1, 1), 2, "zero-by-difference",
                        image_kind="grey", seed=601, group="grey_limits"))
    out.append(GreyCase("one_by_one_open", (2, 30, 40, 3), "open", rect(1, 1), 2, "copy", image_kind="grey", seed=602,
                        group="grey_limits"))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# labelling
# ---------------------------------------------------------------------------------------------------------------------
def m30_limit_width():
    """The widest fully set row whose m30 = sum x^3 = (W (W - 1) / 2)^2 still fits int64 (and, transposed, the tallest
    column for m03)."""
    w = 1
    while ((w + 1) * w // 2) ** 2 <= 2 ** 63 - 1:
        w += 1
    return w


def run_moment_sums(x0, x1, y):
    """The ten raster moments of the pixels x0..x1 of row y, as Python ints."""
    xs = range(x0, x1 + 1)
    s = [sum(x ** k for x in xs) for k in range(4)]
    return {"m00": s[0], "m10": s[1], "m01": y * s[0], "m20": s[2], "m11": y * s[1], "m02": y * y * s[0], "m30": s[3],
            "m21": y * s[2], "m12": y * y * s[1], "m03": y ** 3 * s[0]}


@dataclass
class LabelCase:
    name: str
    masks: np.ndarray = field(repr=False)     # [b, h, w] uint8
    max_blobs: int = None                     # None: every blob fits
    about: str = ""


def label_cases():
    rng = np.random.default_rng(7)
    out = []
    # the scan kernel's rounds of 1024 rows below 4K widths
    for h, w in ((1025, 64), (2049, 33), (3000, 100)):
        m = make_mask("random0.3", (1, h, w), h + w)
        out.append(LabelCase("scan_rounds_%dx%d" % (h, w), m, about="ccl_scan_kernel carries across rounds"))
    # the rank kernel's wbase loop (wpr > 32) at widths that are no multiple of 32
    for w in (1025, 1100, 2047, 3001):
        out.append(LabelCase("rank_wbase_w%d" % w, make_mask("random0.25", (2, 40, w), w), about="ccl_rank_kernel wbase"))
    # the final kernel's partial last warp, with full_words (width % 32 == 0) and without
    for h, w in ((3, 32 * 5), (7, 64), (5, 33), (9, 95)):
        out.append(LabelCase("final_tail_%dx%d" % (h, w), make_mask("random0.5", (1, h, w), 9 * w + h),
                             about="ccl_final_kernel partial warp"))
    # one large blob interleaved with many small ones in the same warp steps (the carried blob hands over)
    m = np.zeros((1, 96, 2048), np.uint8)
    m[0, :, ::2] = 255
    m[0, ::2, :] = 255
    m[0, 1::4, 1::4] = 0
    m[0, 3::4, 3::8] = 0
    big = np.zeros((96, 2048), bool)
    big[10:90, 100:1900] = True
    m2 = ((rng.random((96, 2048)) < 0.08) * 255).astype(np.uint8)
    m2[big] = 255
    m2[10:90:3, 100:1900] = 0          # rows of the big blob cut into strips, tied by one column
    m2[10:90, 1000] = 255
    out.append(LabelCase("carried_interleaved", np.stack([m2, m[0]]), about="carried blob handoff"))
    # dense masks: the k == 0 / k == 33 edges of the 34-bit merge window
    d = np.zeros((1, 64, 256), np.uint8)
    for x in range(31, 256, 32):
        d[0, 1::2, x] = 255           # word-edge pixels on odd rows
        if x + 1 < 256:
            d[0, 0::2, x + 1] = 255   # and their diagonal partners in the next word on even rows
    d[0, 20:30, :] = (rng.random((10, 256)) < 0.7) * 255
    out.append(LabelCase("merge_window_edges", d, about="k == 0 / k == 33 diagonal contacts"))
    out.append(LabelCase("dense_random", make_mask("random0.85", (2, 200, 300), 11), about="dense merge windows"))
    # a batch whose frames differ in blob count and exceed max_blobs by different amounts; max_blobs 0 and 1
    lat = np.zeros((4, 40, 64), np.uint8)
    for f, step in enumerate((2, 3, 4, 8)):
        lat[f, ::step, ::step] = 255
    out.append(LabelCase("overflow_per_frame", lat, max_blobs=150, about="n_blobs beyond max_blobs, different per frame"))
    out.append(LabelCase("max_blobs_0", lat[:2], max_blobs=0))
    out.append(LabelCase("max_blobs_1", lat, max_blobs=1))
    return out
