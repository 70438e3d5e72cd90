"""TEST INFRASTRUCTURE ONLY -- seeded letterbox cases that reach every branch of `bv_letterbox` (csrc/resize.cu).

The YOLO input transform chooses between two kernels and, inside the staged one, between several data-movement
branches: rows copied by the TMA engine or by ordinary loads, padding rows with wide or narrow stores, padding columns,
the single-row identity copy, image descriptors in shared or in global memory.  Landscape frames whose width is a
multiple of 16 reach only a few of them.  Every case here carries the images, the output spec and the set of paths
`expected_paths` says it takes -- a short restatement of `bv_letterbox`'s selection -- together with the paths the
case was written to reach (`wants`), so tests/test_letterbox_cases.py can check that no case lost its purpose.

Paths:
  tma          the staged kernel, some image's source rows copied with cp.async.bulk
  staged       the staged kernel, some image's source rows copied with ordinary loads (row bytes or base address not
               16-byte aligned)
  gather       the per-pixel gather kernel (a source wider than 3840 px, BV_LETTERBOX_GATHER, or a tap table that does
               not fit shared memory)
  smem_gather  the gather kernel, taken only because the tap table does not fit shared memory
  identity     an image that is copied unscaled (its letterboxed size is its own size)
  pad_rows     an image with padding rows above or below it
  pad_cols     an image with padding columns left or right of it
  narrow_rows  the staged kernel writes padding rows with element stores (out_w % 8 != 0, or `out` not 16-byte aligned)
  global_descs the staged kernel reads image descriptors from global memory (more than 64 images)
  cross_images a block of the staged kernel works on rows of more than one image
"""
from dataclasses import dataclass, field

import numpy as np

from .letterbox import letterbox_geometry

# csrc/resize.cu
LB_MAX_ROW_BYTES = 11520      # kLbMaxRowBytes: 3840 px
LB_STAGES = 2                 # kLbStages
LB_SMEM_IMGS = 64             # kLbSmemImgs
LB_MAX_IMGS = 256             # kLbMaxImgs
LB_COEF_BYTES = 8             # sizeof(LbCoef)
# A B200 block may opt in to 227 KB of shared memory; the staged kernel's static tables take a few KB of it.  The
# cases keep their dynamic size clear of the band in between, so the exact static size does not decide a path.
SMEM_SURE_FITS = 200 * 1024
SMEM_SURE_EXCEEDS = 227 * 1024
B200_SMS = 148

ALL_PATHS = ("tma", "staged", "gather", "smem_gather", "identity", "pad_rows", "pad_cols", "narrow_rows",
             "global_descs", "cross_images")


def tma_smem(widths, out_w):
    """Dynamic shared memory of letterbox_tma_kernel: kLbStages x 2 staged rows of the widest image, then the taps."""
    row_stride = (max(widths) * 3 + 127) & ~127
    return LB_STAGES * 2 * row_stride + LB_COEF_BYTES * out_w


def persistent_grid(widths, out_h, out_w, sm_count):
    """Blocks of letterbox_tma_kernel, as bv_letterbox sizes its persistent grid."""
    per_sm = (208 * 1024) // (tma_smem(widths, out_w) + 6 * 1024)
    per_sm = min(max(per_sm, 1), 6)
    return min(sm_count * per_sm, out_h * len(widths))


def expected_paths(shapes, out_h, out_w, offsets=None, out_offset=0, gather_env=False, sm_count=B200_SMS):
    """The paths bv_letterbox takes for sources of `shapes` [(h, w), ...] whose base addresses lie `offsets[i]` bytes
    past a 16-byte boundary, into an output whose base lies `out_offset` bytes past one."""
    n = len(shapes)
    if not 1 <= n <= LB_MAX_IMGS:
        raise ValueError("bv_letterbox takes 1..%d images" % LB_MAX_IMGS)
    offsets = [0] * n if offsets is None else list(offsets)
    widths = [w for _, w in shapes]
    paths = set()
    rows_fit = all(w * 3 <= LB_MAX_ROW_BYTES for w in widths)
    smem = tma_smem(widths, out_w)
    if SMEM_SURE_FITS < smem <= SMEM_SURE_EXCEEDS:
        raise ValueError("shared memory of %d bytes is too close to the device limit to tell the kernel" % smem)
    staged_kernel = rows_fit and not gather_env and smem <= SMEM_SURE_FITS
    if not staged_kernel:
        paths.add("gather")
        if rows_fit and not gather_env:
            paths.add("smem_gather")
    any_pad_rows = False
    for (h, w), off in zip(shapes, offsets):
        uw, uh, top, bottom, left, right = letterbox_geometry(h, w, out_h, out_w)
        if (uw, uh) == (w, h):
            paths.add("identity")
        if top or bottom:
            paths.add("pad_rows")
            any_pad_rows = True
        if left or right:
            paths.add("pad_cols")
        if staged_kernel:
            paths.add("tma" if (w * 3) % 16 == 0 and off % 16 == 0 else "staged")
    if staged_kernel:
        if any_pad_rows and (out_w % 8 != 0 or out_offset % 16 != 0):
            paths.add("narrow_rows")
        if n > LB_SMEM_IMGS:
            paths.add("global_descs")
        n_items = n * out_h
        grid = persistent_grid(widths, out_h, out_w, sm_count)
        per_block = -(-n_items // grid)
        if any((b * per_block) // out_h != (min(n_items, (b + 1) * per_block) - 1) // out_h
               for b in range(grid) if b * per_block < n_items):
            paths.add("cross_images")
    return paths


@dataclass
class Case:
    name: str
    srcs: list                   # (h, w, seed) of each uint8 [H,W,3] BGR source, drawn by `images()`
    out_h: int
    out_w: int
    pad: int = 114
    half: bool = True
    offsets: list = None         # byte offset of each source past a 16-byte boundary (separate allocations)
    stacked: bool = False        # sources are batch[k] of one [n,H,W,3] tensor; offsets follow from k*H*W*3
    out_offset: int = 0          # `out=` given as a view this many elements into its allocation
    wants: set = field(default_factory=set)

    def __post_init__(self):
        n = len(self.srcs)
        if self.stacked:
            h, w = self.srcs[0][:2]
            self.offsets = [(k * h * w * 3) % 16 for k in range(n)]
        elif self.offsets is None:
            self.offsets = [0] * n

    @property
    def shapes(self):
        return [(h, w) for h, w, _ in self.srcs]

    def images(self):
        return [random_image(h, w, seed) for h, w, seed in self.srcs]

    def out_offset_bytes(self):
        return self.out_offset * (2 if self.half else 4)

    def paths(self, gather_env=False, sm_count=B200_SMS):
        return expected_paths(self.shapes, self.out_h, self.out_w, self.offsets, self.out_offset_bytes(), gather_env,
                              sm_count)


def random_image(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


# (h, w) of single sources and the paths each was chosen for (into 640 x 640)
SOURCES = {
    (1242, 2208): {"tma", "pad_rows"},
    (1080, 1920): {"tma", "pad_rows"},
    (479, 641): {"staged", "pad_rows"},
    (641, 479): {"staged", "pad_cols"},
    (640, 320): {"tma", "identity", "pad_cols"},
    (320, 640): {"tma", "identity", "pad_rows"},
    (641, 300): {"staged", "pad_cols"},              # uw == w, uh != h: horizontal scale exactly 1
    (5, 3000): {"staged", "pad_rows"},               # one unpadded row, 319 padding rows above, 320 below
    (3000, 5): {"staged", "pad_cols"},               # one unpadded column
    (1, 1): {"staged"},
    (1, 3): {"staged", "pad_rows"},
    (3, 1): {"staged", "pad_cols"},
    (2, 2): {"staged"},
    (2160, 3840): {"tma", "pad_rows"},               # the widest staged row: exactly kLbMaxRowBytes, no slack
    (2160, 3841): {"gather", "pad_rows"},
    (2160, 4096): {"gather", "pad_rows"},
    (4000, 6000): {"gather", "pad_rows"},            # 106 rows above, 107 below
}
OUTPUTS = [(640, 640), (384, 640), (640, 384), (100, 333), (333, 100), (7, 9), (1, 1), (1280, 1280), (8, 30000)]
OUTPUT_SOURCES = [(1080, 1920), (641, 479), (479, 641), (2160, 3841)]
PADS = [0, 114, 255, -5, 256, 300]


def single_cases():
    """One source per call: every source into 640 x 640, every output size from a few sources, every pad value,
    fp32, a misaligned base address and a misaligned `out=`."""
    cases = []
    for i, (shape, wants) in enumerate(SOURCES.items()):
        cases.append(Case("src%dx%d" % shape, [(*shape, 100 + i)], 640, 640, wants=set(wants)))
    for i, (oh, ow) in enumerate(OUTPUTS):
        for j, shape in enumerate(OUTPUT_SOURCES):
            wants = {"smem_gather"} if ow == 30000 and shape[1] <= 3840 else set()
            cases.append(Case("out%dx%d_src%dx%d" % (oh, ow, *shape), [(*shape, 200 + 10 * i + j)], oh, ow,
                              wants=wants))
    for i, pad in enumerate(PADS):
        for j, shape in enumerate([(1080, 1920), (641, 479), (4000, 6000)]):
            cases.append(Case("pad%d_src%dx%d" % (pad, *shape), [(*shape, 300 + 10 * i + j)], 640, 640,
                              pad=pad))
        cases.append(Case("pad%d_narrow" % pad, [(479, 641, 390 + i)], 333, 100, pad=pad,
                          wants={"narrow_rows"}))
    for j, shape in enumerate([(1242, 2208), (641, 479), (2160, 4096)]):
        cases.append(Case("fp32_src%dx%d" % shape, [(*shape, 400 + j)], 640, 640, half=False))
        for half in (True, False):
            cases.append(Case("outoff_%s_src%dx%d" % ("fp16" if half else "fp32", *shape),
                              [(*shape, 410 + j)], 640, 640, half=half, out_offset=1,
                              wants={"narrow_rows"} if shape == (1242, 2208) else set()))
    for off in range(1, 16):    # 1280 px rows are 16-byte multiples: only the base address makes them staged
        cases.append(Case("offset%d_720x1280" % off, [(720, 1280, 500 + off)], 640, 640, offsets=[off],
                          wants={"staged"}))
    return cases


MIXED_SOURCES = [(1080, 1920), (479, 641), (37, 16), (641, 479), (720, 1280), (30, 37)]


def batch_cases(sm_count=B200_SMS):
    """Several sources per call: mixed kinds of images crossing block boundaries, batch sizes around the shared-memory
    descriptor table and the 256-image limit, and n * out_h around the persistent grid."""
    cases = []
    # aligned (tma), staged and identity images interleaved; 37 rows per image is never a multiple of a block's rows
    for n, seed in ((30, 600), (64, 601), (65, 602), (200, 603)):
        imgs = [(*MIXED_SOURCES[k % len(MIXED_SOURCES)], seed * 1000 + k) for k in range(n)]
        wants = {"tma", "staged", "identity", "pad_rows", "pad_cols", "cross_images"}
        if n > LB_SMEM_IMGS:
            wants.add("global_descs")
        cases.append(Case("mixed_n%d" % n, imgs, 37, 37, wants=wants))
    # batch sizes
    small = [(120, 160), (97, 131), (131, 97), (64, 64), (48, 64)]
    for n in (1, 16, 64, 65, 256):
        imgs = [(*small[k % len(small)], 700 + 1000 * n + k) for k in range(n)]
        cases.append(Case("n%d" % n, imgs, 64, 64, wants={"global_descs"} if n > LB_SMEM_IMGS else set()))
    # batch[k] of one tensor whose image size (97*131*3 bytes) is not a multiple of 16: alignment changes per image
    imgs = [(97, 131, 800 + k) for k in range(12)]
    cases.append(Case("stacked_97x131", imgs, 640, 640, stacked=True, wants={"staged"}))
    # n * out_h at 1, and one below, at and one above the persistent grid
    full = persistent_grid([64], 65535, 48, sm_count)
    for t in (1, full - 1, full, full + 1):
        n = next(d for d in (4, 3, 2, 1) if t % d == 0)
        imgs = [(64, 64, 900 + t + k) for k in range(n)]
        cases.append(Case("items%d" % t, imgs, t // n, 48))
    return cases


def too_many_images():
    """257 sources: one more than bv_letterbox takes."""
    img = random_image(4, 4, 999)
    return [img] * (LB_MAX_IMGS + 1)
