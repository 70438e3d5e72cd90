"""TEST INFRASTRUCTURE ONLY -- seeded cases for the smoothing and warping steps of csrc/filter.cu.

`bv_gaussian_blur` chooses between three kernel families, and inside two of them between unrolled instances:

  fast<CN,NT>     gaussian_blur_fast_kernel: square 3, 5 or 7 tap kernels on rows of a multiple of 4 bytes, source and
                  destination 4-byte aligned; the row is handled as a stream of 32-bit words
  tile<CN,NT>     gaussian_blur_kernel: a tile plus halo staged in dynamic shared memory; NT = 3, 5, 7 unrolled for the
                  square kernels the word path refused, NT = 0 the generic loop; above 48 KiB the launch opts in to
                  more shared memory
  two_launch<CN>  blur_rows16_kernel + blur_cols16_kernel: the tile does not fit 200 KiB, the 16-bit horizontal result
                  goes through a global scratch image.  Only BGR reaches it: the largest grey tile (201 x 201 taps)
                  needs 90 944 bytes.

`expected_blur_path` restates that selection.  Every blur case carries the path it was written for; the warp, remap,
undistortion and local-mean cases carry what they are about.  tests/test_filter_cases.py checks that each case still
reaches its path, that together they reach every reachable one, and that oracle/spec_np.py equals cv2 on them;
tests/test_gpu_filter_paths.py runs them on the device.
"""
from dataclasses import dataclass

import numpy as np

# csrc/filter.cu
BLUR_MAX_TAPS = 201                 # kBlurMaxTaps: the tuner reaches 2 * 100 + 1 (modules/preprocessor.py:110-114)
BLUR_TILE_W, BLUR_TILE_H = 64, 32   # kBlurTileW, kBlurTileH
BLUR_TWO_LAUNCH_SMEM = 200 * 1024   # above this the tile kernel gives way to the two launches
SMEM_DEFAULT = 48 * 1024            # a launch above this opts in with cudaFuncSetAttribute

# Where the BGR square kernels change family (derived by hand from the shared-memory formula, checked by the tests):
BGR_SQUARE_ABOVE_48K = 41           # 39 x 39 needs 48 304 bytes, 41 x 41 needs 50 112
BGR_SQUARE_TWO_LAUNCH = 163         # 161 x 161 needs 202 752 bytes, 163 x 163 needs 206 032
GREY_SQUARE_ABOVE_48K = 125         # 123 x 123 needs 48 368 bytes, 125 x 125 needs 49 296


@dataclass(frozen=True)
class BlurPath:
    kind: str          # "fast", "tile" or "two_launch"
    cn: int
    nt: int = 0        # unrolled tap count of fast / tile (0 = generic tile kernel)
    smem: int = 0      # dynamic shared memory of the tile kernel

    @property
    def above_48k(self):
        return self.smem > SMEM_DEFAULT

    def __str__(self):
        return "two_launch<%d>" % self.cn if self.kind == "two_launch" else "%s<%d,%d>" % (self.kind, self.cn, self.nt)


def blur_tile_smem(cn, kx, ky):
    """Dynamic shared memory of gaussian_blur_kernel: the staged 8-bit tile (padded to 16 bytes), then the 16-bit
    horizontal result."""
    rx, ry = kx // 2, ky // 2
    raw = (BLUR_TILE_W + 2 * rx) * cn * (BLUR_TILE_H + 2 * ry)
    return ((raw + 15) & ~15) + BLUR_TILE_W * cn * (BLUR_TILE_H + 2 * ry) * 2


def expected_blur_path(b, h, w, cn, kx, ky, src_off, dst_off):
    """The kernels bv_gaussian_blur launches for a [b, h, w, cn] image with a kx x ky kernel whose source and
    destination lie src_off / dst_off bytes past a 4-byte boundary (b and h do not matter; they are arguments so a
    case can be passed as it is)."""
    smem = blur_tile_smem(cn, kx, ky)
    if smem > BLUR_TWO_LAUNCH_SMEM:
        return BlurPath("two_launch", cn)
    nt = kx if kx == ky and kx in (3, 5, 7) else 0
    if nt and (w * cn) % 4 == 0 and src_off % 4 == 0 and dst_off % 4 == 0:
        return BlurPath("fast", cn, nt)
    return BlurPath("tile", cn, nt, smem)


def reachable_blur_paths():
    """Every path some input reaches: fast and tile for 1 and 3 channels and each unrolled size, the generic tile
    kernel below and above 48 KiB, and two_launch<3>.  two_launch<1> is not among them."""
    out = set()
    for cn in (1, 3):
        for nt in (3, 5, 7):
            out.add("fast<%d,%d>" % (cn, nt))
            out.add("tile<%d,%d>" % (cn, nt))
        out.add("tile<%d,0>" % cn)
        out.add("tile<%d,0>+48k" % cn)
    out.add("two_launch<3>")
    return out


def path_label(p):
    """str(path), with "+48k" for a generic tile launch that opts in to more shared memory."""
    return str(p) + ("+48k" if p.kind == "tile" and p.above_48k else "")


def by_group(cases):
    """{group: [cases]} in case order."""
    out = {}
    for c in cases:
        out.setdefault(c.group, []).append(c)
    return out


def random_image(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


def smooth_image(shape, seed):
    """Random bytes with some low-frequency structure (a blur of pure noise hides rounding slips in its averages)."""
    rng = np.random.default_rng(seed)
    b, h, w, c = shape
    yy, xx = np.mgrid[0:h, 0:w]
    base = 128 + 90 * np.sin(xx[None, ..., None] * 0.37 + yy[None, ..., None] * 0.23 + rng.random((b, 1, 1, c)) * 6)
    return np.clip(base + rng.normal(0, 25, shape), 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------------------------------
# Gaussian blur
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class BlurCase:
    name: str
    shape: tuple                 # (b, h, w, cn)
    ksize: tuple                 # (kx, ky)
    path: str                    # path_label of the path it was written for
    sigma: tuple = (0.0, 0.0)
    src_off: int = 0             # bytes past a 4-byte (in fact 16-byte) boundary
    dst_off: int = 0
    seed: int = 0
    smem: int = None             # the tile's shared memory the case was written for, where that is its point
    group: str = ""

    def image(self):
        return smooth_image(self.shape, self.seed)

    def predicted(self):
        b, h, w, c = self.shape
        return expected_blur_path(b, h, w, c, self.ksize[0], self.ksize[1], self.src_off, self.dst_off)

    @property
    def pixels(self):
        b, h, w, _ = self.shape
        return b * h * w


def _square_path(cn, n, aligned):
    """The path of an n x n kernel as the constants above place it."""
    if n in (3, 5, 7):
        return "fast<%d,%d>" % (cn, n) if aligned else "tile<%d,%d>" % (cn, n)
    if cn == 3 and n >= BGR_SQUARE_TWO_LAUNCH:
        return "two_launch<3>"
    above = n >= (BGR_SQUARE_ABOVE_48K if cn == 3 else GREY_SQUARE_ABOVE_48K)
    return "tile<%d,0>%s" % (cn, "+48k" if above else "")


def blur_cases():
    cases = []

    def add(group, name, shape, ksize, path, **kw):
        cases.append(BlurCase("%s/%s" % (group, name), tuple(shape), tuple(ksize), path, group=group,
                              seed=len(cases) + 1, **kw))

    # every size the tuner produces, on a small BGR and a small grey frame, rows of 4k bytes and not
    for cn, w_al, w_un in ((3, 20, 21), (1, 24, 23)):
        for k in range(1, 101):
            n = 2 * k + 1
            for w, aligned in ((w_al, True), (w_un, False)):
                add("tuner", "cn%d_w%d_n%d" % (cn, w, n), (1, 19, w, cn), (n, n), _square_path(cn, n, aligned))
    # equal sizes, other taps: sigma x != sigma y on the word path (and on the tile path for unaligned rows)
    for cn, w in ((3, 40), (1, 64), (3, 41)):
        aligned = (w * cn) % 4 == 0
        for n in (3, 5, 7):
            for sx, sy in ((0.6, 2.4), (3.0, 0.9), (1.7, 0.0)):
                add("sigma", "cn%d_w%d_n%d_%g_%g" % (cn, w, n, sx, sy), (1, 45, w, cn), (n, n),
                    "%s<%d,%d>" % ("fast" if aligned else "tile", cn, n), sigma=(sx, sy))
    # sources and destinations off a 4-byte boundary drop to the tile kernel
    for so, do in ((1, 0), (2, 0), (3, 0), (0, 1), (0, 2), (0, 3), (1, 3), (2, 2)):
        for cn, n in ((3, 7), (1, 5), (3, 3)):
            add("offset", "cn%d_n%d_src%d_dst%d" % (cn, n, so, do), (1, 50, 72, cn), (n, n), "tile<%d,%d>" % (cn, n),
                src_off=so, dst_off=do)
    # frames smaller than the kernel radius: several reflections (a 1-pixel side reflects onto itself)
    for (h, w, cn) in ((1, 1, 1), (1, 4, 1), (4, 1, 1), (2, 2, 3), (5, 4, 3)):
        for n in (3, 5, 7, 9, 13, 31):
            for ksize in sorted({(n, n), (n, 3), (3, n)}):
                aligned = (w * cn) % 4 == 0
                if ksize[0] == ksize[1]:
                    path = _square_path(cn, n, aligned)
                else:
                    path = "tile<%d,0>" % cn
                add("tiny", "%dx%dx%d_%dx%d" % (h, w, cn, ksize[0], ksize[1]), (1, h, w, cn), ksize, path)
    # batches on every family, grey as [B, H, W, 1]
    add("batch", "bgr_fast7", (3, 70, 132, 3), (7, 7), "fast<3,7>")
    add("batch", "grey_fast5", (4, 33, 260, 1), (5, 5), "fast<1,5>")
    add("batch", "grey_fast7", (3, 40, 64, 1), (7, 7), "fast<1,7>")
    add("batch", "bgr_tile7", (3, 70, 131, 3), (7, 7), "tile<3,7>")
    add("batch", "grey_tile3", (5, 31, 67, 1), (3, 3), "tile<1,3>")
    add("batch", "bgr_tile_generic", (3, 50, 90, 3), (9, 15), "tile<3,0>")
    add("batch", "grey_tile_generic48k", (3, 60, 70, 1), (151, 151), "tile<1,0>+48k")
    add("batch", "bgr_two_launch", (3, 60, 75, 3), (171, 171), "two_launch<3>")
    add("batch", "bgr_two_launch_rect", (2, 90, 50, 3), (151, 171), "two_launch<3>")
    # tile shared memory on each side of 48 KiB and of the 200 KiB switch
    add("smem", "bgr_39", (1, 70, 100, 3), (39, 39), "tile<3,0>", smem=48304)
    add("smem", "bgr_41", (1, 70, 100, 3), (41, 41), "tile<3,0>+48k", smem=50112)
    add("smem", "grey_123", (1, 70, 130, 1), (123, 123), "tile<1,0>", smem=48368)
    add("smem", "grey_125", (1, 70, 130, 1), (125, 125), "tile<1,0>+48k", smem=49296)
    add("smem", "bgr_151", (1, 90, 170, 3), (151, 151), "tile<3,0>+48k", smem=186736)
    add("smem", "bgr_151x161", (1, 90, 170, 3), (151, 161), "tile<3,0>+48k", smem=196992)
    add("smem", "bgr_151x171", (1, 90, 170, 3), (151, 171), "two_launch<3>")
    add("smem", "bgr_161", (1, 90, 170, 3), (161, 161), "tile<3,0>+48k", smem=202752)
    add("smem", "bgr_163", (1, 90, 170, 3), (163, 163), "two_launch<3>")
    add("smem", "grey_201", (1, 90, 170, 1), (201, 201), "tile<1,0>+48k", smem=90944)
    # a 4K frame at the smallest and the largest tuner size
    add("uhd", "bgr_7", (1, 2160, 3840, 3), (7, 7), "fast<3,7>")
    add("uhd", "bgr_201", (1, 2160, 3840, 3), (201, 201), "two_launch<3>")
    return cases


# ---------------------------------------------------------------------------------------------------------------------
# warpAffine
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class WarpCase:
    name: str
    shape: tuple                  # (b, h, w, cn)
    matrix: np.ndarray            # 2 x 3, float64 (or float32, as the preprocessor builds it)
    dsize: tuple                  # (w, h)
    border: str = "constant"
    border_value: tuple = (0, 0, 0)
    seed: int = 0
    group: str = ""

    def image(self):
        return smooth_image(self.shape, self.seed)


def rotation(center, angle, scale=1.0):
    a = angle * (np.pi / 180)
    alpha, beta = np.cos(a) * scale, np.sin(a) * scale
    return np.array([[alpha, beta, (1 - alpha) * center[0] - beta * center[1]],
                     [-beta, alpha, beta * center[0] + (1 - alpha) * center[1]]], np.float64)


BORDERS = (("replicate", (0, 0, 0)), ("constant", (7, 99, 200)))


def warp_cases():
    cases = []

    def add(group, name, shape, m, dsize=None, border="constant", bval=(0, 0, 0)):
        b, h, w, c = shape
        cases.append(WarpCase("%s/%s_%s" % (group, name, border), tuple(shape), np.asarray(m),
                              (w, h) if dsize is None else tuple(dsize), border, tuple(bval), seed=len(cases) + 1,
                              group=group))

    h, w = 37, 53
    for cn in (1, 3):
        for border, bval in BORDERS:
            for ang in range(360):
                add("rotate_cn%d" % cn, "%d" % ang, (1, h, w, cn), rotation((w / 2, h / 2), ang), border=border, bval=bval)
    for border, bval in BORDERS:
        for cn in (1, 3):
            for s in (0.5, 2.0, -1.0):
                add("scale", "cn%d_%g" % (cn, s), (1, h, w, cn), rotation((w / 2, h / 2), 17, s), border=border, bval=bval)
            m = rotation((w / 2, h / 2), 23, 0.8)
            for dsize in ((100, 80), (10, 7), (1, 1), (1, 40), (90, 1)):
                add("dsize", "cn%d_%dx%d" % (cn, dsize[0], dsize[1]), (1, h, w, cn), m, dsize, border, bval)
            for sh in ((1, 1), (1, 53), (37, 1)):
                for m_, mn in ((rotation((sh[1] / 2, sh[0] / 2), 31), "rot"),
                               (np.array([[1.0, 0, 0.4], [0, 1, -0.3]]), "shift")):
                    add("tiny_src", "cn%d_%dx%d_%s" % (cn, sh[0], sh[1], mn), (1, sh[0], sh[1], cn), m_, (9, 8),
                        border, bval)
            for t in (32767.5, -32767.5, 40000.0, -40000.0, 2.2e6, -2.2e6, -3e6, 3e6):
                add("translate", "cn%d_tx%g" % (cn, t), (1, h, w, cn), np.array([[1.0, 0, t], [0, 1, 2.5]]),
                    border=border, bval=bval)
                add("translate", "cn%d_ty%g" % (cn, t), (1, h, w, cn), np.array([[1.0, 0, -1.5], [0, 1, t]]),
                    border=border, bval=bval)
            # the scale flips sign: adelta falls with x while X0 sits at INT_MIN, the int sums wrap
            add("translate", "cn%d_mirror_-2.2e6" % cn, (1, h, w, cn), np.array([[-1.0, 0, -2.2e6], [0, 1, 0]]),
                border=border, bval=bval)
            for k, bad in enumerate((np.nan, np.inf, -np.inf)):
                for pos in (0, 1, 2, 4, 5):
                    m = rotation((w / 2, h / 2), 12)
                    m.reshape(6)[pos] = bad
                    add("nonfinite", "cn%d_%s_at%d" % (cn, ("nan", "inf", "-inf")[k], pos), (1, h, w, cn), m,
                        border=border, bval=bval)
            # the preprocessor's float32 matrices (modules/preprocessor.py:130-135, 144-149)
            for tx, ty in ((25, 0), (3.3, -2.7), (-300.1, 40.9)):
                add("float32", "cn%d_t%g_%g" % (cn, tx, ty), (1, h, w, cn), np.float32([[1, 0, tx], [0, 1, ty]]),
                    border=border, bval=bval)
            add("float32", "cn%d_rot" % cn, (1, h, w, cn), rotation((w / 2, h / 2), 33.3).astype(np.float32),
                border=border, bval=bval)
        # batches whose frames have an odd byte size: frames 1.. start off a 4-byte boundary
        add("batch", "bgr_479x641", (3, 479, 641, 3), rotation((320.5, 239.5), 10), border=border, bval=bval)
        add("batch", "grey_37x53", (3, 37, 53, 1), rotation((26.5, 18.5), -7, 1.1), border=border, bval=bval)
    return cases


# ---------------------------------------------------------------------------------------------------------------------
# remap
# ---------------------------------------------------------------------------------------------------------------------
F32_SPECIALS = np.array([np.nan, np.inf, -np.inf,
                         2 ** 26 + 1, 2 ** 26 - 1, -(2 ** 26 + 1), -(2 ** 26 - 1),       # all round to +-2^26 in float32
                         2 ** 26 - 4, -(2 ** 26 - 4), 2 ** 26 + 8, 1e9, -1e9, 7e7, -7e7,  # float32 neighbours of 2^26
                         32767, 32768, -32767, -32768, 32767.5, -32768.5, 40000, -40000,
                         1 / 64, 3 / 64, 5 / 64, -1 / 64, -3 / 64, 63 / 64, 65 / 64,   # half steps: cvRound to even
                         -0.01, -0.02, -0.03, -0.5, -1.0, -1.01], np.float64)


@dataclass
class RemapCase:
    name: str
    shape: tuple          # source (b, h, w, cn)
    fixed: bool
    map1: np.ndarray      # float32 x [H, W], or int16 [H, W, 2]
    map2: np.ndarray      # float32 y [H, W], or uint16 [H, W]
    border: str = "constant"
    border_value: tuple = (0, 0, 0)
    seed: int = 0
    group: str = ""

    def image(self):
        return smooth_image(self.shape, self.seed)


def _float_maps(h, w, dh, dw, seed):
    """Ordinary coordinates around and inside the frame, with every special value in x (y ordinary) and in y (x
    ordinary), and both special at once."""
    rng = np.random.default_rng(seed)
    mx = rng.uniform(-3, w + 2, (dh, dw)).astype(np.float32)
    my = rng.uniform(-3, h + 2, (dh, dw)).astype(np.float32)
    sp = F32_SPECIALS.astype(np.float32)
    n = sp.size
    mx[0, :n] = sp
    my[1, :n] = sp
    mx[2, :n], my[2, :n] = sp, sp[::-1]
    mx[3, :n], my[3, :n] = sp, sp
    # interior coordinates on exact 1/64 steps, so the word path sees half-step fractions too
    mx[4] = np.round(rng.uniform(0, max(w - 2, 1), dw) * 32) / 32 + np.float32(1 / 64)
    my[4] = np.round(rng.uniform(0, max(h - 2, 1), dw) * 32) / 32 + np.float32(1 / 64)
    return mx, my


def _fixed_maps(h, w, dh, dw, seed):
    rng = np.random.default_rng(seed)
    xy = np.stack([rng.integers(-3, w + 2, (dh, dw)), rng.integers(-3, h + 2, (dh, dw))], -1).astype(np.int16)
    ext = np.array([-32768, 32767, -32767, -1, 0, w - 2, w - 1, w, 1000], np.int16)
    xy[0, :ext.size, 0] = ext
    xy[1, :ext.size, 1] = ext
    xy[2, :ext.size, 0], xy[2, :ext.size, 1] = ext, ext[::-1]
    frac = rng.integers(0, 65536, (dh, dw)).astype(np.uint16)    # cv2 reads map2 & 1023
    frac[0, :6] = [1023, 1024, 65535, 0, 2047, 33791]
    return xy, frac


def remap_cases():
    cases = []

    def add(group, name, shape, fixed, maps, border, bval):
        cases.append(RemapCase("%s/%s_%s" % (group, name, border), tuple(shape), fixed, maps[0], maps[1], border,
                               tuple(bval), seed=len(cases) + 1, group=group))

    for border, bval in BORDERS:
        for cn in (1, 3):
            for (h, w, dh, dw) in ((23, 37, 9, 48), (40, 64, 12, 64), (1, 1, 6, 48), (5, 1, 6, 48), (1, 7, 6, 48)):
                add("float", "cn%d_%dx%d" % (cn, h, w), (1, h, w, cn), False, _float_maps(h, w, dh, dw, h * w + cn),
                    border, bval)
                add("fixed", "cn%d_%dx%d" % (cn, h, w), (1, h, w, cn), True, _fixed_maps(h, w, dh, dw, h * w + cn),
                    border, bval)
        # a batch whose frames have an odd byte size, sharing one pair of maps
        add("batch", "bgr_odd_float", (3, 45, 77, 3), False, _float_maps(45, 77, 30, 70, 5), border, bval)
        add("batch", "grey_odd_fixed", (3, 45, 77, 1), True, _fixed_maps(45, 77, 30, 70, 6), border, bval)
    return cases


# ---------------------------------------------------------------------------------------------------------------------
# undistortion maps (include/camera_filters.hpp:6-11) and the local mean shift of white_balance_bgr_blur
# ---------------------------------------------------------------------------------------------------------------------
CAM_K = np.array([[904.66192735, 0.0, 481.17596262], [0.0, 902.84000422, 404.82437525], [0.0, 0.0, 1.0]])
CAM_D = np.array([0.48525658, 2.02550297, 0.03807578, -0.02152142, -3.30299241])   # lib/configs/1_camera_matrix_params.yaml

# cv2 builds CV_16SC2 maps with SIMD in groups of 2 * (float64 lanes) columns and the rest of each row with scalar code.
# The vector code saturates the integer part to int16; the scalar code truncates it.  A width that is a multiple of 16
# has no scalar columns with any lane count (2, 4 or 8).  In a 964-wide map the last 4 columns are scalar with 4 or 8
# lanes (AVX2, AVX-512).
CV_SIMD_COLS = 16


@dataclass
class UndistortCase:
    name: str
    new_k: np.ndarray
    size: tuple           # (w, h)
    vector_cols: int      # columns where cv2 takes its vector path on every lane count (see CV_SIMD_COLS)


def undistort_cases():
    wide = np.array([[90.0, 0, 480], [0, 90, 360], [0, 0, 1]])          # focal 90: |u| up to 1.45e9 (beyond 2^26)
    mid = np.array([[300.0, 0, 470], [0, 310, 350], [0, 0, 1]])          # beyond int16, inside int32 after x 32
    return [UndistortCase("wide_960x724", wide, (960, 724), 960),
            UndistortCase("wide_964x724", wide, (964, 724), 960),
            UndistortCase("mid_640x480", mid, (640, 480), 640),
            UndistortCase("mid_321x200", mid, (321, 200), 320)]


@dataclass
class LocalMeanCase:
    name: str
    shape: tuple          # (b, h, w, 3)
    ksize: int
    seed: int = 0

    def image(self):
        return random_image(self.shape, self.seed)


def local_mean_cases():
    out = []
    for k, (shape, ksize) in enumerate((((3, 37, 53, 3), 15), ((3, 20, 30, 3), 4095), ((1, 1, 300, 3), 31),
                                        ((1, 300, 1, 3), 31), ((2, 1, 1, 3), 5), ((1, 1, 70, 3), 4095),
                                        ((1, 70, 1, 3), 4095), ((1, 33, 47, 3), 4095))):
        out.append(LocalMeanCase("%dx%dx%d_k%d" % (shape[0], shape[1], shape[2], ksize), shape, ksize, seed=100 + k))
    return out
