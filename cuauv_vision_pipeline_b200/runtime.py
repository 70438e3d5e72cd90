"""Context object and tensor-level operations over the C ABI.

PyTorch is used only to own device memory and to copy between host and device
(`torch.Tensor.data_ptr()` is what crosses the boundary); every pixel operation is a hand-written
CUDA kernel inside libb200vision.so.  There is no CPU path: creating a Context without a usable
CUDA device raises BVError.
"""
import threading

import numpy as np
import torch

from ._ffi import ffi, lib, check, BVError  # noqa: F401

CVT = {
    "bgr2hsv": lib.BV_BGR2HSV, "bgr2lab": lib.BV_BGR2LAB, "bgr2gray": lib.BV_BGR2GRAY,
    "bgr2ycrcb": lib.BV_BGR2YCRCB, "hsv2bgr": lib.BV_HSV2BGR, "bgr2hls": lib.BV_BGR2HLS,
    "gray2bgr": lib.BV_GRAY2BGR, "bgr2rgb": lib.BV_BGR2RGB, "lab2bgr": lib.BV_LAB2BGR, "bgr2luv": lib.BV_BGR2LUV,
}
MORPH = {"erode": lib.BV_MORPH_ERODE, "dilate": lib.BV_MORPH_DILATE, "open": lib.BV_MORPH_OPEN,
         "close": lib.BV_MORPH_CLOSE, "gradient": lib.BV_MORPH_GRADIENT}
THRESH = {"binary": lib.BV_THRESH_BINARY, "binary_inv": lib.BV_THRESH_BINARY_INV, "trunc": lib.BV_THRESH_TRUNC,
          "tozero": lib.BV_THRESH_TOZERO, "tozero_inv": lib.BV_THRESH_TOZERO_INV}

BLOB_DTYPE = np.dtype([(k, "<i8") for k in ("m00", "m10", "m01", "m20", "m11", "m02", "m30", "m21", "m12", "m03")] +
                      [(k, "<i4") for k in ("x0", "y0", "x1", "y1")])
assert BLOB_DTYPE.itemsize == ffi.sizeof("bv_blob")
CONTOUR_DTYPE = np.dtype([(k, "<i8") for k in ("a00", "a10", "a01")] +
                         [(k, "<i4") for k in ("x0", "y0", "x1", "y1", "start_x", "start_y", "n_points", "n_simple",
                                               "label", "external", "point_offset", "reserved")])
assert CONTOUR_DTYPE.itemsize == ffi.sizeof("bv_contour")
RRECT_DTYPE = np.dtype([(k, "<f4") for k in ("cx", "cy", "width", "height", "angle")] + [("valid", "<i4")])
assert RRECT_DTYPE.itemsize == ffi.sizeof("bv_rrect")
SHAPE_DTYPE = np.dtype([("arc_length", "<f8")] + [(k, "<f4") for k in ("circle_cx", "circle_cy", "circle_r")] +
                       [("rect", RRECT_DTYPE)] + [(k, "<i4") for k in ("n_hull", "n_approx", "approx_convex", "valid",
                                                                      "reserved")])
assert SHAPE_DTYPE.itemsize == ffi.sizeof("bv_shape")


def _u8ptr(t):
    return ffi.cast("uint8_t *", t.data_ptr()) if t is not None else ffi.NULL


class Context:
    """Owns one bv_ctx (one device, one CUDA stream).  Use as a context manager or keep it for the
    life of the module, like the reference's BlockAccessor (core/bindings/...py:388-441)."""

    def __init__(self, device=0):
        out = ffi.new("bv_ctx **")
        check(lib.bv_create(int(device), out))
        self._ctx = out[0]
        self.device = torch.device("cuda", int(device))
        # torch allocations / copies are issued on the context's own stream so that they are
        # ordered with the kernels without any extra synchronisation
        self.torch_stream = torch.cuda.ExternalStream(int(ffi.cast("uintptr_t", lib.bv_stream(self._ctx))),
                                                      device=self.device)
        self._inflight = {}   # slot -> host arrays of an asynchronous stage_host call

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if self._ctx is not None:
            for slot in list(self._inflight):
                lib.bv_stage_host_wait(self._ctx, slot)
            self._inflight.clear()
            lib.bv_destroy(self._ctx)
            self._ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        if self._ctx is None:
            raise BVError(-1, "context is closed")
        return self._ctx

    def sync(self):
        check(lib.bv_sync(self.handle))

    @property
    def launches(self):
        return int(lib.bv_launch_count(self.handle))

    OPTIONS = {"hist_bps": 0, "final_bps": 1, "side_streams": 2, "l2_chunk_mb": 3, "no_hue_table": 4, "contour_pool_chunks": 5,
               "fast_tables": 6, "morph_variant": 7, "no_rcp_tables": 8, "final_sv_tables": 9, "morph_warps": 10}

    def set_option(self, name, value):
        """Tuning knob of the colour-balance passes (include/b200vision.h, BV_OPT_*); 0 = default."""
        check(lib.bv_set_option(self.handle, self.OPTIONS[name], int(value)))

    def profile(self, on=True):
        """Bracket every kernel launch with CUDA events on the context's stream."""
        check(lib.bv_profile_enable(self.handle, 1 if on else 0))

    def profile_dump(self):
        """{kernel: {"launches": n, "ms": total}} since the last dump (synchronises)."""
        import json
        buf = ffi.new("char[]", 1 << 16)
        check(lib.bv_profile_dump(self.handle, buf, 1 << 16))
        return json.loads(ffi.string(buf).decode())

    # -- memory -----------------------------------------------------------------------------
    def empty(self, shape, dtype=torch.uint8):
        with torch.cuda.stream(self.torch_stream):
            return torch.empty(shape, dtype=dtype, device=self.device)

    def upload(self, arr):
        """numpy (or CPU tensor) -> device tensor on this context's stream."""
        if isinstance(arr, torch.Tensor):
            if arr.is_cuda:
                return arr.contiguous()
            src = arr.contiguous()
        else:
            src = torch.from_numpy(np.ascontiguousarray(arr))
        with torch.cuda.stream(self.torch_stream):
            return src.to(self.device, non_blocking=True)

    def download(self, t):
        with torch.cuda.stream(self.torch_stream):
            out = t.cpu()
        return out.numpy()

    # -- operations (device tensors in, device tensors out) ----------------------------------
    @staticmethod
    def _bhw(t, channels=None):
        """Returns (batch, height, width, channels) of a [H,W], [H,W,C], [B,H,W,C] tensor."""
        if t.dtype != torch.uint8 or not t.is_cuda or not t.is_contiguous():
            raise BVError(-1, "expected a contiguous CUDA uint8 tensor")
        if t.dim() == 2:
            return 1, t.shape[0], t.shape[1], 1
        if t.dim() == 3:
            if channels == 1:          # [B,H,W] single-channel batch
                return t.shape[0], t.shape[1], t.shape[2], 1
            return 1, t.shape[0], t.shape[1], t.shape[2]
        if t.dim() == 4:
            return t.shape[0], t.shape[1], t.shape[2], t.shape[3]
        raise BVError(-1, "unsupported tensor rank")

    def _src(self, t):
        """A source image of the filter, morphology and noise steps: a contiguous uint8 tensor on this context's device
        (the kernels read it as packed bytes)."""
        if t.dtype != torch.uint8 or t.device != self.device or not t.is_contiguous():
            raise BVError(-1, "expected a contiguous uint8 tensor on %s" % self.device)
        return t

    def cvt_color(self, src, code, split=False):
        code_i = CVT[code] if isinstance(code, str) else int(code)
        if code_i != lib.BV_GRAY2BGR:
            b, h, w, c = self._bhw(src)
        if code_i == lib.BV_GRAY2BGR:
            if src.dim() not in (2, 3):
                raise BVError(-1, "GRAY2BGR needs [H,W] or [B,H,W]")
            gb = 1 if src.dim() == 2 else src.shape[0]
            dst = self.empty(tuple(src.shape) + (3,))
            check(lib.bv_cvt_color(self.handle, _u8ptr(src), _u8ptr(dst), ffi.NULL, gb, src.shape[-2], src.shape[-1],
                                   code_i))
            return dst
        if c != 3:
            raise BVError(-1, "colour conversion needs a 3-channel image")
        one = code_i == lib.BV_BGR2GRAY
        lead = tuple(src.shape[:-1])
        dst = self.empty(lead if one else lead + (3,))
        planes = None
        if split and not one:
            planes = [self.empty(lead) for _ in range(3)]
            pp = ffi.new("uint8_t *[3]", [_u8ptr(p) for p in planes])
        else:
            pp = ffi.NULL
        check(lib.bv_cvt_color(self.handle, _u8ptr(src), _u8ptr(dst), pp, b, h, w, code_i))
        return (dst, planes) if split else dst

    @staticmethod
    def _cv_bounds(lo, hi, channels):
        """cv2.inRange's reading of its bounds on an 8-bit image: cvRound (half to even) of each value; a bare scalar is
        cv::Scalar(v, 0, 0, 0), i.e. on a 3-channel image it bounds channel 0 only and channels 1, 2 get [0, 0]."""
        lo = np.rint(np.atleast_1d(np.asarray(lo, dtype=np.float64))).astype(np.int64)
        hi = np.rint(np.atleast_1d(np.asarray(hi, dtype=np.float64))).astype(np.int64)
        if channels == 3:
            if lo.size == 1:
                lo = np.array([lo[0], 0, 0], np.int64)
            if hi.size == 1:
                hi = np.array([hi[0], 0, 0], np.int64)
        return lo, hi

    def in_range(self, src, lo, hi):
        n_lo = np.size(lo)
        if src.dim() == 2 or (src.dim() == 3 and n_lo == 1 and src.shape[-1] != 3):
            b, h, w, c = self._bhw(src, channels=1)
        else:
            b, h, w, c = self._bhw(src)
        if c not in (1, 3):
            raise BVError(-1, "inRange needs 1 or 3 channels")
        lo, hi = self._cv_bounds(lo, hi, c)
        # cv2.inRange compares in the scalar's domain: bounds outside [0,255] saturate harmlessly
        empty = bool(np.any(lo > 255) or np.any(hi < 0))
        lo8 = np.clip(lo, 0, 255).astype(np.uint8)
        hi8 = np.clip(hi, 0, 255).astype(np.uint8)
        if empty:
            lo8[:] = 255
            hi8[:] = 0
        mask = self.empty((b, h, w) if (src.dim() == 4 or (src.dim() == 3 and c == 1)) else (h, w))
        check(lib.bv_in_range(self.handle, _u8ptr(src), _u8ptr(mask), b, h, w, c,
                              ffi.from_buffer("uint8_t[]", lo8), ffi.from_buffer("uint8_t[]", hi8)))
        return mask

    def cvt_in_range(self, src, code, lo, hi):
        """cvtColor + inRange in one pass (modules/bins.py:13-16): device BGR [H,W,3] / [B,H,W,3] -> mask."""
        b, h, w, c = self._bhw(src)
        if c != 3:
            raise BVError(-1, "cvt_in_range needs a 3-channel image")
        lo8 = np.clip(np.broadcast_to(np.asarray(lo), (3,)), 0, 255).astype(np.uint8)
        hi8 = np.clip(np.broadcast_to(np.asarray(hi), (3,)), 0, 255).astype(np.uint8)
        mask = self.empty(tuple(src.shape[:-1]))
        check(lib.bv_cvt_in_range(self.handle, _u8ptr(src), _u8ptr(mask), b, h, w, CVT[code] if isinstance(code, str) else int(code),
                                  ffi.from_buffer("uint8_t[]", lo8), ffi.from_buffer("uint8_t[]", hi8)))
        return mask

    def threshold(self, src, thresh, maxval, kind):
        dst = self.empty(tuple(src.shape))
        check(lib.bv_threshold(self.handle, _u8ptr(src), _u8ptr(dst), src.numel(), int(np.floor(thresh)), int(maxval),
                               THRESH[kind]))
        return dst

    def apply_lut(self, src, lut):
        lut = np.ascontiguousarray(lut, dtype=np.uint8)
        channels = 1 if lut.ndim == 1 else lut.shape[0]
        dst = self.empty(tuple(src.shape))
        check(lib.bv_apply_lut(self.handle, _u8ptr(src), _u8ptr(dst), src.numel() // channels, channels,
                               ffi.from_buffer("uint8_t[]", lut)))
        return dst

    def color_distance(self, planes, color, weights, use, max_dist_sq):
        """planes: 3 device uint8 tensors of equal shape.  Returns (mask, dist) device tensors."""
        n = planes[0].numel()
        mask = self.empty(tuple(planes[0].shape))
        dist = self.empty(tuple(planes[0].shape))
        pp = ffi.new("uint8_t *[3]", [_u8ptr(p) for p in planes])
        check(lib.bv_color_distance(self.handle, ffi.cast("const uint8_t *const *", pp), n,
                                    ffi.new("double[3]", [float(c) for c in color]),
                                    ffi.new("double[3]", [float(w) for w in weights]),
                                    ffi.new("int32_t[3]", [int(u) for u in use]), float(max_dist_sq),
                                    _u8ptr(mask), _u8ptr(dist)))
        return mask, dist

    def color_distance_f32(self, planes, color, weights, use):
        """The float32 squared-distance image (utils/color.py:94-97) as a device tensor."""
        n = planes[0].numel()
        d = self.empty(tuple(planes[0].shape), torch.float32)
        pp = ffi.new("uint8_t *[3]", [_u8ptr(p) for p in planes])
        check(lib.bv_color_distance_f32(self.handle, ffi.cast("const uint8_t *const *", pp), n,
                                        ffi.new("double[3]", [float(c) for c in color]),
                                        ffi.new("double[3]", [float(w) for w in weights]),
                                        ffi.new("int32_t[3]", [int(u) for u in use]), ffi.cast("float *", d.data_ptr())))
        return d

    def select_kth(self, values, k):
        """k-th smallest (0-based) of a float32 device tensor, as np.float32."""
        out = ffi.new("float *")
        n = values.numel()
        check(lib.bv_select_kth_f32(self.handle, ffi.cast("float *", values.data_ptr()), n, int(k) % n, out))
        return np.float32(out[0])

    def morph(self, src, op, kernel, iterations=1):
        self._src(src)
        kernel = np.ascontiguousarray(np.asarray(kernel) != 0, dtype=np.uint8)
        kh, kw = kernel.shape
        if src.dim() == 2:
            b, h, w, c = 1, src.shape[0], src.shape[1], 1
        elif src.dim() == 3:
            b, h, w, c = 1, src.shape[0], src.shape[1], src.shape[2]
        else:
            b, h, w, c = src.shape
        dst = self.empty(tuple(src.shape))
        check(lib.bv_morph(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, c, MORPH[op] if isinstance(op, str) else op,
                           ffi.from_buffer("uint8_t[]", kernel), kw, kh, int(iterations)))
        return dst

    def canny(self, src, threshold1, threshold2, aperture_size=3, l2_gradient=False):
        """cv2.Canny(src, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of a device image
        [H,W], [H,W,3], [B,H,W] or [B,H,W,3] (a rank-3 tensor whose last dimension is 3 is one BGR frame) -> uint8 0/255
        [.., H, W], bit-exact (bv_canny).  BVError for an aperture other than 3, 5 or 7, as cv2 raises."""
        self._src(src)
        if src.dim() == 2:
            b, h, w, c = 1, src.shape[0], src.shape[1], 1
        elif src.dim() == 3:
            b, h, w, c = (1, src.shape[0], src.shape[1], 3) if src.shape[2] == 3 else (src.shape[0], src.shape[1],
                                                                                        src.shape[2], 1)
        elif src.dim() == 4 and src.shape[3] in (1, 3):
            b, h, w, c = src.shape
        else:
            raise BVError(-1, "canny takes [H,W], [H,W,3], [B,H,W] or [B,H,W,3]")
        dst = self.empty((b, h, w) if src.dim() == 4 or (src.dim() == 3 and c == 1) else (h, w))
        check(lib.bv_canny(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, c, float(threshold1), float(threshold2),
                           int(aperture_size), 1 if l2_gradient else 0))
        return dst

    def color_balance(self, src, want_stats=False, **flags):
        b, h, w, c = self._bhw(src)
        if c != 3:
            raise BVError(-1, "colour balance needs BGR input")
        prm = ffi.new("bv_balance_params *")
        lib.bv_balance_default(prm)
        for k, v in flags.items():
            setattr(prm, k, int(v))
        dst = self.empty(tuple(src.shape))
        stats = ffi.new("bv_balance_stats[]", b) if want_stats else ffi.NULL
        check(lib.bv_color_balance(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, prm, stats))
        if want_stats:
            out = []
            for i in range(b):
                s = stats[i]
                out.append(dict(bgr_min=tuple(s.bgr_min), bgr_max=tuple(s.bgr_max), bgr_avg=tuple(s.bgr_avg),
                                dominant=s.dominant, s_min=s.s_min, s_max=s.s_max, v_min=s.v_min, v_max=s.v_max,
                                degenerate=s.degenerate))
            return dst, out
        return dst

    def label(self, mask, max_blobs=4096, want_labels=True):
        if mask.dim() == 2:
            b, h, w = 1, mask.shape[0], mask.shape[1]
        else:
            b, h, w = mask.shape[0], mask.shape[1], mask.shape[2]
        labels = self.empty(tuple(mask.shape), torch.int32) if want_labels else None
        blobs = self.empty((b, max_blobs, BLOB_DTYPE.itemsize), torch.uint8) if max_blobs else None
        nb = self.empty((b,), torch.int32)
        check(lib.bv_label(self.handle, _u8ptr(mask), ffi.cast("int32_t *", labels.data_ptr()) if want_labels else ffi.NULL,
                           b, h, w, ffi.cast("bv_blob *", blobs.data_ptr()) if max_blobs else ffi.NULL, max_blobs,
                           ffi.cast("int32_t *", nb.data_ptr())))
        return labels, blobs, nb

    def outer_contours(self, mask, max_contours=4096, max_points=0):
        """Device mask [H,W] or [B,H,W] -> (contour table as uint8 [B,max,72], count [B], points
        int32 [B,max_points,2] or None, points needed [B] or None)."""
        if mask.dim() == 2:
            b, h, w = 1, mask.shape[0], mask.shape[1]
        else:
            b, h, w = mask.shape[0], mask.shape[1], mask.shape[2]
        table = self.empty((b, max_contours, CONTOUR_DTYPE.itemsize), torch.uint8)
        nb = self.empty((b,), torch.int32)
        points = self.empty((b, max_points, 2), torch.int32) if max_points else None
        npts = self.empty((b,), torch.int32) if max_points else None
        check(lib.bv_outer_contours(self.handle, _u8ptr(mask), b, h, w, ffi.cast("bv_contour *", table.data_ptr()),
                                    max_contours, ffi.cast("int32_t *", nb.data_ptr()),
                                    ffi.cast("int32_t *", points.data_ptr()) if max_points else ffi.NULL, max_points,
                                    ffi.cast("int32_t *", npts.data_ptr()) if max_points else ffi.NULL))
        return table, nb, points, npts

    RETR = {"list": lib.BV_RETR_LIST, "ccomp": lib.BV_RETR_CCOMP, "tree": lib.BV_RETR_TREE}
    CHAIN = {"none": lib.BV_CHAIN_APPROX_NONE, "simple": lib.BV_CHAIN_APPROX_SIMPLE}

    def find_contours(self, mask, mode="tree", method="simple", max_contours=4096, max_points=0):
        """cv2.findContours(mask, RETR_LIST / CCOMP / TREE, CHAIN_APPROX_NONE / SIMPLE) of a device mask [H,W] or
        [B,H,W] -> (contour table as uint8 [B,max,72]: outer borders then hole borders, hierarchy int32
        [B,max,4], counts int32 [B,2] = (outer, holes), points int32 [B,max_points,2] or None, points needed [B]
        or None).  `mode` / `method` take the names or the BV_* values."""
        mode = self.RETR[mode] if isinstance(mode, str) else int(mode)
        method = self.CHAIN[method] if isinstance(method, str) else int(method)
        b, h, w, _ = self._bhw(mask, channels=1)
        table = self.empty((b, max_contours, CONTOUR_DTYPE.itemsize), torch.uint8)
        hier = self.empty((b, max_contours, 4), torch.int32)
        nc = self.empty((b, 2), torch.int32)
        points = self.empty((b, max_points, 2), torch.int32) if max_points else None
        npts = self.empty((b,), torch.int32) if max_points else None
        check(lib.bv_find_contours(self.handle, _u8ptr(mask), b, h, w, mode, method,
                                   ffi.cast("bv_contour *", table.data_ptr()), ffi.cast("int32_t *", hier.data_ptr()),
                                   max_contours, ffi.cast("int32_t *", nc.data_ptr()),
                                   ffi.cast("int32_t *", points.data_ptr()) if max_points else ffi.NULL, max_points,
                                   ffi.cast("int32_t *", npts.data_ptr()) if max_points else ffi.NULL))
        return table, hier, nc, points, npts

    def min_area_rects(self, table, nb, points):
        """cv2.minAreaRect of every external contour of `outer_contours(..., max_points > 0)`: structured numpy
        array [B, max_contours] with fields cx, cy, width, height, angle, valid."""
        b, max_contours = table.shape[0], table.shape[1]
        max_points = points.shape[1]
        rects = self.empty((b, max_contours, RRECT_DTYPE.itemsize), torch.uint8)
        check(lib.bv_min_area_rects(self.handle, ffi.cast("bv_contour *", table.data_ptr()), ffi.cast("int32_t *", nb.data_ptr()),
                                    ffi.cast("int32_t *", points.data_ptr()), b, max_contours, max_points,
                                    ffi.cast("bv_rrect *", rects.data_ptr())))
        return self.download(rects).view(RRECT_DTYPE).reshape(b, max_contours)

    def contour_shapes(self, table, counts, points, method, approx_epsilon=0.0, approx_relative=0.0, hull=True,
                       approx=True):
        """Shape descriptors of every record of a contour table (bv_contour_shapes): `table`, `counts` and `points` as
        find_contours (counts [B,2]) or outer_contours (counts [B], SIMPLE) returned them.  Returns (shapes as uint8
        [B,max_contours,SHAPE_DTYPE.itemsize], hull int32 [B,max_points,2] or None, approx int32 [B,max_points,2] or
        None); a record's hull and approximation start at its point_offset."""
        method = self.CHAIN[method] if isinstance(method, str) else int(method)
        b, max_contours = table.shape[0], table.shape[1]
        max_points = points.shape[1]
        counts_per_frame = 1 if counts.dim() == 1 else 2
        shapes = self.empty((b, max_contours, SHAPE_DTYPE.itemsize), torch.uint8)
        hull_t = self.empty((b, max_points, 2), torch.int32) if hull else None
        approx_t = self.empty((b, max_points, 2), torch.int32) if approx else None
        check(lib.bv_contour_shapes(self.handle, ffi.cast("bv_contour *", table.data_ptr()),
                                    ffi.cast("int32_t *", counts.data_ptr()), counts_per_frame,
                                    ffi.cast("int32_t *", points.data_ptr()), b, max_contours, max_points, method,
                                    float(approx_epsilon), float(approx_relative), ffi.cast("bv_shape *", shapes.data_ptr()),
                                    ffi.cast("int32_t *", hull_t.data_ptr()) if hull else ffi.NULL,
                                    ffi.cast("int32_t *", approx_t.data_ptr()) if approx else ffi.NULL))
        return shapes, hull_t, approx_t

    def blobs_to_numpy(self, blobs, nb):
        """Device blob table -> list (per frame) of structured numpy arrays."""
        n = self.download(nb)
        raw = self.download(blobs)
        out = []
        for f in range(raw.shape[0]):
            k = int(min(n[f], raw.shape[1]))
            out.append(raw[f, :k].copy().view(BLOB_DTYPE).reshape(k))
        return n, out

    def resize(self, src, width, height):
        b, sh, sw, c = self._bhw(src)
        shape = (height, width) if src.dim() == 2 else ((height, width, c) if src.dim() == 3 else (b, height, width, c))
        dst = self.empty(shape)
        check(lib.bv_resize_linear(self.handle, _u8ptr(src), sh, sw, _u8ptr(dst), height, width, c, b))
        return dst

    @staticmethod
    def _bhwc(src):
        if src.dim() == 2:
            return 1, src.shape[0], src.shape[1], 1
        if src.dim() == 3:
            return 1, src.shape[0], src.shape[1], src.shape[2]
        return tuple(src.shape)

    def gaussian_blur(self, src, ksize, sigma_x=0.0, sigma_y=0.0):
        """cv2.GaussianBlur(src, ksize=(kw, kh), sigma_x, sigma_y) on uint8 (BORDER_REFLECT_101)."""
        b, h, w, c = self._bhwc(self._src(src))
        dst = self.empty(tuple(src.shape))
        check(lib.bv_gaussian_blur(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, c, int(ksize[0]), int(ksize[1]),
                                   float(sigma_x), float(sigma_y)))
        return dst

    def warp_affine(self, src, matrix, dsize=None, border="constant", border_value=(0, 0, 0)):
        """cv2.warpAffine(src, matrix, dsize, flags=INTER_LINEAR, borderMode=..., borderValue=...) on uint8."""
        b, h, w, c = self._bhwc(self._src(src))
        dw, dh = (w, h) if dsize is None else (int(dsize[0]), int(dsize[1]))
        m = np.ascontiguousarray(np.asarray(matrix, dtype=np.float64).reshape(6))
        bv_ = np.ascontiguousarray(np.asarray(list(border_value)[:c] + [0] * max(0, c - len(border_value)), dtype=np.uint8))
        shape = (dh, dw) if src.dim() == 2 else ((dh, dw, c) if src.dim() == 3 else (b, dh, dw, c))
        dst = self.empty(shape)
        check(lib.bv_warp_affine(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, c, dh, dw, ffi.from_buffer("double[]", m),
                                 {"constant": 0, "replicate": 1}[border], ffi.from_buffer("uint8_t[]", bv_)))
        return dst

    def remap(self, src, map1, map2, border="constant", border_value=(0, 0, 0)):
        """cv2.remap(src, map1, map2, INTER_LINEAR, borderMode, borderValue) on uint8.  Device maps: two float32 [H,W]
        planes (x, y) or int16 [H,W,2] + uint16 [H,W] (fixed point)."""
        b, h, w, c = self._bhwc(self._src(src))
        fixed = map1.dtype == torch.int16
        if fixed:
            if map1.dim() != 3 or map1.shape[2] != 2 or map2.dtype not in (torch.uint16, torch.int16) or tuple(map2.shape) != tuple(map1.shape[:2]):
                raise BVError(-1, "fixed-point maps are int16 [H,W,2] + uint16 [H,W]")
        elif map1.dtype != torch.float32 or map2.dtype != torch.float32 or map1.dim() != 2 or tuple(map1.shape) != tuple(map2.shape):
            raise BVError(-1, "float maps are two float32 [H,W] planes")
        if not (map1.device == self.device == map2.device and map1.is_contiguous() and map2.is_contiguous()):
            raise BVError(-1, "maps must be contiguous tensors on %s" % self.device)
        dh, dw = int(map1.shape[0]), int(map1.shape[1])
        bv_ = np.ascontiguousarray(np.asarray(list(border_value)[:c] + [0] * max(0, c - len(border_value)), dtype=np.uint8))
        shape = (dh, dw) if src.dim() == 2 else ((dh, dw, c) if src.dim() == 3 else (b, dh, dw, c))
        dst = self.empty(shape)
        check(lib.bv_remap(self.handle, _u8ptr(src), _u8ptr(dst), b, h, w, c, dh, dw, ffi.cast("void *", map1.data_ptr()),
                           ffi.cast("void *", map2.data_ptr()), 1 if fixed else 0, {"constant": 0, "replicate": 1}[border],
                           ffi.from_buffer("uint8_t[]", bv_)))
        return dst

    def undistort_maps(self, camera_matrix, dist_coeffs, inv_new_camera_rot, size, fixed=False):
        """Device maps of cv2.initUndistortRectifyMap: float32 (x, y) planes, or with fixed=True the int16 [H,W,2] +
        uint16 [H,W] pair cv2.undistort uses.  size = (width, height)."""
        w, h = int(size[0]), int(size[1])
        km = np.ascontiguousarray(np.asarray(camera_matrix, np.float64).reshape(9))
        ir = np.ascontiguousarray(np.asarray(inv_new_camera_rot, np.float64).reshape(9))
        d = np.ascontiguousarray(np.asarray(dist_coeffs if dist_coeffs is not None else [], np.float64).ravel())
        null = ffi.NULL
        if fixed:
            m1, m2 = self.empty((h, w, 2), torch.int16), self.empty((h, w), torch.uint16)
            check(lib.bv_undistort_maps(self.handle, ffi.from_buffer("double[]", km), ffi.from_buffer("double[]", d) if d.size else null,
                                        int(d.size), ffi.from_buffer("double[]", ir), w, h, null, null,
                                        ffi.cast("int16_t *", m1.data_ptr()), ffi.cast("uint16_t *", m2.data_ptr())))
        else:
            m1, m2 = self.empty((h, w), torch.float32), self.empty((h, w), torch.float32)
            check(lib.bv_undistort_maps(self.handle, ffi.from_buffer("double[]", km), ffi.from_buffer("double[]", d) if d.size else null,
                                        int(d.size), ffi.from_buffer("double[]", ir), w, h, ffi.cast("float *", m1.data_ptr()),
                                        ffi.cast("float *", m2.data_ptr()), null, null))
        return m1, m2

    def lab_shift_local_mean(self, lab, ksize):
        """a, b of a uint8 LAB image minus (their ksize x ksize box mean - 128), numpy-cast to uint8 (white_balance_bgr_blur)."""
        b, h, w, c = self._bhwc(self._src(lab))
        if c != 3:
            raise BVError(-1, "lab_shift_local_mean needs a 3-channel image")
        dst = self.empty(tuple(lab.shape))
        check(lib.bv_lab_shift_local_mean(self.handle, _u8ptr(lab), _u8ptr(dst), b, h, w, int(ksize)))
        return dst

    def add_gaussian_noise(self, src, sigma, random_state=None):
        """clip(src + randn(*src.shape) * sigma, 0, 255).astype(uint8) with the values numpy's legacy generator would
        draw: numpy's global one (as modules/preprocessor.py:115-119 uses) unless a RandomState is given.  The
        generator is advanced exactly as numpy.random.randn would advance it."""
        self._src(src)
        rs = np.random if random_state is None else random_state
        name, key, pos, has_gauss, cached = rs.get_state()
        if name != "MT19937":
            raise BVError(-1, "add_gaussian_noise needs numpy's legacy MT19937 generator")
        st = ffi.new("bv_mt19937_state *")
        ffi.buffer(st.key)[:] = np.ascontiguousarray(key, dtype=np.uint32).tobytes()
        st.pos, st.has_gauss, st.gauss = int(pos), int(has_gauss), float(cached)
        dst = self.empty(tuple(src.shape))
        check(lib.bv_add_gaussian_noise(self.handle, _u8ptr(src), _u8ptr(dst), src.numel(), float(sigma), st))
        rs.set_state((name, np.frombuffer(ffi.buffer(st.key), dtype=np.uint32).copy(), int(st.pos), int(st.has_gauss),
                      float(st.gauss)))
        return dst

    def letterbox(self, images, out_h=640, out_w=640, pad=114, half=True, out=None):
        """images: contiguous CUDA uint8 [H,W,3] BGR frames.  out: None, or a contiguous [n,3,out_h,out_w] fp16 (half) /
        fp32 tensor on this context's device.  pad is saturated to 0..255."""
        n = len(images)
        for im in images:
            if im.dim() != 3 or im.shape[2] != 3 or im.dtype != torch.uint8 or not im.is_cuda or not im.is_contiguous():
                raise BVError(-1, "letterbox needs contiguous CUDA uint8 [H,W,3] tensors")
        if out is not None:
            if (tuple(out.shape) != (n, 3, out_h, out_w) or out.dtype != (torch.float16 if half else torch.float32)
                    or not out.is_contiguous() or out.device != self.device):
                raise BVError(-1, "out= must be a contiguous %s [%d,3,%d,%d] tensor on %s"
                              % ("float16" if half else "float32", n, out_h, out_w, self.device))
        srcs = ffi.new("uint8_t *[]", [_u8ptr(im) for im in images])
        hs = ffi.new("int32_t[]", [int(im.shape[0]) for im in images])
        ws = ffi.new("int32_t[]", [int(im.shape[1]) for im in images])
        if out is None:
            out = self.empty((n, 3, out_h, out_w), torch.float16 if half else torch.float32)
        check(lib.bv_letterbox(self.handle, ffi.cast("const uint8_t *const *", srcs), hs, ws, n,
                               ffi.cast("void *", out.data_ptr()), out_h, out_w, pad, 1 if half else 0))
        return out

    # -- ZED auxiliary planes --------------------------------------------------------------------
    def rgba_to_rgb(self, src):
        dst = self.empty(tuple(src.shape[:-1]) + (3,))
        check(lib.bv_rgba_to_rgb(self.handle, _u8ptr(src), _u8ptr(dst), src.numel() // 4))
        return dst

    def normals_to_rgb01(self, src):
        dst = self.empty(tuple(src.shape[:-1]) + (3,), torch.float32)
        check(lib.bv_normals_to_rgb01(self.handle, ffi.cast("float *", src.data_ptr()), ffi.cast("float *", dst.data_ptr()),
                                      src.numel() // 4))
        return dst

    def f32_to_u8(self, src, sub=None, div=None, clip_before_scale=False):
        dst = self.empty(tuple(src.shape))
        affine = sub is not None
        check(lib.bv_f32_to_u8(self.handle, ffi.cast("float *", src.data_ptr()), _u8ptr(dst), src.numel(), 1 if affine else 0,
                               float(sub or 0.0), float(div if div is not None else 1.0), 1 if clip_before_scale else 0))
        return dst

    def channel_means(self, src):
        """np.mean(img, axis=(0, 1)) of a uint8 [H,W,C] device image: exact integer sums / count."""
        c = src.shape[-1] if src.dim() == 3 else 1
        sums = self.empty((c,), torch.int64)
        npx = src.numel() // c
        check(lib.bv_channel_sums(self.handle, _u8ptr(src), npx, c, ffi.cast("uint64_t *", sums.data_ptr())))
        return self.download(sums).astype(np.float64) / npx

    # -- fused stage ---------------------------------------------------------------------------
    @staticmethod
    def make_stage(balance=None, cvt=None, lo=(0, 0, 0), hi=(255, 255, 255), morph=(), label=False):
        """Builds a bv_stage_desc.  balance: None or dict of process_frame flags ({} = defaults);
        cvt: None or conversion name; morph: sequence of (op, kw, kh, iterations)."""
        d = ffi.new("bv_stage_desc *")
        d.do_balance = 0 if balance is None else 1
        lib.bv_balance_default(ffi.addressof(d, "balance"))
        if balance:
            for k, v in balance.items():
                setattr(d.balance, k, int(v))
        d.cvt_code = -1 if cvt is None else (CVT[cvt] if isinstance(cvt, str) else int(cvt))
        lo, hi = Context._cv_bounds(lo, hi, 3)          # same convention as in_range / cv2.inRange
        if np.any(lo > 255) or np.any(hi < 0) or np.any(lo > hi):
            lo, hi = np.array([255, 255, 255]), np.array([0, 0, 0])     # empty range
        for k in range(3):
            d.lo[k] = int(np.clip(lo[k], 0, 255))
            d.hi[k] = int(np.clip(hi[k], 0, 255))
        if len(morph) > 4:
            raise BVError(-1, "at most 4 morphology steps")
        d.n_morph = len(morph)
        for i, (op, kw, kh, it) in enumerate(morph):
            d.morph_op[i] = MORPH[op] if isinstance(op, str) else int(op)
            d.morph_kw[i], d.morph_kh[i], d.morph_iters[i] = int(kw), int(kh), int(it)
        d.do_label = 1 if label else 0
        return d

    def stage(self, desc, src, want=("mask",), max_blobs=1024, out=None):
        """Runs the fused stage on a device tensor [B,H,W,3] (or [H,W,3]).  `want` selects the
        outputs among balanced, converted, mask, labels, blobs; returns a dict of device tensors.
        `out` may carry preallocated tensors to reuse."""
        b, h, w, c = self._bhw(src)
        lead = tuple(src.shape[:-1])
        out = dict(out or {})
        one = desc.cvt_code == lib.BV_BGR2GRAY

        def get(name, shape, dtype=torch.uint8):
            if name not in want:
                return None
            if name not in out:
                out[name] = self.empty(shape, dtype)
            return out[name]
        balanced = get("balanced", lead + (3,))
        converted = get("converted", lead if one else lead + (3,))
        mask = get("mask", lead)
        labels = get("labels", lead, torch.int32)
        blobs = get("blobs", (b, max_blobs, BLOB_DTYPE.itemsize))
        if desc.do_label and "n_blobs" not in out:
            out["n_blobs"] = self.empty((b,), torch.int32)
        nb = out.get("n_blobs")
        check(lib.bv_stage(self.handle, desc, _u8ptr(src), b, h, w, _u8ptr(balanced), _u8ptr(converted), _u8ptr(mask),
                           ffi.cast("int32_t *", labels.data_ptr()) if labels is not None else ffi.NULL,
                           ffi.cast("bv_blob *", blobs.data_ptr()) if blobs is not None else ffi.NULL,
                           max_blobs if blobs is not None else 0,
                           ffi.cast("int32_t *", nb.data_ptr()) if nb is not None else ffi.NULL))
        return out

    def stage_host(self, desc, src, want=("mask",), max_blobs=1024, out=None, slot=None):
        """Same stage on HOST arrays (numpy, ideally pinned): upload, run, download, blocking.
        Returns a dict of numpy arrays; `out` may carry preallocated (pinned) arrays.
        slot = 0 or 1: asynchronous form (bv_stage_host_submit): returns at once, the arrays of the returned dict are
        complete after `stage_host_wait(slot)`; two calls (one per slot) may be in flight.  The caller keeps `src` and
        the returned arrays alive (and unmodified) until then."""
        src = np.ascontiguousarray(src, dtype=np.uint8)
        if src.ndim == 3:
            b, (h, w, c) = 1, src.shape
        else:
            b, h, w, c = src.shape
        lead = tuple(src.shape[:-1])
        out = dict(out or {})
        one = desc.cvt_code == lib.BV_BGR2GRAY

        def get(name, shape, dtype=np.uint8):
            if name not in want:
                return None
            if name not in out:
                out[name] = np.empty(shape, dtype)
            return out[name]
        balanced = get("balanced", lead + (3,))
        converted = get("converted", lead if one else lead + (3,))
        mask = get("mask", lead)
        labels = get("labels", lead, np.int32)
        blobs = get("blobs", (b, max_blobs), BLOB_DTYPE)
        if desc.do_label and "n_blobs" not in out:
            out["n_blobs"] = np.zeros((b,), np.int32)
        nb = out.get("n_blobs")

        def p(a, ctype):
            return ffi.cast(ctype, a.ctypes.data) if a is not None else ffi.NULL
        if slot is None:
            check(lib.bv_stage_host(self.handle, desc, p(src, "uint8_t *"), b, h, w, p(balanced, "uint8_t *"),
                                    p(converted, "uint8_t *"), p(mask, "uint8_t *"), p(labels, "int32_t *"),
                                    p(blobs, "bv_blob *"), max_blobs if blobs is not None else 0, p(nb, "int32_t *")))
        else:
            check(lib.bv_stage_host_submit(self.handle, int(slot), desc, p(src, "uint8_t *"), b, h, w, p(balanced, "uint8_t *"),
                                           p(converted, "uint8_t *"), p(mask, "uint8_t *"), p(labels, "int32_t *"),
                                           p(blobs, "bv_blob *"), max_blobs if blobs is not None else 0, p(nb, "int32_t *")))
            self._inflight[int(slot)] = (src, out)   # keeps the buffers alive until the wait
        return out

    def stage_host_wait(self, slot):
        """Blocks until the call submitted on `slot` has delivered its results to the host arrays."""
        check(lib.bv_stage_host_wait(self.handle, int(slot)))
        self._inflight.pop(int(slot), None)


# ---- pinned numpy buffers --------------------------------------------------------------------
class _PinnedBlock:
    """Owner of one cudaHostAlloc'ed block; numpy views made from it keep it (and so the memory) alive."""

    def __init__(self, nbytes):
        self._ptr = lib.bv_host_alloc(max(nbytes, 1))
        if self._ptr == ffi.NULL:
            raise BVError(-4, ffi.string(lib.bv_last_error()).decode())
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "version": 3,
                                    "data": (int(ffi.cast("uintptr_t", self._ptr)), False)}

    def __del__(self):
        try:
            if self._ptr is not None and self._ptr != ffi.NULL:
                lib.bv_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass


class PinnedArray:
    """numpy array over cudaHostAlloc'ed memory (full-speed PCIe for the *_host entry points).  `.array` (and any view
    of it) owns a reference to the block: the memory is released when the last of them is gone."""

    def __init__(self, shape, dtype=np.uint8):
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        block = _PinnedBlock(nbytes)
        self.array = np.asarray(block)[:nbytes].view(dtype).reshape(shape)

    def free(self):
        self.array = None


# ---- default contexts (one per device, created on first use) ----------------------------------
_default = {}
_default_lock = threading.Lock()


def default_context(device=0):
    with _default_lock:
        ctx = _default.get(device)
        if ctx is None:
            ctx = _default[device] = Context(device)
        return ctx
