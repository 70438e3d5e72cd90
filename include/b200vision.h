/*
 * b200vision.h -- C ABI of libb200vision.so: the per-frame pixel hot path of
 * ayf7/cuauv-vision-pipeline as hand-written CUDA for NVIDIA B200 (sm_100a).
 *
 * Style follows the reference's own FFI (lib/camera_message_framework_c.cpp:20-102, bound from
 * core/bindings/camera_message_framework.py:13-70 with cffi in ABI mode): extern "C", opaque
 * handles, plain pointers and sizes, int status codes.  No torch / C++ types cross this boundary.
 *
 * Conventions
 *   - Images are uint8, interleaved HWC, tightly packed (row stride = width * channels), a batch is
 *     `batch` such images back to back.  This is the layout ModuleBase hands to process()
 *     (core/base.py:762-768: C-contiguous np.uint8[H,W,3], BGR).
 *   - Pointers named *_dev are CUDA device pointers (e.g. torch.Tensor.data_ptr()); pointers named
 *     *_host are host pointers.  Small parameter arrays (bounds, structuring elements) are host.
 *   - Every bv_* call on a context enqueues on that context's CUDA stream and returns without
 *     waiting, unless stated otherwise; call bv_sync() (or synchronise the stream) before reading
 *     results on the host.  A context is bound to one device and must be used by one thread at a
 *     time (the reference runs process() calls strictly serially on one worker thread per module,
 *     core/base.py:701-703).
 *   - Return value: BV_OK (0) or a negative bv_status.  bv_last_error() gives the message for
 *     the calling thread.  The library never aborts or exits the process.
 *   - There is no CPU fallback: when no CUDA device is usable, bv_create fails.
 */
#ifndef B200VISION_H
#define B200VISION_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BV_VERSION 100 /* 0.1.0 */

typedef struct bv_ctx bv_ctx;

typedef enum bv_status {
    BV_OK = 0,
    BV_ERR_INVALID = -1,     /* bad argument                                            */
    BV_ERR_CUDA = -2,        /* a CUDA runtime call failed; see bv_last_error()          */
    BV_ERR_UNSUPPORTED = -3, /* valid in the reference but not implemented here          */
    BV_ERR_NOMEM = -4,       /* device or host allocation failed                         */
    BV_ERR_CAPACITY = -5,    /* caller-provided table too small                          */
    BV_ERR_NOT_READY = -6    /* bv_ingest_seqlock: nothing published yet, or torn on every try */
} bv_status;

/* Colour conversions.  Replaces cv2.cvtColor as called from utils/color.py:11-32
 * (_convert_colorspace and the bgr_to_* / *_to_bgr family), modules/bins.py:13,
 * modules/preprocessor.py:56-86.  Values are private to this ABI (not cv2's enum). */
typedef enum bv_cvt_code {
    BV_BGR2HSV = 0,   /* 8-bit, H in [0,180)                                               */
    BV_BGR2LAB = 1,
    BV_BGR2GRAY = 2,  /* 3 -> 1 channel                                                  */
    BV_BGR2YCRCB = 3,
    BV_HSV2BGR = 4,   /* float32 path of OpenCV incl. its 32-px vector/tail rounding rule  */
    BV_BGR2HLS = 5,
    BV_GRAY2BGR = 6,  /* 1 -> 3 channels                                                 */
    BV_BGR2RGB = 7,
    BV_LAB2BGR = 8,   /* OpenCV's 8-bit fixed-point Lab2RGBinteger (utils/color.py:27-29 lab_to_bgr) */
    BV_BGR2LUV = 9    /* OpenCV's 33^3 trilinear table (utils/color.py:30 bgr_to_luv); <= 1 LSB on 0.004 % of colours */
} bv_cvt_code;

/* cv2.threshold types used by utils/color.py:124-201. */
typedef enum bv_thresh_type {
    BV_THRESH_BINARY = 0,     /* x >  t ? maxval : 0   */
    BV_THRESH_BINARY_INV = 1, /* x >  t ? 0 : maxval   */
    BV_THRESH_TRUNC = 2,      /* x >  t ? t : x        */
    BV_THRESH_TOZERO = 3,     /* x >  t ? x : 0        */
    BV_THRESH_TOZERO_INV = 4  /* x >  t ? 0 : x        */
} bv_thresh_type;

/* Morphology.  Replaces cv2.erode / cv2.dilate / cv2.morphologyEx as called from
 * utils/transform.py:80-164 and modules/preprocessor.py:120-129. */
typedef enum bv_morph_op {
    BV_MORPH_ERODE = 0,
    BV_MORPH_DILATE = 1,
    BV_MORPH_OPEN = 2,    /* erode^n then dilate^n */
    BV_MORPH_CLOSE = 3,   /* dilate^n then erode^n */
    BV_MORPH_GRADIENT = 4 /* dilate^n - erode^n    */
} bv_morph_op;

/* Flags of the reference's process_frame (utils/color_correction/color_balance.hpp:9-14), in the
 * same order.  bv_balance_default() fills the defaults of balance()
 * (modules/color_balance.py:93-96). */
typedef struct bv_balance_params {
    int32_t equalize_rgb;
    int32_t rgb_contrast_correct;
    int32_t hsv_contrast_correct;
    int32_t hsi_contrast_correct; /* color_balance.cpp:702-774, <= 1 LSB (csrc/hsi.cu); frame by frame, ~10x the default cost */
    int32_t rgb_extrema_clipping;
    int32_t adaptive_cast_correction;
    int32_t horizontal_blocks;
    int32_t vertical_blocks;
} bv_balance_params;

/* Per-frame statistics the colour balance derived on the device (optional output, host side). */
typedef struct bv_balance_stats {
    int32_t bgr_min[3], bgr_max[3]; /* percentile (or extrema) clip bounds, order B,G,R */
    double bgr_avg[3];              /* exact means of the clipped channels              */
    int32_t dominant;               /* 0=B 1=G 2=R (whole-frame tile)                   */
    int32_t s_min, s_max, v_min, v_max;
    int32_t degenerate;             /* 1 if s_max==s_min or v_max==v_min (reference: SIGFPE) */
} bv_balance_stats;

/* One labelled blob: exact integer raster moments up to third order and the bounding box
 * (inclusive), exact while every sum fits int64 (the widest fully set row whose m30 fits has 77 936 px, and so has the
 * tallest column for m03).  Labels are 1..n in raster order of each blob's first pixel.  Plays the role of
 * outer_contours + contour_centroid + contour_area (utils/feature.py:5-21,240-265). */
typedef struct bv_blob {
    int64_t m00, m10, m01, m20, m11, m02, m30, m21, m12, m03;
    int32_t x0, y0, x1, y1;
} bv_blob;

/* Description of the fused per-frame stage: [colour balance] -> colour conversion -> inRange ->
 * up to 4 morphology steps -> [labelling + moments].  This is modules/bins.py:13-27 and
 * modules/red_buoy.py:21-44 with an optional balance() in front (modules/preprocessor.py:87-88). */
typedef struct bv_stage_desc {
    int32_t do_balance;           /* run colour balance first                             */
    bv_balance_params balance;
    int32_t cvt_code;             /* bv_cvt_code applied to the (balanced) BGR frame;       */
                                  /* -1 = threshold the BGR frame itself                  */
    uint8_t lo[3], hi[3];         /* inclusive bounds per converted channel; a channel is  */
                                  /* ignored by giving lo=0, hi=255                       */
    int32_t n_morph;              /* 0..4 steps on the mask                               */
    int32_t morph_op[4];          /* bv_morph_op                                          */
    int32_t morph_kw[4], morph_kh[4]; /* rectangular structuring element, anchor = centre  */
    int32_t morph_iters[4];
    int32_t do_label;             /* label the final mask and accumulate blob moments      */
} bv_stage_desc;

/* ---- library / context ------------------------------------------------------------------- */
int bv_version(void);
const char *bv_last_error(void);
int bv_device_count(void);
int bv_create(int device, bv_ctx **out);
void bv_destroy(bv_ctx *ctx);
int bv_sync(bv_ctx *ctx);
/* The context's cudaStream_t as an opaque pointer (to wrap it, e.g. torch.cuda.ExternalStream). */
void *bv_stream(bv_ctx *ctx);
/* Use a caller-owned cudaStream_t (NULL restores the context's own stream). */
int bv_set_stream(bv_ctx *ctx, void *cuda_stream);
/* Number of kernels this context has launched so far (bench.py reports it as gpu_launches). */
uint64_t bv_launch_count(const bv_ctx *ctx);

/* Tuning knobs of the colour-balance passes (no reference counterpart).  value <= 0 restores the
 * built-in default.  Each knob is also read once, at bv_create, from the environment variable of
 * the same name (BV_HIST_BPS, BV_FINAL_BPS, BV_SIDE_STREAMS, BV_L2_CHUNK_MB, BV_NO_HUE_TABLE). */
enum {
    BV_OPT_HIST_BPS = 0,     /* blocks per SM of the histogram passes */
    BV_OPT_FINAL_BPS = 1,    /* blocks per SM of the final pass */
    BV_OPT_SIDE_STREAMS = 2, /* independent chunks of one call in flight (1..4) */
    BV_OPT_L2_CHUNK_MB = 3,  /* input bytes per chunk: the chunk and its H,S,V scratch stay in L2 across the passes */
    BV_OPT_NO_HUE_TABLE = 4, /* 1: always do the HSV round trip arithmetically (testing) */
    BV_OPT_CONTOUR_POOL_CHUNKS = 5, /* chunks of the contour walk's vertex pool per frame (testing the second-walk fallback) */
    BV_OPT_FAST_TABLES = 6, /* 1: passes 2 and 3 with per-lane replicated (bank-conflict-free) shared-memory tables; measured slower in a real step, see DESIGN.md */
    BV_OPT_MORPH_VARIANT = 7, /* binary morphology chain: 0 register-rolling warps (default), 1 shared-memory tile filled with plain loads,
                                 2 shared-memory tile filled by one TMA bulk copy (A-B timing, profiles/r02_morph_variants.log) */
    BV_OPT_NO_RCP_TABLES = 8, /* 1: pass 2 looks sdiv / hdiv up in shared memory instead of computing them with the reciprocal unit (A-B timing) */
    BV_OPT_FINAL_SV_TABLES = 9, /* pass 3 of balance -> BGR2LAB: 0 byte S'/V' tables (default); 1 float32 s, v tables; 2 8-byte {s, 1-s} / {v, trunc(255 v)} tables (A-B timing, DESIGN.md 4b) */
    BV_OPT_MORPH_WARPS = 10, /* register-rolling morphology: row strips (= warps) per SM over the whole launch; taller strips re-compute less halo */
    BV_OPT_COUNT = 11
};
int bv_set_option(bv_ctx *ctx, int option, int value);
void bv_balance_default(bv_balance_params *p);
/* Per-kernel timing: while enabled, every kernel launch is bracketed by CUDA events on the
 * context's stream.  bv_profile_dump synchronises, writes a JSON object
 * {"kernel": {"launches": n, "ms": total}, ...} into buf and clears the records. */
int bv_profile_enable(bv_ctx *ctx, int on);
int bv_profile_dump(bv_ctx *ctx, char *buf, size_t cap);

/* ---- colour balance: replaces process_frame (color_balance.cpp:343-780) ------------------- */
/* src_dev -> dst_dev (may alias), batch frames of height x width BGR.  stats_host (optional, may
 * be NULL) receives `batch` records; asking for it forces a stream synchronisation. */
int bv_color_balance(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                     const bv_balance_params *params, bv_balance_stats *stats_host);

/* ---- colour conversion / thresholds -------------------------------------------------------- */
/* planes_dev: optional 3 device pointers receiving the split channels (cv2.split of the result,
 * utils/color.py:22), each batch*height*width bytes; pass NULL to skip.  dst_dev may be NULL when
 * only the planes are wanted. */
int bv_cvt_color(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, uint8_t *const *planes_dev, int batch,
                 int height, int width, int code);
/* cv2.inRange (utils/color.py:121, modules/bins.py:16): channels = 1 or 3. */
int bv_in_range(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *mask_dev, int batch, int height, int width,
                int channels, const uint8_t *lo_host, const uint8_t *hi_host);
/* cv2.threshold on uint8 (utils/color.py:124-201); n = number of bytes. */
int bv_threshold(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n, int thresh, int maxval,
                 int type);
/* cvtColor + inRange in one pass, nothing but the mask is written. */
int bv_cvt_in_range(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *mask_dev, int batch, int height, int width,
                    int code, const uint8_t *lo_host, const uint8_t *hi_host);
/* Per-channel 256-entry look-up tables (lut_host: channels*256 bytes).  Carries the bias /
 * contrast / brightness steps of modules/preprocessor.py:89-109, composed on the host. */
int bv_apply_lut(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n_pixels, int channels,
                 const uint8_t *lut_host);

/* Weighted squared colour distance threshold (thresh_color_distance, utils/color.py:66-103; the percentile
 * option is composed from the two calls below).  planes_dev: the 3 split channels; weights_host: per-channel weights
 * already normalised as the reference does (ignored channels zeroed, divided by the 2-norm of the
 * un-zeroed weights); use_host[c] = 0 skips channel c.  mask_dev: 255 where 0 <= d <= max_dist_sq;
 * dist_dev: uint8(sqrt(d)).  Either output may be NULL. */
int bv_color_distance(bv_ctx *ctx, const uint8_t *const *planes_dev, size_t n, const double *color_host,
                      const double *weights_host, const int32_t *use_host, double max_dist_sq, uint8_t *mask_dev,
                      uint8_t *dist_dev);
/* The float32 squared-distance image itself (the `dists` of utils/color.py:94-97), and the k-th
 * smallest value of a float32 device array (k = 0: the minimum; NaN-free input): the two order
 * statistics np.percentile interpolates between for auto_distance_percentile (utils/color.py:98-99);
 * the interpolation itself is numpy's scalar arithmetic, done by the host mirror (color.py). */
int bv_color_distance_f32(bv_ctx *ctx, const uint8_t *const *planes_dev, size_t n, const double *color_host,
                          const double *weights_host, const int32_t *use_host, float *dists_dev);
int bv_select_kth_f32(bv_ctx *ctx, const float *values_dev, size_t n, size_t k, float *value_host);

/* ---- morphology ------------------------------------------------------------------------------ */
/* se_host: kh*kw bytes (non-zero = member), anchor = centre; channels 1..4 (per channel); src_dev == dst_dev is allowed.
 * Border handling is cv2's default (BORDER_CONSTANT with morphologyDefaultBorderValue).  Iterations as cv2 counts them:
 * a negative count is read as 1; 0 returns the source, and for GRADIENT all zeros.  A rectangle of any size and count is
 * computed (its n iterations are one rectangle with n-fold extents); any other element may have at most 256 horizontal
 * runs (BV_ERR_UNSUPPORTED beyond).  In bv_stage_desc a negative count is rejected (BV_ERR_INVALID) and 0 follows the
 * same rule. */
int bv_morph(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
             int channels, int op, const uint8_t *se_host, int kw, int kh, int iterations);

/* ---- edges ------------------------------------------------------------------------------------ */
/* cv2.Canny(src, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of every frame, bit-exact
 * against OpenCV 4.13.0 (a module's edge detection, cv2.Canny on the host, moved to the device).  src_dev: uint8
 * [batch,H,W,channels], channels 1 or 3; dst_dev: uint8 [batch,H,W] of 0/255.  The rules:
 *   1. dx, dy = Sobel(src, CV_16S, ksize = aperture_size, BORDER_REPLICATE) of each channel; aperture 7 scales them by
 *      1/16 (rounded half to even) and divides both thresholds by 16 first.
 *   2. magnitude |dx| + |dy| (L1) or dx^2 + dy^2 (L2); on 3 channels the channel with the largest magnitude (the first
 *      on a tie) gives the pixel's magnitude, dx and dy.
 *   3. L2: each threshold becomes min(t, 32767), squared when positive; low > high swaps them; both are floored
 *      (INT_MIN for NaN or beyond int32, as cvFloor on x86-64).
 *   4. non-maximum suppression across the gradient direction (tan 22.5 deg in 15-bit fixed point; magnitude 0 outside
 *      the frame): a kept pixel with magnitude > low is a candidate, a candidate with magnitude > high is strong.
 *   5. 255 on every candidate whose 8-connected component of candidates holds a strong pixel (union-find, not a stack).
 * Frames are independent.  BV_ERR_INVALID (as cv2 raises) for an aperture other than 3, 5 or 7; also for overlapping
 * src / dst ranges and for frames or batches past bv_label's 32-bit index limits. */
int bv_canny(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width, int channels,
             double threshold1, double threshold2, int aperture_size, int l2_gradient);

/* ---- connected components + moments ------------------------------------------------------- */
/* 8-connected labelling of mask != 0.  labels_dev: int32[batch,H,W] (0 = background).
 * blobs_dev: bv_blob[batch * max_blobs] (may be NULL), n_blobs_dev: int32[batch] total blob
 * count per frame (blobs beyond max_blobs are labelled but have no table entry). */
int bv_label(bv_ctx *ctx, const uint8_t *mask_dev, int32_t *labels_dev, int batch, int height, int width,
             bv_blob *blobs_dev, int max_blobs, int32_t *n_blobs_dev);

/* One outer border as cv2.findContours(mask, RETR_EXTERNAL, ...) follows it (utils/feature.py:5-21),
 * reduced to what the reference consumes: the Green's-theorem sums of cv2.moments(contour)
 * (contour_centroid, utils/feature.py:240-252) and cv2.contourArea (255-265):
 *   m00 = |a00| / 2,   m10 = a10 / 6,   m01 = a01 / 6   (signs flipped when a00 < 0). */
typedef struct bv_contour {
    int64_t a00, a10, a01;
    int32_t x0, y0, x1, y1;   /* bounding box of the border pixels (inclusive)                    */
    int32_t start_x, start_y; /* first border pixel = the component's first pixel in raster order */
                              /* (hole border, bv_find_contours: the pixel left of the hole's)    */
    int32_t n_points;         /* border pixels visited (length of the CHAIN_APPROX_NONE contour)  */
    int32_t n_simple;         /* vertices kept by CHAIN_APPROX_SIMPLE (utils/feature.py:20)       */
    int32_t label;            /* the component's label in bv_label's numbering (hole border: the  */
                              /* label of the component around the hole)                          */
    int32_t external;         /* 1: reported by RETR_EXTERNAL; 0: lies inside another blob's hole */
                              /* or is a hole border                                              */
    int32_t point_offset;     /* index of its first vertex in the frame's point list, -1 if the   */
                              /* list was not requested or is full                                */
    int32_t reserved;
} bv_contour;

/* contours_dev: bv_contour[batch * max_contours], one record per 8-connected component in raster
 * order of its first pixel (filter on .external for the RETR_EXTERNAL set); n_contours_dev:
 * int32[batch] number of components (may exceed max_contours; may be NULL).
 * points_dev (optional): int32[batch][max_points][2] receiving the CHAIN_APPROX_SIMPLE vertices
 * (x, y) of the external contours in cv2's order, contour after contour; n_points_dev (optional):
 * int32[batch] vertices needed per frame (may exceed max_points: contours that do not fit get
 * point_offset = -1). */
int bv_outer_contours(bv_ctx *ctx, const uint8_t *mask_dev, int batch, int height, int width,
                      bv_contour *contours_dev, int max_contours, int32_t *n_contours_dev, int32_t *points_dev,
                      int max_points, int32_t *n_points_dev);

/* Every border of cv2.findContours(mask, mode, method) with its hierarchy (utils/feature.py:25-40
 * all_contours; vision_common.py Hierarchy / fill_ratio).  Values are cv2's. */
typedef enum bv_retr_mode {
    BV_RETR_LIST = 1,  /* no hierarchy: every parent and child is -1                                */
    BV_RETR_CCOMP = 2, /* outer borders at the top level, each hole a child of its component's border */
    BV_RETR_TREE = 3   /* the full nesting                                                           */
} bv_retr_mode;
typedef enum bv_chain_approx {
    BV_CHAIN_APPROX_NONE = 1,  /* every border pixel                                               */
    BV_CHAIN_APPROX_SIMPLE = 2 /* the pixels where the chain turns (cyclically, so the start of a  */
                               /* hole border is dropped when the chain runs straight through it)  */
} bv_chain_approx;
/* The same set of borders as cv2 (one outer border per 8-connected component, one hole border per
 * 4-connected background region that does not touch the image edge), in this order, per frame:
 *   records 0 .. n_outer-1: the outer borders, in bv_label's label order, equal to the records
 *     bv_outer_contours writes;
 *   records n_outer .. n_outer+n_holes-1: the hole borders, in raster order of the hole's first
 *     pixel; start_x/start_y = the pixel left of it, label = the enclosing component's label,
 *     external = 0.
 * cv2 lists the same borders in an order of its own; each border's vertex list is identical.
 * contours_dev: bv_contour[batch * max_contours].  hierarchy_dev (optional, 16-byte aligned):
 * int32[batch][max_contours][4] = cv2's (next, prev, first_child, parent) over this record order;
 * siblings are linked in increasing record order and first_child is the smallest child.
 * n_contours_dev (optional): int32[batch][2] = (n_outer, n_holes), which may exceed max_contours:
 * records past max_contours are not written, and hierarchy links then reach only written records.
 * points_dev (optional): int32[batch][max_points][2] receiving the vertices (x, y) of every record
 * in cv2's order, record after record; n_points_dev (optional): int32[batch] vertices the written
 * records need per frame (may exceed max_points: records that do not fit get point_offset = -1).
 * mode = BV_RETR_EXTERNAL (cv2's 0) is bv_outer_contours. */
int bv_find_contours(bv_ctx *ctx, const uint8_t *mask_dev, int batch, int height, int width, int mode, int method,
                     bv_contour *contours_dev, int32_t *hierarchy_dev, int max_contours, int32_t *n_contours_dev,
                     int32_t *points_dev, int max_points, int32_t *n_points_dev);

/* cv2.minAreaRect of every external contour (modules/bins.py:60-69; utils/feature.py:301-312), from
 * the vertex lists bv_outer_contours wrote (same contours_dev / n_contours_dev / points_dev /
 * max_contours / max_points).  rects_dev: bv_rrect[batch * max_contours], entry i belongs to contour
 * record i; valid = 0 for records that are not external or whose vertices did not fit.
 * ((cx, cy), (width, height), angle) as cv2 4.13.0 reports them (angle in [-90, 0) degrees);
 * float32, tolerance 1e-4 relative on the area (see csrc/rects.cu). */
typedef struct bv_rrect {
    float cx, cy, width, height, angle;
    int32_t valid;
} bv_rrect;
int bv_min_area_rects(bv_ctx *ctx, const bv_contour *contours_dev, const int32_t *n_contours_dev,
                      const int32_t *points_dev, int batch, int max_contours, int max_points, bv_rrect *rects_dev);

/* Shape descriptors of every record of a contour table, from bv_find_contours (any mode, NONE or SIMPLE:
 * counts_per_frame = 2, n_contours_dev = its (n_outer, n_holes) pairs) or bv_outer_contours (SIMPLE,
 * counts_per_frame = 1), with the same contours_dev / points_dev / max_contours / max_points.  method (bv_chain_approx)
 * selects each record's vertex count: n_points (NONE) or n_simple (SIMPLE); counts_per_frame = 1 takes SIMPLE only
 * (BV_ERR_INVALID otherwise).  shapes_dev: bv_shape[batch *
 * max_contours], entry i belongs to record i; valid = 0 for records past the count or max_contours and for records
 * whose vertices did not fit (point_offset < 0), and nothing else is written for them.
 * hull_dev / approx_dev (optional, NULL skips; a NULL approx_dev skips the Douglas-Peucker work): int32[batch]
 * [max_points][2], shaped as points_dev; a record's hull and approximation start at its own point_offset (both have at
 * most as many vertices as the record; the rest of the record's slots in approx_dev are overwritten as scratch).
 * Each record's approximation accuracy is eps = approx_epsilon + approx_relative * arc_length (double, no fused
 * multiply-add), the value `k * cv2.arcLength(c, True)` gives a caller.  Exactness against cv2 4.13.0:
 *   arc_length      cv2.arcLength(c, True): bit-exact (float32 steps, summed exactly in double)
 *   hull, n_hull    cv2.convexHull(c) (clockwise=False): the same vertices in the same order; the same first vertex
 *                   for every contour that visits no pixel twice (cv2's first vertex depends on the order its
 *                   unstable sort leaves repeated pixels in; the library takes the first visit of each pixel)
 *   rect            cv2.minAreaRect(c), hole borders included; outer records bit-equal to bv_min_area_rects
 *   approx          cv2.approxPolyDP(c, eps, True): bit-exact (OpenCV 4.13's algorithm, which splits a slice at the
 *                   point farthest from its chord segment, in the same double operations)
 *   approx_convex   cv2.isContourConvex(approx): exact
 *   circle          cv2.minEnclosingCircle(c): the exact circle of the hull in double, radius + 1e-4, rounded to
 *                   float32; cv2 itself is within ~1.3e-4 px of it (stated tolerance 2e-3 px) */
typedef struct bv_shape {
    double arc_length;
    float circle_cx, circle_cy, circle_r;
    bv_rrect rect;
    int32_t n_hull;
    int32_t n_approx;
    int32_t approx_convex;
    int32_t valid;
    int32_t reserved;
} bv_shape;
int bv_contour_shapes(bv_ctx *ctx, const bv_contour *contours_dev, const int32_t *n_contours_dev, int counts_per_frame,
                      const int32_t *points_dev, int batch, int max_contours, int max_points, int method,
                      double approx_epsilon, double approx_relative, bv_shape *shapes_dev, int32_t *hull_dev,
                      int32_t *approx_dev);

/* ---- resize / YOLO input ------------------------------------------------------------------ */
/* cv2.resize(..., INTER_LINEAR) on uint8 (utils/transform.py:179, modules/preprocessor.py:136-143). */
int bv_resize_linear(bv_ctx *ctx, const uint8_t *src_dev, int src_h, int src_w, uint8_t *dst_dev, int dst_h,
                     int dst_w, int channels, int batch);
/* Letterbox + BGR->RGB + HWC->CHW + /255 for n frames of possibly different sizes
 * (the Ultralytics pre-transform behind modules/yolo.py:112).  srcs_host: n device pointers;
 * out_dev: [n,3,out_h,out_w] of fp16 (out_fp16 != 0) or fp32.  n <= 256.  pad_value is saturated
 * to 0..255 as cv2.copyMakeBorder does on uint8 (300 pads with 255, -5 with 0). */
int bv_letterbox(bv_ctx *ctx, const uint8_t *const *srcs_host, const int32_t *heights_host,
                 const int32_t *widths_host, int n, void *out_dev, int out_h, int out_w, int pad_value,
                 int out_fp16);

/* ---- smoothing / warping steps of the preprocessor ------------------------------------------- */
/* cv2.GaussianBlur(src, (ksize_x, ksize_y), sigma_x, sigma_y) on uint8, BORDER_REFLECT_101
 * (modules/preprocessor.py:110-114 calls it with ksize = 2k+1 and sigma 0).  sigma <= 0: derived
 * from the kernel size as OpenCV does.  OpenCV's 8.8 fixed-point arithmetic, bit-exact. */
int bv_gaussian_blur(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                     int channels, int ksize_x, int ksize_y, double sigma_x, double sigma_y);
/* cv2.warpAffine(src, M, (dst_width, dst_height), flags=INTER_LINEAR, borderMode, borderValue) on
 * uint8; m_host: the 2x3 forward matrix in row-major doubles, as cv2 takes it
 * (modules/preprocessor.py:130-135 rotate with BORDER_REPLICATE, 144-149 translate with the default
 * BORDER_CONSTANT 0).  border_value_host: `channels` bytes or NULL (0). */
typedef enum bv_border_mode { BV_BORDER_CONSTANT = 0, BV_BORDER_REPLICATE = 1 } bv_border_mode;
int bv_warp_affine(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                   int channels, int dst_height, int dst_width, const double *m_host, int border_mode,
                   const uint8_t *border_value_host);
/* Lens undistortion (include/camera_filters.hpp:6-11 declares the maps and their initialiser; the reference holds no
 * definition or call site, so parity is pinned to the cv2 calls such a definition makes).
 * bv_remap == cv2.remap(src, map1, map2, INTER_LINEAR, borderMode, borderValue) on uint8; the maps live on the device and
 * serve every frame of the batch.  BV_MAP_F32: map1 / map2 are float32 x / y planes (CV_32FC1); BV_MAP_FIXED: map1 is
 * int16 (x, y) pairs, map2 uint16 (fy * 32 + fx, read & 1023 as cv2 does) (CV_16SC2 + CV_16UC1, what cv2.convertMaps and
 * cv2.undistort use).  A float map value becomes cvRound(x * 32) as OpenCV computes it on x86-64: round half to even, and
 * INT_MIN for NaN, +-inf and |x * 32| >= 2^31 (such a tap lands on the left / top border, whichever its sign); the
 * integer part is then saturated to int16.  Bit-exact in both formats.  src_dev != dst_dev. */
typedef enum bv_map_format { BV_MAP_F32 = 0, BV_MAP_FIXED = 1 } bv_map_format;
int bv_remap(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width, int channels,
             int dst_height, int dst_width, const void *map1_dev, const void *map2_dev, int map_format, int border_mode,
             const uint8_t *border_value_host);
/* cv2.initUndistortRectifyMap(camera_matrix, dist_coeffs, R, new_camera_matrix, (width, height), ...): float32 maps
 * (mapx_dev / mapy_dev, CV_32FC1) and / or the fixed-point pair (map_xy_dev / map_frac_dev) that cv2.undistort derives
 * straight from the float64 coordinates; either pair may be NULL.  camera_matrix_host: 3x3 row-major; dist_coeffs_host:
 * n_dist = 0, 4, 5 or 8 values k1 k2 p1 p2 [k3 [k4 k5 k6]]; inv_new_camera_rot_host: inverse of
 * (new_camera_matrix x R), 3x3 row-major.  float64 arithmetic in OpenCV's order: identical maps on the reference's
 * camera files (lib/configs/<n>_camera_matrix_params.yaml); in general to the last float32 bit.  Fixed-point pair:
 * saturate_cast<int>(u * 32) (INT_MIN for NaN and values beyond int32, as cvRound on x86-64), integer part saturated to
 * int16 as cv2's vector code does (cv2's scalar code for the last width mod (2 x float64 lanes) columns of a row
 * truncates instead; the two agree wherever a ray stays within int16). */
int bv_undistort_maps(bv_ctx *ctx, const double *camera_matrix_host, const double *dist_coeffs_host, int n_dist,
                      const double *inv_new_camera_rot_host, int width, int height, float *mapx_dev, float *mapy_dev,
                      int16_t *map_xy_dev, uint16_t *map_frac_dev);
/* The middle step of white_balance_bgr_blur (utils/color.py:381-391) on an 8-bit LAB image: a and b are moved by
 * their local mean, `a - (cv2.blur(a, (ksize, ksize), BORDER_REPLICATE) - 128)` in float32, then cast the way
 * numpy's astype(uint8) casts (truncation, wrap-around); L is copied.  The BGR2LAB before and the LAB2BGR after are
 * bv_cvt_color calls.  Bit-exact (cv2.blur of a float plane sums in double, exact for 8-bit values). */
int bv_lab_shift_local_mean(bv_ctx *ctx, const uint8_t *lab_dev, uint8_t *dst_dev, int batch, int height, int width,
                            int ksize);

/* Gaussian-noise step of the preprocessor (modules/preprocessor.py:115-119):
 *   dst = clip(src + numpy.random.randn(n_values) * sigma, 0, 255).astype(uint8)
 * with the values numpy's legacy global generator (MT19937 + polar method) would draw from `state`, which is
 * numpy.random.get_state() in C form and is advanced exactly as numpy.random.randn advances it (hand it back with
 * numpy.random.set_state).  Synchronous.  The random values go through the device's double-precision log, which
 * may differ from the host libm's in the last bit of ~0.1 % of the values; a pixel changes only if its sum lies
 * within that bit of an integer (stated tolerance: <= 1 LSB, expected on < 1e-10 of the pixels). */
typedef struct bv_mt19937_state {
    uint32_t key[624];
    int32_t pos;
    int32_t has_gauss;
    double gauss;
} bv_mt19937_state;
int bv_add_gaussian_noise(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n_values, double sigma,
                          bv_mt19937_state *state);

/* ---- shared-memory ingest (replaces Block::read_frame's memcpy, lib/camera_message_framework.cpp:423-453, and the
 *      writable copy of core/base.py:762-768) -------------------------------------------------------------------------
 * A ring of `slots` frame slots in host memory that a writer fills round robin and guards with a sequence lock, described
 * by plain pointers so that the header does not depend on the transport's private struct (lib/camera_message_framework.cpp
 * :39-54): `uid` = frames published so far, the newest one lives in slot uid % slots; slot i's sequence words are at
 * v_begin + i * meta_stride (FrameMetadata::v_a, stamped after the payload is in place) and v_end + i * meta_stride
 * (FrameMetadata::v_b, stamped last); its payload starts at data + i * slot_stride.  The memory should be pinned
 * (bv_host_register on the mapping) for full-speed DMA. */
typedef struct bv_seqlock_ring {
    const volatile uint64_t *uid;
    const volatile uint64_t *v_begin;
    const volatile uint64_t *v_end;
    size_t meta_stride;
    const uint8_t *data;
    size_t slot_stride;
    int slots;
} bv_seqlock_ring;
/* Copies the newest frame (height x width x src_channels bytes at payload_offset inside its slot) to dst_dev as packed
 * 3-channel pixels: one H2D DMA on the context's stream, then the slot is re-validated (v_begin == v_end as the reference
 * reader does, and uid has not advanced far enough for the writer to be back in this slot); a torn copy is repeated up to
 * max_retries times.  src_channels == 4 drops the fourth byte on the device (swap_rb: RGBA -> BGR).  Blocking (the
 * validation needs the copy to be complete); the frame is ready on the context's stream when it returns.
 * BV_ERR_NOT_READY: nothing published yet / still torn after max_retries. */
int bv_ingest_seqlock(bv_ctx *ctx, const bv_seqlock_ring *ring, size_t payload_offset, uint8_t *dst_dev, int height,
                      int width, int src_channels, int swap_rb, int max_retries, uint64_t *uid_out, int *retries_out);

/* ---- ZED auxiliary planes (capture_sources/zed.{py,cpp}, modules/poster.py, modules/record.py) ----- */
/* Drop the alpha byte (cv2.cvtColor(RGBA2RGB), capture_sources/zed.py:49-50; zed.cpp:54-71). */
int bv_rgba_to_rgb(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n_pixels);
/* float4 normals -> 3 floats (v + 1) * 0.5 (capture_sources/zed.cpp:73-91). */
int bv_normals_to_rgb01(bv_ctx *ctx, const float *src_xyzw_dev, float *dst_rgb_dev, size_t n_pixels);
/* float32 plane -> uint8 for display.  y = apply_affine ? (x - sub) / div : x, then
 * clip_before_scale == 0: clip(y * 255, 0, 255)   (modules/poster.py:41-47, modules/calibrate.py:111)
 * clip_before_scale != 0: clip(y, 0, 1) * 255      (modules/record.py:106-109)
 * truncated to uint8 like numpy's astype.  NaN -> 0 (undefined in numpy). */
int bv_f32_to_u8(bv_ctx *ctx, const float *src_dev, uint8_t *dst_dev, size_t n, int apply_affine, float sub, float div,
                 int clip_before_scale);
/* Exact per-channel sums of an interleaved uint8 image: the numerators of np.mean(img, axis=(0,1))
 * (modules/auto_calibrate_zed.py:82).  sums_dev: uint64[channels]. */
int bv_channel_sums(bv_ctx *ctx, const uint8_t *src_dev, size_t n_pixels, int channels, uint64_t *sums_dev);

/* ---- fused stage --------------------------------------------------------------------------- */
/* Any output pointer may be NULL to skip it.  balanced_dev: BGR after colour balance;
 * converted_dev: image after desc->cvt_code; mask_dev: uint8 0/255 after the morphology steps;
 * labels_dev / blobs_dev / n_blobs_dev as in bv_label. */
int bv_stage(bv_ctx *ctx, const bv_stage_desc *desc, const uint8_t *src_dev, int batch, int height, int width,
             uint8_t *balanced_dev, uint8_t *converted_dev, uint8_t *mask_dev, int32_t *labels_dev,
             bv_blob *blobs_dev, int max_blobs, int32_t *n_blobs_dev);
/* Same stage fed from and returning to HOST memory (pinned memory gives full PCIe speed):
 * uploads, runs, downloads, and returns after the results are in the host buffers. */
int bv_stage_host(bv_ctx *ctx, const bv_stage_desc *desc, const uint8_t *src_host, int batch, int height,
                  int width, uint8_t *balanced_host, uint8_t *converted_host, uint8_t *mask_host,
                  int32_t *labels_host, bv_blob *blobs_host, int max_blobs, int32_t *n_blobs_host);
/* The same call split in two, for a caller that has the next batch ready while the previous one is still being returned
 * (the vision daemon runs one module process per camera, core/base.py:669-844; a process that serves several cameras, or
 * works on frame k's results while frame k+1 is on its way, uses this).  bv_stage_host_submit enqueues the uploads, the
 * kernels and the downloads and returns; the host output buffers are complete after bv_stage_host_wait(ctx, slot).
 * slot is 0 or 1: each has its own device staging, so two calls can be in flight and the uploads of one overlap the
 * downloads of the other (PCIe is full duplex).  Calls execute in submission order.  Submitting on a slot first waits
 * for that slot's previous call.  Host buffers must stay valid until the wait returns and should be pinned
 * (bv_host_alloc / bv_host_register): a copy from or to pageable memory makes the submit block. */
int bv_stage_host_submit(bv_ctx *ctx, int slot, const bv_stage_desc *desc, const uint8_t *src_host, int batch, int height,
                         int width, uint8_t *balanced_host, uint8_t *converted_host, uint8_t *mask_host,
                         int32_t *labels_host, bv_blob *blobs_host, int max_blobs, int32_t *n_blobs_host);
int bv_stage_host_wait(bv_ctx *ctx, int slot);

/* ---- pinned host memory (so the *_host entry points run at full PCIe speed) ---------------- */
void *bv_host_alloc(size_t bytes);               /* cudaHostAlloc; NULL on failure            */
void bv_host_free(void *p);
int bv_host_register(void *p, size_t bytes);      /* pin an existing buffer (e.g. a CMF frame) */
int bv_host_unregister(void *p);

/* ---- legacy symbol ------------------------------------------------------------------------- */
/* Exact signature of the reference's libauv-color-balance.so entry point
 * (utils/color_correction/color_balance.hpp:9-14), so modules/color_balance.py:93-110 works
 * unchanged: host buffer, in place, blocking.  Returns 0 on success (the reference always
 * returns 0, color_balance.cpp:779), non-zero bv_status on failure.  Uses a process-wide context
 * on device $BV_DEVICE (default 0), serialised by a mutex. */
int process_frame(unsigned char *arr, size_t height, size_t width, size_t depth, bool equalize_rgb,
                  bool rgb_contrast_correct, bool hsv_contrast_correct, bool hsi_contrast_correct,
                  bool rgb_extrema_clipping, bool adaptive_cast_correction, int horizontal_blocks,
                  int vertical_blocks);

#ifdef __cplusplus
}
#endif
#endif /* B200VISION_H */
