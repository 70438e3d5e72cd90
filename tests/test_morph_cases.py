"""CPU: the morphology and labelling cases of oracle/morph_cases.py reach the paths they were written for, and the cv2
facts the device's morphology rules rely on hold (cv2 4.13.0)."""
import cv2
import numpy as np
import pytest

from oracle import morph_cases as mc

STAGE = mc.stage_cases()
GREY = mc.grey_cases()


def test_every_stage_case_reaches_its_path():
    wrong = [(c.name, c.path, str(c.predicted())) for c in STAGE if str(c.predicted()) != c.path]
    assert not wrong, wrong


def test_stage_cases_reach_every_binary_path():
    assert mc.reachable_morph_paths() <= {str(c.predicted()) for c in STAGE}


def test_roll_strip_split_at_its_edges():
    paths = {c.name: c.predicted() for c in STAGE if c.predicted().kind == "roll"}
    assert paths["roll_one_strip_per_frame"].strips == 1                        # batch >= sm_count * 8
    assert {p.strip_rows for n, p in paths.items() if n.startswith("roll_height")} == {1, 2, 3, 4}
    assert any(c.warps not in (0, 8) for c in STAGE)
    assert any(c.predicted().strips > 1 for c in STAGE if c.predicted().kind == "roll")


def test_step_cases_take_two_and_three_passes_in_both_directions():
    seen = set()
    for c in STAGE:
        p = c.predicted()
        if p.kind != "step":
            continue
        for entry in p.passes:
            if entry in ("zero", ()):
                continue
            op, hp, vp = entry
            basics = {"erode": ("erode",), "dilate": ("dilate",)}.get(op, ("erode", "dilate"))
            for b in basics:
                if hp > vp:
                    seen.add((b, "h", hp))
                if vp > hp:
                    seen.add((b, "v", vp))
                if hp == vp:
                    seen.add((b, "hv", hp))
    for b in ("erode", "dilate"):
        for d in ("h", "v", "hv"):
            for p in (2, 3):
                assert (b, d, p) in seen, (b, d, p)


def test_step_cases_cover_gradient_and_identity_steps():
    passes = [e for c in STAGE if c.predicted().kind == "step" for e in c.predicted().passes]
    assert "zero" in passes and () in passes
    assert any(c.predicted().kind == "step" and c.predicted().family is None for c in STAGE)    # a memset only
    assert any(e[0] == "gradient" and max(e[1:]) > 1 for e in passes if isinstance(e, tuple) and e)
    for op in mc.OPS:       # 1x1 and zero-iteration steps of every op
        assert any(c.steps == [(op, 1, 1, 1)] for c in STAGE) and any(c.steps == [(op, 5, 5, 0)] for c in STAGE)


def test_tma_cases_stage_some_tiles_by_bulk_copy_and_some_by_loads():
    staged = []
    for c in STAGE:
        p = c.predicted()
        if c.variant == 2 and p.kind == "chain":
            b, h, w = c.shape
            staged += mc.tma_staged_tiles(p, b, h, w, mc.halo_up(c.steps)).values()
    assert True in staged and False in staged


def test_stage_cases_cover_widths_heights_batches_and_entries():
    widths = {c.shape[2] for c in STAGE}
    assert {1, 31, 32, 33, 63, 64, 65, 1025, 2048, 2049, 4096, 4097, 6145} <= widths and max(widths) > 25600
    assert {1, 2, 3, 4, 1025} <= {c.shape[1] for c in STAGE}
    assert {1, 3} <= {c.shape[0] for c in STAGE} and max(c.shape[0] for c in STAGE) > mc.SM_COUNT * 8
    assert {True, False} == {c.bits_direct() for c in STAGE}
    assert any(c.mask_off and c.shape[2] % 16 == 0 for c in STAGE)       # aligned width, unaligned buffer


def test_large_element_cases_are_neither_empty_nor_full():
    """A zero-versus-zero comparison proves nothing: the big erosions see bars, the big dilations a few points."""
    for c in STAGE:
        if c.nontrivial:
            for f, m in enumerate(c.masks()):
                r = mc.cv2_steps(m, c.steps)
                assert r.any() and not r.all(), (c.name, f)
    for c in GREY:
        if c.group == "grey_large":
            r = c.want(c.image())
            assert r.any() and not r.all(), c.name


def test_every_grey_case_reaches_its_path():
    wrong = [(c.name, c.path, str(c.predicted())) for c in GREY if str(c.predicted()) != c.path]
    assert not wrong, wrong
    kinds = {str(c.predicted()) for c in GREY}
    assert {"copy", "zero", "zero-by-difference", "rect/1", "rect/2", "rect/3", "runs"} <= kinds
    for op in mc.OPS:
        assert any(c.op == op and c.in_place for c in GREY), op
    assert {1, 2, 3, 4} <= {c.shape[3] for c in GREY} and {1, 2, 3} <= {c.dst_off for c in GREY}
    assert any(c.shape[0] > 1 for c in GREY)
    assert any(mc.horizontal_runs(c.se) == mc.GREY_MAX_RUNS for c in GREY)
    # the horizontal extent of a rectangle passes int16 in at least one case
    assert any(c.se.all() and (c.se.shape[1] // 2) * c.iterations > 32767 for c in GREY)
    assert {0, 1, 2, 3, -1, -7} <= {c.iterations for c in GREY}


# ---------------------------------------------------------------------------------------------------------------------
# the cv2 facts behind the device's rules
# ---------------------------------------------------------------------------------------------------------------------
def _masks(seed, n=6):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        h, w = rng.integers(1, 60, 2)
        yield ((rng.random((h, w)) < rng.uniform(0.3, 0.95)) * 255).astype(np.uint8)


@pytest.mark.parametrize("vertical", [False, True])
@pytest.mark.parametrize("fn", [cv2.erode, cv2.dilate])
def test_segments_with_inner_anchors_compose_under_the_ignored_border(fn, vertical):
    """bv_morph applies the column taps y-U .. y+D in passes of at most 256 rows: with out-of-image taps ignored, an
    erosion (dilation) by a segment that contains its anchor, followed by one by another such segment, is the erosion
    (dilation) by the summed segment.  Checked against cv2 on random masks and random splits, frames smaller than the
    segments included."""
    rng = np.random.default_rng(5 if vertical else 6)
    for m in _masks(1 if vertical else 2, 40):
        parts = [(int(rng.integers(0, 30)), int(rng.integers(0, 30))) for _ in range(int(rng.integers(2, 4)))]
        U, D = sum(p[0] for p in parts), sum(p[1] for p in parts)

        def seg(u, d, m):
            k = np.ones((u + d + 1, 1) if vertical else (1, u + d + 1), np.uint8)
            return fn(m, k, anchor=(0, u) if vertical else (u, 0))
        step = m
        for u, d in parts:
            step = seg(u, d, step)
        assert np.array_equal(step, seg(U, D, m)), (m.shape, parts)


def test_cv2_gradient_with_zero_iterations_is_all_zero():
    """Fix 1: cv2.morphologyEx(GRADIENT, iterations=0) returns zeros; the other ops return the source."""
    img = np.random.default_rng(3).integers(0, 256, (30, 41, 3), dtype=np.uint8)
    for m in (img, img[..., 0] > 127):
        m = np.ascontiguousarray(m.astype(np.uint8) * (255 if m.dtype == bool else 1))
        k = np.ones((3, 3), np.uint8)
        assert not cv2.morphologyEx(m, cv2.MORPH_GRADIENT, k, iterations=0).any()
        for op in ("erode", "dilate", "open", "close"):
            assert np.array_equal(cv2.morphologyEx(m, mc.CV_OP[op], k, iterations=0), m), op


@pytest.mark.parametrize("op", mc.OPS)
def test_cv2_reads_negative_iterations_as_one(op):
    """Fix 2: bv_morph clamps a negative count to 1, as cv2 does for erode, dilate and morphologyEx."""
    img = np.random.default_rng(4).integers(0, 256, (33, 47), dtype=np.uint8)
    for k in (np.ones((3, 5), np.uint8), cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (5, 5))):
        one = cv2.morphologyEx(img, mc.CV_OP[op], k, iterations=1)
        for it in (-1, -7):
            assert np.array_equal(cv2.morphologyEx(img, mc.CV_OP[op], k, iterations=it), one), it
    assert np.array_equal(cv2.erode(img, np.ones((3, 3), np.uint8), iterations=-2), cv2.erode(img, np.ones((3, 3), np.uint8)))
    assert np.array_equal(cv2.dilate(img, np.ones((3, 3), np.uint8), iterations=-2), cv2.dilate(img, np.ones((3, 3), np.uint8)))


def _window_reduce(m, L, R, axis, erode):
    """Binary erosion / dilation of rows (axis 1) or columns (axis 0) by the taps -L .. R, out-of-image taps ignored."""
    a = np.moveaxis(m != 0, axis, -1)
    n = a.shape[-1]
    bad = ~a if erode else a
    c = np.concatenate([np.zeros(a.shape[:-1] + (1,), np.int64), np.cumsum(bad, axis=-1)], axis=-1)
    idx = np.arange(n)
    lo, hi = np.clip(idx - L, 0, n), np.clip(idx + R + 1, 0, n)
    cnt = c[..., hi] - c[..., lo]
    out = (cnt == 0) if erode else (cnt > 0)
    return np.moveaxis(out, -1, axis).astype(np.uint8) * 255


def test_cv2_computes_rectangles_past_int16_and_256_rows():
    """Fix 4: cv2 computes a 255-wide rectangle at 259 iterations (taps 32 893 px either side, past int16) and a 255-tall
    one at 2 iterations (509 rows, past one 256-row launch): n iterations of a rectangle are one rectangle with n-fold
    extents, out-of-image taps ignored."""
    wide = mc.make_mask("rows", (1, 6, 40000), 8)[0]
    assert np.array_equal(cv2.erode(wide, np.ones((1, 255), np.uint8), iterations=259), _window_reduce(wide, 32893, 32893, 1, True))
    pts = mc.make_mask("points", (1, 4, 40000), 9)[0]
    assert np.array_equal(cv2.dilate(pts, np.ones((1, 255), np.uint8), iterations=259), _window_reduce(pts, 32893, 32893, 1, False))
    tall = mc.make_mask("cols", (1, 700, 20), 10)[0]
    assert np.array_equal(cv2.erode(tall, np.ones((255, 1), np.uint8), iterations=2), _window_reduce(tall, 254, 254, 0, True))
    even = np.ones((254, 1), np.uint8)      # anchor 127: taps 2 * 127 above, 2 * 126 below
    assert np.array_equal(cv2.dilate(tall, even, iterations=2), _window_reduce(tall, 254, 252, 0, False))


def test_int64_moment_limits():
    """bv_blob moments are exact while they fit int64: a fully set row of W px has m30 = (W (W - 1) / 2)^2, the widest
    such row (and, for m03, the tallest column) is the limit frame of the GPU tests."""
    w = mc.m30_limit_width()
    s3 = (w * (w - 1) // 2) ** 2
    assert s3 <= 2 ** 63 - 1 < ((w + 1) * w // 2) ** 2
    assert w < 2 ** 17
    assert mc.run_moment_sums(0, w - 1, 0)["m30"] == s3 == sum(x ** 3 for x in range(w))
    m = mc.run_moment_sums(5, 9, 3)
    xs = np.arange(5, 10)
    assert m == {"m00": 5, "m10": int(xs.sum()), "m01": 15, "m20": int((xs ** 2).sum()), "m11": 3 * int(xs.sum()), "m02": 45,
                 "m30": int((xs ** 3).sum()), "m21": 3 * int((xs ** 2).sum()), "m12": 9 * int(xs.sum()), "m03": 135}


def test_label_cases_cover_the_labelling_paths():
    cases = {c.name: c for c in mc.label_cases()}
    assert any(c.masks.shape[1] > 1024 and c.masks.shape[2] < 3840 for c in cases.values())
    assert any(c.masks.shape[2] > 1024 and c.masks.shape[2] % 32 for c in cases.values())
    tails = [c.masks.shape[1] * mc.words_per_row(c.masks.shape[2]) % 32 for c in cases.values()]
    assert any(tails)
    assert {0, 1} <= {c.max_blobs for c in cases.values()}
    ov = cases["overflow_per_frame"]
    counts = [cv2.connectedComponents(f, connectivity=8)[0] - 1 for f in ov.masks]
    assert len(set(counts)) == len(counts) and sum(n > ov.max_blobs for n in counts) >= 2 and min(counts) < ov.max_blobs
