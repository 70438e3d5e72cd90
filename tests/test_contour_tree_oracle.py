"""cv2.findContours(RETR_LIST / CCOMP / TREE) against scipy labellings: the facts oracle/contour_tree.py relies on to put
cv2's borders into bv_find_contours' record order (CPU only)."""
import cv2
import numpy as np
import pytest

from oracle import contour_tree as ct
from oracle import synth


def _random_masks():
    """300 seeded masks: blurred noise at random thresholds, salt-and-pepper, sizes 1x1 .. 90x90."""
    out = []
    for seed in range(300):
        rng = np.random.default_rng(1000 + seed)
        h, w = int(rng.integers(1, 91)), int(rng.integers(1, 91))
        if seed % 3 == 0:
            m = (rng.random((h, w)) < rng.uniform(0.2, 0.8)).astype(np.uint8) * 255
        else:
            f = cv2.GaussianBlur(rng.random((h, w)).astype(np.float32), (0, 0), rng.uniform(0.7, 3.0))
            m = (f > np.quantile(f, rng.uniform(0.2, 0.8))).astype(np.uint8) * 255
        out.append(("random%d" % seed, m))
    return out


def _special_masks():
    out = [("1x1_on", np.full((1, 1), 255, np.uint8)), ("1x1_off", np.zeros((1, 1), np.uint8)),
           ("all0", np.zeros((20, 30), np.uint8)), ("all255", np.full((20, 30), 255, np.uint8))]
    one_hole = np.full((20, 30), 255, np.uint8)
    one_hole[7, 11] = 0
    out.append(("one_hole", one_hole))
    for n in (1, 2, 5, 31):
        out.append(("row%d" % n, synth.mask_random(1, n, n, 0.6)))
        out.append(("col%d" % n, synth.mask_random(n, 1, n, 0.6)))
    # diagonal-only contacts: the holes of a diagonal lattice touch each other only at corners
    d = np.zeros((24, 24), np.uint8)
    d[(np.add.outer(np.arange(24), np.arange(24)) % 4) == 0] = 255
    d[(np.subtract.outer(np.arange(24), np.arange(24)) % 4) == 0] = 255
    out.append(("diagonal_lattice", d))
    out.append(("diagonals", synth.mask_diagonals(40, 50)))
    out.append(("rings", synth.mask_rings(61, 70, step=3)))
    ring = np.zeros((9, 9), np.uint8)
    cv2.rectangle(ring, (1, 1), (7, 7), 255, 1)
    out.append(("ring", ring))
    edge = np.full((10, 12), 255, np.uint8)
    edge[3:6, 0:4] = 0                                            # background reaching the edge: no hole border
    edge[0:2, 6] = 0
    out.append(("edge_regions", edge))
    return out


MASKS = _random_masks() + _special_masks()


@pytest.mark.parametrize("name,mask", MASKS, ids=[n for n, _ in MASKS])
def test_findcontours_facts(name, mask):
    reg = ct.regions(mask)
    n = len(reg["outer_start"]) + len(reg["hole_start"])
    hier = {}
    for mode in ("list", "ccomp", "tree"):
        none, h_none = cv2.findContours(mask, ct.MODES[mode], cv2.CHAIN_APPROX_NONE)
        simple, h_simple = cv2.findContours(mask, ct.MODES[mode], cv2.CHAIN_APPROX_SIMPLE)
        # 1 + 2: one border per component and per hole, starting where regions() says (record_order asserts both)
        assert len(none) == n
        perm = ct.record_order(mask, none, reg)
        # 5: NONE and SIMPLE list the borders in the same order with the same hierarchy
        assert len(simple) == n
        if n:
            assert np.array_equal(h_none, h_simple)
        # 4: SIMPLE is NONE without the points where the step direction does not change, cyclically
        for a, b in zip(none, simple):
            assert np.array_equal(ct.simple_from_none(a), b)
        # 3: the parents
        parent = ct.remap_hierarchy(h_none, perm)[:, 3].tolist() if n else []
        assert parent == ct.expected_parent(reg, mode), mode
        hier[mode] = parent
        # the restatement round-trips
        for method in ("none", "simple"):
            canon = ct.canonical(mask, mode, method, reg)
            back, back_h = ct.restore(canon)
            assert len(back) == len(canon["cv_contours"])
            assert all(np.array_equal(x, y) for x, y in zip(back, canon["cv_contours"]))
            if n:
                assert np.array_equal(back_h, canon["cv_hierarchy"])
    # every outer border's start pixel is a turn of the chain; only hole borders lose their start under SIMPLE
    none, _ = cv2.findContours(mask, cv2.RETR_TREE, cv2.CHAIN_APPROX_NONE)
    for r, i in enumerate(ct.record_order(mask, none, reg)[:len(reg["outer_start"])]):
        s = ct.simple_from_none(none[i])
        assert tuple(s[0, 0]) == tuple(none[i][0, 0])


def test_hole_start_pixel_is_dropped_by_simple_on_some_masks():
    """The start of a hole border is not always a vertex of CHAIN_APPROX_SIMPLE (the chain can run straight through)."""
    dropped = 0
    for _, mask in MASKS:
        reg = ct.regions(mask)
        canon = ct.canonical(mask, "tree", "simple", reg)
        for r in range(canon["n_outer"], canon["n_outer"] + canon["n_holes"]):
            dropped += tuple(canon["contours"][r][0, 0]) != tuple(canon["none"][r][0, 0])
    assert dropped > 0


def test_record_links_rule():
    parent = [-1, -1, 4, -1, 0, 0, 1]
    links = ct.record_links(parent)
    assert links.tolist() == [[1, -1, 4], [3, 0, 6], [-1, -1, -1], [-1, 1, -1], [5, -1, 2], [-1, 4, -1], [-1, -1, -1]]
