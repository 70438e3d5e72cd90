"""Edge frames of the colour balance's statistics (oracle/edge_frames.py): each generator has the property it claims,
the restatement's zero-width option is the device's stated rule, and -- where oracle/_ref is built -- the compiled
reference equals the restatement on every edge frame on which it is defined."""
import cv2
import numpy as np
import pytest

from oracle import color_balance_np as cb
from oracle import edge_frames as ef
from oracle import ref_balance

# shapes on which the float32 bounds differ from the float64 ones: two of the issue's, one with H*W mod 16 != 0 and
# one above 2^24 pixels, where (float)n itself rounds
BOUND_SHAPES = [(214, 2208), (281, 1920), (203, 601), (4097, 4099)]
SMALL_BOUND_SHAPES = [(1, 500), (1, 501), (480, 640)]


def hsv_limits(img):
    hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
    return cb.percentile_min_max(hsv[..., 1]), cb.percentile_min_max(hsv[..., 2])


def limits_with(ch, bounds):
    return cb.percentile_from_counts(np.bincount(ch.reshape(-1), minlength=256), *bounds)


@pytest.mark.parametrize("shape", BOUND_SHAPES)
def test_float32_bounds_differ_from_float64_on_the_bound_shapes(shape):
    n = shape[0] * shape[1]
    assert ef.f32_bounds(n) != ef.f64_bounds(n)


@pytest.mark.parametrize("shape", BOUND_SHAPES + SMALL_BOUND_SHAPES)
def test_exact_bound_frame_has_its_counts_and_limits(shape):
    img, claim = ef.exact_bound_frame(shape[0], shape[1], seed=1)
    n = shape[0] * shape[1]
    assert (claim["lb"], claim["hb"]) == ef.f32_bounds(n) == (int(np.float32(0.002) * np.float32(n)),
                                                              n - int(np.float32(0.998) * np.float32(n)))
    for c in range(3):
        ch = img[..., c]
        low, high = claim["low"][c], claim["high"][c]
        assert int((ch == low).sum()) == claim["n_low"][c] == claim["lb"] + ef.BGR_OFFSETS[c][0]
        assert int((ch == high).sum()) == claim["n_high"][c] == claim["hb"] + ef.BGR_OFFSETS[c][1]
        assert int(ch.min()) >= low and int(ch.max()) <= high
        assert cb.percentile_min_max(ch) == claim["limits"][c]
    if ef.f32_bounds(n) != ef.f64_bounds(n):
        # the frame tells the two bound computations apart: some channel clips differently under the float64 bounds
        assert any(limits_with(img[..., c], ef.f64_bounds(n)) != claim["limits"][c] for c in range(3))


@pytest.mark.parametrize("shape", BOUND_SHAPES[:3] + [(480, 640)])
def test_exact_bound_sv_frame_has_its_counts_and_limits(shape):
    img, claim = ef.exact_bound_sv_frame(shape[0], shape[1], seed=2)
    hsv = cv2.cvtColor(img, cv2.COLOR_BGR2HSV)
    s, v = hsv[..., 1], hsv[..., 2]
    ts = claim["tail_sv"]
    assert int((s == ts["s_low"][0]).sum()) == claim["counts"]["s_low"] and int(s.min()) == ts["s_low"][0]
    assert int((s == ts["s_high"][0]).sum()) == claim["counts"]["s_high"] and int(s.max()) == ts["s_high"][0]
    assert int((v == ts["v_low"][1]).sum()) == claim["counts"]["v_low"] and int(v.min()) == ts["v_low"][1]
    assert int((v == ts["v_high"][1]).sum()) == claim["counts"]["v_high"] and int(v.max()) == ts["v_high"][1]
    assert hsv_limits(img) == (claim["s_limits"], claim["v_limits"])
    _, st = cb.process_frame_np(img, return_stats=True, **ef.SV_FLAGS)
    assert ((st["s_min"], st["s_max"]), (st["v_min"], st["v_max"])) == (claim["s_limits"], claim["v_limits"])
    n = img.shape[0] * img.shape[1]
    if ef.f32_bounds(n) != ef.f64_bounds(n):
        assert (limits_with(s, ef.f64_bounds(n)), limits_with(v, ef.f64_bounds(n))) != (claim["s_limits"], claim["v_limits"])


@pytest.mark.parametrize("pattern", ef.TIE_PATTERNS)
def test_tie_frame_has_equal_clipped_means(pattern):
    img, claim = ef.tie_frame(240, 320, 5, pattern)
    _, st = cb.process_frame_np(img, return_stats=True)
    avg = dict(zip("bgr", st["bgr_avg"]))
    eq = claim["equal"]
    assert len(eq) >= 2 and all(avg[k] == avg[eq[0]] for k in eq)
    for hi in claim["higher"]:
        for lo in claim["lower"]:
            assert avg[hi] > avg[lo]
    # the tie holds in every tile of a 2x2 tiling too (each tile's mean is taken over the clipped channel)
    _, st2 = cb.process_frame_np(img, return_stats=True, horizontal_blocks=2, vertical_blocks=2)
    for tile in st2["tiles"]:
        loc = dict(zip("bgr", tile["local"]))
        assert all(loc[k] == loc[eq[0]] for k in eq)


@pytest.mark.parametrize("kind", ef.ZERO_WIDTH_KINDS)
def test_zero_width_frame_has_an_empty_range(kind):
    img, claim = ef.zero_width_frame(240, 320, 5, kind)
    flags = claim["flags"]
    base = cb.process_frame_np(img, hsv_contrast_correct=False, **flags)
    (s_lo, s_hi), (v_lo, v_hi) = hsv_limits(base)
    assert (s_lo == s_hi) == ("s" in claim["zero"]) and (v_lo == v_hi) == ("v" in claim["zero"])
    with pytest.raises(ZeroDivisionError):
        cb.process_frame_np(img, **flags)
    if kind == "sparse_red":
        n = img.shape[0] * img.shape[1]
        assert 0 < int((img[..., 2] > 0).sum()) < 0.002 * n


def test_glare_frame_sums_exceed_32_bits():
    img, claim = ef.glare_frame(*ef.GLARE_SHAPE, seed=7)
    n = img.shape[0] * img.shape[1]
    assert n > 1 << 24 and claim["n_white"] >= 0.9 * n
    assert int(np.all(img == 255, axis=2).sum()) >= claim["n_white"]
    for c in range(3):
        assert int(img[..., c].sum(dtype=np.int64)) == claim["sums"][c] > 1 << 32
        assert int(np.bincount(img[..., c].reshape(-1), minlength=256)[255]) >= claim["n_white"]


def test_hsi_edge_frame_has_its_bands():
    img, claim = ef.hsi_edge_frame(384, 512, 3)
    assert img.shape[0] * img.shape[1] >= 128 * 1024
    b, g, r = (img[..., c].astype(int) for c in range(3))
    assert int(((b == g) & (g == r)).sum()) >= claim["grey"] + claim["black"]
    assert int((img.max(axis=2) == 0).sum()) >= claim["black"]
    prim = np.isin(img.reshape(-1, 3).view(np.dtype((np.void, 3))), np.array(ef.PRIMARIES, np.uint8).view(np.dtype((np.void, 3))))
    assert int(prim.sum()) >= claim["primaries"]


# ---------------------------------------------------------------------------------------------------------------------
# the restatement's zero-width option
# ---------------------------------------------------------------------------------------------------------------------
def direct_zero_width_rule(img, **flags):
    """The device's definition stated directly: pass-1 result -> cv2 HSV -> per channel, a zero-width range maps to 0,
    any other range to (x - lo) * 255 / (hi - lo) in integers -> cv2 HSV2BGR."""
    hsv = cv2.cvtColor(cb.process_frame_np(img, hsv_contrast_correct=False, **flags), cv2.COLOR_BGR2HSV)
    out = hsv.copy()
    for k in (1, 2):
        lo, hi = cb.percentile_min_max(hsv[..., k])
        x = np.clip(hsv[..., k].astype(np.int64), lo, hi)
        out[..., k] = 0 if hi == lo else (x - lo) * 255 // (hi - lo)
    return cv2.cvtColor(out, cv2.COLOR_HSV2BGR)


@pytest.mark.parametrize("kind", ef.ZERO_WIDTH_KINDS)
def test_zero_width_option_is_the_stated_rule(kind):
    img, claim = ef.zero_width_frame(240, 320, 5, kind)
    got = cb.process_frame_np(img, zero_width_stretch="zero", **claim["flags"])
    assert np.array_equal(got, direct_zero_width_rule(img, **claim["flags"]))
    if claim["zero"] == "s":      # S -> 0, V still stretched: a grey frame whose levels span the stretched V
        assert np.array_equal(got[..., 0], got[..., 1]) and np.array_equal(got[..., 1], got[..., 2])
        assert int(got.min()) == 0 and int(got.max()) == 255
    else:                         # V -> 0: black
        assert not got.any()


def test_zero_width_option_changes_nothing_on_ordinary_frames():
    img, _ = ef.exact_bound_frame(214, 2208, seed=1)
    want = cb.process_frame_np(img)
    assert np.array_equal(cb.process_frame_np(img, zero_width_stretch="zero"), want)
    assert np.array_equal(direct_zero_width_rule(img), want)
    with pytest.raises(ValueError):
        cb.process_frame_np(img, zero_width_stretch="identity")


def test_nan_and_out_of_range_casts_are_defined():
    # constrain (equalize_lut): NaN -> 0, +inf -> 255, -inf -> 0
    assert cb.constrain([np.nan, np.inf, -np.inf, -0.5, 254.99, 255.5]).tolist() == [0, 255, 0, 0, 254, 255]
    with np.errstate(invalid="ignore"):
        assert cb.equalize_lut(np.inf, False).tolist() == [0] + [255] * 255      # 0 * inf = NaN -> 0
        assert cb.equalize_lut(np.nan, False).tolist() == [0] * 256
        assert cb.equalize_lut(np.nan, True).tolist() == [0] * 256
    # (unsigned char)(int)double: NaN and values outside the int32 range -> INT_MIN -> low byte 0
    assert cb._uchar_cast(np.array([np.nan, np.inf, -np.inf, 2.0 ** 31, 2.0 ** 31 - 1, 300.7, -1.5])).tolist() == \
        [0, 0, 0, 0, 255, 44, 255]


# ---------------------------------------------------------------------------------------------------------------------
# compiled reference == restatement on the edge frames it is defined on
# ---------------------------------------------------------------------------------------------------------------------
def defined_edge_cases():
    cases = [("bound_%dx%d" % s, lambda s=s: ef.exact_bound_frame(s[0], s[1], seed=1)[0], {}) for s in BOUND_SHAPES[:3]]
    cases += [("bound_%dx%d_rgbcc" % s, lambda s=s: ef.exact_bound_frame(s[0], s[1], seed=1)[0], dict(rgb_contrast_correct=True))
              for s in BOUND_SHAPES[:2]]
    cases += [("sv_214x2208", lambda: ef.exact_bound_sv_frame(214, 2208, seed=2)[0], ef.SV_FLAGS)]
    cases += [("tie_%s" % p, lambda p=p: ef.tie_frame(240, 320, 5, p)[0], dict(rgb_contrast_correct=True)) for p in ef.TIE_PATTERNS]
    cases += [("tie_%s_2x2" % p, lambda p=p: ef.tie_frame(240, 320, 5, p)[0], dict(horizontal_blocks=2, vertical_blocks=2))
              for p in ef.TIE_PATTERNS]
    return cases


@pytest.mark.skipif(not ref_balance.available(), reason="oracle/_ref not built")
@pytest.mark.parametrize("name,make,flags", defined_edge_cases(), ids=lambda x: x if isinstance(x, str) else "")
def test_compiled_reference_equals_restatement_on_edge_frames(name, make, flags):
    img = make()
    assert np.array_equal(ref_balance.balance(img, **flags), cb.process_frame_np(img, **flags)), name
