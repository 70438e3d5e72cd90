"""GPU: bv_hough_lines against cv2.HoughLinesWithAccumulator with 0 differing bits and cv2's counts on every case of
oracle/hough_cases.py (each batch in one call, guard bytes around the outputs, the launch list of the shared-memory and
the global-atomic vote paths checked by the profiler), truncation at max_lines, the arguments it rejects, the wrappers'
shapes, stream ordering from a side stream, and the device chain hough_lines(canny(...))."""
import math

import cv2
import numpy as np
import pytest
import torch

from cuauv_vision_pipeline_b200 import BVError, feature
from oracle import canny_cases as cc
from oracle import hough_cases as hc
from oracle import hough_np as hn

pytestmark = pytest.mark.gpu

CASES = hc.by_group(hc.all_cases())
GUARD = 16          # float32 / int32 words on each side of the outputs
POISON = -12345


def lib():
    from cuauv_vision_pipeline_b200.runtime import ffi, lib as lib_
    return ffi, lib_


def cv2_rows(frame, c):
    rho, theta, thr, mn, mx, ev = c.args
    got = cv2.HoughLinesWithAccumulator(frame, rho, theta, thr, min_theta=mn, max_theta=mx, use_edgeval=ev)
    return np.zeros((0, 3), np.float32) if got is None else got.reshape(-1, 3)


def expected_launches(c, h, w):
    """One edge, one vote, one peak and one sort kernel; the vote kernel is the global-atomic one when a row of
    numrho + 2 int32 bins does not fit in the opt-in shared memory; no peak kernel when there is no rho bin."""
    na, nr = hn.counts(h, w, c.rho, c.theta, c.min_theta, c.max_theta)
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    vote = "hough_vote_kernel" if (nr + 2) * 4 <= optin else "hough_vote_global_kernel"
    out = {"hough_edges_kernel": 1, vote: 1, "hough_sort_kernel": 1}
    if nr > 0:
        out["hough_peaks_kernel"] = 1
    return out


def call(ctx, frames, c, max_lines, profile=False):
    """One C-ABI call for the whole batch into outputs with guard words on both sides -> (status, rows, counts,
    launches)."""
    ffi, L = lib()
    b, h, w = frames.shape
    src = ctx.upload(frames)
    with torch.cuda.stream(ctx.torch_stream):
        lines = torch.full((GUARD + b * max_lines * 3 + GUARD,), float(POISON), dtype=torch.float32, device=ctx.device)
        counts = torch.full((GUARD + b + GUARD,), POISON, dtype=torch.int32, device=ctx.device)
    if profile:
        ctx.profile(True)
        ctx.profile_dump()
    try:
        rc = L.bv_hough_lines(ctx.handle, ffi.cast("uint8_t *", src.data_ptr()), b, h, w, float(c.rho), float(c.theta),
                              int(c.threshold), float(c.min_theta), float(c.max_theta), int(c.use_edgeval),
                              ffi.cast("float *", lines.data_ptr() + 4 * GUARD), max_lines,
                              ffi.cast("int32_t *", counts.data_ptr() + 4 * GUARD))
        kernels = {k: v["launches"] for k, v in ctx.profile_dump().items()} if profile else None
    finally:
        if profile:
            ctx.profile(False)
    host_lines, host_counts = ctx.download(lines), ctx.download(counts)
    assert (host_lines[:GUARD] == POISON).all() and (host_lines[GUARD + b * max_lines * 3:] == POISON).all(), \
        "wrote outside lines_dev"
    assert (host_counts[:GUARD] == POISON).all() and (host_counts[GUARD + b:] == POISON).all(), "wrote outside n_lines_dev"
    return rc, host_lines[GUARD:GUARD + b * max_lines * 3].reshape(b, max_lines, 3), host_counts[GUARD:GUARD + b], kernels


def run_case(ctx, c):
    frames = c.frames()
    b, h, w = frames.shape
    want = [cv2_rows(f, c) for f in frames]
    max_lines = max(1, max(len(x) for x in want))
    rc, rows, counts, kernels = call(ctx, frames, c, max_lines, profile=True)
    if rc != 0:
        ffi, L = lib()
        return "%s: status %d: %s" % (c.name, rc, ffi.string(L.bv_last_error()).decode())
    for k in range(b):
        if counts[k] != len(want[k]):
            return "%s frame %d: %d lines, cv2 has %d" % (c.name, k, counts[k], len(want[k]))
        got = rows[k, :len(want[k])]
        bad = np.argwhere(got.view(np.int32) != want[k].view(np.int32))
        if bad.size:
            i, j = bad[0]
            return "%s frame %d: %d differing values, first row %d col %d: got %r, want %r" % (
                c.name, k, len(bad), i, j, got[i], want[k][i])
        if (rows[k, len(want[k]):] != POISON).any():
            return "%s frame %d: wrote rows past its lines" % (c.name, k)
    if kernels != expected_launches(c, h, w):
        return "%s: ran %s" % (c.name, kernels)
    return None


@pytest.mark.parametrize("group", sorted(CASES))
def test_cases_match_cv2(ctx, group):
    failures = [f for f in (run_case(ctx, c) for c in CASES[group]) if f]
    assert not failures, "%d failing cases:\n  %s" % (len(failures), "\n  ".join(failures[:20]))


def test_both_vote_paths_are_exercised():
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    paths = set()
    for c in hc.all_cases():
        _, h, w = c.frames().shape
        paths |= set(expected_launches(c, h, w))
    assert {"hough_vote_kernel", "hough_vote_global_kernel"} <= paths, optin


def test_truncation_reports_every_line(ctx):
    """max_lines smaller than the line count: the first max_lines rows of each frame in cv2's order, nothing written
    past them, and n_lines still the full count; max_lines = 0 writes counts only."""
    c = [x for x in CASES["batch"] if x.name == "batch5"][0]
    frames = c.frames()
    want = [cv2_rows(f, c) for f in frames]
    for cap in (0, 1, 7):
        rc, rows, counts, _ = call(ctx, frames, c, cap)
        assert rc == 0
        assert list(counts) == [len(x) for x in want]
        for k in range(len(frames)):
            m = min(cap, len(want[k]))
            assert np.array_equal(rows[k, :m].view(np.int32), want[k][:m].view(np.int32))
            assert (rows[k, m:] == POISON).all()


def test_rejects_what_cv2_rejects_and_past_the_limits(ctx):
    ffi, L = lib()
    buf = ctx.upload(np.zeros(64 * 64 * 2, np.uint8))
    out = ctx.empty((2 * 10 * 3,), torch.float32)
    cnt = ctx.empty((2,), torch.int32)
    src = ffi.cast("uint8_t *", buf.data_ptr())
    lines = ffi.cast("float *", out.data_ptr())
    n = ffi.cast("int32_t *", cnt.data_ptr())

    def rc(rho=1.0, theta=math.pi / 180, mn=0.0, mx=math.pi, ev=0, b=1, h=64, w=64, s=src, li=lines, nl=n, cap=10):
        return L.bv_hough_lines(ctx.handle, s, b, h, w, rho, theta, 10, mn, mx, ev, li, cap, nl)
    n0 = ctx.launches
    bad = [dict(rho=0.0), dict(rho=-1.0), dict(rho=1e-50), dict(rho=float("nan")), dict(rho=float("inf")),
           dict(theta=0.0), dict(theta=-0.1), dict(theta=1e-50), dict(theta=float("nan")),
           dict(mn=1.0, mx=0.5), dict(mn=float("nan")), dict(mx=float("inf")),
           dict(b=0), dict(h=0), dict(w=-1), dict(cap=-1), dict(h=65536, w=1), dict(h=1, w=65536),
           dict(h=3000, w=3000, ev=1),                                   # 255 * H * W past INT32_MAX
           dict(theta=1e-9),                                             # past 2^31 accumulator bins
           dict(s=ffi.NULL), dict(nl=ffi.NULL), dict(li=ffi.NULL),
           dict(li=ffi.cast("float *", buf.data_ptr() + 64)),            # lines inside the source
           dict(nl=ffi.cast("int32_t *", out.data_ptr() + 8)),           # counts inside the lines
           dict(nl=ffi.cast("int32_t *", buf.data_ptr() + 4096 - 4))]
    for kw in bad:
        assert rc(**kw) == L.BV_ERR_INVALID, kw
    assert ctx.launches == n0
    # accepted at the edges: an empty angle range, a range past pi, 4K with use_edgeval, no line buffer with cap 0
    assert rc(mn=0.2, mx=0.2) == 0 and rc(mn=-0.5, mx=4.0) == 0 and rc(li=ffi.NULL, cap=0) == 0
    big = ctx.empty((2160 * 3840,))
    assert rc(s=ffi.cast("uint8_t *", big.data_ptr()), h=2160, w=3840, ev=1) == 0
    with pytest.raises(BVError):
        ctx.hough_lines(buf.view(2, 64, 64), 1, 0, 10)


def test_wrapper_shapes_and_none(ctx):
    frame = hc.canny_underwater(1, 120, 160, 800)[0]
    ref = cv2.HoughLines(frame, 1, np.pi / 180, 15)
    got = feature.hough_lines(frame, 1, np.pi / 180, 15)
    assert isinstance(got, np.ndarray) and got.shape == ref.shape and got.dtype == np.float32
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    acc = cv2.HoughLinesWithAccumulator(frame, 1, np.pi / 180, 15)
    got = feature.hough_lines(frame, 1, np.pi / 180, 15, votes=True)
    assert got.shape == acc.shape == (len(ref), 1, 3) and np.array_equal(got.view(np.int32), acc.view(np.int32))
    assert feature.hough_lines(np.zeros((30, 40), np.uint8), 1, np.pi / 180, 0) is None
    assert feature.hough_lines(frame, 1, np.pi / 180, 10 ** 6) is None
    # max_lines is a first guess: a frame with more lines is served in full by one more call
    got = feature.hough_lines(frame, 1, np.pi / 180, 15, max_lines=3)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    batch = np.stack([frame, np.zeros_like(frame), hc.canny_underwater(1, 120, 160, 801)[0]])
    out = feature.hough_lines(batch, 1, np.pi / 180, 15, max_lines=2)
    assert isinstance(out, list) and len(out) == 3 and out[1] is None
    for k in (0, 2):
        assert np.array_equal(out[k].view(np.int32), cv2.HoughLines(batch[k], 1, np.pi / 180, 15).view(np.int32))
    dev = feature.hough_lines(ctx.upload(frame), 1, np.pi / 180, 15)
    assert dev.is_cuda and dev.dtype == torch.float32 and tuple(dev.shape) == ref.shape
    lines, n = ctx.hough_lines(ctx.upload(frame), 1, np.pi / 180, 15, max_lines=8)
    assert tuple(lines.shape) == (8, 3) and int(n) == len(ref)
    with pytest.raises(ValueError):
        feature.hough_lines(frame, 1, np.pi / 180, 15, srn=2)
    with pytest.raises(ValueError):
        feature.hough_lines(frame, 1, np.pi / 180, 15, stn=2)
    with pytest.raises(TypeError):
        feature.hough_lines(frame.astype(np.float32), 1, np.pi / 180, 15)
    with pytest.raises(BVError):
        feature.hough_lines(frame, 0, np.pi / 180, 15)
    with pytest.raises(BVError):
        feature.hough_lines(frame, 1, np.pi / 180, 15, min_theta=1.0, max_theta=0.5)
    for bad in (ctx.upload(frame)[:, 10:50], ctx.upload(frame).float(), ctx.upload(frame)[None, None]):
        with pytest.raises(BVError):
            ctx.hough_lines(bad, 1, np.pi / 180, 15)


def test_feature_hough_lines_on_a_side_stream():
    """A CUDA tensor produced on the caller's side stream -> CUDA tensors the caller can consume on that stream with no
    synchronisation of its own."""
    edges = hc.canny_underwater(2, 270, 480, 810)
    want = [cv2.HoughLinesWithAccumulator(f, 1, np.pi / 180, 40) for f in edges]
    side = torch.cuda.Stream()
    pinned = torch.from_numpy(edges).pin_memory()
    for rep in range(3):
        with torch.cuda.stream(side):
            acc = pinned.to("cuda", non_blocking=True).to(torch.int32)
            for _ in range(40):
                acc = acc + 3
            for _ in range(40):
                acc = acc - 3
            out = feature.hough_lines(acc.to(torch.uint8), 1, np.pi / 180, 40, votes=True)
            host = [(t + 0).cpu() for t in out]                           # the caller's stream again
        side.synchronize()
        for k in range(2):
            assert want[k] is not None and np.array_equal(host[k].numpy().view(np.int32), want[k].view(np.int32)), (rep, k)


def test_hough_lines_of_device_canny_matches_cv2(ctx):
    """hough_lines(canny(device frame)) stays on the device until the lines come back, and equals
    cv2.HoughLines(cv2.Canny(frame)) bit for bit."""
    for h, w, seed in ((1080, 1920, 820), (480, 640, 821)):
        frame = cc.underwater(1, h, w, seed)[0]
        edges = feature.canny(ctx.upload(frame), 50, 150)
        assert edges.is_cuda
        got = feature.hough_lines(edges, 1, np.pi / 180, 80)
        ref = cv2.HoughLines(cv2.Canny(frame, 50, 150), 1, np.pi / 180, 80)
        if ref is None:
            assert got is None
        else:
            assert got.is_cuda and np.array_equal(got.cpu().numpy().view(np.int32), ref.view(np.int32))
