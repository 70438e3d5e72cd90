#!/usr/bin/env python3
"""bv_contour_shapes (arcLength, convexHull, minAreaRect, minEnclosingCircle, approxPolyDP at 0.02 of the arc length,
isContourConvex) timed with CUDA events on a device-resident RETR_TREE / CHAIN_APPROX_SIMPLE table, next to the cv2 host
loop over the same contours on this machine's CPU: a 1920x1080 bins-style mask, a 3840x2160 mask, and eight 4K masks
with thousands of borders.  Prints the card's name and power limit of the same run.

    python tools/contour_shapes_time.py [out.log]"""
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import cuauv_vision_pipeline_b200 as bv  # noqa: E402
from oracle import synth  # noqa: E402  (input generator only)


def bins_mask(h, w, seed):
    hsv = cv2.cvtColor(synth.gen_underwater(h, w, seed), cv2.COLOR_BGR2HSV)
    m = cv2.inRange(hsv, np.array([0, 40, 60]), np.array([179, 255, 255]))
    return cv2.morphologyEx(m, cv2.MORPH_OPEN, np.ones((3, 3), np.uint8))


def noise_4k(seed):
    m = np.full((2160, 3840), 255, np.uint8)
    rng = np.random.default_rng(seed)
    m[rng.random(m.shape) < 0.02] = 0
    m[::97, :] = 0
    return m


def host_loop(masks):
    """The per-contour cv2 calls a module makes today (cv2.findContours itself is not timed)."""
    n = 0
    per = []
    for m in masks:
        per.append(cv2.findContours(m, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)[0])
    t0 = time.perf_counter()
    for cs in per:
        for c in cs:
            a = cv2.arcLength(c, True)
            cv2.approxPolyDP(c, 0.02 * a, True)
            cv2.convexHull(c)
            cv2.minAreaRect(c)
            cv2.minEnclosingCircle(c)
            n += 1
    return (time.perf_counter() - t0) * 1e3, n


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else sys.stdout
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print("gpu: %s" % (smi[0] if smi else torch.cuda.get_device_name(0)), file=out)
    ctx = bv.Context(0)
    cases = [("1920x1080 bins b1", [bins_mask(1080, 1920, 31)]), ("3840x2160 bins b1", [bins_mask(2160, 3840, 32)]),
             ("3840x2160 noise b8", [noise_4k(s) for s in range(8)])]
    for name, masks in cases:
        arr = np.stack(masks)
        dev = ctx.upload(arr)
        table, _, nc, pts, npts = ctx.find_contours(dev, "tree", "simple", 1 << 16, 1 << 22)
        n_rec = int(ctx.download(nc).sum())
        for _ in range(3):
            ctx.contour_shapes(table, nc, pts, "simple", 0.0, 0.02)
        ctx.sync()
        times = []
        for _ in range(20):
            with torch.cuda.stream(ctx.torch_stream):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ctx.contour_shapes(table, nc, pts, "simple", 0.0, 0.02)
                b.record()
            b.synchronize()
            times.append(a.elapsed_time(b))
        host_ms, n_host = host_loop(masks)
        print("%-20s records %6d  bv_contour_shapes median %8.3f ms (min %.3f, max %.3f)  |  cv2 host loop %9.2f ms "
              "over %d contours" % (name, n_rec, float(np.median(times)), min(times), max(times), host_ms, n_host),
              file=out)
        out.flush()
    ctx.close()


if __name__ == "__main__":
    main()
