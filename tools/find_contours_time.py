#!/usr/bin/env python3
"""bv_find_contours (RETR_TREE, CHAIN_APPROX_SIMPLE) and bv_outer_contours timed with CUDA events on device-resident
masks, against cv2.findContours(RETR_TREE, CHAIN_APPROX_SIMPLE) on the host, at 1920x1080 and 3840x2160, batch 1 and 8.

    python tools/find_contours_time.py [--baseline-lib other/libb200vision.so]

--baseline-lib times bv_outer_contours of another build of the library (e.g. the previous commit's) in the same run,
alternating with this one, so that the RETR_EXTERNAL path can be compared without a second process."""
import argparse
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import cuauv_vision_pipeline_b200 as bv  # noqa: E402
from cuauv_vision_pipeline_b200._ffi import ffi, lib  # noqa: E402
from oracle import synth  # noqa: E402  (input generator only)


def mask_for(h, w, seed):
    """bins-style mask: HSV inRange of a synthetic underwater frame, OPEN 3x3 (many blobs, many holes)."""
    hsv = cv2.cvtColor(synth.gen_underwater(h, w, seed), cv2.COLOR_BGR2HSV)
    m = cv2.inRange(hsv, np.array([0, 40, 60]), np.array([179, 255, 255]))
    return cv2.morphologyEx(m, cv2.MORPH_OPEN, np.ones((3, 3), np.uint8))


class Runner:
    """One library + one context; buffers sized for the batch."""

    def __init__(self, library, b, h, w, max_contours, max_points):
        self.lib = library
        out = ffi.new("bv_ctx **")
        check_status = library.bv_create(0, out)
        assert check_status == 0, check_status
        self.ctx = out[0]
        self.stream = torch.cuda.ExternalStream(int(ffi.cast("uintptr_t", library.bv_stream(self.ctx))))
        dev = torch.device("cuda", 0)
        self.b, self.h, self.w, self.mc, self.mp = b, h, w, max_contours, max_points
        self.table = torch.empty((b, max_contours, ffi.sizeof("bv_contour")), dtype=torch.uint8, device=dev)
        self.hier = torch.empty((b, max_contours, 4), dtype=torch.int32, device=dev)
        self.nc = torch.empty((b, 2), dtype=torch.int32, device=dev)
        self.pts = torch.empty((b, max_points, 2), dtype=torch.int32, device=dev)
        self.npts = torch.empty((b,), dtype=torch.int32, device=dev)

    def p(self, t, kind):
        return ffi.cast(kind, t.data_ptr())

    def outer(self, mask):
        return self.lib.bv_outer_contours(self.ctx, self.p(mask, "uint8_t *"), self.b, self.h, self.w,
                                          self.p(self.table, "bv_contour *"), self.mc, self.p(self.nc, "int32_t *"),
                                          self.p(self.pts, "int32_t *"), self.mp, self.p(self.npts, "int32_t *"))

    def tree(self, mask):
        return self.lib.bv_find_contours(self.ctx, self.p(mask, "uint8_t *"), self.b, self.h, self.w, lib.BV_RETR_TREE,
                                         lib.BV_CHAIN_APPROX_SIMPLE, self.p(self.table, "bv_contour *"),
                                         self.p(self.hier, "int32_t *"), self.mc, self.p(self.nc, "int32_t *"),
                                         self.p(self.pts, "int32_t *"), self.mp, self.p(self.npts, "int32_t *"))

    def time(self, fn, mask, reps):
        for _ in range(3):
            assert fn(mask) == 0
        self.lib.bv_sync(self.ctx)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(reps):
            fn(mask)
        e1.record(self.stream)
        self.lib.bv_sync(self.ctx)
        return e0.elapsed_time(e1) * 1e3 / reps   # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print("GPU:", smi)
    print("cv2 %s, %d host threads (cv2.findContours is single-threaded)" % (cv2.__version__, cv2.getNumThreads()))
    base = ffi.dlopen(args.baseline_lib) if args.baseline_lib else None
    for (h, w) in ((1080, 1920), (2160, 3840)):
        for b in (1, 8):
            masks = np.stack([mask_for(h, w, 40 + i) for i in range(b)])
            ref = [cv2.findContours(m, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE) for m in masks]
            n_max = max(len(c) for c, _ in ref)
            p_max = max(sum(len(x) for x in c) for c, _ in ref)
            t0 = time.perf_counter()
            for m in masks:
                cv2.findContours(m, cv2.RETR_TREE, cv2.CHAIN_APPROX_SIMPLE)
            cpu_us = (time.perf_counter() - t0) * 1e6
            mc, mp = n_max + 1024, p_max + 65536
            cur = Runner(lib, b, h, w, mc, mp)
            dev = torch.from_numpy(masks).cuda()
            torch.cuda.synchronize()
            assert cur.tree(dev) == 0
            cur.lib.bv_sync(cur.ctx)
            nc = cur.nc.cpu().numpy()
            assert all(int(nc[f].sum()) == len(ref[f][0]) for f in range(b)), "border counts differ from cv2"
            tree_us, outer_us, base_us = [], [], []
            other = Runner(base, b, h, w, mc, mp) if base is not None else None
            for _ in range(args.rounds):
                tree_us.append(cur.time(cur.tree, dev, args.reps))
                outer_us.append(cur.time(cur.outer, dev, args.reps))
                if other is not None:
                    base_us.append(other.time(other.outer, dev, args.reps))
            line = ("%4dx%-4d b=%d  borders/frame<=%6d  find_contours TREE/SIMPLE %8.1f us/batch (rounds %s)  "
                    "outer_contours %8.1f us/batch (rounds %s)" %
                    (w, h, b, n_max, min(tree_us), [round(x, 1) for x in tree_us], min(outer_us),
                     [round(x, 1) for x in outer_us]))
            if base_us:
                line += "  baseline outer_contours %8.1f us/batch (rounds %s)" % (min(base_us), [round(x, 1) for x in base_us])
            line += "  cv2 RETR_TREE host %9.1f us/batch" % cpu_us
            print(line, flush=True)
            lib.bv_destroy(cur.ctx)
            if other is not None:
                base.bv_destroy(other.ctx)


if __name__ == "__main__":
    main()
