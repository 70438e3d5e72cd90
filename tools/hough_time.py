#!/usr/bin/env python3
"""bv_hough_lines timed with CUDA events on device-resident edge maps, next to cv2.HoughLines on the host: Canny maps of
underwater frames (sparse, 0.5 % edge pixels) and of blurred noise (dense, ~33 %) at 1920x1080, 2208x1242 and 3840x2160,
rho = 1, theta = pi / 180, batch 1 and 8.

    python tools/hough_time.py [out.log]

The edge maps stay on the device; they and the accumulators (4-9 MB a frame) are L2-resident after the warm-up, as
they are when the Canny step of the same frame has just written the map.  cv2.HoughLines runs on the first frame of
each batch, in host memory, with its default threads, and the device rows of that frame are checked against it.  The
per-kernel split of one call comes from the library's profiler (serialised launches).  The card's name and power limit
are read in the same run."""
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

SIZES = ((1080, 1920), (1242, 2208), (2160, 3840))
THRESHOLD = 150
REPS = 20
MAX_LINES = 1 << 20


def edge_maps(kind, h, w, b):
    if kind == "underwater":
        return np.stack([cv2.Canny(synth.gen_underwater(h, w, 60 + i), 50, 150) for i in range(b)])
    rng = np.random.default_rng(7)
    return np.stack([cv2.Canny(cv2.GaussianBlur(rng.integers(0, 256, (h, w), dtype=np.uint8), (5, 5), 2.0), 40, 120)
                     for _ in range(b)])


def main():
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else None

    def say(line):
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    say("GPU: %s" % smi)
    say("cv2 %s, %d host threads (cv2.HoughLines(edges, 1, pi/180, %d) per frame, host memory)" %
        (cv2.__version__, cv2.getNumThreads(), THRESHOLD))
    ctx = bv.Context(0)
    for kind in ("underwater", "noise"):
        for h, w in SIZES:
            maps8 = edge_maps(kind, h, w, 8)
            for b in (1, 8):
                maps = np.ascontiguousarray(maps8[:b])
                src = ctx.upload(maps)
                lines = ctx.empty((b, MAX_LINES, 3), torch.float32)
                counts = ctx.empty((b,), torch.int32)

                def call():
                    return lib.bv_hough_lines(ctx.handle, ffi.cast("uint8_t *", src.data_ptr()), b, h, w, 1.0,
                                              np.pi / 180, THRESHOLD, 0.0, np.pi, 0,
                                              ffi.cast("float *", lines.data_ptr()), MAX_LINES,
                                              ffi.cast("int32_t *", counts.data_ptr()))
                for _ in range(3):
                    assert call() == 0, ffi.string(lib.bv_last_error()).decode()
                ctx.sync()
                n0 = int(ctx.download(counts)[0])
                t0 = time.perf_counter()
                want = cv2.HoughLines(maps[0], 1, np.pi / 180, THRESHOLD)
                cpu_ms = (time.perf_counter() - t0) * 1e3
                want = np.zeros((0, 1, 2), np.float32) if want is None else want
                got = ctx.download(lines[0, :n0, :2]).reshape(-1, 1, 2)
                assert got.shape == want.shape and np.array_equal(got.view(np.int32), want.view(np.int32)), \
                    "bv_hough_lines differs from cv2.HoughLines"
                rounds = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(ctx.torch_stream)
                    for _ in range(REPS):
                        call()
                    e1.record(ctx.torch_stream)
                    ctx.sync()
                    rounds.append(e0.elapsed_time(e1) / REPS)
                best = min(rounds)
                ctx.profile(True)
                ctx.profile_dump()
                call()
                split = ctx.profile_dump()
                ctx.profile(False)
                say("%-10s %4dx%-4d b=%d edges %8d lines %6d  device %7.3f ms/batch %7.3f ms/frame (rounds %s)  "
                    "cv2 host %8.2f ms/frame  split %s" %
                    (kind, w, h, b, int((maps[0] > 0).sum()), n0, best, best / b, [round(x, 3) for x in rounds], cpu_ms,
                     " ".join("%s %.3f" % (k.replace("hough_", "").replace("_kernel", ""), v["ms"])
                              for k, v in sorted(split.items()))))
                del src, lines, counts
                torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
