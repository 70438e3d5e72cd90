#!/usr/bin/env python3
"""bv_threshold_auto and bv_adaptive_threshold timed with CUDA events on device-resident grey frames, next to
cv2.threshold / cv2.adaptiveThreshold on the host: Otsu, Triangle, MEAN_C at k = 11, 51, 201, 1001 and GAUSSIAN_C at
k = 11, 51, on 1920x1080, 2208x1242 and 3840x2160, batch 1 and 8.

    python tools/threshold_time.py [out.log]

Each timed call reads a different copy of its batch, and the copies together hold at least 256 MB, more than the
B200's 126 MB of L2: the source comes from HBM as it does for a fresh camera frame.  The device output is checked
against cv2 before timing (GAUSSIAN_C k = 51 may differ at proven ties).  The per-kernel split of one batch-8 call comes
from the library's profiler (serialised launches).  The card's name and power limit are read in the same run."""
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
from oracle import threshold_np as tn  # noqa: E402  (tie proof only)

SIZES = ((1080, 1920), (1242, 2208), (2160, 3840))
VARIANTS = (("otsu", None), ("triangle", None), ("mean", 11), ("mean", 51), ("mean", 201), ("mean", 1001),
            ("gaussian", 11), ("gaussian", 51))
WORKING_SET = 256 << 20
REPS = 20


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
    say("cv2 %s, %d host threads (one cv2 call per frame, host memory)" % (cv2.__version__, cv2.getNumThreads()))
    ctx = bv.Context(0)
    th = ctx.empty((8,), torch.float64)
    for h, w in SIZES:
        grey8 = np.stack([cv2.cvtColor(synth.gen_underwater(h, w, 70 + i), cv2.COLOR_BGR2GRAY) for i in range(8)])
        for b in (1, 8):
            frames = np.ascontiguousarray(grey8[:b])
            copies = max(2, -(-WORKING_SET // frames.nbytes))
            srcs = [ctx.upload(frames) for _ in range(copies)]
            dst = ctx.empty((b, h, w))
            for name, k in VARIANTS:
                def call(src):
                    s, d = ffi.cast("uint8_t *", src.data_ptr()), ffi.cast("uint8_t *", dst.data_ptr())
                    if k is None:
                        return lib.bv_threshold_auto(ctx.handle, s, d, b, h, w, 255.0, 0,
                                                     8 if name == "otsu" else 16, ffi.cast("double *", th.data_ptr()))
                    return lib.bv_adaptive_threshold(ctx.handle, s, d, b, h, w, 255.0, 0 if name == "mean" else 1, 0, k,
                                                     2.0)

                def host(f):
                    if k is None:
                        return cv2.threshold(f, 0, 255, 8 if name == "otsu" else 16)[1]
                    return cv2.adaptiveThreshold(f, 255, 0 if name == "mean" else 1, 0, k, 2.0)
                for s in srcs:                      # warm-up: every copy once, scratch allocated
                    assert call(s) == 0, ffi.string(lib.bv_last_error()).decode()
                ctx.sync()
                got = ctx.download(dst)
                t0 = time.perf_counter()
                want = [host(f) for f in frames]
                cpu_ms = (time.perf_counter() - t0) * 1e3 / b
                ties = 0
                for i in range(b):
                    bad = got[i] != want[i]
                    if bad.any():
                        assert name == "gaussian" and k >= 11 and tn.gaussian_ties(frames[i], k)[bad].all(), \
                            "%s k=%s differs from cv2" % (name, k)
                        ties += int(bad.sum())
                rounds = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(ctx.torch_stream)
                    for r in range(REPS):
                        call(srcs[r % copies])
                    e1.record(ctx.torch_stream)
                    ctx.sync()
                    rounds.append(e0.elapsed_time(e1) / REPS)
                best = min(rounds)
                line = ("%4dx%-4d b=%d %-8s k=%-4s device %7.3f ms/batch %7.3f ms/frame (rounds %s)  cv2 host %8.3f "
                        "ms/frame  ties %d  working set %d MB" %
                        (w, h, b, name, k or "-", best, best / b, [round(x, 3) for x in rounds], cpu_ms, ties,
                         copies * frames.nbytes >> 20))
                if b == 8:
                    ctx.profile(True)
                    ctx.profile_dump()
                    call(srcs[0])
                    split = ctx.profile_dump()
                    ctx.profile(False)
                    line += "  split " + " ".join("%s %.3f" % (kk.replace("_kernel", ""), v["ms"])
                                                  for kk, v in sorted(split.items()))
                say(line)
            del srcs, dst
            torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
