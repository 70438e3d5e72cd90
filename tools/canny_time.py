#!/usr/bin/env python3
"""bv_canny timed with CUDA events on device-resident frames, next to cv2.Canny on the host: 1920x1080, 2208x1242 and
3840x2160, grey and BGR, batch 1 and 8, aperture 3 with L1 and aperture 5 with L2.

    python tools/canny_time.py [out.log]

Each timed call reads a different copy of its batch, and the copies together hold at least 256 MB, more than the
B200's 126 MB of L2: the source comes from HBM as it does for a fresh camera frame.  "GB/s" is the algorithmic traffic,
(channels + 1) bytes per pixel (the source read once, the 0/255 edges written once), over the device time.  The
per-kernel split of one batch-8 call comes from the library's profiler (serialised launches).  The card's name and
power limit are read in the same run."""
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
VARIANTS = ((50.0, 150.0, 3, False), (400.0, 1200.0, 5, True))
WORKING_SET = 256 << 20
REPS = 30


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
    say("cv2 %s, %d host threads (cv2.Canny per frame, host memory)" % (cv2.__version__, cv2.getNumThreads()))
    ctx = bv.Context(0)
    for h, w in SIZES:
        bgr8 = np.stack([synth.gen_underwater(h, w, 60 + i) for i in range(8)])
        grey8 = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr8])
        for frames8 in (grey8, bgr8):
            ch = 3 if frames8.ndim == 4 else 1
            for b in (1, 8):
                frames = np.ascontiguousarray(frames8[:b])
                nbytes = frames.nbytes
                copies = max(2, -(-WORKING_SET // nbytes))
                srcs = [ctx.upload(frames) for _ in range(copies)]
                dst = ctx.empty((b, h, w))
                for t1, t2, ap, l2 in VARIANTS:
                    def call(src):
                        return lib.bv_canny(ctx.handle, ffi.cast("uint8_t *", src.data_ptr()),
                                            ffi.cast("uint8_t *", dst.data_ptr()), b, h, w, ch, t1, t2, ap, int(l2))
                    for s in srcs:                      # warm-up: every copy once, scratch allocated
                        assert call(s) == 0, ffi.string(lib.bv_last_error()).decode()
                    ctx.sync()
                    got = ctx.download(dst)
                    t0 = time.perf_counter()
                    want = [cv2.Canny(f, t1, t2, apertureSize=ap, L2gradient=l2) for f in frames]
                    cpu_ms = (time.perf_counter() - t0) * 1e3 / b
                    assert all(np.array_equal(got[k], want[k]) for k in range(b)), "bv_canny differs from cv2.Canny"
                    rounds = []
                    for _ in range(3):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(ctx.torch_stream)
                        for r in range(REPS):
                            call(srcs[r % copies])
                        e1.record(ctx.torch_stream)
                        ctx.sync()
                        rounds.append(e0.elapsed_time(e1) / REPS)      # ms per call
                    best = min(rounds)
                    gbs = b * h * w * (ch + 1) / (best * 1e-3) / 1e9
                    line = ("%4dx%-4d %s b=%d ap%d %s  device %7.3f ms/batch %7.3f ms/frame (rounds %s)  %6.1f GB/s  "
                            "cv2 host %7.3f ms/frame  working set %d MB" %
                            (w, h, "BGR " if ch == 3 else "grey", b, ap, "L2" if l2 else "L1", best, best / b,
                             [round(x, 3) for x in rounds], gbs, cpu_ms, copies * nbytes >> 20))
                    if b == 8:
                        ctx.profile(True)
                        ctx.profile_dump()
                        call(srcs[0])
                        split = ctx.profile_dump()
                        ctx.profile(False)
                        line += "  split " + " ".join("%s %.3f" % (k.replace("_kernel", ""), v["ms"])
                                                      for k, v in sorted(split.items()))
                    say(line)
                del srcs, dst
                torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
