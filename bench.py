#!/usr/bin/env python3
"""bench.py -- frames/s of the per-frame pixel hot path on N B200s, with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], "C2"): ZED 2208x1242 stereo frames through balance() (default
flags, modules/color_balance.py:93-96) and BGR2LAB (utils/color.py:26).  One step = one batch of
64 frames (32 stereo pairs, 526 MB > L2) per GPU taken from a ring of 128 synthetic frames (1.05 GB;
consecutive steps use different batches).  Frames shard by index across GPUs with no collective
("weak" scaling: 64 frames per GPU per step).  The host-buffer legs move 32 frames per call.

One JSON line on stdout (rank 0).  `value`: device-resident frames/s, CUDA events on the library's
stream.  `e2e`: same stage through bv_stage_host_submit / _wait (and, beside it, the blocking bv_stage_host) with pinned HOST buffers, H2D + D2H inside the
timed region.  `roofline`: dominant kernel, per-launch CUDA-event time from the library's own
profiler; `stage_roofline`: the whole step against the algorithmic 6 B/px.  `cpu_baseline`: the
reference's compiled process_frame + cv2.cvtColor on the host cores (reported, not a target).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 1242, 2208
BATCH = 64       # frames per device-resident call: the join at the end of a call drains the side streams; long calls amortise it
                 # and take 8-frame chunks (tools/batch_sweep.py: 16 / 32 / 64 frames per call = 64.7 / 68.9 / 71.8 k frames/s)
E2E_BATCH = 32   # frames per host-buffer call (pinned buffers: 4 x 263 MB)
RING = 128       # 64 generated frames + 64 cyclic shifts of them (same statistics, every pixel somewhere else)
BPP_C2 = 6          # SURVEY.md 8d: BGR in (3) + LAB image out (3)
METRIC = "frames/sec at 2208x1242"


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self, wait_s=5.0):
        """Starts nvidia-smi and waits for its first sample, so that even a short timed region is
        covered (nvidia-smi needs ~0.5 s to come up)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < wait_s:
                time.sleep(0.02)
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark(self):
        """Index of the next sample: samples[mark_a:mark_b] belong to a timed region."""
        return len(self.lines)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, first=0, last=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # the device-resident region can be shorter than one sampling period: widen by one sample
        # on each side, the rest of the window (profile + end-to-end legs) is under load as well
        lines = self.lines[max(0, first - 1):(None if last is None else last + 1)] or self.lines
        for ln in lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_ring(n, h=H, w=W, seed0=2000):
    from oracle import synth  # synthetic inputs only (generators live with the test infrastructure)
    return np.stack([synth.gen_underwater(h, w, seed0 + i) for i in range(n)])


# image rows that --dump-outputs writes of every frame: a fixed, seeded sample (64 frames x 16 rows of LAB = 27 MB float32)
DUMP_ROWS = np.sort(np.random.default_rng(0).permutation(H)[:16])


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference_step(frames, pool):
    import cv2
    from oracle import ref_balance, color_balance_np

    def one(img):
        # the reference's own translation unit as fast as this host runs it: -O3 -mavx2 build when the CPU has AVX2, its
        # cv::cvtColor calls served by real OpenCV (oracle/ref_balance.py::fastest); identical bytes to the parity oracle
        bal = ref_balance.balance_timed(img) if ref_balance.available() else color_balance_np.process_frame_np(img)
        return cv2.cvtColor(bal, cv2.COLOR_BGR2LAB)
    return list(pool.map(one, frames))


def reference_build_note():
    from oracle import ref_balance
    if not ref_balance.available():
        return "numpy restatement of color_balance.cpp (oracle/color_balance_np.py)"
    import numpy as np_
    from oracle import synth
    probe = synth.gen_underwater(120, 160, 1)
    assert np_.array_equal(ref_balance.balance_timed(probe), ref_balance.balance(probe)), "timed reference build differs from the oracle"
    return "color_balance.cpp compiled unmodified (" + ref_balance.fastest()[1] + "); cv::split / merge / mean of oracle/cvshim"


def cpu_baseline(frames, cores):
    import cv2
    from concurrent.futures import ThreadPoolExecutor
    from oracle import ref_balance
    cv2.setNumThreads(1)
    with ThreadPoolExecutor(max_workers=cores) as pool:
        cpu_reference_step(frames[:min(len(frames), cores)], pool)     # warm-up
        t0 = time.perf_counter()
        cpu_reference_step(frames, pool)
        dt = time.perf_counter() - t0
    cv2.setNumThreads(0)
    return {"value": len(frames) / dt, "unit": "frames/s", "cores": cores,
            "kind": "reference" if ref_balance.available() else "port",
            "sample": "%d frames 2208x1242: compiled reference process_frame (default flags, marshalled as "
                      "modules/color_balance.py:93-110) + cv2.cvtColor(BGR2LAB), one frame per thread, %.2f s wall; %s"
                      % (len(frames), dt, reference_build_note())}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import cv2
    from concurrent.futures import ThreadPoolExecutor
    from oracle import ref_balance
    cores = os.cpu_count() or 1
    per_step = max(2, cores)            # one frame per host thread: every core works in every step
    ring = make_ring(per_step * 2)
    cv2.setNumThreads(1)
    times = []
    with ThreadPoolExecutor(max_workers=cores) as pool:
        for s in range(args.warmup + args.steps):
            frames = ring[(s % 2) * per_step:(s % 2 + 1) * per_step]
            t0 = time.perf_counter()
            converted = cpu_reference_step(frames, pool)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"converted": np.stack(converted[:BATCH])[:, DUMP_ROWS]})
    total = sum(times)
    value = per_step * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "C2: ZED 2208x1242 stereo frames, balance() default flags -> BGR2LAB image "
                               "(BASELINE.json configs[1])",
                   "reference_sample": "each step = %d frames on the host cores (compiled reference process_frame + "
                                       "cv2.cvtColor), one frame per thread" % per_step,
                   "reference_build": reference_build_note(),
                   "frames_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores,
                         "kind": "reference" if ref_balance.available() else "port",
                         "sample": "%d steps x %d frames, one frame per thread over %d threads" % (args.steps, per_step, cores)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_side_baselines(cores, budget_s=4.0):
    """The reference's CPU OpenCV path for the other BASELINE configs, on this box's host cores (cv2's own
    thread pool, `cores` threads), each a bounded sample (about `budget_s` seconds).  oracle/cv_ops.py holds the
    literal calls of the reference's call sites; used here only as the timed baseline."""
    import cv2
    from oracle import cv_ops, synth, letterbox, ref_balance, color_balance_np
    cv2.setNumThreads(cores)
    res = {}

    def timed(name, fn, frames, unit="frames/s", note="", per_thread=False):
        """per_thread: one frame per host thread with cv2 single-threaded (for the chains that contain process_frame,
        which uses two threads at most); otherwise one frame at a time with cv2's own pool over all cores."""
        from concurrent.futures import ThreadPoolExecutor
        fn(frames[0])
        n, t0 = 0, time.perf_counter()
        if per_thread:
            cv2.setNumThreads(1)
            with ThreadPoolExecutor(max_workers=cores) as pool:
                while True:
                    list(pool.map(fn, [frames[(n + i) % len(frames)] for i in range(cores)]))
                    n += cores
                    dt = time.perf_counter() - t0
                    if dt > budget_s:
                        break
            cv2.setNumThreads(cores)
        else:
            while True:
                fn(frames[n % len(frames)])
                n += 1
                dt = time.perf_counter() - t0
                if dt > budget_s or n >= 400:
                    break
        res[name] = {"value": n / dt, "unit": unit, "cores": cores, "kind": "reference",
                     "sample": "%d frames in %.2f s, %s%s" % (n, dt, ("one frame per thread over %d threads" % cores) if per_thread
                                                              else ("cv2.setNumThreads(%d)" % cores), note)}

    # C1: modules/red_buoy.py:21-44 at 640x480 -- CPU OpenCV is the subject of this config
    def c1(img):
        threshed, cleaned = cv_ops.buoy_mask(img, 150, 255)
        cs = cv_ops.outer_contours(threshed)                  # red_buoy.py:38 uses `threshed`
        return [(cv_ops.contour_centroid(c), cv_ops.contour_area(c)) for c in cs]
    timed("c1_red_buoy_640x480", c1, [synth.gen_underwater(480, 640, 3400 + i) for i in range(8)])

    # C3: modules/bins.py:13-27 at 1920x1080 (+ the declared labelling oracle's cv2 call)
    def c3(img):
        _, cleaned = cv_ops.bins_mask(img)
        return cv2.connectedComponentsWithStats(cleaned, connectivity=8, ltype=cv2.CV_32S)
    timed("c3_hsv_inrange_open_label_1920x1080", c3, [synth.gen_underwater(1080, 1920, 3100 + i) for i in range(4)])

    # C3 as the reference literally does it: findContours + polygon moments (utils/feature.py:5-21,240-265)
    def c3c(img):
        _, cleaned = cv_ops.bins_mask(img)
        return [(cv_ops.contour_centroid(c), cv2.minAreaRect(c)) for c in cv_ops.outer_contours(cleaned)]
    timed("c3_hsv_inrange_open_contours_1920x1080", c3c, [synth.gen_underwater(1080, 1920, 3100 + i) for i in range(4)])

    # C4: letterbox + normalise, per image as Ultralytics does it (modules/yolo.py:112-114 "we don't batch")
    imgs = [synth.gen_underwater(H, W, 3300 + i) for i in range(4)]
    timed("c4_letterbox_16x2208x1242_to_640_fp16", lambda im: letterbox.yolo_input([im], 640, 640, half=True), imgs,
          unit="images/s", note=", oracle/letterbox.py (Ultralytics restated; parity unpinned)")

    # C5: balance() + bins chain + labelling at 3840x2160, one frame per call (reference process_frame is
    # internally 2-threaded at most, color_balance.cpp:398-418)
    bal = ref_balance.balance_timed if ref_balance.available() else color_balance_np.process_frame_np

    def c5(img):
        _, cleaned = cv_ops.bins_mask(bal(img))
        return cv2.connectedComponentsWithStats(cleaned, connectivity=8, ltype=cv2.CV_32S)
    timed("c5_balance_threshold_label_3840x2160", c5, [synth.gen_c5_frame(3200 + i) for i in range(2)],
          note=", compiled reference process_frame (fastest build, real cv2 conversions) + cv2", per_thread=True)

    # north-star fused stage at 2208x1242 on the CPU: balance -> HSV -> inRange -> OPEN
    def fused(img):
        return cv_ops.bins_mask(bal(img), (0, 40, 60), (179, 255, 255))[1]
    timed("fused_balance_hsv_inrange_open_2208x1242", fused, imgs, per_thread=True)
    cv2.setNumThreads(0)
    return res


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def time_device(ctx, fn, steps, warmup):
    """fn(step) enqueues one step on ctx's stream.  CUDA events on that stream."""
    import torch
    for s in range(warmup):
        fn(s)
    ctx.sync()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ctx.torch_stream):
        e0.record()
    for s in range(steps):
        fn(warmup + s)
    with torch.cuda.stream(ctx.torch_stream):
        e1.record()
    ctx.sync()
    return e0.elapsed_time(e1) / 1e3


def side_workloads(ctx, peak_gbs):
    """Short device-resident measurements of the other BASELINE configs (not the headline)."""
    import torch
    from oracle import synth
    res = {}

    def fps(name, fn, frames, bpp_px, steps=10, warmup=3):
        dt = time_device(ctx, fn, steps, warmup)
        v = frames * steps / dt
        res[name] = {"frames_per_s": v, "ms_per_step": 1e3 * dt / steps,
                     "algorithmic_gbs": bpp_px * v / 1e9, "frac_of_hbm": bpp_px * v / 1e9 / peak_gbs}
    # north-star stage at 2208x1242: balance -> HSV -> inRange -> OPEN 5x5, mask out (4 B/px)
    base = [synth.gen_underwater(H, W, 3000 + i) for i in range(16)]
    ring = ctx.upload(np.stack(base + [np.roll(b, 131, axis=1) for b in base]))     # 32 frames per call, 263 MB > L2
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(0, 40, 60), hi=(179, 255, 255), morph=[("open", 5, 5, 1)])
    out = {}
    fps("fused_balance_hsv_inrange_open_2208x1242", lambda s: out.update(ctx.stage(desc, ring, want=("mask",), out=out)),
        32, 4 * H * W)
    res["fused_balance_hsv_inrange_open_2208x1242"]["frames_per_call"] = 32
    ring = ring[:16]
    # C3: 1920x1080 HSV inRange -> OPEN -> CCL + moments (8 B/px)
    ring3 = ctx.upload(np.stack([synth.gen_underwater(1080, 1920, 3100 + i) for i in range(16)]))
    d3 = ctx.make_stage(cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)], label=True)
    o3 = {}
    fps("c3_hsv_inrange_open_label_1920x1080",
        lambda s: o3.update(ctx.stage(d3, ring3, want=("mask", "labels", "blobs"), max_blobs=4096, out=o3)), 16, 8 * 1080 * 1920)
    # C1: 640x480 red_buoy chain (modules/red_buoy.py:21-44): LAB a-channel inRange -> OPEN -> CLOSE, mask out (4 B/px);
    # the config's subject is the CPU path, its number sits beside this one as cpu_baseline
    ring1 = ctx.upload(np.stack([synth.gen_underwater(480, 640, 3400 + i) for i in range(64)]))
    d1 = ctx.make_stage(cvt="bgr2lab", lo=(0, 150, 0), hi=(255, 255, 255), morph=[("open", 5, 5, 1), ("close", 5, 5, 1)])
    o1 = {}
    fps("c1_red_buoy_640x480", lambda s: o1.update(ctx.stage(d1, ring1, want=("mask",), out=o1)), 64, 4 * 480 * 640)
    # C4: 16 frames -> letterbox 640x640 fp16
    imgs = [ctx.upload(synth.gen_underwater(H, W, 3300 + i)) for i in range(16)]
    bytes_batch = 16 * H * W * 3 + 16 * 3 * 640 * 640 * 2
    dt = time_device(ctx, lambda s: ctx.letterbox(imgs), 10, 3)
    res["c4_letterbox_16x2208x1242_to_640_fp16"] = {"images_per_s": 160 / dt, "ms_per_step": 1e2 * dt,
                                                   "algorithmic_gbs": bytes_batch * 10 / dt / 1e9,
                                                   "frac_of_hbm": bytes_batch * 10 / dt / 1e9 / peak_gbs}
    # pure streaming kernels (what the HBM roofline looks like on this path when the arithmetic is light)
    rgba = ctx.upload(np.random.default_rng(0).integers(0, 256, (16, H, W, 4), dtype=np.uint8))
    gray_out = {}
    dt = time_device(ctx, lambda s: ctx.rgba_to_rgb(rgba), 10, 3)
    res["stream_rgba_to_rgb_16x2208x1242"] = {"frames_per_s": 160 / dt, "ms_per_step": 1e2 * dt,
                                              "algorithmic_gbs": 7 * H * W * 160 / dt / 1e9,
                                              "frac_of_hbm": 7 * H * W * 160 / dt / 1e9 / peak_gbs}
    dt = time_device(ctx, lambda s: ctx.cvt_color(ring, "bgr2gray"), 10, 3)
    res["stream_bgr2gray_16x2208x1242"] = {"frames_per_s": 160 / dt, "ms_per_step": 1e2 * dt,
                                           "algorithmic_gbs": 4 * H * W * 160 / dt / 1e9,
                                           "frac_of_hbm": 4 * H * W * 160 / dt / 1e9 / peak_gbs}
    del ring, ring1, ring3, imgs, rgba
    torch.cuda.empty_cache()
    return res


C5_STREAMS = 8
C5_H, C5_W = 2160, 3840
C5_FRAMES_PER_STREAM = 8      # consecutive frames of every stream per step (a GPU that owns one stream still gets 8 frames = two L2 chunks per call)


def c5_leg(ctx, world, rank, peak_gbs, steps=10, warmup=3):
    """BASELINE.json configs[4]: 8 camera streams of 3840x2160 through balance -> BGR2HSV -> inRange -> OPEN 5x5 ->
    labels + moments (modules/bins.py:13-27 behind preprocessor.py:87-88), stream s on GPU s mod N, no collective.
    The 8 streams are fixed, so this leg scales STRONGLY with N.  One step = C5_FRAMES_PER_STREAM consecutive new frames
    from every stream (64 frames in all), so that a GPU owning a single stream at N = 8 is still handed 8 frames per call."""
    import torch
    import torch.distributed as dist
    from oracle import synth
    from cuauv_vision_pipeline_b200.sharding import streams_for_rank   # stream s -> rank s mod N (tested with gloo, world 2)
    mine = streams_for_rank(C5_STREAMS, rank, world)
    base = [synth.gen_c5_frame(3200 + i, C5_H, C5_W, big_target=(i == 0)) for i in range(2)]
    # two alternating step batches; frame j of stream s is a cyclic shift of a base frame (same statistics, every pixel
    # somewhere else), laid out stream-major: [stream][frame of the step]
    rings = [ctx.upload(np.stack([np.roll(base[(i + j) % 2], 97 * (s + 1) + 13 * (2 * i + j) + 7 * j, axis=1)
                                  for s in mine for j in range(C5_FRAMES_PER_STREAM)])) for i in range(2)] if mine else []
    desc = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)], label=True)
    out = {}

    def step(s):
        if mine:
            out.update(ctx.stage(desc, rings[s % 2], want=("mask", "labels", "blobs"), max_blobs=8192, out=out))
    for s in range(warmup):
        step(s)
    ctx.sync()
    if world > 1:
        dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ctx.torch_stream):
        e0.record()
    for s in range(steps):
        step(warmup + s)
    with torch.cuda.stream(ctx.torch_stream):
        e1.record()
    ctx.sync()
    dt = e0.elapsed_time(e1) / 1e3
    if world > 1:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    fps = C5_STREAMS * C5_FRAMES_PER_STREAM * steps / dt
    gbs = 8 * C5_H * C5_W * fps / 1e9
    n_blobs = int(ctx.download(out["n_blobs"])[0]) if mine else None
    del rings
    out.clear()
    torch.cuda.empty_cache()
    return {"frames_per_s": fps, "ms_per_step": 1e3 * dt / steps, "streams": C5_STREAMS, "steps": steps,
            "frames_per_stream_per_step": C5_FRAMES_PER_STREAM,
            "streams_per_gpu": [len(streams_for_rank(C5_STREAMS, r, world)) for r in range(world)],
            "scaling": "strong", "shape": "%dx%d" % (C5_W, C5_H), "algorithmic_gbs": gbs,
            "frac_of_hbm": gbs / (peak_gbs * min(world, C5_STREAMS)), "blobs_in_first_frame": n_blobs,
            "workload": "C5: 8 streams 3840x2160, balance -> BGR2HSV -> inRange([10,20,60],[30,100,255]) -> OPEN 5x5 -> "
                        "labels + moments, mask + labels + blob table out (8 B/px), stream s -> GPU s mod N"}


def load_static_profile():
    """Per-kernel numbers that only ncu can give (steady-state DRAM bytes, executed instructions), from the
    committed capture of the same workload; bench.py measures the kernel TIME live."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f), name
        except Exception:  # noqa: BLE001
            continue
    return None, None


def run_ours(args):
    import torch
    import torch.distributed as dist
    import cuauv_vision_pipeline_b200 as bv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = []
    if world > 1:
        torch.cuda.set_device(local)
        # one process per GPU: stay on the CPUs next to that GPU so the pinned buffers of the end-to-end leg
        # are allocated on its NUMA node (at N=1 the process keeps every core for the CPU baseline leg)
        from cuauv_vision_pipeline_b200.sharding import bind_to_gpu_numa
        numa_cpus = bind_to_gpu_numa(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = bv.Context(local)
    peak_gbs, peak_src = read_peaks()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # synthetic ring, distinct per rank (frame f of the global stream goes to rank f mod world)
    ring_np = make_ring(RING // 2, seed0=2000 + 100 * rank)
    ring = torch.cat([ctx.upload(ring_np), ctx.upload(np.roll(ring_np, 211, axis=2))])
    dump_rows = torch.from_numpy(DUMP_ROWS).to(ring.device) if (args.dump_outputs and rank == 0) else None
    n_batches = RING // BATCH
    desc = ctx.make_stage(balance={}, cvt="bgr2lab")
    out = {}

    def step(s):
        b = s % n_batches
        out.update(ctx.stage(desc, ring[b * BATCH:(b + 1) * BATCH], want=("converted",), out=out))

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed_steps(n, first):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ctx.torch_stream):
            e0.record()
        for s in range(n):
            step(first + s)
        with torch.cuda.stream(ctx.torch_stream):
            e1.record()
        barrier()
        return allmax(e0.elapsed_time(e1) / 1e3)

    # ---- device-resident throughput ----
    for s in range(args.warmup):
        step(s)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        for s in range(args.warmup):   # keep the GPU busy while the sampler came up
            step(s)
        ctx.sync()
    barrier()
    mark_a = sampler.mark()
    launches0 = ctx.launches
    elapsed = timed_steps(args.steps, args.warmup)
    launches = ctx.launches - launches0
    if dump_rows is not None:
        # the LAB images the last timed step returned: a device copy of the sampled rows, taken before the sustained
        # repetition below overwrites `out` and written to disk once the clock-sampled window is over
        with torch.cuda.stream(ctx.torch_stream):
            dumped = out["converted"].index_select(1, dump_rows)
    value = world * BATCH * args.steps / elapsed
    # the same step repeated for >= ~1.5 s: what a continuously running consumer sees (clocks, power cap)
    sus_steps = int(min(20000, max(args.steps, args.sustain_s / (elapsed / args.steps))))
    sus_elapsed = timed_steps(sus_steps, args.warmup + args.steps)
    sustained = {"value": world * BATCH * sus_steps / sus_elapsed, "unit": "frames/s", "steps": sus_steps,
                 "seconds": sus_elapsed}
    mark_b = sampler.mark()
    if dump_rows is not None:
        write_outputs(args.dump_outputs, {"converted": ctx.download(dumped)})
        del dumped

    # ---- per-kernel timing (library profiler: CUDA events around every launch) ----
    ctx.profile(True)
    for s in range(4):
        step(s)
    prof = ctx.profile_dump()
    ctx.profile(False)
    total_ms = sum(v["ms"] for v in prof.values()) or 1.0
    dom = max(prof, key=lambda k: prof[k]["ms"])
    # one launch of any pass covers one chunk of frames (the library sizes it: L2, call length): 4 profiled steps of BATCH
    # frames went through `launches` launches of the dominant kernel
    chunk_frames = max(1, (4 * BATCH) // max(1, prof[dom]["launches"]))
    dom_ms = prof[dom]["ms"] / prof[dom]["launches"]
    achieved = BPP_C2 * H * W * chunk_frames / (dom_ms / 1e3) / 1e9
    static, static_name = load_static_profile()
    traffic, traffic_src, issue = None, None, None
    sm_clock_hz = 1.965e9
    if static:
        k = static.get("kernels", {}).get(dom)
        if k:
            if k.get("dram_bytes_per_launch") is not None:
                traffic = k["dram_bytes_per_launch"] / k["frames_per_launch"] * chunk_frames
                traffic_src = "profiles/%s: %s" % (static_name, static.get("source", ""))
            if k.get("warp_instructions_per_launch"):
                ipp = k["warp_instructions_per_launch"] * 32.0 / (k["frames_per_launch"] * H * W)
                bound_us = ipp * H * W * chunk_frames / (148 * 4 * 32 * sm_clock_hz) * 1e6
                issue = {"thread_instr_per_px": ipp, "issue_bound_us_per_launch": bound_us,
                         "measured_us_per_launch": dom_ms * 1e3, "frac_of_issue_bound": bound_us / (dom_ms * 1e3),
                         "note": "instr/px x px / (148 SM x 4 schedulers x 32 lanes x 1.965 GHz); instr from ncu "
                                 "smsp__inst_executed.sum of profiles/%s" % static_name}
        st = (static.get("steady_state") or {}).get("c2")
    else:
        st = None
    # `traffic`: what the frames of one launch really move through HBM in steady state (ncu range replay over a whole
    # concurrent step, all three passes: they cannot be attributed to one kernel when chunks overlap); the
    # kernel-replay figure of the dominant kernel alone (caches kept warm by the serialised passes before it, so it
    # UNDER-counts) is kept beside it
    steady_traffic = st["dram_bytes_per_frame"] * chunk_frames if st else None
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": steady_traffic if steady_traffic is not None else traffic,
                "traffic_kind": ("steady-state DRAM bytes of the whole step (passes 1-3, ncu --replay-mode range, kernels "
                                 "concurrent) per frame x frames per launch" if steady_traffic is not None
                                 else "kernel replay of the dominant kernel"),
                "traffic_kernel_replay": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel_ms_per_launch": dom_ms, "kernel_share_of_step": prof[dom]["ms"] / total_ms,
                "algorithmic_bytes_per_launch": BPP_C2 * H * W * chunk_frames, "issue": issue,
                "note": "achieved = 6 B/px (BGR in + LAB out) x frames in one launch / that kernel's CUDA-event time"}
    stage_gbs = BPP_C2 * H * W * value / world / 1e9
    stage_roofline = {"achieved": stage_gbs, "peak": peak_gbs, "unit": "GB/s", "frac": stage_gbs / peak_gbs,
                      "steady_state_dram_bytes_per_frame": st,
                      "per_kernel_ms": {k: round(v["ms"] / 4, 4) for k, v in sorted(prof.items())},
                      "frames_per_launch": chunk_frames}

    # ---- C5: 8 x 4K streams sharded by stream (strong scaling), every rank ----
    c5 = None if args.no_side else c5_leg(ctx, world, rank, peak_gbs)

    # ---- end to end through the host-buffer entry point (pinned memory) ----
    pin_in = bv.PinnedArray((2, E2E_BATCH, H, W, 3))
    pin_in.array[0] = ring_np[:E2E_BATCH]
    pin_in.array[1] = ring_np[E2E_BATCH:2 * E2E_BATCH]
    pin_out = bv.PinnedArray((E2E_BATCH, H, W, 3))
    host_out = {"converted": pin_out.array}
    e2e_steps = max(3, min(args.steps, 30))   # a step moves 263 MB over PCIe (~3 ms): 30 steps amortise the first upload / last download
    for s in range(2):
        ctx.stage_host(desc, pin_in.array[s % 2], want=("converted",), out=host_out)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        ctx.stage_host(desc, pin_in.array[s % 2], want=("converted",), out=host_out)
    barrier()
    e2e_dt = allmax(time.perf_counter() - t0)
    # the same work through the asynchronous pair (bv_stage_host_submit / _wait): two batches in flight, one per staging
    # slot, so that the uploads of batch k+1 run while batch k is still being returned (PCIe is full duplex)
    pin_out2 = bv.PinnedArray((E2E_BATCH, H, W, 3))
    host_outs = [host_out, {"converted": pin_out2.array}]

    def pipelined(steps):
        for s in range(steps):
            ctx.stage_host(desc, pin_in.array[s % 2], want=("converted",), out=host_outs[s % 2], slot=s % 2)
        ctx.stage_host_wait(0)
        ctx.stage_host_wait(1)
    pipelined(2)
    barrier()
    t0 = time.perf_counter()
    pipelined(e2e_steps)
    barrier()
    e2e_pipe_dt = allmax(time.perf_counter() - t0)
    # module-realistic end to end (modules/bins.py: a frame goes in, a blob table comes out): the D2H side is KBs
    desc_bins = ctx.make_stage(balance={}, cvt="bgr2hsv", lo=(10, 20, 60), hi=(30, 100, 255), morph=[("open", 5, 5, 1)], label=True)
    bins_out = {}
    for s in range(2):
        bins_out = ctx.stage_host(desc_bins, pin_in.array[s % 2], want=("blobs",), max_blobs=1024, out=bins_out)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        ctx.stage_host(desc_bins, pin_in.array[s % 2], want=("blobs",), max_blobs=1024, out=bins_out)
    barrier()
    bins_dt = allmax(time.perf_counter() - t0)
    pin_blobs = [bv.PinnedArray((E2E_BATCH, 1024), bv.BLOB_DTYPE) for _ in range(2)]
    pin_nb = [bv.PinnedArray((E2E_BATCH,), np.int32) for _ in range(2)]
    bins_outs = [{"blobs": pin_blobs[i].array, "n_blobs": pin_nb[i].array} for i in range(2)]

    def bins_pipelined(steps):
        for s in range(steps):
            ctx.stage_host(desc_bins, pin_in.array[s % 2], want=("blobs",), max_blobs=1024, out=bins_outs[s % 2], slot=s % 2)
        ctx.stage_host_wait(0)
        ctx.stage_host_wait(1)
    bins_pipelined(2)
    barrier()
    t0 = time.perf_counter()
    bins_pipelined(e2e_steps)
    barrier()
    bins_pipe_dt = allmax(time.perf_counter() - t0)
    # single-frame latency of the drop-in call (what a module's process() pays per frame)
    one_out = {"converted": pin_out.array[:1]}
    for s in range(3):
        ctx.stage_host(desc, pin_in.array[0][:1], want=("converted",), out=one_out)
    t0 = time.perf_counter()
    for s in range(20):
        ctx.stage_host(desc, pin_in.array[0][s % E2E_BATCH:s % E2E_BATCH + 1], want=("converted",), out=one_out)
    single_ms = (time.perf_counter() - t0) / 20 * 1e3
    # the box's own host<->device copy ceiling, measured with the same pinned buffers and EVERY rank copying at the
    # same time (the host memory system is shared by all GPUs of the box; it differs between boxes of the pool)
    d_in = torch.empty(pin_in.array[0].shape, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(pin_out.array.shape, dtype=torch.uint8, device="cuda")
    t_in, t_out = torch.from_numpy(pin_in.array[0]), torch.from_numpy(pin_out.array)
    s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()

    def copies(up, down):
        if up:
            with torch.cuda.stream(s_up):
                d_in.copy_(t_in, non_blocking=True)
        if down:
            with torch.cuda.stream(s_down):
                t_out.copy_(d_out, non_blocking=True)

    def copy_rate(up, down, reps=5):
        copies(up, down)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            copies(up, down)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        return allmax(dt) / reps
    both_dt = copy_rate(True, True)
    up_dt = copy_rate(True, False)
    nbytes_in, nbytes_out = t_in.numel(), t_out.numel()
    pcie = {"both_directions_gbs": world * (nbytes_in + nbytes_out) / both_dt / 1e9,
            "h2d_only_gbs": world * nbytes_in / up_dt / 1e9,
            "ceiling_frames_per_s": world * E2E_BATCH / both_dt,
            "h2d_only_ceiling_frames_per_s": world * E2E_BATCH / up_dt,
            "ranks_copying_concurrently": world}
    del d_in, d_out
    clocks = sampler.stop(mark_a, mark_b) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "device-resident timed region + the sustained repetition (%.1f s)" % sus_elapsed
    e2e = {"value": world * E2E_BATCH * e2e_steps / e2e_pipe_dt, "unit": "frames/s",
           "h2d_bytes_per_step": E2E_BATCH * H * W * 3, "d2h_bytes_per_step": E2E_BATCH * H * W * 3,
           "api": "bv_stage_host_submit / bv_stage_host_wait (C ABI, pinned host buffers, two %d-frame batches in flight: "
                  "every step uploads its frames and returns their LAB images inside the timed region)" % E2E_BATCH,
           "steps": e2e_steps,
           "blocking_call": {"value": world * E2E_BATCH * e2e_steps / e2e_dt, "unit": "frames/s",
                             "api": "bv_stage_host (one blocking call per %d-frame batch)" % E2E_BATCH},
           "single_frame_latency_ms": single_ms,
           "pcie_note": "8.23 MB in + 8.23 MB out per frame, copied in both directions at once; `pcie` is this box's own "
                        "ceiling for that (plain cudaMemcpyAsync of the same pinned buffers on every rank at once, no kernels)",
           "pcie": pcie,
           "bins_module": {"value": world * E2E_BATCH * e2e_steps / bins_pipe_dt, "unit": "frames/s",
                           "blocking_call": world * E2E_BATCH * e2e_steps / bins_dt,
                           "h2d_bytes_per_step": E2E_BATCH * H * W * 3, "d2h_bytes_per_step": E2E_BATCH * (1024 * 96 + 4),
                           "frac_of_h2d_ceiling": (world * E2E_BATCH * e2e_steps / bins_pipe_dt) / pcie["h2d_only_ceiling_frames_per_s"],
                           "workload": "frames in, blob tables out: balance -> BGR2HSV -> inRange -> OPEN 5x5 -> labels + "
                                       "moments (modules/bins.py:13-27), bv_stage_host_submit / _wait (blocking_call: bv_stage_host)"}}
    pcie["e2e_frac_of_ceiling"] = e2e["value"] / pcie["ceiling_frames_per_s"]

    if rank == 0:
        cores = os.cpu_count() or 1
        cpu = cpu_baseline(list(ring_np[:min(32, max(8, cores))]), cores) if (world == 1 and not args.no_cpu) else None
        others = side_workloads(ctx, peak_gbs) if (world == 1 and not args.no_side) else None
        if others is not None and not args.no_cpu:
            for k, v in cpu_side_baselines(cores).items():
                if k.startswith("c5_") and c5 is not None:
                    c5["cpu_baseline"] = v
                else:
                    others.setdefault(k, {})["cpu_baseline"] = v
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "C2: ZED 2208x1242 stereo frames, balance() default flags -> BGR2LAB image "
                                   "(BASELINE.json configs[1])",
                       "frames_per_step_per_gpu": BATCH, "ring_frames": RING,
                       "l2": ("inputs larger than L2 (%d MB per step from a 1.05 GB ring; consecutive steps use "
                              "different batches)") % (BATCH * H * W * 3 // 1000000),
                       "parallelism": "frames sharded by index over %d GPU(s), no collective" % world,
                       "host_affinity": ("%d CPUs local to each GPU" % len(numa_cpus)) if numa_cpus else "default"},
            "sustained": sustained,
            "roofline": roofline, "stage_roofline": stage_roofline, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": launches, "clocks": clocks, "c5": c5, "other_workloads": others,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-side", action="store_true", help="skip the short measurements of the other configs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (tuning sweeps only)")
    ap.add_argument("--sustain-s", dest="sustain_s", type=float, default=1.5,
                    help="seconds of back-to-back steps for the `sustained` value")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/<name>.npy (float32, a fixed sample of 16 image "
                         "rows of every frame, at most 27 MB; rank 0 only).  --impl reference: the first 64 frames of "
                         "its last step, which holds one frame per host core, so its frames follow the host")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
