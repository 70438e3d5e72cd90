#!/usr/bin/env python3
"""Generates tests/golden/*.npz from the REFERENCE ITSELF, run in the build container:

  * balance_*.npz   input frame + output of the reference's process_frame, i.e. the unmodified
                    /root/reference/utils/color_correction/color_balance.cpp compiled by
                    oracle/Makefile and called exactly like modules/color_balance.py:93-110;
  * cv_*.npz        input + outputs of the literal cv2 calls the reference makes (oracle/cv_ops.py)
                    with the installed cv2 (third-party dependency of the reference);
  * process_frame_outputs.npz
                    process_frame on the frames of the compiled-reference tests in tests/test_oracle_ref.py
                    (larger frames, HSI branch), too large to store whole: per frame the SHA-256 of input and
                    output, four full output rows and the source of the output.  `python tests/golden/make_golden.py
                    process_frame_outputs` takes them from the compiled reference; with --from-restatement (no
                    reference checkout at hand) from oracle/color_balance_np.py, which those tests compare with the
                    compiled reference byte for byte.  The stored file says which; test_compiled_reference_reproduces_golden
                    re-checks it against the compiled reference wherever that is built.

The reference repository has no tests or fixtures of its own (build.ninja:72-73), so these
vectors are what pins the oracle; they travel to the GPU box, /root/reference does not.
Run from the repo root:  python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np
import cv2

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_balance, cv_ops, synth, ccl, letterbox  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def load_reference_color():
    """Imports the reference's utils/color.py itself (stubbing the two external CUAUV modules it
    pulls in at import time) so that golden vectors come from the reference function, not from a
    restatement."""
    import importlib.util
    import types
    sys.modules.setdefault("auv_python_helpers", types.SimpleNamespace(load_library=lambda n: None))
    for name in ("vision", "vision.utils"):
        sys.modules.setdefault(name, types.ModuleType(name))
    helpers = types.ModuleType("vision.utils.helpers")
    helpers.as_mat = lambda m: m
    sys.modules["vision.utils.helpers"] = helpers
    spec = importlib.util.spec_from_file_location("ref_utils_color", "/root/reference/utils/color.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def write_process_frame_outputs(from_restatement):
    sys.path.insert(0, os.path.dirname(OUT))
    from oracle import color_balance_np
    from test_oracle_ref import STORED_OUTPUTS, sha256, stored_cases, synth_frame
    if from_restatement:
        balance = color_balance_np.process_frame_np
        source = ("oracle/color_balance_np.py (equal byte for byte to the compiled color_balance.cpp on this input in "
                  "test_restatement_matches_compiled_reference / test_hsi_branch_restatement_matches_compiled_reference)")
    else:
        assert ref_balance.available(), "build oracle/_ref first (make -C oracle), or pass --from-restatement"
        balance, source = ref_balance.balance, "compiled color_balance.cpp (oracle/_ref)"
    d = {}
    for key, (kind, shape, seed, flags) in stored_cases().items():
        img = synth_frame(kind, shape, seed)
        out = balance(img, **flags)
        rows = np.linspace(0, shape[0] - 1, 4).round().astype(np.int64)
        d.update({key + "__src_sha256": np.array(sha256(img)), key + "__out_sha256": np.array(sha256(out)),
                  key + "__row_index": rows, key + "__rows": out[rows], key + "__source": np.array(source)})
    np.savez_compressed(STORED_OUTPUTS, **d)
    print("wrote", STORED_OUTPUTS, "from", source)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "process_frame_outputs":
        write_process_frame_outputs("--from-restatement" in sys.argv)
        return
    assert ref_balance.available(), "build oracle/_ref first (make -C oracle)"
    # colour balance: default flags on three shapes (one with width % 32 != 0), plus flag variants
    cases = [("default_96x160", 96, 160, 11, {}),
             ("default_120x161", 120, 161, 12, {}),
             ("default_64x64_notargets", 64, 64, 13, {}),
             ("nohsv_96x160", 96, 160, 14, dict(hsv_contrast_correct=False)),
             ("noclip_96x160", 96, 160, 15, dict(rgb_extrema_clipping=False)),
             ("rgbcc_96x160", 96, 160, 16, dict(rgb_contrast_correct=True)),
             ("adaptive_96x160", 96, 160, 17, dict(adaptive_cast_correction=True)),
             ("noeq_96x160", 96, 160, 18, dict(equalize_rgb=False)),
             ("tiles4x2_96x160", 96, 160, 19, dict(horizontal_blocks=4, vertical_blocks=2)),
             ("tiles2x3_adaptive_96x160", 96, 160, 20, dict(horizontal_blocks=2, vertical_blocks=3, adaptive_cast_correction=True))]
    for name, h, w, seed, flags in cases:
        img = synth.gen_underwater(h, w, seed, targets=(name != "default_64x64_notargets"))
        if name.startswith("tiles"):   # make one quadrant differ enough for the fall-back rule (line 474) to matter
            img[:h // 2, :w // 2] = np.clip(img[:h // 2, :w // 2].astype(int) + np.array([25, 5, 0]), 0, 255).astype(np.uint8)
        out = ref_balance.balance(img, **flags)
        np.savez_compressed(os.path.join(OUT, "balance_%s.npz" % name), src=img, out=out,
                            flags=np.array(sorted(flags.items()), dtype=object) if flags else np.array([], dtype=object))
    # cv2 call sites on one small frame
    img = synth.gen_underwater(72, 128, 21)
    d = dict(src=img)
    for code in ("bgr2lab", "bgr2hsv", "bgr2hls", "bgr2ycrcb", "bgr2gray"):
        d[code] = cv_ops.convert(img, code)[0]
    d["hsv2bgr"] = cv2.cvtColor(d["bgr2hsv"], cv2.COLOR_HSV2BGR)
    mask, cleaned = cv_ops.bins_mask(img)
    d["bins_mask"], d["bins_cleaned"] = mask, cleaned
    th, cl = cv_ops.buoy_mask(img, 140, 255)
    d["buoy_threshed"], d["buoy_cleaned"] = th, cl
    d["resize_50x37"] = cv_ops.resize(img, 50, 37)
    d["ellipse_erode_2"] = cv_ops.ellipse_erode(img, 2)
    d["ellipse_dilate_3"] = cv_ops.ellipse_dilate(img, 3)
    d["contrast_1p7"] = cv_ops.contrast(img, 1.7)
    d["brightness_m40"] = cv_ops.brightness(img, -40)
    d["bias_r25"] = cv_ops.channel_bias(img, 2, 25)
    np.savez_compressed(os.path.join(OUT, "cv_calls_72x128.npz"), **d)
    # thresh_color_distance: outputs of the reference function itself (utils/color.py:66-103)
    ref_color = load_reference_color()
    lab = cv2.cvtColor(img, cv2.COLOR_BGR2LAB)
    split = cv2.split(lab)
    cases = [dict(color=(120, 150, 140), distance=30), dict(color=(60, 128, 128), distance=45, weights=(0.2, 1, 1)),
             dict(color=(200, 110, 170), distance=25.5, ignore_channels=[0]),
             dict(color=(10, 240, 20), distance=400, weights=(3, 1, 2))]
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for k, kw in enumerate(cases):
            m, dimg = ref_color.thresh_color_distance(list(split), **kw)
            d["tcd%d_mask" % k], d["tcd%d_dist" % k] = m, dimg
    np.savez_compressed(os.path.join(OUT, "cv_calls_72x128.npz"), **d)
    # labelling oracle on a small blob mask
    m = synth.mask_blobs(90, 160, 5, sigma=4.0)
    n, lab, tab = ccl.label_and_moments(m)
    np.savez_compressed(os.path.join(OUT, "ccl_90x160.npz"), mask=m, n=np.int32(n), labels=lab,
                        **{k: v for k, v in tab.items()})
    # letterbox restatement (parity unpinned, see oracle/letterbox.py)
    im = synth.gen_underwater(90, 160, 31)
    np.savez_compressed(os.path.join(OUT, "letterbox_90x160_to_64.npz"), src=im,
                        u8=letterbox.letterbox_u8(im, 64, 64), f16=letterbox.yolo_input([im], 64, 64))
    print("wrote", sorted(f for f in os.listdir(OUT) if f.endswith(".npz")))


if __name__ == "__main__":
    main()
