#!/usr/bin/env python3
"""Static SASS census of the library's hot kernels for profiles/: per kernel the instruction total and the counts that
prove the claims made in DESIGN.md (UBLKCP = cp.async.bulk TMA copies, SYNCS = mbarrier arrive/wait, ATOMS = shared-memory
atomics, LDS / STS, LDG / STG widths, HMMA / UTC*MMA = tensor cores: must be absent on this path).
    python tools/sass_census.py > profiles/r02_sass_census.md"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "cuauv_vision_pipeline_b200", "lib", "libb200vision.so")
KEYS = ["UBLKCP", "UTMALDG", "SYNCS", "ATOMS", "ATOMG", "RED", "LDS", "STS", "LDG", "STG", "SHFL", "BAR", "IMAD", "FFMA", "LOP3",
        "PRMT", "VIMNMX3", "HMMA", "UTCHMMA", "MUFU", "I2F", "F2I"]
WANT = ["hist_bgr_kernel", "hist_sv_kernel", "final_kernel", "mask_from_hsv_kernel",
        "ivl_build_kernel", "morph_roll_kernel", "morph_chain_kernel", "letterbox_tma_kernel", "resize_kernel", "cvt_kernel",
        "ccl_merge_kernel", "ccl_final_kernel", "contour_kernel", "min_area_rect_kernel", "rgba_to_rgb_kernel"]

out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
fn, counts, wide = None, {}, {}
for line in out.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        fn = m.group(1)
        counts[fn], wide[fn] = collections.Counter(), collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
    if m and fn:
        ins = m.group(1).split()
        op = ins[1] if ins[0].startswith("@") else ins[0]
        counts[fn][op.split(".")[0]] += 1
        counts[fn]["_total"] += 1
        if op.startswith(("LDG", "STG")) and ".128" in op:
            wide[fn][op.split(".")[0] + ".128"] += 1
names = subprocess.run(["cu++filt"] + list(counts), capture_output=True, text=True).stdout.splitlines()
print("# r02 -- static SASS census of libb200vision.so (cuobjdump -sass, sm_100a)\n")
print("Per kernel instantiation: total instructions, then the opcodes that matter for the design claims. `UBLKCP` is the SASS of "
      "`cp.async.bulk` (TMA bulk copy), `SYNCS` of mbarrier operations, `ATOMS` of shared-memory atomics; no `HMMA` / `UTC*MMA` "
      "(tensor cores) and no `UTMALDG` (tensor-map TMA) anywhere on this path.\n")
print("| kernel | total | " + " | ".join(KEYS) + " | LDG.128 | STG.128 |")
print("|---|---:|" + "---:|" * (len(KEYS) + 2))
for fn, dem in sorted(zip(counts, names), key=lambda t: t[1]):
    short = re.sub(r"^(void )?bv::", "", dem)
    base = short.split("<")[0].split("(")[0]
    if base not in WANT:
        continue
    c = counts[fn]
    cut = short.find(">(")
    tmpl = short[:cut + 1] if cut >= 0 else (short[:short.index("(")] if "(" in short else short)
    print("| `%s` | %d | %s | %d | %d |" % (tmpl[:70], c["_total"], " | ".join(str(c[k]) for k in KEYS), wide[fn]["LDG.128"], wide[fn]["STG.128"]))
tot = collections.Counter()
for c in counts.values():
    tot.update(c)
print("\nWhole library: %d functions, %d instructions; UBLKCP %d, UTMALDG %d, SYNCS %d, ATOMS %d, HMMA %d, UTCHMMA %d."
      % (len(counts), tot["_total"], tot["UBLKCP"], tot["UTMALDG"], tot["SYNCS"], tot["ATOMS"], tot["HMMA"], tot["UTCHMMA"]))
