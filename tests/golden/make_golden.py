"""Generates tests/golden/*.npz and kat.json by EXECUTING THE REFERENCE (oracle/_ref/libfsr1_ref.so =
the reference's own ffx_fsr1.h source compiled for the host, see oracle/build_ref.sh).  Needs
FSR1_REFERENCE_DIR; the outputs are committed so the tests run where the reference is absent.

    python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle_lib as ol  # noqa: E402
import fsr1_b200 as F  # noqa: E402

R = ol.ref()
assert R is not None, "reference build missing: set FSR1_REFERENCE_DIR to a checkout of the reference and run oracle/build_ref.sh"

IW, IH = 32, 18
SIZES = {"x2.0": (64, 36), "x1.5": (48, 27), "x1.3": (41, 23), "x1.0": (32, 18), "x2.0x1.5": (64, 27)}
fix = {}
for kind, gen in (("uniform", F.uniform), ("structured", F.structured)):
    src = gen(IW, IH, 777)
    src_h = F.to_half(src)
    fix[kind + "_in_f32"] = src
    fix[kind + "_in_f16"] = src_h.view(np.uint16)
    for tag, (ow, oh) in SIZES.items():
        econ = ol.easu_con(IW, IH, ow, oh, lib=R)
        e = ol.easu(src, ow, oh, econ, lib=R)
        fix["%s_%s_easu_f32" % (kind, tag)] = e
        eh = ol.easu(src_h, ow, oh, econ, lib=R)
        fix["%s_%s_easu_h16" % (kind, tag)] = eh.view(np.uint16)
        # fp32 algorithm on the half-quantised input: what the fp16 kernels are held to (1e-2)
        eq = ol.easu(src_h.astype(np.float32), ow, oh, econ, lib=R)
        fix["%s_%s_easu_f32_of_f16" % (kind, tag)] = eq
        for sharp in (0.0, 0.25, 2.0):
            rcon = ol.rcas_con(sharp, lib=R)
            for clamp in (0, 1):
                key = "%s_%s_rcas_s%g_c%d" % (kind, tag, sharp, clamp)
                if tag in ("x2.0", "x1.3") or (sharp == 0.25 and clamp == 0):
                    fix[key + "_f32"] = ol.rcas(e, rcon, bool(clamp), lib=R)
                    fix[key + "_h16"] = ol.rcas(eh, rcon, bool(clamp), lib=R).view(np.uint16)
np.savez_compressed(os.path.join(HERE, "fsr1_golden.npz"), **fix)

# Known-answer table: constants from the reference's UNMODIFIED header (#define A_CPU) and spot pixels /
# checksums of the 96x54 LCG frame of SURVEY.md §8(c).
kat = {"easu_con": {}, "rcas_con": {}, "easu_con_offset": {}, "f32_to_f16": {}}
for (iw, ih, ow, oh) in [(960, 540, 1920, 1080), (1920, 1080, 3840, 2160), (2560, 1440, 3840, 2160),
                         (2953, 1661, 3840, 2160), (3840, 2160, 7680, 4320), (96, 54, 192, 108), (1, 1, 4, 4)]:
    kat["easu_con"]["%d,%d,%d,%d" % (iw, ih, ow, oh)] = ["%08x" % v for v in ol.easu_con(iw, ih, ow, oh, lib=R)]
kat["easu_con_offset"]["1280,720,1920,1080,2560,1440,16,8"] = [
    "%08x" % v for v in ol.easu_con(1920, 1080, 2560, 1440, vw=1280, vh=720, lib=R, off=(16.0, 8.0))]
for s in (0.0, 0.2, 0.25, 0.5, 1.0, 2.0, 3.3, 10.0, 20.0):
    kat["rcas_con"][repr(s)] = ["%08x" % v for v in ol.rcas_con(s, lib=R)]
for v in (0.0, 1.0, 0.870550563, 65504.0, 65520.0, 1e-5, 6e-8, 5.9e-8, 2.9e-8, 1e-8, -0.333, 1e9, float("inf"), 0.1):
    kat["f32_to_f16"][repr(v)] = "%04x" % R.fsr1ref_cpu_f32_to_f16(v)
frame = F.uniform(96, 54, 12345)
kat["lcg_96x54"] = {}
for tag, (ow, oh) in {"x2": (192, 108), "x1.5": (144, 81)}.items():
    e = ol.easu(frame, ow, oh, lib=R)
    d = {"easu_sum": float(e[..., :3].astype(np.float64).sum())}
    for (x, y) in [(0, 0), (1, 1), (100, 50), (ow - 1, oh - 1)]:
        d["easu_%d_%d" % (x, y)] = ["%08x" % v for v in e[y, x, :3].view(np.uint32)]
    for clamp in (0, 1):
        r = ol.rcas(e, ol.rcas_con(0.25, lib=R), bool(clamp), lib=R)
        d["rcas_sum_c%d" % clamp] = float(r[..., :3].astype(np.float64).sum())
        d["rcas_100_50_c%d" % clamp] = ["%08x" % v for v in r[50, 100, :3].view(np.uint32)]
        d["rcas_0_0_c%d" % clamp] = ["%08x" % v for v in r[0, 0, :3].view(np.uint32)]
    kat["lcg_96x54"][tag] = d
with open(os.path.join(HERE, "kat.json"), "w") as f:
    json.dump(kat, f, indent=1, sort_keys=True)
print("wrote", len(fix), "arrays;", os.path.getsize(os.path.join(HERE, "fsr1_golden.npz")) // 1024, "KiB")
