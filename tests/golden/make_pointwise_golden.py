"""Generates tests/golden/fsr1_pointwise_golden.npz by EXECUTING THE REFERENCE's own FsrSrtmF / FsrSrtmInvF / FsrLfgaF /
FsrTepdDitF / FsrTepdC8F / FsrTepdC10F (oracle/_ref/libfsr1_ref.so, see oracle/build_ref.sh).  Needs
FSR1_REFERENCE_DIR; the output is committed so the tests run where the reference is absent.

    python tests/golden/make_pointwise_golden.py
"""
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

W, H = 300, 11                                  # wider than one 256-thread CTA row, no multiple of any tile size
fix = {}
sdr = F.structured(W, H, 4242)
sdr[0, 0, :3] = (0.0, 1.0, 0.5)
hdr = sdr.copy()
hdr[..., :3] = hdr[..., :3] ** 3 * 60.0
hdr[::7, ::5, :3] = 0.0
hdr[3::11, 2::3, :3] = 1.0
grain = (F.uniform(12, 5, 99) - 0.5).astype(np.float32)      # 12 x 5 tile: exercises the wrap in both directions
noise = F.uniform(9, 7, 98)
noise[0, 0, 3], noise[0, 1, 3] = -0.5, 1.5
fix["sdr"], fix["hdr"], fix["grain"], fix["noise"] = sdr, hdr, grain, noise
fix["srtm"] = ol.srtm(hdr, lib=R)
fix["srtm_inv"] = ol.srtm(fix["srtm"], inverse=True, lib=R)
for amount in (0.0, 0.35, 1.0):
    fix["lfga_%g" % amount] = ol.lfga(sdr, grain, amount, lib=R)
fix["dit_f5"] = ol.tepd_dit(W, H, 5, lib=R)
for bits in (8, 10):
    fix["tepd%d_f5" % bits] = ol.tepd(sdr, bits, frame=5, lib=R)
    fix["tepd%d_noise" % bits] = ol.tepd(sdr, bits, dither=noise, lib=R)
np.savez_compressed(os.path.join(HERE, "fsr1_pointwise_golden.npz"), **fix)
print("wrote", len(fix), "arrays;", os.path.getsize(os.path.join(HERE, "fsr1_pointwise_golden.npz")) // 1024, "KiB")
