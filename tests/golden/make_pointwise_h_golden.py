"""Generates tests/golden/fsr1_pointwise_h_golden.npz by EXECUTING THE REFERENCE's own half-precision functions FsrSrtmH /
FsrSrtmInvH / FsrLfgaH / FsrTepdDitH / FsrTepdC8H / FsrTepdC10H and their packed Hx2 forms, plus FsrRcasHx2 with the
compile-time options (oracle/_ref/libfsr1_ref.so built with A_HALF, see oracle/build_ref.sh).  The H and the Hx2 results are
asserted bit-identical before one copy is stored.  Needs FSR1_REFERENCE_DIR; the output is committed so the
checks also run where the reference build is absent.

    python tests/golden/make_pointwise_h_golden.py
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


def u16(a):
    return np.ascontiguousarray(a).view(np.uint16)


def both(fn, *args, **kw):
    a, b = fn(*args, lib=R, **kw), fn(*args, lib=R, hx2=True, **kw)
    assert np.array_equal(u16(a), u16(b)), "the reference's H and Hx2 forms disagree"
    return u16(a)


W, H = 300, 7                                   # wider than one 256-pixel CTA row, ends inside the first half of a 16-pixel strip
sdr = F.structured(W, H, 4242).copy()
sdr[0, 0, :3] = (0.0, 1.0, 0.5)
hdr = sdr.copy()
hdr[..., :3] = hdr[..., :3] ** 3 * 60.0
hdr[::7, ::5, :3] = 0.0
hdr[3::11, 2::3, :3] = 1.0
grain = (F.uniform(12, 5, 99) - 0.5).astype(np.float32)
noise = F.uniform(9, 7, 98)
noise[0, 0, 3], noise[0, 1, 3] = -0.5, 1.5
sdr, hdr, grain, noise = F.to_half(sdr), F.to_half(hdr), F.to_half(grain), F.to_half(noise)
fix = {"sdr": u16(sdr), "hdr": u16(hdr), "grain": u16(grain), "noise": u16(noise)}
fix["srtm"] = both(ol.srtm_h, hdr)
fix["srtm_inv"] = both(ol.srtm_h, fix["srtm"].view(np.float16), inverse=True)
for amount in (0.0, 0.35, 1.0):
    fix["lfga_%g" % amount] = both(ol.lfga_h, sdr, grain, amount)
fix["dit_f5"] = both(ol.tepd_dit_h, W, H, 5)
for bits in (8, 10):
    fix["tepd%d_f5" % bits] = both(ol.tepd_h, sdr, bits, frame=5)
    fix["tepd%d_noise" % bits] = both(ol.tepd_h, sdr, bits, dither=noise)
rc = ol.rcas_con(0.25)
for dn in (False, True):
    for pa in (False, True):
        for clamp in (False, True):
            a = ol.rcas_hx2(sdr, rc, clamp, denoise=dn, alpha=pa)
            assert np.array_equal(u16(a), u16(ol.rcas(sdr, rc, clamp, lib=R, denoise=dn, alpha=pa)))
            fix["rcas_hx2_dn%d_pa%d_c%d" % (dn, pa, clamp)] = u16(a)
np.savez_compressed(os.path.join(HERE, "fsr1_pointwise_h_golden.npz"), **fix)
print("wrote", len(fix), "arrays;", os.path.getsize(os.path.join(HERE, "fsr1_pointwise_h_golden.npz")) // 1024, "KiB")
