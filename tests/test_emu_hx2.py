"""The packed Hx2 calling-convention kernels (csrc/fsr1_hx2.cu: FsrRcasHx2, FsrSrtmHx2, FsrLfgaHx2, FsrTepdC8Hx2 / C10Hx2,
FsrTepdDitHx2) compiled for the HOST (tests/emu, one rounding per emulated half operation) and compared BIT FOR BIT with the
oracle's half restatement and, where it was built, with the reference's own H and Hx2 source (oracle/_ref).  The emulator
executes the kernels' own statements, so lane pairing (ip, ip + (8,0)), the AoS <-> SoA shuffles, right-edge strips, row windows,
tile wrap and both out-of-image rules are checked without a GPU; tests/test_gpu_pointwise.py and test_gpu_parity.py repeat the
comparison on the hardware."""
import ctypes

import numpy as np
import pytest

import fsr1_b200 as F
import oracle_lib as ol
from test_emu import emu_lib

P, LL = ctypes.c_void_p, ctypes.c_longlong


def bits(a):
    return np.ascontiguousarray(a).view(np.uint16)


def emu_rcas_hx2(img, con, clamp=False, y0=0, y1=None, opts=0, window=None):
    """window=(row0, rows): hand the kernel only those rows of the image (a row slab)."""
    h, w = img.shape[:2]
    y1 = h if y1 is None else y1
    r0, nr = window if window else (0, h)
    src = np.ascontiguousarray(bits(img)[r0:r0 + nr])
    out = np.zeros((h, w, 4), np.uint16)
    rc = emu_lib().emu_rcas_hx2(P(src.ctypes.data), r0, nr, P(out.ctypes.data), w, h, LL(src.strides[0]), LL(out.strides[0]),
                                (ctypes.c_uint32 * 4)(*con), 1 if clamp else 0, y0, y1, opts)
    assert rc == 0
    return out.view(np.float16)


def emu_point(op, img, aux=None, amount=0.0, frame=0, y0=0, y1=None):
    h, w = img.shape[:2]
    y1 = h if y1 is None else y1
    src = np.ascontiguousarray(bits(img))
    out = np.zeros((h, w, 4), np.uint16)
    if aux is not None:
        a = np.ascontiguousarray(bits(aux))
        args = (P(a.ctypes.data), a.shape[1], a.shape[0], LL(a.strides[0]))
    else:
        args = (P(0), 0, 0, LL(0))
    rc = emu_lib().emu_pointwise_hx2(op, P(src.ctypes.data), LL(src.strides[0]), P(out.ctypes.data), LL(out.strides[0]), w, h, *args,
                                     ctypes.c_float(amount), ctypes.c_uint32(frame), y0, y1)
    assert rc == 0
    return out.view(np.float16)


@pytest.mark.parametrize("size", [(96, 20), (37, 9), (16, 3), (5, 4), (300, 5)])
@pytest.mark.parametrize("gen", ["uniform", "structured"])
def test_emulated_rcas_hx2_bit_identical_to_the_half_oracle(size, gen):
    """Widths that end inside a 16-pixel strip, inside its first half, and wider than one CTA (256 px)."""
    w, h = size
    img = F.to_half(getattr(F, gen)(w, h, 321))
    R = ol.ref()
    for sharp in (0.0, 0.25, 2.0):
        rc = ol.rcas_con(sharp)
        for clamp in (False, True):
            got = emu_rcas_hx2(img, rc, clamp)
            assert np.array_equal(bits(got), bits(ol.rcas(img, rc, clamp)))
            if sharp == 0.25:         # the reference's own FsrRcasHx2 and FsrRcasH, live or through their stored digests
                ol.pinned(ol.rcas_key("h16", gen, w, h, 321, sharp, clamp), got,
                          lambda: ol.rcas_hx2(img, rc, clamp), lambda: ol.rcas(img, rc, clamp, lib=R))


@pytest.mark.parametrize("denoise,alpha", [(True, False), (False, True), (True, True)])
def test_emulated_rcas_hx2_options(denoise, alpha):
    w, h = 53, 11
    img = F.to_half(F.structured(w, h, 77))
    rc = ol.rcas_con(0.25)
    opts = (1 if denoise else 0) | (2 if alpha else 0)
    for clamp in (False, True):
        got = emu_rcas_hx2(img, rc, clamp, opts=opts)
        assert np.array_equal(bits(got), bits(ol.rcas(img, rc, clamp, denoise=denoise, alpha=alpha)))
        ol.pinned(ol.rcas_key("h16", "structured", w, h, 77, 0.25, clamp, denoise, alpha), got,
                  lambda: ol.rcas_hx2(img, rc, clamp, denoise=denoise, alpha=alpha))
        if alpha:
            assert np.array_equal(bits(got[..., 3]), bits(img[..., 3]))


def test_emulated_rcas_hx2_row_range_and_window():
    w, h = 70, 24
    img = F.to_half(F.uniform(w, h, 9))
    rc = ol.rcas_con(0.25)
    full = emu_rcas_hx2(img, rc)
    part = emu_rcas_hx2(img, rc, y0=7, y1=15, window=(6, 10))          # rows 7..14 read rows 6..15 only
    assert np.array_equal(bits(part[7:15]), bits(full[7:15]))
    assert not bits(part[:7]).any() and not bits(part[15:]).any()


def _frames(w, h):
    sdr = F.structured(w, h, 4242).copy()
    sdr[0, 0, :3] = (0.0, 1.0, 0.5)
    hdr = sdr.copy()
    hdr[..., :3] = hdr[..., :3] ** 3 * 60.0
    hdr[::7, ::5, :3] = 0.0
    hdr[3::11, 2::3, :3] = 1.0
    grain = (F.uniform(12, 5, 99) - 0.5).astype(np.float32)       # 12 x 5 tile: wraps in both directions
    noise = F.uniform(9, 7, 98)
    noise[0, 0, 3], noise[0, 1, 3] = -0.5, 1.5                     # saturated on use
    return F.to_half(sdr), F.to_half(hdr), F.to_half(grain), F.to_half(noise)


@pytest.mark.parametrize("size", [(96, 12), (33, 17), (5, 4), (300, 3)])
def test_emulated_pointwise_hx2_bit_identical_to_the_half_oracle(size):
    w, h = size
    sdr, hdr, grain, noise = _frames(w, h)
    R = ol.ref()
    k = "emu_frames %dx%d " % (w, h)      # the reference's H (and Hx2) functions: live or through their stored digests
    # SRTM and its inverse (incl. the c = 1.0 case the extra max solves)
    t = emu_point(1, hdr)
    assert np.array_equal(bits(t), bits(ol.srtm_h(hdr)))
    ol.pinned(k + "srtm", t, lambda: ol.srtm_h(hdr, lib=R), lambda: ol.srtm_h(hdr, lib=R, hx2=True))
    ti = emu_point(2, t)
    one = F.to_half(np.ones((2, 20, 4), np.float32))
    t1 = emu_point(2, one)
    assert np.array_equal(bits(ti), bits(ol.srtm_h(t, inverse=True)))
    assert np.array_equal(bits(t1), bits(ol.srtm_h(one, inverse=True)))
    ol.pinned(k + "srtm_inv", ti, lambda: ol.srtm_h(t, inverse=True, lib=R))
    ol.pinned("emu_frames ones 20x2 srtm_inv", t1, lambda: ol.srtm_h(one, inverse=True, lib=R))
    assert np.array_equal(bits(t[..., 3]), bits(hdr[..., 3]))      # alpha carried through
    # LFGA
    for amount in (0.0, 0.35, 1.0):
        got = emu_point(3, sdr, aux=grain, amount=amount)
        assert np.array_equal(bits(got), bits(ol.lfga_h(sdr, grain, amount)))
        ol.pinned(k + "lfga %g" % amount, got, lambda: ol.lfga_h(sdr, grain, amount, lib=R),
                  lambda: ol.lfga_h(sdr, grain, amount, lib=R, hx2=True))
    # TEPD, positional dither (FsrTepdDitHx2: p and p + (8,0)) and a blue-noise tile
    for nbits, op in ((8, 4), (10, 5)):
        for frame in (0, 5):
            got = emu_point(op, sdr, frame=frame)
            assert np.array_equal(bits(got), bits(ol.tepd_h(sdr, nbits, frame=frame)))
            ol.pinned(k + "tepd%d f%d positional" % (nbits, frame), got, lambda: ol.tepd_h(sdr, nbits, frame=frame, lib=R),
                      lambda: ol.tepd_h(sdr, nbits, frame=frame, lib=R, hx2=True))
        got = emu_point(op, sdr, aux=noise)
        assert np.array_equal(bits(got), bits(ol.tepd_h(sdr, nbits, dither=noise)))
        ol.pinned(k + "tepd%d noise" % nbits, got, lambda: ol.tepd_h(sdr, nbits, dither=noise, lib=R))


def test_emulated_pointwise_hx2_row_range_in_place_semantics():
    w, h = 40, 9
    sdr, hdr, grain, noise = _frames(w, h)
    full = emu_point(1, hdr)
    part = emu_point(1, hdr, y0=2, y1=6)
    assert np.array_equal(bits(part[2:6]), bits(full[2:6]))
    assert not bits(part[:2]).any() and not bits(part[6:]).any()
