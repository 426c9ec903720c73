"""GPU parity of the reference's packed calling convention (csrc/fsr1_hx2.cu): FSR1_FLAG_RCAS_HX2 on fsr1_rcas and the
half-precision pointwise entry points fsr1_srtm_h / fsr1_lfga_h / fsr1_tepd_h.

Every operation of these kernels rounds to half once, in the reference's order, so the bar is BIT-EXACTNESS against the half
oracle — which tests/test_oracle.py pins to the reference's own FsrRcasH / FsrRcasHx2 / Fsr*H / Fsr*Hx2 source and to
tests/golden/fsr1_pointwise_h_golden.npz.  The same kernels run bit-exactly on the CPU emulator (tests/test_emu_hx2.py)."""
import os

import numpy as np
import pytest
import torch

import fsr1_b200 as F
import oracle_lib as ol

pytestmark = pytest.mark.gpu
api = F.api
GH = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fsr1_pointwise_h_golden.npz"))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint16)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def gpu_rcas(img, sharp, flags, y0=0, y1=0):
    out = torch.zeros(img.shape, dtype=torch.float16, device="cuda")
    api.rcas(dev(img), out, api.rcas_con(sharp), y0=y0, y1=y1, flags=flags)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def run(fn, src, **kw):
    d = dev(src)
    o = torch.zeros_like(d)
    fn(d, o, **kw)
    torch.cuda.synchronize()
    return o.cpu().numpy()


@pytest.mark.parametrize("size", [(96, 54), (37, 9), (16, 3), (5, 4), (300, 20), (1, 1)])
@pytest.mark.parametrize("gen", ["uniform", "structured"])
def test_rcas_hx2_flag_is_bit_identical_to_the_half_source(size, gen):
    w, h = size
    img = F.to_half(getattr(F, gen)(w, h, 321))
    for sharp in (0.0, 0.25, 2.0):
        rc = ol.rcas_con(sharp)
        for clamp in (0, api.FLAG_RCAS_CLAMP):
            got = gpu_rcas(img, sharp, api.FLAG_RCAS_HX2 | clamp)
            assert api.last_kernel().startswith("rcas_hx2")
            assert np.array_equal(bits(got), bits(ol.rcas(img, rc, bool(clamp))))
            assert np.array_equal(bits(got), bits(gpu_rcas(img, sharp, api.FLAG_H_REFERENCE | clamp)))   # Hx2 == H on the GPU too
            if sharp == 0.25:                                                                           # the reference's FsrRcasHx2
                ol.pinned(ol.rcas_key("h16", gen, w, h, 321, sharp, bool(clamp)), got, lambda: ol.rcas_hx2(img, rc, bool(clamp)))


def test_rcas_hx2_options_golden_vectors_row_ranges_and_rejections():
    sdr = GH["sdr"].view(np.float16)
    for dn in (False, True):
        for pa in (False, True):
            for clamp in (False, True):
                fl = api.FLAG_RCAS_HX2 | (api.FLAG_RCAS_DENOISE if dn else 0) | (api.FLAG_RCAS_PASSTHROUGH_ALPHA if pa else 0)
                got = gpu_rcas(sdr, 0.25, fl | (api.FLAG_RCAS_CLAMP if clamp else 0))
                assert np.array_equal(bits(got), GH["rcas_hx2_dn%d_pa%d_c%d" % (dn, pa, clamp)])
    # a row range writes only its rows; a row-slab window of the input is enough
    img = F.to_half(F.uniform(70, 24, 9))
    full = gpu_rcas(img, 0.25, api.FLAG_RCAS_HX2)
    part = gpu_rcas(img, 0.25, api.FLAG_RCAS_HX2, y0=7, y1=15)
    assert np.array_equal(bits(part[7:15]), bits(full[7:15])) and not bits(part[:7]).any() and not bits(part[15:]).any()
    out = torch.zeros((24, 70, 4), dtype=torch.float16, device="cuda")
    slab = dev(img[6:16])                                              # rows 6..15: what rows 7..14 read
    api.rcas(api.image(slab, height=24, row0=6), out, api.rcas_con(0.25), y0=7, y1=15, flags=api.FLAG_RCAS_HX2)
    torch.cuda.synchronize()
    assert np.array_equal(bits(out.cpu().numpy()[7:15]), bits(full[7:15]))
    # the Sample.x square still applies (as a separate pass, like the H-reference kernel)
    sq = gpu_rcas(img, 0.25, api.FLAG_RCAS_HX2 | api.FLAG_OUTPUT_SQUARE).astype(np.float32)
    want = full.astype(np.float32)
    want[..., :3] = (want[..., :3] * want[..., :3]).astype(np.float16).astype(np.float32)
    assert np.array_equal(sq[..., :3], want[..., :3])
    # half images only
    with pytest.raises(F._lib.Fsr1Error):
        out32 = torch.zeros((24, 70, 4), dtype=torch.float32, device="cuda")
        api.rcas(dev(F.uniform(70, 24, 9)), out32, api.rcas_con(0.25), flags=api.FLAG_RCAS_HX2)


def test_pointwise_h_against_the_reference_golden_vectors():
    sdr, hdr, grain, noise = (GH[k].view(np.float16) for k in ("sdr", "hdr", "grain", "noise"))
    t = run(api.srtm_h, hdr)
    assert api.last_kernel() == "pointwise_hx2<FsrSrtmHx2>"
    assert np.array_equal(bits(t), GH["srtm"])
    assert np.array_equal(bits(run(lambda a, b: api.srtm_h(a, b, inverse=True), GH["srtm"].view(np.float16))), GH["srtm_inv"])
    grain_d, noise_d = dev(grain), dev(noise)
    for amount in (0.0, 0.35, 1.0):
        got = run(lambda a, b: api.lfga_h(a, grain_d, b, amount), sdr)
        assert np.array_equal(bits(got), GH["lfga_%g" % amount])
    for b_ in (8, 10):
        assert np.array_equal(bits(run(lambda a, b: api.tepd_h(a, b, b_, frame=5), sdr)), GH["tepd%d_f5" % b_])
        assert np.array_equal(bits(run(lambda a, b: api.tepd_h(a, b, b_, dither=noise_d), sdr)), GH["tepd%d_noise" % b_])
    assert api.last_kernel() == "pointwise_hx2<FsrTepdC10Hx2>"


@pytest.mark.parametrize("size", [(96, 54), (33, 17), (5, 4), (300, 9), (257, 130)])
def test_pointwise_h_bit_identical_to_the_half_oracle(size):
    w, h = size
    sdr32 = F.structured(w, h, 5).copy()
    sdr32[0, 0, :3] = (0.0, 1.0, 0.5)
    hdr32 = F.structured(w, h, 6).copy()
    hdr32[..., :3] = hdr32[..., :3] ** 3 * 60.0
    hdr32[::7, ::5, :3] = 0.0
    hdr32[3::11, 2::3, :3] = 1.0
    grain32 = (F.uniform(16, 8, 77) - 0.5).astype(np.float32)
    noise32 = F.uniform(8, 8, 3)
    noise32[0, 0, 3], noise32[0, 1, 3] = -0.5, 1.5
    sdr, hdr, grain, noise = F.to_half(sdr32), F.to_half(hdr32), F.to_half(grain32), F.to_half(noise32)
    grain_d, noise_d = dev(grain), dev(noise)
    t = run(api.srtm_h, hdr)
    assert np.array_equal(bits(t), bits(ol.srtm_h(hdr)))
    assert np.array_equal(bits(run(lambda a, b: api.srtm_h(a, b, inverse=True), t)), bits(ol.srtm_h(t, inverse=True)))
    for amount in (0.0, 0.35, 1.0):
        assert np.array_equal(bits(run(lambda a, b: api.lfga_h(a, grain_d, b, amount), sdr)), bits(ol.lfga_h(sdr, grain, amount)))
    for nbits in (8, 10):
        for frame in (0, 9):
            assert np.array_equal(bits(run(lambda a, b: api.tepd_h(a, b, nbits, frame=frame), sdr)), bits(ol.tepd_h(sdr, nbits, frame=frame)))
        assert np.array_equal(bits(run(lambda a, b: api.tepd_h(a, b, nbits, dither=noise_d), sdr)), bits(ol.tepd_h(sdr, nbits, dither=noise)))
    # in place, on a row range only: rows outside [y0,y1) keep their content
    if h >= 9:
        d = dev(hdr)
        api.srtm_h(d, d, y0=2, y1=h - 3)
        torch.cuda.synchronize()
        got = d.cpu().numpy()
        assert np.array_equal(bits(got[2:h - 3]), bits(ol.srtm_h(hdr)[2:h - 3]))
        assert np.array_equal(bits(got[:2]), bits(hdr[:2])) and np.array_equal(bits(got[h - 3:]), bits(hdr[h - 3:]))


def test_pointwise_h_takes_half_images_only():
    f32 = dev(F.uniform(16, 8, 1))
    with pytest.raises(F._lib.Fsr1Error):
        api.srtm_h(f32, torch.zeros_like(f32))
    h16 = dev(F.to_half(F.uniform(16, 8, 1)))
    with pytest.raises(F._lib.Fsr1Error):
        api.lfga_h(h16, f32, torch.zeros_like(h16), 0.5)       # the grain tile must be RGBA16F too
    with pytest.raises(F._lib.Fsr1Error):
        api.tepd_h(h16, torch.zeros_like(h16), 9)             # bits must be 8 or 10
