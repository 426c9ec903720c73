"""ctypes access to the CPU oracle (oracle/libfsr1_oracle.so) and, when it was built, to the reference's
own source compiled for the host (oracle/_ref/libfsr1_ref.so).  TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "libfsr1_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libfsr1_ref.so")
P, F, Z, U = ctypes.c_void_p, ctypes.c_float, ctypes.c_size_t, ctypes.c_uint32


def build():
    src = os.path.join(ROOT, "oracle", "fsr1_oracle.c")
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "libfsr1_oracle.so"],
                              stdout=subprocess.DEVNULL)
    ref_dir = os.environ.get("FSR1_REFERENCE_DIR")
    if not os.path.exists(REF_SO) and ref_dir and os.path.exists(os.path.join(ref_dir, "ffx-fsr", "ffx_fsr1.h")):
        subprocess.check_call([os.path.join(ROOT, "oracle", "build_ref.sh")], stdout=subprocess.DEVNULL)


_o = _r = None


def oracle():
    global _o
    if _o is None:
        build()
        _o = ctypes.CDLL(ORACLE_SO)
        _o.fsr1o_f32_to_f16_trunc.restype = ctypes.c_uint32
        _o.fsr1o_f32_to_f16_trunc.argtypes = [F]
    return _o


def ref():
    """The reference-source build, or None where it is not available."""
    global _r
    if _r is None:
        build()
        if not os.path.exists(REF_SO):
            return None
        _r = ctypes.CDLL(REF_SO)
        _r.fsr1ref_cpu_f32_to_f16.restype = ctypes.c_uint32
        _r.fsr1ref_cpu_f32_to_f16.argtypes = [F]
    return _r


DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
_digests, _recorded = None, {}


def _record_at_exit():
    with open(os.environ["FSR1_RECORD_DIGESTS"], "w") as f:
        json.dump(dict(sorted(_recorded.items())), f, indent=0)


if os.environ.get("FSR1_RECORD_DIGESTS"):
    atexit.register(_record_at_exit)


def pinned(key, got, *live):
    """`got` (array-like) must be what the reference's own source computes for the inputs `key` names.  Where the reference build
    exists, every live() is computed and compared bit for bit.  Always, the SHA-256 of got's bytes is compared with the one stored
    for `key` in tests/golden/reference_digests.json, so the comparison also runs where the reference is absent.  Those digests were
    recorded from the oracle (FSR1_RECORD_DIGESTS=<file> python -m pytest tests/test_oracle.py tests/test_constants.py
    tests/test_emu_hx2.py), which these same tests hold bit-equal to the reference build wherever it is present."""
    got = np.ascontiguousarray(got)
    if ref() is not None:
        for fn in live:
            want = np.ascontiguousarray(fn())
            assert want.shape == got.shape and want.tobytes() == got.tobytes(), key
    d = hashlib.sha256(got.tobytes()).hexdigest()
    if os.environ.get("FSR1_RECORD_DIGESTS"):
        assert _recorded.setdefault(key, d) == d, key
        return
    global _digests
    if _digests is None:
        with open(DIGESTS) as f:
            _digests = json.load(f)
    assert _digests.get(key) == d, key


def rcas_key(prec, gen, w, h, seed, sharp, clamp, denoise=False, alpha=False):
    """The `pinned` key of an RCAS of frames.<gen>(w, h, seed) (prec "h16": quantised to half)."""
    return "rcas_%s %s %dx%d seed%d s%g c%d dn%d pa%d" % (prec, gen, w, h, seed, sharp, clamp, denoise, alpha)


def _con(n):
    return (ctypes.c_uint32 * n)()


def easu_con(iw, ih, ow, oh, vw=None, vh=None, lib=None, off=None):
    c = _con(16)
    vw, vh = (iw if vw is None else vw), (ih if vh is None else vh)
    if lib is None or lib is oracle():
        if off is None:
            oracle().fsr1o_easu_con(c, F(vw), F(vh), F(iw), F(ih), F(ow), F(oh))
        else:
            oracle().fsr1o_easu_con_offset(c, F(vw), F(vh), F(iw), F(ih), F(ow), F(oh), F(off[0]), F(off[1]))
    else:
        if off is None:
            lib.fsr1ref_cpu_easu_con(c, F(vw), F(vh), F(iw), F(ih), F(ow), F(oh))
        else:
            lib.fsr1ref_cpu_easu_con_offset(c, F(vw), F(vh), F(iw), F(ih), F(ow), F(oh), F(off[0]), F(off[1]))
    return list(c)


def rcas_con(sharp, lib=None):
    c = _con(4)
    if lib is None or lib is oracle():
        oracle().fsr1o_rcas_con(c, F(sharp))
    else:
        lib.fsr1ref_cpu_rcas_con(c, F(sharp))
    return list(c)


def _arr(con):
    return (ctypes.c_uint32 * len(con))(*con)


def _pitch(a):
    assert a.strides[2] == a.itemsize and a.strides[1] == 4 * a.itemsize
    return a.strides[0] // a.itemsize


def easu(img, ow, oh, con=None, y0=0, y1=None, lib=None):
    """EASU of a [H,W,4] float32 (F path) or uint16/float16 (H-path model) image on the CPU."""
    lib = lib or oracle()
    ih, iw = img.shape[:2]
    con = con or easu_con(iw, ih, ow, oh)
    y1 = oh if y1 is None else y1
    half = img.dtype != np.float32
    src = img.view(np.uint16) if half else img
    out = np.zeros((oh, ow, 4), np.uint16 if half else np.float32)
    name = {(False, True): "fsr1o_easu_f32", (True, True): "fsr1o_easu_h16", (False, False): "fsr1ref_easu_f",
            (True, False): "fsr1ref_easu_h"}[(half, lib is oracle())]
    getattr(lib, name)(P(src.ctypes.data), iw, ih, Z(_pitch(src)), P(out.ctypes.data), ow, oh, Z(_pitch(out)), _arr(con),
                       y0, y1)
    return out.view(np.float16) if half else out


def rcas(img, con, clamp=False, y0=0, y1=None, lib=None, denoise=False, alpha=False):
    """RCAS; denoise / alpha = the reference's compile-time options FSR_RCAS_DENOISE / FSR_RCAS_PASSTHROUGH_ALPHA."""
    lib = lib or oracle()
    h, w = img.shape[:2]
    y1 = h if y1 is None else y1
    half = img.dtype != np.float32
    src = img.view(np.uint16) if half else img
    out = np.zeros((h, w, 4), np.uint16 if half else np.float32)
    args = [P(src.ctypes.data), w, h, Z(_pitch(src)), P(out.ctypes.data), Z(_pitch(out)), _arr(con), 1 if clamp else 0, y0, y1]
    if lib is oracle():
        getattr(lib, "fsr1o_rcas_h16_opt" if half else "fsr1o_rcas_f32_opt")(*args, (1 if denoise else 0) | (2 if alpha else 0))
    else:
        suffix = {(False, False): "", (True, False): "_dn", (False, True): "_pa", (True, True): "_dnpa"}[(denoise, alpha)]
        getattr(lib, ("fsr1ref_rcas_h" if half else "fsr1ref_rcas_f") + suffix)(*args)
    return out.view(np.float16) if half else out


def rcas_hx2(img, con, clamp=False, denoise=False, alpha=False):
    """The reference's packed calling convention FsrRcasHx2 (two pixels per call), reference build only."""
    lib = ref()
    h, w = img.shape[:2]
    src = img.view(np.uint16)
    out = np.zeros((h, w, 4), np.uint16)
    suffix = {(False, False): "", (True, False): "_dn", (False, True): "_pa", (True, True): "_dnpa"}[(denoise, alpha)]
    getattr(lib, "fsr1ref_rcas_hx2" + suffix)(P(src.ctypes.data), w, h, Z(_pitch(src)), P(out.ctypes.data), Z(_pitch(out)), _arr(con),
                                              1 if clamp else 0, 0, h)
    return out.view(np.float16)


# ---- pointwise companions (LFGA / SRTM / TEPD), fp32 images [H,W,4] --------------------------------------------
def lfga(img, grain, amount, lib=None):
    h, w = img.shape[:2]
    if lib is None or lib is oracle():
        out = np.zeros_like(img)
        oracle().fsr1o_lfga_f32(P(img.ctypes.data), Z(_pitch(img)), P(grain.ctypes.data), grain.shape[1], grain.shape[0],
                                Z(_pitch(grain)), P(out.ctypes.data), Z(_pitch(out)), w, h, F(amount))
        return out
    out = np.ascontiguousarray(img).copy()
    gy, gx = np.arange(h) % grain.shape[0], np.arange(w) % grain.shape[1]
    tiled = np.ascontiguousarray(grain[gy][:, gx])
    lib.fsr1ref_lfga_f(P(out.ctypes.data), P(tiled.ctypes.data), Z(h * w), F(amount))
    return out


def srtm(img, inverse=False, lib=None):
    h, w = img.shape[:2]
    if lib is None or lib is oracle():
        out = np.zeros_like(img)
        oracle().fsr1o_srtm_f32(P(img.ctypes.data), Z(_pitch(img)), P(out.ctypes.data), Z(_pitch(out)), w, h,
                                1 if inverse else 0)
        return out
    out = np.ascontiguousarray(img).copy()
    lib.fsr1ref_srtm_f(P(out.ctypes.data), Z(h * w), 1 if inverse else 0)
    return out


def tepd_dit(w, h, frame, lib=None):
    if lib is None or lib is oracle():
        oracle().fsr1o_tepd_dit.restype = ctypes.c_float
        oracle().fsr1o_tepd_dit.argtypes = [U, U, U]
        return np.array([[oracle().fsr1o_tepd_dit(x, y, frame) for x in range(w)] for y in range(h)], np.float32)
    out = np.zeros((h, w), np.float32)
    lib.fsr1ref_tepd_dit_f(P(out.ctypes.data), w, h, U(frame))
    return out


def tepd(img, bits, frame=0, dither=None, lib=None):
    """dither: None -> FsrTepdDitF(position, frame); else a tiled [h,w,4] image whose .w channel is the dither."""
    h, w = img.shape[:2]
    if lib is None or lib is oracle():
        out = np.zeros_like(img)
        d = (P(dither.ctypes.data), dither.shape[1], dither.shape[0], Z(_pitch(dither))) if dither is not None else (P(0), 0, 0, Z(0))
        oracle().fsr1o_tepd_f32(P(img.ctypes.data), Z(_pitch(img)), *d, P(out.ctypes.data), Z(_pitch(out)), w, h, bits, U(frame))
        return out
    out = np.ascontiguousarray(img).copy()
    if dither is None:
        dit = tepd_dit(w, h, frame, lib=lib)
    else:
        gy, gx = np.arange(h) % dither.shape[0], np.arange(w) % dither.shape[1]
        dit = np.ascontiguousarray(np.clip(dither[gy][:, gx][..., 3], 0.0, 1.0).astype(np.float32))
    lib.fsr1ref_tepd_f(P(out.ctypes.data), P(dit.ctypes.data), Z(h * w), bits)
    return out


# ---- pointwise companions in half precision: RGBA16F images [H,W,4] (numpy float16) -------------------------------
# lib=None: the C restatement; lib=ref(): the reference's own FsrLfgaH / FsrSrtmH / FsrTepdC*H, or with hx2=True its packed
# calling convention (FsrLfgaHx2 / FsrSrtmHx2 / FsrTepdDitHx2 / FsrTepdC*Hx2).
def _tile16(aux, h, w):
    gy, gx = np.arange(h) % aux.shape[0], np.arange(w) % aux.shape[1]
    return np.ascontiguousarray(aux[gy][:, gx])


def lfga_h(img, grain, amount, lib=None, hx2=False):
    h, w = img.shape[:2]
    src, g = np.ascontiguousarray(img).view(np.uint16), np.ascontiguousarray(grain).view(np.uint16)
    if lib is None or lib is oracle():
        out = np.zeros_like(src)
        oracle().fsr1o_lfga_h16(P(src.ctypes.data), Z(_pitch(src)), P(g.ctypes.data), g.shape[1], g.shape[0], Z(_pitch(g)),
                                P(out.ctypes.data), Z(_pitch(out)), w, h, F(amount))
        return out.view(np.float16)
    out, tiled = src.copy(), _tile16(g, h, w)
    getattr(lib, "fsr1ref_lfga_hx2" if hx2 else "fsr1ref_lfga_h")(P(out.ctypes.data), P(tiled.ctypes.data), Z(h * w), F(amount))
    return out.view(np.float16)


def srtm_h(img, inverse=False, lib=None, hx2=False):
    h, w = img.shape[:2]
    src = np.ascontiguousarray(img).view(np.uint16)
    if lib is None or lib is oracle():
        out = np.zeros_like(src)
        oracle().fsr1o_srtm_h16(P(src.ctypes.data), Z(_pitch(src)), P(out.ctypes.data), Z(_pitch(out)), w, h, 1 if inverse else 0)
        return out.view(np.float16)
    out = src.copy()
    getattr(lib, "fsr1ref_srtm_hx2" if hx2 else "fsr1ref_srtm_h")(P(out.ctypes.data), Z(h * w), 1 if inverse else 0)
    return out.view(np.float16)


def tepd_dit_h(w, h, frame, lib=None, hx2=False):
    if lib is None or lib is oracle():
        oracle().fsr1o_tepd_dit_h16.restype = ctypes.c_uint16
        oracle().fsr1o_tepd_dit_h16.argtypes = [U, U, U]
        return np.array([[oracle().fsr1o_tepd_dit_h16(x, y, frame) for x in range(w)] for y in range(h)], np.uint16).view(np.float16)
    out = np.zeros((h, w), np.uint16)
    getattr(lib, "fsr1ref_tepd_dit_hx2" if hx2 else "fsr1ref_tepd_dit_h")(P(out.ctypes.data), w, h, U(frame))
    return out.view(np.float16)


def tepd_h(img, bits, frame=0, dither=None, lib=None, hx2=False):
    """dither: None -> FsrTepdDitH(position, frame); else a tiled [h,w,4] float16 image whose .w channel is the dither."""
    h, w = img.shape[:2]
    src = np.ascontiguousarray(img).view(np.uint16)
    if lib is None or lib is oracle():
        out = np.zeros_like(src)
        if dither is not None:
            d16 = np.ascontiguousarray(dither).view(np.uint16)
            d = (P(d16.ctypes.data), d16.shape[1], d16.shape[0], Z(_pitch(d16)))
        else:
            d = (P(0), 0, 0, Z(0))
        oracle().fsr1o_tepd_h16(P(src.ctypes.data), Z(_pitch(src)), *d, P(out.ctypes.data), Z(_pitch(out)), w, h, bits, U(frame))
        return out.view(np.float16)
    out = src.copy()
    if dither is None:
        dit = np.ascontiguousarray(tepd_dit_h(w, h, frame, lib=lib, hx2=hx2)).view(np.uint16)
    else:
        t = _tile16(np.ascontiguousarray(dither), h, w)[..., 3].astype(np.float32)
        dit = np.ascontiguousarray(np.clip(t, 0.0, 1.0).astype(np.float16)).view(np.uint16)
    getattr(lib, "fsr1ref_tepd_hx2" if hx2 else "fsr1ref_tepd_h")(P(out.ctypes.data), P(dit.ctypes.data), Z(h * w), bits)
    return out.view(np.float16)
