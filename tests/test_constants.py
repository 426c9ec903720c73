"""FsrEasuCon / FsrEasuConOffset / FsrRcasCon of include/fsr1_host.h (exported through the C ABI) against the
reference's unmodified header compiled with #define A_CPU (golden table + live where available)."""
import ctypes
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

import fsr1_b200 as F
import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KAT = json.load(open(os.path.join(HERE, "golden", "kat.json")))


def hexes(con):
    return ["%08x" % v for v in con]


def test_easu_con_known_answers():
    for key, want in KAT["easu_con"].items():
        iw, ih, ow, oh = map(int, key.split(","))
        assert hexes(F.api.easu_con(iw, ih, iw, ih, ow, oh)) == want, key
        assert hexes(ol.easu_con(iw, ih, ow, oh)) == want, key
    # values quoted in SURVEY.md §8(a)/(c)
    assert KAT["easu_con"]["1920,1080,3840,2160"][:4] == ["3f000000", "3f000000", "be800000", "be800000"]
    assert KAT["easu_con"]["2953,1661,3840,2160"][:4] == ["3f44dddf", "3f44dbf8", "bdec8884", "bdec9020"]


def test_easu_con_offset_known_answer():
    (key, want), = KAT["easu_con_offset"].items()
    vw, vh, iw, ih, ow, oh, ox, oy = map(float, key.split(","))
    assert hexes(F.api.easu_con_offset(vw, vh, iw, ih, ow, oh, ox, oy)) == want


def test_rcas_con_known_answers():
    for key, want in KAT["rcas_con"].items():
        assert hexes(F.api.rcas_con(float(key))) == want, key
        assert hexes(ol.rcas_con(float(key))) == want, key
    assert KAT["rcas_con"]["0.25"][:2] == ["3f5744fd", "3aba3aba"]
    assert KAT["rcas_con"]["0.0"][:2] == ["3f800000", "3c003c00"]
    # the CPU packer TRUNCATES (ffx_a.h:549): 0.2 -> 3af6, not the round-to-nearest 3af7
    assert KAT["rcas_con"]["0.2"][:2] == ["3f5edc67", "3af63af6"]


def test_truncating_half_packer_known_answers():
    for key, want in KAT["f32_to_f16"].items():
        assert "%04x" % ol.oracle().fsr1o_f32_to_f16_trunc(float(key)) == want, key


def test_constants_against_live_reference_sweep():
    """Live against the reference build where it exists, else against the stored digests of its results (ol.pinned)."""
    R = ol.ref()
    rng = np.random.default_rng(3)
    shapes = []
    for _ in range(300):
        ow, oh = int(rng.integers(1, 8000)), int(rng.integers(1, 5000))
        iw, ih = int(rng.integers(1, ow + 1)), int(rng.integers(1, oh + 1))
        shapes.append((iw, ih, ow, oh))
    ol.pinned("easu_con sweep rng3 x300", np.array([F.api.easu_con(iw, ih, iw, ih, ow, oh) for iw, ih, ow, oh in shapes], np.uint32),
              lambda: np.array([ol.easu_con(iw, ih, ow, oh, lib=R) for iw, ih, ow, oh in shapes], np.uint32))
    sharps = [float(s) for s in np.linspace(0, 40, 401)]
    ol.pinned("rcas_con sweep 0..40 x401", np.array([F.api.rcas_con(s) for s in sharps], np.uint32),
              lambda: np.array([ol.rcas_con(s, lib=R) for s in sharps], np.uint32))
    # packer: every exponent, a spread of mantissas, both signs (arithmetic vs the reference's tables); NaN inputs excluded
    vals = (np.arange(0, 2 ** 32, 65521, dtype=np.uint64)).astype(np.uint32)[::97]
    fs = [float(f) for f in vals.view(np.float32) if not np.isnan(f)]
    ol.pinned("f32_to_f16_trunc sweep", np.array([ol.oracle().fsr1o_f32_to_f16_trunc(f) for f in fs], np.uint32),
              lambda: np.array([R.fsr1ref_cpu_f32_to_f16(f) for f in fs], np.uint32))


def test_host_header_compiles_as_c_and_matches(tmp_path):
    """include/fsr1_host.h is usable from plain C exactly like the reference's header pair."""
    src = tmp_path / "t.c"
    src.write_text('#include <stdio.h>\n#include "fsr1_host.h"\nint main(void){AU1 c0[4],c1[4],c2[4],c3[4],r[4];'
                   'FsrEasuCon(c0,c1,c2,c3,1920.0f,1080.0f,1920.0f,1080.0f,3840.0f,2160.0f);FsrRcasCon(r,0.25f);'
                   'printf("%08x %08x %08x %08x %08x %08x\\n",c0[0],c0[2],c1[1],c3[1],r[0],r[1]);return 0;}\n')
    exe = tmp_path / "t"
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-O1", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), "-lm"])
    out = subprocess.check_output([str(exe)]).decode().split()
    assert out == ["3f000000", "be800000", "3a72b9d6", "3b72b9d6", "3f5744fd", "3aba3aba"]
    # the compat headers keep the reference's include lines working
    src2 = tmp_path / "u.c"
    src2.write_text('#include <stdint.h>\n#include <math.h>\n#define A_CPU\n#include "ffx_a.h"\n#include "ffx_fsr1.h"\n'
                    'int main(void){AU1 r[4];FsrRcasCon(r,(AF1)1.0);return r[0]==0x3f000000u?0:1;}\n')
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-I", os.path.join(ROOT, "include", "compat"), str(src2), "-o",
                           str(tmp_path / "u"), "-lm"])
    assert subprocess.call([str(tmp_path / "u")]) == 0


def test_unorm_decode_refinement_is_correctly_rounded_for_every_code():
    """unorm_to_float (csrc/fsr1_common.cuh): q = c * (1/s) followed by one FMA refinement equals the correctly rounded c / s for
    every 8- and 10-bit code (the plain product is an ulp off for half of the 8-bit codes, and an ulp of luma flips EASU's exact-tie
    0/0 length term).  The device function itself runs in tests/test_emu.py (host build) and on the GPU."""
    for s in (255, 1023):
        c = np.arange(0, s + 1, dtype=np.float32)
        want = (c / np.float32(s)).astype(np.float32)
        k = np.float32(1.0) / np.float32(s)
        q = (c * k).astype(np.float32)
        assert (q != want).any()                      # the shortcut really is inexact
        r = (c.astype(np.float64) - q.astype(np.float64) * np.float64(s)).astype(np.float32)          # fma(-q, s, c): exact
        q2 = (r.astype(np.float64) * np.float64(k) + q.astype(np.float64)).astype(np.float32)         # fma(r, 1/s, q)
        assert np.array_equal(q2, want)
