"""CPU suite: ComputeMSE and the IsAlphaAllOpaque scan in the host emulator (tests/emul/analysis_emul.cpp: the kernels' own headers,
dxb_analyze.cuh) against the reference's recorded answers (tests/golden/analysis_calls.npz, tests/analysis_lib.py), the numerical contract against an fp64 sum in numpy, and the CMSE_FLAGS enumerators of
the C++ mirror against the reference header.  tests/analysis_cases.py is the case table the GPU suite replays too."""
import os
import subprocess

import numpy as np
import pytest

from directxtex_b200 import formats as F
from tests import analysis_cases as AC
from tests.analysis_lib import analysis_oracle, analysis_emul  # noqa: F401  (fixtures)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("DXB_REFERENCE_SRC", "")
SNAP_CMSE = os.path.join(ROOT, "tests", "golden", "cmse_reference.txt")
CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
GAMMA = 0x1 | 0x2


def check_vs_reference(got, want):
    """mseV and mse within 2e-3 relative of the reference's running fp32 sum (images <= 256^2)"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.all(np.abs(got - want) <= 2e-3 * np.abs(want) + 1e-30), (got, want)


@pytest.mark.parametrize("case", AC.mse_cases(), ids=lambda c: c[0])
def test_emulated_mse_matches_the_reference(case, analysis_oracle, analysis_emul):
    cid, fa, fb, w, h, fl, pad = case
    a, b = AC.mse_inputs(case)
    hr, want = analysis_oracle.compute_mse(a, fa, b, fb, w, h, fl, full=True)
    assert hr == 0
    pa, pitch_a = AC.padded(a, fa, w, h, pad)
    pb, pitch_b = AC.padded(b, fb, w, h, pad)
    hr, got = analysis_emul.compute_mse(pa, fa, pb, fb, w, h, fl, pitch_a, pitch_b)
    assert hr == 0
    check_vs_reference(got, want)
    assert got[0] == np.float32(((got[1] + got[2]) + got[3]) + got[4])


def _decoded(fmt, img, w, h, emul):
    """the fp32 pixels ComputeMSE_ compares for the formats numpy can load exactly"""
    if fmt in F.BLOCK_BYTES:
        return emul.decode_blocks(fmt, img, w, h).reshape(-1, 4)
    if fmt == 28:
        return np.asarray(img, np.uint8).reshape(-1, 4).astype(np.float32) * np.float32(1.0 / 255.0)
    if fmt == 2:
        return np.asarray(img).view(np.float32).reshape(-1, 4)
    if fmt == 10:
        return np.asarray(img).view(np.float16).reshape(-1, 4).astype(np.float32)
    raise ValueError(fmt)


@pytest.mark.parametrize("cid", ["pair_28_28", "pair_2_10", "flags_80", "flags_100", "flags_200", "bc_98_vs_rgba32f", "bc_71_vs_rgba32f",
                                 "size_rgba8_256x256", "size_f16_256", "size_bc1_256", "pitch_rgba8"])
def test_mse_is_within_4_ulp_of_the_fp64_sum_of_the_reference_squares(cid, emul, analysis_emul):
    case = [c for c in AC.mse_cases() if c[0] == cid][0]
    _, fa, fb, w, h, fl, pad = case
    a, b = AC.mse_inputs(case)
    v1, v2 = _decoded(fa, a, w, h, emul), _decoded(fb, b, w, h, emul)
    if fl & 0x100:
        v1 = v1 * np.float32(2) + np.float32(-1)
    if fl & 0x200:
        v2 = v2 * np.float32(2) + np.float32(-1)
    d = (v1 - v2).astype(np.float32)
    for k, bit in enumerate((0x10, 0x20, 0x40, 0x80)):
        if fl & bit:
            d[:, k] = 0
    sq = (d * d).astype(np.float32)                                   # the reference's fp32 squares
    exact = (sq.astype(np.float64).sum(0) / 1.0).astype(np.float64)
    want = (exact.astype(np.float32) / np.float32(w * h)).astype(np.float32)
    pa, pitch_a = AC.padded(a, fa, w, h, pad)
    pb, pitch_b = AC.padded(b, fb, w, h, pad)
    hr, got = analysis_emul.compute_mse(pa, fa, pb, fb, w, h, fl, pitch_a, pitch_b)
    assert hr == 0
    ulp = np.spacing(np.abs(want)).astype(np.float64)
    assert np.all(np.abs(got[1:].astype(np.float64) - want) <= 4 * ulp), (got[1:], want)


@pytest.mark.parametrize("case", AC.opaque_cases(), ids=lambda c: c[0])
def test_emulated_alpha_scan_matches_the_reference(case, analysis_oracle, analysis_emul):
    cid, fmt, w, h, levels, px = case
    hr, want = analysis_oracle.is_alpha_all_opaque(px, fmt, w, h, 1, levels)
    assert hr == 0
    hr, scan = analysis_emul.is_alpha_all_opaque(px, AC.opaque_layout(fmt, w, h, levels), fmt)
    assert hr == 0
    # ScratchImage::IsAlphaAllOpaque: formats without alpha answer true before the scan (BC4 / BC5 / BC6H scan as "not opaque")
    got = 1 if fmt in AC.NO_ALPHA else scan
    assert got == want, (cid, got, want)
    if fmt in (80, 83, 95):
        assert scan == 0


def test_alpha_scan_thresholds(analysis_emul):
    """the cases the table is built around give the answers the thresholds imply (0.997 uncompressed, 0.99 BC)"""
    want = {"rgba8_opaque_chain": 1, "rgba8_last_level": 0, "rgba8_254": 0, "rgba32f_0997": 1, "rgba32f_below_0997": 0, "bc3_alpha_252": 0,
            "bc3_alpha_253": 1, "bc3_padding_only": 1, "bc1_transparent_index": 0, "bc1_four_colour": 1, "bc7_modes_0_3": 1}
    for cid, fmt, w, h, levels, px in AC.opaque_cases():
        if cid in want:
            hr, v = analysis_emul.is_alpha_all_opaque(px, AC.opaque_layout(fmt, w, h, levels), fmt)
            assert hr == 0 and v == want[cid], cid


def _cmse_probe(tmp_path, reference):
    exe = str(tmp_path / ("cmse_ref" if reference else "cmse_ours"))
    inc = ["-DPROBE_REFERENCE", "-msse2", "-I", os.path.join(ROOT, "oracle", "compat"), "-I", REF] if reference else ["-I", os.path.join(ROOT, "directxtex_b200", "host")]
    subprocess.run([CXX, "-std=c++17", "-w"] + inc + [os.path.join(ROOT, "tests", "cpp", "cmse_probe.cpp"), "-o", exe], check=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def test_cmse_flags_match_the_reference_header(tmp_path):
    ours = _cmse_probe(tmp_path, False)
    if os.path.isdir(REF):
        theirs = _cmse_probe(tmp_path, True)
        if not os.path.exists(SNAP_CMSE) or open(SNAP_CMSE).read() != theirs:
            open(SNAP_CMSE, "w").write(theirs)               # snapshot for machines without the reference tree (committed)
    else:
        theirs = open(SNAP_CMSE).read()
    assert len(ours.splitlines()) == 9 and ours.splitlines() == theirs.splitlines()
