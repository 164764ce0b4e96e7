"""SURVEY 8(f) rank 3: the DDS container either side of the hot path (host-side code, no GPU): byte-for-byte against the
reference's SaveToDDSMemory / LoadFromDDSMemory (DirectXTexDDS.cpp) for the formats this library implements."""
import numpy as np
import pytest

from directxtex_b200 import capi, formats as F
from tests.oracle_lib import same

DX10, DX10_MISC2, IGNORE_MIPS = 0x10000, 0x20000, 0x100
CUBE = 0x4
CASES = [
    # fmt, w, h, arraySize, mipLevels, miscFlags, miscFlags2, flags
    (28, 16, 8, 1, 1, 0, 0, 0), (28, 16, 8, 1, 5, 0, 0, 0), (28, 16, 8, 1, 1, 0, 0, DX10), (29, 16, 16, 1, 3, 0, 0, 0),
    (87, 9, 7, 1, 1, 0, 0, 0), (88, 8, 8, 1, 1, 0, 0, 0), (2, 8, 4, 1, 1, 0, 0, 0), (10, 8, 4, 3, 2, 0, 0, 0),
    (11, 4, 4, 1, 1, 0, 0, 0), (13, 4, 4, 1, 1, 0, 0, 0), (16, 4, 4, 1, 1, 0, 0, 0), (34, 4, 4, 1, 1, 0, 0, 0),
    (41, 5, 3, 1, 1, 0, 0, 0), (54, 5, 3, 1, 1, 0, 0, 0), (35, 6, 2, 1, 1, 0, 0, 0), (37, 6, 2, 1, 1, 0, 0, 0),
    (49, 6, 2, 1, 1, 0, 0, 0), (51, 6, 2, 1, 1, 0, 0, 0), (56, 6, 2, 1, 1, 0, 0, 0), (61, 7, 3, 1, 1, 0, 0, 0),
    (65, 7, 3, 1, 1, 0, 0, 0), (31, 4, 4, 1, 1, 0, 0, 0), (24, 4, 4, 1, 1, 0, 0, 0),
    (71, 16, 16, 1, 5, 0, 0, 0), (72, 16, 16, 1, 1, 0, 0, 0), (74, 8, 8, 1, 1, 0, 0, 0), (74, 8, 8, 1, 1, 0, 2, 0),
    (77, 8, 8, 1, 1, 0, 0, 0), (77, 8, 8, 1, 1, 0, 2, 0), (80, 12, 12, 1, 1, 0, 0, 0), (81, 12, 12, 1, 1, 0, 0, 0),
    (83, 12, 12, 1, 1, 0, 0, 0), (84, 12, 12, 1, 1, 0, 0, 0), (95, 8, 8, 1, 4, 0, 0, 0), (98, 20, 12, 2, 3, 0, 0, 0),
    (85, 8, 8, 1, 1, 0, 0, 0), (86, 8, 8, 1, 3, 0, 0, 0), (115, 6, 6, 1, 1, 0, 0, 0), (26, 8, 4, 1, 1, 0, 0, 0), (67, 8, 4, 2, 2, 0, 0, 0), (85, 8, 8, 1, 1, 0, 0, DX10),
    (28, 8, 8, 6, 1, CUBE, 0, 0), (28, 8, 8, 12, 2, CUBE, 0, 0), (98, 8, 8, 1, 1, 0, 1, DX10_MISC2), (71, 5, 5, 4, 1, 0, 0, 0),
]


def _pixels(fmt, w, h, n, m, seed):
    _, total = capi.texture_layout(fmt, w, h, n, m)
    return np.random.default_rng(seed).integers(0, 256, total, dtype=np.uint8)


@pytest.mark.parametrize("case", CASES)
def test_dds_save_matches_reference_and_round_trips(oracle, case):
    fmt, w, h, n, m, misc, misc2, flags = case
    px = _pixels(fmt, w, h, n, m, hash(case) & 0xFFFF)
    hr, want = oracle.dds_save(px, fmt, w, h, n, m, misc, misc2, flags)
    assert hr == 0, hex(hr)
    got = capi.dds_save(px, fmt, w, h, n, m, misc, misc2, flags)
    assert same(got, want), case
    # load the reference's file (the same bytes) with this library and this library's file with the reference
    md, back = capi.dds_load(got)
    hr, rmeta, rback = oracle.dds_load(got)
    assert hr == 0
    assert [md.width, md.height, md.arraySize, md.mipLevels, md.format, md.miscFlags, md.miscFlags2] == rmeta, case
    assert same(back, rback) and same(back, px)


DX9, RXGB = 0x40000, 0x80000


@pytest.mark.parametrize("case", [(29, 8, 8, 1, 1, 0, 0, DX9), (91, 8, 8, 1, 2, 0, 0, DX9), (93, 8, 8, 1, 1, 0, 0, DX9), (72, 8, 8, 1, 1, 0, 0, DX9),
                                  (75, 8, 8, 1, 1, 0, 2, DX9), (78, 8, 8, 1, 1, 0, 0, DX9), (80, 8, 8, 1, 1, 0, 0, DX9), (83, 8, 8, 1, 1, 0, 0, DX9),
                                  (28, 8, 8, 1, 1, 0, 0, DX9), (77, 8, 8, 1, 1, 0, 0, RXGB), (28, 8, 8, 6, 1, CUBE, 0, DX9)])
def test_dds_legacy_flags_match_reference(oracle, case):
    fmt, w, h, n, m, misc, misc2, flags = case
    px = _pixels(fmt, w, h, n, m, 5)
    hr, want = oracle.dds_save(px, fmt, w, h, n, m, misc, misc2, flags)
    assert hr == 0, hex(hr)
    got = capi.dds_save(px, fmt, w, h, n, m, misc, misc2, flags)
    assert same(got, want), case
    if flags != RXGB:                                   # the reference itself cannot read its RXGB files back as BC3
        md, back = capi.dds_load(got)                  # the reference's file: the same bytes
        hr, rmeta, rback = oracle.dds_load(got)
        assert hr == 0 and [md.width, md.height, md.arraySize, md.mipLevels, md.format, md.miscFlags, md.miscFlags2] == rmeta
        assert same(back, rback)


def test_dds_legacy_flag_failures_match_reference(oracle):
    for fmt, n, misc, flags in [(98, 1, 0, DX9), (95, 1, 0, DX9), (28, 3, 0, DX9), (28, 1, 0, DX9 | DX10)]:
        px = _pixels(fmt, 8, 8, n, 1, 2)
        hr = oracle.dds_save(px, fmt, 8, 8, n, 1, misc, 0, flags)[0]
        with pytest.raises(capi.DxTexError) as e:
            capi.dds_save(px, fmt, 8, 8, n, 1, misc, 0, flags)
        assert e.value.hr == hr == 0x80070052, (fmt, n, hex(flags), hex(hr))      # HRESULT_E_CANNOT_MAKE


def test_dds_ignore_mips_and_errors(oracle):
    px = _pixels(28, 16, 16, 1, 5, 3)
    data = capi.dds_save(px, 28, 16, 16, 1, 5)
    md, top = capi.dds_load(data, IGNORE_MIPS)
    hr, rmeta, rtop = oracle.dds_load(data, IGNORE_MIPS)
    assert hr == 0 and md.mipLevels == 1 == rmeta[3] and same(top, rtop)
    with pytest.raises(capi.DxTexError) as e:
        capi.dds_load(data[:100])
    assert e.value.hr == 0x8007000D                        # HRESULT_E_INVALID_DATA, as the reference (:336-339)
    assert oracle.dds_load(data[:100])[0] == 0x8007000D
    bad = data.copy(); bad[0] = 0
    with pytest.raises(capi.DxTexError) as e:
        capi.dds_load(bad)
    assert e.value.hr == F.E_FAIL and oracle.dds_load(bad)[0] == F.E_FAIL
    with pytest.raises(capi.DxTexError) as e:
        capi.dds_load(data[:-8])                           # truncated pixel data
    assert e.value.hr == 0x80070026 and oracle.dds_load(data[:-8])[0] == 0x80070026


def test_cpp_dds_mirror_round_trip(tmp_path, oracle):
    """SaveToDDSMemory / LoadFromDDSMemory / SaveToDDSFile / LoadFromDDSFile / Blob of the C++ mirror, from a C++ caller
    (no GPU involved); the file it writes is then read by the reference."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "directxtex_b200", "_lib")
    exe = str(tmp_path / "dds_roundtrip")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(root, "directxtex_b200", "host"),
                    os.path.join(root, "tests", "cpp", "dds_roundtrip.cpp"), "-L", libdir, "-ldxtex_b200",
                    "-Wl,-rpath," + libdir, "-o", exe], check=True)
    out = str(tmp_path / "pm.dds")
    r = subprocess.run([exe, out], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr
    hr, meta, pixels = oracle.dds_load(np.fromfile(out, np.uint8))
    assert hr == 0 and meta[:5] == [16, 8, 1, 1, 77] and (meta[6] & 7) == 2          # BC3, premultiplied (DXT4)
    assert same(pixels, (np.arange(pixels.size, dtype=np.uint32) * 13).astype(np.uint8))
