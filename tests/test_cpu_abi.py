"""CPU suite: the C++ mirror against the reference's OWN public header.
(1) tests/cpp/abi_probe.cpp is compiled against directxtex_b200/host/DirectXTexB200.h: sizeof / offsetof of Image, TexMetadata, ScratchImage,
    Blob, CompressOptions, ConvertOptions and the values of every public enumerator the path uses must print what the same probe prints
    compiled against the reference's DirectXTex.h (through oracle/compat).
(2) the mangled symbols libdxtex_b200.so exports for the mirrored functions must be exported by the reference build
    (oracle/_ref/libdxtex_ref.so) under exactly the same name, i.e. the signatures match the reference's.
The reference side is the committed snapshots under tests/golden/.  With DXB_REFERENCE_SRC=<the reference's DirectXTex directory> (and
oracle/_ref built from it) the probes are also built against the reference and the snapshots rewritten from them."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("DXB_REFERENCE_SRC", "")
SNAP = os.path.join(ROOT, "tests", "golden", "abi_reference.txt")
SNAP_SYMS = os.path.join(ROOT, "tests", "golden", "abi_reference_symbols.txt")
CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def _probe(tmp_path, reference):
    exe = str(tmp_path / ("probe_ref" if reference else "probe_ours"))
    inc = ["-DPROBE_REFERENCE", "-I", os.path.join(ROOT, "oracle", "compat"), "-I", REF] if reference else ["-I", os.path.join(ROOT, "directxtex_b200", "host")]
    subprocess.run([CXX, "-std=c++17", "-w", "-msse2"] + inc + [os.path.join(ROOT, "tests", "cpp", "abi_probe.cpp"), "-o", exe], check=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def test_struct_layout_and_enumerators_match_the_reference_header(tmp_path):
    ours = _probe(tmp_path, False)
    if os.path.isdir(REF):
        theirs = _probe(tmp_path, True)
        if not os.path.exists(SNAP) or open(SNAP).read() != theirs:
            open(SNAP, "w").write(theirs)               # snapshot for machines without the reference tree (committed)
    else:
        theirs = open(SNAP).read()
    assert ours.splitlines() == theirs.splitlines()


SNAP_FMT = os.path.join(ROOT, "tests", "golden", "format_reference.txt")


def test_format_utilities_answer_like_the_reference_for_every_dxgi_value(tmp_path):
    """tests/cpp/format_probe.cpp prints IsValid / IsCompressed / IsPacked / IsVideo / IsPlanar / IsPalettized / IsDepthStencil / IsSRGB / IsBGR /
    IsTypeless / HasAlpha / BitsPerPixel / BitsPerColor / FormatDataType / Make{SRGB,Linear,Typeless,TypelessUNORM,TypelessFLOAT} / ComputeScanlines for the values
    0..200: linked against the mirror (name-driven classification, DirectXTexB200.cpp) and against the reference build the output is identical."""
    lib_dir = os.path.join(ROOT, "directxtex_b200", "_lib")
    exe = str(tmp_path / "fmt_ours")
    subprocess.run([CXX, "-std=c++17", "-w", "-I", os.path.join(ROOT, "directxtex_b200", "host"), os.path.join(ROOT, "tests", "cpp", "format_probe.cpp"), "-o", exe,
                    os.path.join(lib_dir, "libdxtex_b200.so"), "-Wl,-rpath," + lib_dir], check=True)
    ours = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(REF) and os.path.exists(os.path.join(ref_dir, "libdxtex_ref.so")):
        exe = str(tmp_path / "fmt_ref")
        subprocess.run([CXX, "-std=c++17", "-w", "-msse2", "-DPROBE_REFERENCE", "-I", os.path.join(ROOT, "oracle", "compat"), "-I", REF,
                        os.path.join(ROOT, "tests", "cpp", "format_probe.cpp"), "-o", exe, os.path.join(ref_dir, "libdxtex_ref.so"), "-Wl,-rpath," + ref_dir], check=True)
        theirs = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
        if not os.path.exists(SNAP_FMT) or open(SNAP_FMT).read() != theirs:
            open(SNAP_FMT, "w").write(theirs)            # snapshot for machines without the reference tree (committed)
    else:
        theirs = open(SNAP_FMT).read()
    assert len(ours.splitlines()) == 201
    assert ours.splitlines() == theirs.splitlines()


SNAP_CONT = os.path.join(ROOT, "tests", "golden", "container_reference.txt")


def _linked_probe(tmp_path, source, reference):
    lib_dir = os.path.join(ROOT, "oracle", "_ref") if reference else os.path.join(ROOT, "directxtex_b200", "_lib")
    lib = os.path.join(lib_dir, "libdxtex_ref.so" if reference else "libdxtex_b200.so")
    inc = ["-msse2", "-DPROBE_REFERENCE", "-I", os.path.join(ROOT, "oracle", "compat"), "-I", REF] if reference else ["-I", os.path.join(ROOT, "directxtex_b200", "host")]
    exe = str(tmp_path / (os.path.splitext(source)[0] + ("_ref" if reference else "_ours")))
    subprocess.run([CXX, "-std=c++17", "-w"] + inc + [os.path.join(ROOT, "tests", "cpp", source), "-o", exe, lib, "-Wl,-rpath," + lib_dir], check=True)
    return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def test_scratchimage_constructors_match_the_reference(tmp_path):
    """Initialize1D / 2D / Cube, InitializeFromImage (1D and 2D), InitializeArrayFromImages, InitializeCubeFromImages and OverrideFormat: HRESULTs,
    metadata, per-image layout and a checksum of the copied pixels equal the reference build's (tests/cpp/container_probe.cpp)."""
    ours = _linked_probe(tmp_path, "container_probe.cpp", False)
    if os.path.isdir(REF) and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libdxtex_ref.so")):
        theirs = _linked_probe(tmp_path, "container_probe.cpp", True)
        if not os.path.exists(SNAP_CONT) or open(SNAP_CONT).read() != theirs:
            open(SNAP_CONT, "w").write(theirs)
    else:
        theirs = open(SNAP_CONT).read()
    assert len(ours.splitlines()) > 80 and ours.splitlines() == theirs.splitlines()


SNAP_PITCH = os.path.join(ROOT, "tests", "golden", "pitch_reference.txt.gz")


def test_compute_pitch_with_every_cp_flag_matches_the_reference(tmp_path):
    """ComputePitch over the values 0..200 x 5 sizes x 11 CP_FLAGS settings (alignment, BAD_DXTN_TAILS, forced bits per pixel) and a ScratchImage
    laid out with alignment flags: 11 107 lines identical to the reference build's (tests/cpp/pitch_probe.cpp)."""
    import gzip
    ours = _linked_probe(tmp_path, "pitch_probe.cpp", False)
    if os.path.isdir(REF) and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libdxtex_ref.so")):
        theirs = _linked_probe(tmp_path, "pitch_probe.cpp", True)
        if not os.path.exists(SNAP_PITCH) or gzip.open(SNAP_PITCH, "rt").read() != theirs:
            with gzip.open(SNAP_PITCH, "wt") as f:
                f.write(theirs)
    else:
        theirs = gzip.open(SNAP_PITCH, "rt").read()
    assert len(ours.splitlines()) > 11000 and ours.splitlines() == theirs.splitlines()


def _exports(path):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return {l.split()[-1] for l in out.splitlines() if l.strip()}


MIRRORED = ["Compress", "CompressEx", "Decompress", "Convert", "ConvertEx", "GenerateMipMaps", "Resize", "PremultiplyAlpha",
            "ScaleMipMapsAlphaForCoverage", "ComputePitch", "CalculateMipLevels", "IsCompressed", "IsSRGB", "BitsPerPixel",
            "SaveToDDSMemory", "SaveToDDSFile", "LoadFromDDSMemory", "LoadFromDDSFile", "GetMetadataFromDDSMemory", "GetMetadataFromDDSFile",
            "IsValid", "IsPacked", "IsVideo", "IsPlanar", "IsPalettized", "IsDepthStencil", "IsBGR", "IsTypeless", "HasAlpha", "BitsPerColor", "FormatDataType",
            "ComputeScanlines", "MakeSRGB", "MakeLinear", "MakeTypeless", "MakeTypelessUNORM", "MakeTypelessFLOAT",
            "ScratchImage", "Blob", "TexMetadata"]


def test_exported_cpp_symbols_exist_in_the_reference_build():
    lib = os.path.join(ROOT, "directxtex_b200", "_lib", "libdxtex_b200.so")
    mine = {s for s in _exports(lib) if s.startswith("_ZN7DirectX") or s.startswith("_ZNK7DirectX")}
    assert len(mine) > 40
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libdxtex_ref.so")
    if os.path.isdir(REF) and os.path.exists(ref_so):
        theirs = {s for s in _exports(ref_so) if "7DirectX" in s}
        open(SNAP_SYMS, "w").write("\n".join(sorted(theirs)) + "\n")
    else:
        theirs = set(open(SNAP_SYMS).read().split())
    dem = subprocess.run(["c++filt"], input="\n".join(sorted(mine)), capture_output=True, text=True, check=True).stdout.splitlines()
    missing = [d for s, d in zip(sorted(mine), dem) if s not in theirs]
    # the only symbols the reference build does not export: narrow-character DDS file paths (our addition; the reference is wchar_t
    # only, DirectXTex.h:588-616) and the functions the reference defines inline (DirectXTex.inl:63, 112, 135, 150)
    inline_in_reference = ("DirectX::IsCompressed(DXGI_FORMAT)", "DirectX::IsSRGB(DXGI_FORMAT)", "DirectX::IsValid(DXGI_FORMAT)", "DirectX::IsPalettized(DXGI_FORMAT)",
                           "DirectX::SaveToDDSMemory(DirectX::Image const&, DirectX::DDS_FLAGS, DirectX::Blob&)",
                           "DirectX::SaveToDDSFile(DirectX::Image const&, DirectX::DDS_FLAGS, wchar_t const*)")
    allowed = [m for m in missing if ("char const*" in m and "DDSFile" in m and "wchar_t" not in m) or m in inline_in_reference]
    assert sorted(missing) == sorted(allowed), "exported but not in the reference build (signature differs?):\n" + "\n".join(m for m in missing if m not in allowed)
    # and every mirrored entry point is there at all
    names = " ".join(dem)
    for fn in MIRRORED:
        assert ("DirectX::" + fn) in names, fn
