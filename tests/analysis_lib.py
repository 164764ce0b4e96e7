"""TEST INFRASTRUCTURE for ComputeMSE / IsAlphaAllOpaque: the reference's answers (tests/golden/analysis_calls.npz, replayed through
oracle_lib.Recorded), the reference build that records them (ComputeMSE through oracle/_ref/libdxtex_ref.so, ScratchImage::IsAlphaAllOpaque
through tests/cpp/alpha_probe.cpp compiled against the reference's header and linked with that build), the host emulator of the
kernels' arithmetic (tests/emul/analysis_emul.cpp) and the same probe linked with the C++ mirror.  Never imported by the product.

Recording: DXB_RECORD_ANALYSIS=<file> DXB_REFERENCE_SRC=<the reference's DirectXTex directory> python -m pytest tests/test_cpu_analysis.py
(with oracle/_ref built, `make -C oracle`) sends the calls to the reference build and records them into <file>."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from directxtex_b200 import formats as F
from tests import oracle_lib

ROOT = oracle_lib.ROOT
CALLS = os.path.join(ROOT, "tests", "golden", "analysis_calls.npz")
CSRC = os.path.join(ROOT, "directxtex_b200", "csrc")
EMUL_SRC = os.path.join(ROOT, "tests", "emul", "analysis_emul.cpp")
EMUL_SO = os.path.join(ROOT, "tests", "emul", "_build", "libdxb_emul_analysis.so")
PROBE_SRC = os.path.join(ROOT, "tests", "cpp", "alpha_probe.cpp")
CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def _stale(out, srcs):
    return not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs)


def build_emul(out=EMUL_SO):
    """the analysis emulator, with the flags of tests/emul/build.sh; into a temporary directory when the tree is not writable"""
    srcs = [EMUL_SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if not _stale(out, srcs):
        return out
    try:
        os.makedirs(os.path.dirname(out), exist_ok=True)
        probe = open(out + ".tmp", "w")
        probe.close()
        os.remove(out + ".tmp")
    except OSError:
        out = os.path.join(tempfile.mkdtemp(prefix="dxb_emul_"), os.path.basename(out))
    subprocess.run([CXX, "-std=c++17", "-O2", "-msse2", "-mfpmath=sse", "-mfma", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-x", "c++",
                    "-I", CSRC, EMUL_SRC, "-o", out], check=True)
    return out


def build_probe(reference):
    """tests/cpp/alpha_probe.cpp as a shared library linked with the reference build (reference=True) or with libdxtex_b200.so"""
    out = os.path.join(tempfile.mkdtemp(prefix="dxb_probe_"), "libalpha_probe_%s.so" % ("ref" if reference else "ours"))
    if reference:
        ref_dir, ref_src = os.path.join(ROOT, "oracle", "_ref"), os.environ.get("DXB_REFERENCE_SRC", "")
        inc = ["-msse2", "-DPROBE_REFERENCE", "-I", os.path.join(ROOT, "oracle", "compat"), "-I", ref_src]
        lib = [os.path.join(ref_dir, "libdxtex_ref.so"), "-Wl,-rpath," + ref_dir]
    else:
        lib_dir = os.path.join(ROOT, "directxtex_b200", "_lib")
        inc = ["-I", os.path.join(ROOT, "directxtex_b200", "host")]
        lib = [os.path.join(lib_dir, "libdxtex_b200.so"), "-Wl,-rpath," + lib_dir]
    subprocess.run([CXX, "-std=c++17", "-O1", "-w", "-fPIC", "-shared"] + inc + [PROBE_SRC, "-o", out] + lib, check=True)
    return out


class Probe:
    """ScratchImage::IsAlphaAllOpaque and ComputeMSE of one DirectXTex build (the reference's or the C++ mirror)"""

    def __init__(self, path):
        L = self.L = C.CDLL(path)
        sz, u32, vp = C.c_size_t, C.c_uint32, C.c_void_p
        L.probe_is_alpha_all_opaque.argtypes = [vp, sz, u32, sz, sz, sz, sz, C.POINTER(C.c_int32)]
        L.probe_compute_mse.argtypes = [vp, u32, vp, u32, sz, sz, u32, vp]
        L.probe_is_alpha_all_opaque.restype = L.probe_compute_mse.restype = C.c_int32

    def compute_mse(self, a, fmt_a, b, fmt_b, w, h, flags=0):
        """DirectX::ComputeMSE of two tightly packed images: (hr, float32[5] = mse, mseV[0..3])"""
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        out = np.zeros(5, np.float32)
        hr = self.L.probe_compute_mse(a.ctypes.data, fmt_a, b.ctypes.data, fmt_b, w, h, flags, out.ctypes.data)
        return F.hr_u32(hr), out

    def is_alpha_all_opaque(self, pixels, fmt, w, h, array_size=1, mip_levels=1):
        """ScratchImage::IsAlphaAllOpaque of a 2D texture packed in ScratchImage order: (hr, 1 / 0)"""
        pixels = np.ascontiguousarray(pixels).view(np.uint8).reshape(-1)
        v = C.c_int32(-1)
        hr = self.L.probe_is_alpha_all_opaque(pixels.ctypes.data, pixels.size, fmt, w, h, array_size, mip_levels, C.byref(v))
        return F.hr_u32(hr), v.value


class AnalysisEmul:
    def __init__(self, path):
        L = self.L = C.CDLL(path)
        sz, u32, vp = C.c_size_t, C.c_uint32, C.c_void_p
        L.emul_compute_mse.argtypes = [vp, u32, sz, vp, u32, sz, sz, sz, u32, vp]
        L.emul_is_alpha_all_opaque.argtypes = [vp] + [C.POINTER(sz)] * 4 + [sz, u32, C.POINTER(C.c_int32)]

    def compute_mse(self, a, fmt_a, b, fmt_b, w, h, flags=0, pitch_a=0, pitch_b=0):
        """the emulated ComputeMSE (same tile arithmetic and fp64 tree as the kernels): (hr, float32[5] = mse, mseV[0..3])"""
        a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
        out = np.zeros(5, np.float32)
        hr = self.L.emul_compute_mse(a.ctypes.data, fmt_a, pitch_a, b.ctypes.data, fmt_b, pitch_b, w, h, flags, out.ctypes.data)
        return F.hr_u32(hr), out

    def is_alpha_all_opaque(self, pixels, layout, fmt):
        """the emulated scan of the images at the (offset, w, h, rowPitch, slicePitch) entries of `layout`: (hr, 1 / 0)"""
        pixels = np.ascontiguousarray(pixels).view(np.uint8).reshape(-1)
        A = C.c_size_t * len(layout)
        off, ws, hs, ps = A(*[l[0] for l in layout]), A(*[l[1] for l in layout]), A(*[l[2] for l in layout]), A(*[l[3] for l in layout])
        v = C.c_int32(-1)
        hr = self.L.emul_is_alpha_all_opaque(pixels.ctypes.data, off, ws, hs, ps, len(layout), fmt, C.byref(v))
        return F.hr_u32(hr), v.value


def load_reference_answers():
    """Recorded answers, or a Recorder on the reference build when DXB_RECORD_ANALYSIS names the file to record into"""
    if os.environ.get("DXB_RECORD_ANALYSIS"):
        oracle_lib.build_ref()
        return oracle_lib.Recorder(Probe(build_probe(True)))
    return oracle_lib.Recorded(CALLS)


@pytest.fixture(scope="session")
def analysis_oracle():
    ref = load_reference_answers()
    yield ref
    if isinstance(ref, oracle_lib.Recorder):
        ref.save(os.environ["DXB_RECORD_ANALYSIS"])


@pytest.fixture(scope="session")
def analysis_emul():
    return AnalysisEmul(build_emul())
