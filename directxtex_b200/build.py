"""Build libdxtex_b200.so (CUDA kernels + C ABI) in-tree for sm_100a.

nvcc cross-compiles without a GPU.  Numeric contract of the build (DESIGN.md):
  -fmad=false            no multiply-add contraction: the BC1-5 / convert / mip kernels must be
                         bit-exact against the reference CPU build (which has no FMA either)
  (default) -prec-div=true -prec-sqrt=true, no --use_fast_math
  -Xcompiler -ffp-contract=off   same for the host code that builds the triangle-filter tables
"""
import os, subprocess, sys, shutil

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
OUT = os.path.join(OUT_DIR, "libdxtex_b200.so")
SOURCES = [os.path.join(CSRC, f) for f in ("dxb_api.cu", "dxb_k_bc7.cu", "dxb_k_bc6h.cu", "dxb_k_bc15.cu", "dxb_k_decode.cu", "dxb_k_rows.cu", "dxb_k_analyze.cu")]
HOST_SOURCES = [os.path.join(HERE, "host", "DirectXTexB200.cpp"), os.path.join(HERE, "host", "dxb_dds.cpp")]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _deps():
    deps = list(SOURCES) + [os.path.join(HERE, "..", "include", "dxtex_b200.h")]
    for root in (CSRC, os.path.join(HERE, "host")):
        if os.path.isdir(root):
            deps += [os.path.join(root, f) for f in os.listdir(root)]
    return deps


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in _deps() if os.path.exists(d))


def _flags():
    return ["-std=c++17", "-O3", "-lineinfo",
            "-gencode", "arch=compute_100a,code=sm_100a",
            "-fmad=false",
            "-Xcompiler", "-fPIC,-ffp-contract=off,-fvisibility=hidden",
            "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++",
            "-I", os.path.join(HERE, "..", "include"), "-I", CSRC, "-DDXB_BUILDING_LIB"]


def build_variant(tag, defines, only=("dxb_k_bc7.cu",)):
    """Experiment helper: rebuild the TUs in `only` with extra -D flags and link _lib/variants/libdxtex_b200_<tag>.so
    (all other objects are reused from the main build)."""
    vdir = os.path.join(OUT_DIR, "variants")
    os.makedirs(vdir, exist_ok=True)
    build()
    nvcc = _nvcc()
    objs = []
    for src in SOURCES + [s for s in HOST_SOURCES if os.path.exists(s)]:
        base = os.path.splitext(os.path.basename(src))[0]
        if os.path.basename(src) in only:
            obj = os.path.join(vdir, base + "_" + tag + ".o")
            r = subprocess.run([nvcc] + _flags() + list(defines) + ["-c", src, "-o", obj], capture_output=True, text=True)
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("variant build failed")
        else:
            obj = os.path.join(OUT_DIR, base + ".o")
        objs.append(obj)
    out = os.path.join(vdir, "libdxtex_b200_%s.so" % tag)
    r = subprocess.run([nvcc, "-shared", "-cudart", "static", "-ccbin", "/usr/bin/g++", "-o", out] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("variant link failed")
    return out


def build(force=False, verbose=False):
    """Compile each translation unit (in parallel, only the stale ones) and link libdxtex_b200.so."""
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OUT_DIR, exist_ok=True)
    srcs = SOURCES + [s for s in HOST_SOURCES if os.path.exists(s)]
    import re

    def dep_time(path, seen=None):
        """newest mtime of `path` and every local header it includes (recursively)"""
        seen = seen if seen is not None else set()
        if path in seen or not os.path.exists(path):
            return 0.0
        seen.add(path)
        t = os.path.getmtime(path)
        for inc in re.findall(r'#include\s+"([^"]+)"', open(path).read()):
            for base in (os.path.dirname(path), CSRC, os.path.join(HERE, "..", "include")):
                cand = os.path.normpath(os.path.join(base, inc))
                if os.path.exists(cand):
                    t = max(t, dep_time(cand, seen))
                    break
        return t
    objs, todo = [], []
    for src in srcs:
        obj = os.path.join(OUT_DIR, os.path.splitext(os.path.basename(src))[0] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < dep_time(src):
            todo.append((src, obj))
    if not todo and os.path.exists(OUT) and not force:
        return OUT
    nvcc = _nvcc()

    def cc(job):
        src, obj = job
        cmd = [nvcc] + _flags() + (["-Xptxas=-v"] if verbose else []) + ["-c", src, "-o", obj]
        return src, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=4) as ex:
        for src, r in ex.map(cc, todo):
            if verbose or r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on " + src)
    r = subprocess.run([nvcc, "-shared", "-cudart", "static", "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++",
                        "-o", OUT] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
