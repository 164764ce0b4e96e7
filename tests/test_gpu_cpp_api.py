"""GPU suite: the C++ `namespace DirectX` mirror (directxtex_b200/host) driven by a caller written like a DirectXTex
user's program (tests/cpp/texconv_mini.cpp); outputs compared with the oracle."""
import os
import subprocess

import numpy as np
import pytest

from directxtex_b200 import formats as F, synth
from tests import oracle_lib
from tests.oracle_lib import same, same_concat

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "directxtex_b200", "_lib")


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("cpp") / "texconv_mini")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "directxtex_b200", "host"), "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "texconv_mini.cpp"), "-L", LIBDIR, "-ldxtex_b200",
                    "-Wl,-rpath," + LIBDIR, "-o", out], check=True)
    return out


def run(exe, tmp_path, op, src, w, h, sf, arg, flags=0, items=1, expect_fail=False, env=None):
    fin, fout = str(tmp_path / "in.raw"), str(tmp_path / "out.raw")
    np.ascontiguousarray(src).tofile(fin)
    r = subprocess.run([exe, op, fin, fout, str(w), str(h), str(sf), str(arg), str(flags), str(items)], capture_output=True, text=True,
                       env=dict(os.environ, **(env or {})))
    if expect_fail:
        return r
    assert r.returncode == 0, r.stdout + r.stderr
    return np.fromfile(fout, np.uint8)


def test_cpp_compress_matches_oracle(exe, tmp_path, oracle):
    img = synth.c1_rgba8(96, 64, seed=4)
    for fmt in (71, 77, 83):
        got = run(exe, tmp_path, "compress", img, 96, 64, 28, fmt)
        hr, want = oracle.compress(img, 96, 64, 28, fmt)
        assert hr == 0 and same(got, want)
    got = run(exe, tmp_path, "compress_cb", img, 96, 64, 28, 71)       # status callback: called (0,h) and (h,h)
    hr, want = oracle.compress(img, 96, 64, 28, 71)
    assert same(got, want)


def test_cpp_compress_array_and_errors(exe, tmp_path, oracle):
    rng = np.random.default_rng(3)
    imgs = np.stack([oracle_lib.random_image(28, 32, 16, rng) for _ in range(5)])
    got = run(exe, tmp_path, "compress", imgs, 32, 16, 28, 77, 0, 5)
    want = [oracle.compress(imgs[i], 32, 16, 28, 77)[1] for i in range(5)]
    assert same_concat(got, want, [F.compute_pitch(77, 32, 16)[1]] * 5)
    r = run(exe, tmp_path, "compress", imgs[0], 32, 16, 28, 28, expect_fail=True)          # destination not BC -> E_INVALIDARG
    assert "hr=0x80070057" in r.stdout and r.returncode == 1


def test_cpp_convert_and_mips(exe, tmp_path, oracle):
    rng = np.random.default_rng(5)
    src = oracle_lib.random_image(61, 128, 32, rng)
    got = run(exe, tmp_path, "convert", src, 128, 32, 61, 41)
    hr, want = oracle.convert(src, 128, 32, 61, 41)
    assert hr == 0 and same(got, want)
    src = oracle_lib.random_image(28, 64, 64, rng)
    for fl in (F.TEX_FILTER_BOX, F.TEX_FILTER_CUBIC, 0):
        got = run(exe, tmp_path, "mips", src, 64, 64, 28, fl)
        hr, want = oracle.generate_mipmaps(src, 64, 64, 28, fl)
        assert hr == 0 and same(got, want), hex(fl)


def test_cpp_pipeline_writes_dds_files_the_reference_reads(exe, tmp_path, oracle):
    """mips -> .dds and compress -> .dds through the C++ API (SaveToDDSFile / LoadFromDDSFile, SURVEY 8(f) rank 3): the
    reference's LoadFromDDSMemory must return the same metadata and the pixels the reference computes itself."""
    rng = np.random.default_rng(8)
    src = oracle_lib.random_image(28, 64, 32, rng)
    fin, fout = str(tmp_path / "in.raw"), str(tmp_path / "chain.dds")
    src.tofile(fin)
    r = subprocess.run([exe, "mips", fin, fout, "64", "32", "28", str(F.TEX_FILTER_BOX), "0", "1"], capture_output=True, text=True)
    assert r.returncode == 0 and "dds hr=0x00000000" in r.stdout, r.stdout + r.stderr
    hr, meta, pixels = oracle.dds_load(np.fromfile(fout, np.uint8))
    hr2, want = oracle.generate_mipmaps(src, 64, 32, 28, F.TEX_FILTER_BOX)
    assert hr == 0 and hr2 == 0 and meta[:5] == [64, 32, 1, 7, 28] and same(pixels, want)
    fout = str(tmp_path / "bc3.dds")
    r = subprocess.run([exe, "compress", fin, fout, "64", "32", "28", "77", "0", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    hr, meta, pixels = oracle.dds_load(np.fromfile(fout, np.uint8))
    assert hr == 0 and meta[:5] == [64, 32, 1, 1, 77] and same(pixels, oracle.compress(src, 64, 32, 28, 77)[1])


def test_cpp_status_callback_per_band_and_abort(exe, tmp_path, oracle):
    """CompressEx status callback (DirectXTexCompress.cpp:115-121): called before every band of block rows with (rows done, height),
    monotone, (height, height) at the end; returning false stops the call between bands with E_ABORT."""
    img = synth.c1_rgba8(4096, 4096, seed=6)           # 64 MiB: several 32 MiB bands
    r = run(exe, tmp_path, "compress_cb", img, 4096, 4096, 28, 71, expect_fail=True)
    assert r.returncode == 0, r.stdout + r.stderr
    calls = int(r.stdout.split("callbacks=")[1].split()[0])
    assert calls >= 3 and "last=4096" in r.stdout, r.stdout          # one call per band of ~32 MiB + the final (height, height)
    got = np.fromfile(str(tmp_path / "out.raw"), np.uint8)
    hr, want = oracle.compress(img, 4096, 4096, 28, 71)
    assert hr == 0 and same(got, want)
    r = run(exe, tmp_path, "compress_cb", img, 4096, 4096, 28, 71, expect_fail=True, env={"TEXCONV_MINI_ABORT_AT": "2"})
    assert "hr=0x80004004" in r.stdout and r.returncode == 1, r.stdout          # E_ABORT


def test_cpp_array_compress_uses_every_initialised_gpu(exe, tmp_path, oracle):
    """DirectX::Compress(array) from a C++ caller after dxb200_init_devices: contiguous image ranges per GPU, same bytes as one GPU."""
    from directxtex_b200 import capi
    rng = np.random.default_rng(13)
    imgs = np.stack([oracle_lib.random_image(28, 256, 128, rng) for _ in range(25)])      # 3 n + 1 images for up to 8 GPUs
    want = [oracle.compress(imgs[i], 256, 128, 28, 77)[1] for i in range(len(imgs))]
    one = synth.c1_rgba8(4096, 4096, seed=7)           # one large image: its bands are spread over the GPUs
    hr, want_one = oracle.compress(one, 4096, 4096, 28, 71)
    n = capi.lib.dxb200_device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    imgs = imgs[:3 * n + 1]
    devs = ",".join(str(i) for i in range(n))
    got = run(exe, tmp_path, "compress", imgs, 256, 128, 28, 77, 0, len(imgs), env={"TEXCONV_MINI_DEVICES": devs})
    assert same_concat(got, want[:len(imgs)], [F.compute_pitch(77, 256, 128)[1]] * len(imgs))
    got = run(exe, tmp_path, "compress", one, 4096, 4096, 28, 71, env={"TEXCONV_MINI_DEVICES": devs})
    assert hr == 0 and same(got, want_one)
