"""BC7 / BC6H tolerance contract (tests/tolerance.py) for the host lock-step emulator of the CUDA encoders, on every content
class of the corpus at 256x256, against tests/golden/golden_bc67_v2.npz (per-block errors of the unmodified reference
encoder, tests/golden/make_golden_bc67.py).  The GPU suite checks that the device output is bit-identical to the emulator's
on the same inputs and re-checks the contract on the device output."""
import numpy as np
import pytest

from directxtex_b200 import synth
from tests import tolerance


@pytest.mark.parametrize("kind,flags", tolerance.bc7_cases())
def test_bc7_contract_per_class(emul, kind, flags):
    img = synth.content_ldr(kind, tolerance.SIZE, tolerance.SIZE, tolerance.SEED)
    he, blocks = emul.compress(img, tolerance.SIZE, tolerance.SIZE, 2, 98, flags)
    assert he == 0
    ratio, bad = tolerance.check_bc7(emul, kind, flags, blocks)
    print("bc7 %-13s ratio %.4f  blocks > 2x+16: %.2f%%" % (kind, ratio, 100 * bad))


@pytest.mark.parametrize("kind,fmt", tolerance.bc6h_cases())
def test_bc6h_contract_per_class(emul, kind, fmt):
    img = synth.content_hdr(kind, tolerance.SIZE, tolerance.SIZE, tolerance.SEED)
    he, blocks = emul.compress(img, tolerance.SIZE, tolerance.SIZE, 2, fmt, 0)
    assert he == 0
    ratio, bad, fratio = tolerance.check_bc6h(emul, kind, fmt, blocks)
    print("bc6h %-13s %d ratio %.4f  blocks > 2x+768: %.2f%%  float mse ratio %.3f" % (kind, fmt, ratio, 100 * bad, fratio))


def test_golden_is_the_reference(oracle):
    """the recorded reference answers give finite per-block BC7 errors (the measure the golden's tolerance anchors are stored in)"""
    kind = "text"
    img = synth.content_ldr(kind, 64, 64, tolerance.SEED)
    hr, sse = oracle.bc7_block_sse(img, 64, 64, 0, full=True)
    assert hr == 0 and np.isfinite(sse).all()
