"""Out-of-bounds evidence without compute-sanitizer (closed on the GPU pool): `make bounds` compiles the same sources with
-DB200PC_BOUNDS, which turns every B200PC_DEV_ASSERT (index checks on the device, csrc/common.cuh) into a trap.
tools/bounds_sweep.py drives every kernel family through small, ragged, tied, split, non-finite and forced-variant shapes
against that build in a child process; a violated check kills the child with a CUDA error."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "point-cloud-interpolation-_b200")
BOUNDS_LIB = os.path.join(PKG, "b200pc", "libb200pc_bounds.so")


@pytest.mark.gpu
def test_every_kernel_family_under_the_bounds_checked_build():
    assert os.path.exists(BOUNDS_LIB), "libb200pc_bounds.so is not built (make -C point-cloud-interpolation-_b200 bounds)"
    env = dict(os.environ, B200PC_LIBRARY="bounds")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bounds_sweep.py")], env=env, capture_output=True, text=True, timeout=900)
    out = p.stdout + p.stderr
    assert "library: libb200pc_bounds.so" in out, out[-2000:]
    assert "device assert failed" not in out, out[-4000:]
    assert p.returncode == 0 and "bounds sweep ok" in out, out[-4000:]


@pytest.mark.gpu
def test_a_violated_check_traps_the_launch():
    """the checks are live: b200pc_fma_peak launched with an index its check rejects (B200PC_BOUNDS_TRIP=1) must fail loudly
    under the bounds build and run normally under the shipped one"""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import torch; from b200pc import ops; "
            "print(ops.fma_peak(1 << 10)); torch.cuda.synchronize(); print('survived')") % (ROOT, PKG)
    bad = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, B200PC_LIBRARY="bounds", B200PC_BOUNDS_TRIP="1"),
                         capture_output=True, text=True, timeout=300)
    assert bad.returncode != 0 and "device assert failed" in bad.stdout + bad.stderr, (bad.stdout + bad.stderr)[-2000:]
    shipped = {k: v for k, v in os.environ.items() if k != "B200PC_LIBRARY"}     # also when the suite itself runs the bounds build
    ok = subprocess.run([sys.executable, "-c", code], env=dict(shipped, B200PC_BOUNDS_TRIP="1"), capture_output=True, text=True, timeout=300)
    assert ok.returncode == 0 and "survived" in ok.stdout, (ok.stdout + ok.stderr)[-2000:]


def test_bounds_build_has_the_checks_and_the_shipped_library_does_not():
    """CPU: the asserts exist in the bounds build only (the shipped library pays nothing for them)"""
    shipped = os.path.join(PKG, "b200pc", "libb200pc.so")
    if not (os.path.exists(BOUNDS_LIB) and os.path.exists(shipped)):
        pytest.skip("libraries not built")
    needle = b"b200pc device assert failed"
    assert needle in open(BOUNDS_LIB, "rb").read()
    assert needle not in open(shipped, "rb").read()
    import ctypes
    lib = ctypes.CDLL(BOUNDS_LIB)
    from b200pc import _lib
    for name in _lib.SIGNATURES:
        assert hasattr(lib, name), name
