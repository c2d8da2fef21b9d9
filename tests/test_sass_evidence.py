"""Static evidence that the built library is Blackwell-native (no GPU needed): the SASS of
liblogreg_b200.so contains the tcgen05 / TMEM / TMA instructions of the many-chain kernel and the
128-bit streaming loads of the fused kernel."""
import os
import re
import shutil
import subprocess

import pytest


def cuobjdump():
    """cuobjdump from PATH, else the one installed beside the nvcc the library is built with."""
    from logreg_b200 import build
    try:
        path = shutil.which("cuobjdump") or os.path.join(os.path.dirname(build.nvcc_path()), "cuobjdump")
    except RuntimeError:
        return None
    return path if os.path.exists(path) else None


@pytest.mark.skipif(cuobjdump() is None, reason="cuobjdump not available")
def test_sass_contains_tcgen05_tmem_tma_and_vector_loads():
    from logreg_b200 import _native as N
    N.load()
    sass = subprocess.run([cuobjdump(), "-sass", N.library_path()], capture_output=True, text=True, timeout=600).stdout
    assert "sm_100a" in sass or "SM100" in sass.upper() or "EF_CUDA_SM100" in sass
    count = lambda pat: len(re.findall(pat, sass))
    assert count(r"\bUTCHMMA\b") >= 48          # tcgen05.mma.kind::tf32 (3xTF32: 24 + 24 per tile)
    assert count(r"\bLDTM\b") >= 2 and count(r"\bSTTM\b") >= 2   # tcgen05.ld / tcgen05.st
    assert count(r"\bUTMALDG\b") >= 2           # cp.async.bulk.tensor (TMA tile loads, two swizzles)
    assert count(r"\bUBLKCP\b") >= 1            # cp.async.bulk (the y bytes)
    assert count(r"LDG\.E\.NA\.128\.CONSTANT") >= 100   # ld.global.nc.L1::no_allocate.v4 / .v2.f64 streaming loads
    assert "HGMMA" not in sass and "wgmma" not in sass   # nothing Hopper-only slipped in
