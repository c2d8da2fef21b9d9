"""The C-ABI library loads on a CPU-only box, exports every symbol include/logreg_b200.h
declares, and refuses to compute without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "logreg_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lrb_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    from logreg_b200 import _native as N
    lib = N.load()
    names = declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    # the ctypes table covers the header exactly (nothing bound that is not declared, and vice versa)
    assert sorted(N.SIGNATURES) == names
    assert lib.lrb_abi_version() == 2


def test_struct_layouts_match_header():
    from logreg_b200 import _native as N
    # lrb_sampler_params: int32 int32 double ptr uint64 int32 int32 double int64 = 56 bytes on LP64 (ABI 2 added t0)
    assert C.sizeof(N.SamplerParams) == 56
    assert N.SamplerParams.scale.offset == 16 and N.SamplerParams.flags.offset == 36 and N.SamplerParams.init_lpost.offset == 40
    assert N.SamplerParams.t0.offset == 48
    # lrb_info: int64 + 8*int32 + 3*int64 = 64 bytes
    assert C.sizeof(N.Info) == 64 and N.Info.bytes_per_eval.offset == 40


def test_key_child_is_host_arithmetic_and_matches_the_philox_spec():
    """lrb_key_child (the split of the keyed front-end) needs no GPU and equals words (x, y) of
    Philox4x32-10 at counter (i_lo, i_hi, 0, 4) under the parent key."""
    from logreg_b200 import _native as N
    from tests.test_host_logic import philox_ref
    lib = N.load()
    for key in (0, 42, 0xDEADBEEFCAFEF00D, 2 ** 64 - 1):
        for i in (0, 1, 7, 2 ** 32 + 5):
            r = philox_ref([i & 0xFFFFFFFF, i >> 32, 0, 4], [key & 0xFFFFFFFF, key >> 32])
            assert lib.lrb_key_child(key, i) == ((r[1] << 32) | r[0])
    import logreg_b200.jaxlike as J
    assert J.split(42, 4) == [lib.lrb_key_child(42, i) for i in range(4)]


NO_GPU_CHECK = """
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import pytest
import logreg_b200 as lr
from logreg_b200 import _native as N
try:
    have = N.device_count() > 0
except lr.LogregB200Error as e:
    have = False
    assert e.code == N.E_NO_DEVICE
    assert "no CPU fallback" in str(e)
assert not have
with pytest.raises(lr.LogregB200Error):
    lr.Problem(0)
with pytest.raises(lr.LogregB200Error):
    lr.bind_data(np.ones((4, 2)), np.zeros(4, dtype=np.float32))
with pytest.raises(lr.LogregB200Error, match="bind_data"):
    lr.use(None)
    lr.lpost(np.zeros(2))
print("NO_GPU_OK")
"""


def test_no_gpu_means_loud_failure():
    """On a box without a CUDA device the product path must raise, not fall back.  Runs in a child
    process that sees no device (CUDA_VISIBLE_DEVICES empty), so it also runs where a GPU is present."""
    import subprocess
    import sys
    from logreg_b200 import _native as N
    N.load()
    r = subprocess.run([sys.executable, "-c", NO_GPU_CHECK, ROOT], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and "NO_GPU_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_product_code_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under logreg_b200/ may import or call it."""
    pkg = os.path.join(ROOT, "logreg_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.lower().replace("# oracle", ""), os.path.join(dirpath, f)


def test_header_is_plain_c_and_links(tmp_path):
    """The ABI header compiles as strict C99 and the demo links against the library (no run:
    running needs a GPU)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    from logreg_b200 import _native as N
    N.load()
    libdir = os.path.dirname(N.library_path())
    exe = tmp_path / "c_abi_demo"
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-o", str(exe), "-L", libdir, "-llogreg_b200",
           f"-Wl,-rpath,{libdir}", "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    # without a GPU the demo must fail loudly through the error convention, not crash
    try:
        have_gpu = N.device_count() > 0
    except Exception:
        have_gpu = False
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    if have_gpu:
        assert run.returncode == 0 and "lpost" in run.stdout, run.stderr
    else:
        assert run.returncode == 1 and "no CUDA device" in run.stderr


def test_newton_cholesky_solve_on_the_host():
    """lrb_map's Cholesky solve is __host__ __device__ code: check it here against NumPy
    (A + diag(pscale^-2)) step = g, and its not-positive-definite report."""
    from logreg_b200 import _native as N
    lib = N.load()
    rs = np.random.RandomState(0)
    for p in (1, 2, 8, 64, 130):
        M = rs.randn(p + 5, p)
        A = M.T @ M
        ps = 0.5 + rs.rand(p)
        g = rs.randn(p)
        ld = p + 3
        buf = np.zeros((p, ld))
        buf[:, :p] = A
        step = np.zeros(p)
        rc = lib.lrb_debug_chol_solve(N.as_dp(buf), ld, p, N.as_dp(ps), N.as_dp(g), N.as_dp(step))
        assert rc == 0
        np.testing.assert_allclose(step, np.linalg.solve(A + np.diag(1 / ps ** 2), g), rtol=1e-9, atol=1e-12)
    bad = np.array([[1.0, 2.0], [2.0, 1.0]]) - np.eye(2)      # minus the prior term: indefinite
    step = np.zeros(2)
    assert lib.lrb_debug_chol_solve(N.as_dp(bad), 2, 2, N.as_dp(np.ones(2)), N.as_dp(np.ones(2)), N.as_dp(step)) == 2
