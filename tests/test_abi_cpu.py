"""CPU: the C-ABI library builds for sm_100a, loads, exports every symbol the header declares,
and refuses to run without a GPU (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re
import subprocess
import sys


def test_library_exports_every_header_symbol(pkg):
    L = pkg.lib()
    syms = pkg.exported_symbols()
    assert len(syms) >= 40
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    # and the binding table covers the header exactly
    assert sorted(pkg._SIGS) == syms


def test_library_is_sm100a_and_has_the_kernels(pkg):
    out = subprocess.run(["cuobjdump", "-lelf", pkg.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out
    sass = subprocess.run(["cuobjdump", "-sass", pkg.LIB_PATH], capture_output=True, text=True).stdout
    for k in ("k_send", "k_recv", "k_poll_scan"):
        assert k in sass
    # bulk traffic is 128-bit vector loads/stores
    assert re.search(r"LDG\.E\.128", sass) and re.search(r"STG\.E\.128", sass)


def test_product_does_not_touch_the_oracle(pkg):
    """The product path must not import, link or call anything under oracle/."""
    root = pkg.ROOT
    for dirpath, _, files in os.walk(os.path.join(root, "grpc-rdma_b200")):
        for f in files:
            if f.endswith((".cu", ".cuh", ".cc", ".h", ".py", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "rb_oracle" not in txt and "liboracle" not in txt and "orlib" not in txt, f
    ldd = subprocess.run(["ldd", pkg.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd


NO_GPU_CHECK = """
import sys
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as ge
pkg = ge.load_package()
L = pkg.lib()
assert L.b200_init(0) == -1
assert b"no CPU fallback" in L.b200_last_error()
assert not L.b200_pool_take(b"x")
try:
    pkg.init(0)
except RuntimeError:
    print("refused")
"""


def test_no_gpu_means_loud_failure(pkg):
    # a child process with every GPU hidden, so that the check also runs on a machine that has one
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", NO_GPU_CHECK, pkg.ROOT], capture_output=True, text=True, env=env,
                         timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.strip() == "refused", out.stdout


def test_workload_shape_helpers(pkg):
    lens = pkg.chttp2_slice_lens(4 * 1024 * 1024)
    assert len(lens) == 514 and lens[0] == 9 and lens[1] == 16384 and lens[-1] == 5
    assert sum(lens[1::2]) == 4 * 1024 * 1024 + 5
    tx, rx = pkg.frame_hbm_bytes([9, 16384])
    assert tx == (9 + 32) + (16384 + 16400) and rx == (32 + 9 + 32) + (16400 + 16384 + 16400)
