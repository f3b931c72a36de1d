"""CPU: the drop-in claim checked against the reference's own sources.  integration/shim/ replaces the
reference's src/core/lib/ibverbs/{pair,poller}.h with forwards to include/b200_pair.h; with it in front of the
include path the reference's endpoint (rdma_bp_posix.cc) and BPEV engine (ev_epollex_rdma_bpev_linux.cc) must
compile UNCHANGED, and every b200_* symbol their objects then need must be exported by libb200rdma.so.
The compile needs the reference source tree; the symbols it yields are stored in tests/golden/ and checked
without it."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
NEEDED = os.path.join(ROOT, "tests", "golden", "reference_needed_b200_symbols.txt")
SHIM = os.path.join(ROOT, "integration", "shim", "src", "core", "lib", "ibverbs")


def stored_needed():
    return [s for s in open(NEEDED).read().splitlines() if s and not s.startswith("#")]


def test_library_exports_what_the_reference_endpoint_and_engine_need(pkg):
    """The entry points the reference's endpoint + engine were compiled to need are forwarded to by the shim
    headers, and every entry point the shim forwards to is exported by libb200rdma.so."""
    needed = stored_needed()
    assert len(needed) == 17
    shim = set()
    for h in ("pair.h", "poller.h"):
        shim.update(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", open(os.path.join(SHIM, h)).read()))
    assert set(needed) <= shim, sorted(set(needed) - shim)
    L = pkg.lib()
    assert not [s for s in sorted(shim) if not hasattr(L, s)]


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "src/core/lib/iomgr")), reason="reference tree not present")
def test_reference_endpoint_and_engine_compile_unchanged_against_the_shim(pkg):
    out = subprocess.run(["make", "-C", os.path.join(ROOT, "integration"), "check"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("compiled unchanged") == 2
    needed = open(os.path.join(ROOT, "integration", "_obj", "needed_b200_symbols.txt")).read().split()
    assert sorted(needed) == sorted(stored_needed())
    # the surface the endpoint + engine + Poller use on a pair (SURVEY.md section 8b)
    for s in ("b200_pair_send", "b200_pair_recv", "b200_pair_has_message", "b200_pair_has_pending_writes",
              "b200_pair_status", "b200_pair_readable", "b200_pair_wakeup_read_fd", "b200_pool_take", "b200_poller_add"):
        assert s in needed, s
    L = pkg.lib()
    assert not [s for s in needed if not hasattr(L, s)]
    # the objects reference the reference's own symbols (they ARE the reference's code), not copies of ours
    nm = subprocess.run(["nm", "-C", os.path.join(ROOT, "integration", "_obj", "rdma_bp_posix.o")],
                        capture_output=True, text=True).stdout
    assert "grpc_rdma_bp_create" in nm and "grpc_fd_set_arg" in nm
