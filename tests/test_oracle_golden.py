"""CPU: pin the plain-C oracle (oracle/rb_oracle.c).

1. against tests/golden/traces.json, generated from the reference's own code
   (tests/golden/make_golden.py);
2. when oracle/_ref exists (built from /root/reference), against the reference itself on
   random traces, state by state, ring image by ring image.
"""
import json
import os

import numpy as np
import pytest

import orlib
import trace

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "traces.json")))


def _ops(raw):
    return [tuple(o) for o in raw]


@pytest.mark.parametrize("name", sorted(GOLDEN["traces"]))
def test_oracle_matches_golden(oracle, name):
    t = GOLDEN["traces"][name]
    recs = trace.run_trace(oracle, t["cap"], _ops(t["ops"]), GOLDEN["max_sge"])
    assert len(recs) == len(t["records"])
    for i, (got, want) in enumerate(zip(recs, t["records"])):
        assert got == want, "trace %s op %d (%s)" % (name, i, want["op"])


GOLDEN_FULL = json.load(open(os.path.join(HERE, "golden", "traces_full.json")))


@pytest.mark.parametrize("name", sorted(GOLDEN_FULL["traces"]))
def test_oracle_matches_golden_full_size(oracle, name):
    """BASELINE size: 16 MiB ring, 4 MiB chttp2-shaped messages, the ring wrapped more than twice."""
    t = GOLDEN_FULL["traces"][name]
    recs = trace.run_trace(oracle, t["cap"], _ops(t["ops"]), GOLDEN_FULL["max_sge"], ring_images=False)
    assert len(recs) == len(t["records"])
    for i, (got, want) in enumerate(zip(recs, t["records"])):
        assert got == want, "trace %s op %d (%s)" % (name, i, want["op"])
    assert sum(r["ret"] for r in recs if r["op"] in ("recv", "recv_drain", "stream")) > 2 * t["cap"]


def test_golden_covers_required_cases():
    names = set(GOLDEN["traces"])
    for need in ["frame_sizes_64k", "max_frames_4k", "wrap_walk_1k", "partial_reads_1k", "max_sge_cut_64k",
                 "zero_len_slice_4k", "credit_2k", "chttp2_300k_128k"]:
        assert need in names
    for t in GOLDEN["traces"].values():
        for r in t["records"]:
            if r["op"] == "stream":
                assert r["intact"]


def test_helpers_known_answers(oracle):
    L = oracle.L
    # SURVEY.md appendix A, observed on the reference build
    assert [L.orb_calc_writable(s) for s in (0, 23, 24, 31, 32, 33, 40, 47, 48)] == [0, 0, 0, 0, 8, 8, 16, 16, 24]
    assert [L.orb_encoded_size(p) for p in (1, 8, 9, 16384)] == [24, 24, 32, 16400]
    assert L.orb_free_size(64, 0, 0) == 64 and L.orb_free_size(64, 8, 0) == 8
    assert L.orb_writable_size(64, 0, 40) == 0 and L.orb_writable_size(64, 0, 8) == 32


def test_appendix_a_read_sequence(oracle):
    """13-byte frame at offset 32 of a 64-byte ring then a 5-byte frame wrapping to 0:
    reads with cap 4,4,32 return 4,4,5 with internal bytes 12,4,16; ring is all zero after."""
    import ctypes as C
    L = oracle.L
    buf = np.zeros(64, dtype=np.uint8)
    ring = orlib.OrbRing()
    L.orb_ring_init(C.byref(ring), buf.ctypes.data, 64)
    ring.head = ring.moving_head = 32

    def frame(p, fill):
        e = np.zeros(16 + (p + 7) // 8 * 8, dtype=np.uint8)
        e[:8] = np.frombuffer(np.uint64(p).tobytes(), dtype=np.uint8)
        e[8:8 + p] = fill
        e[-8:] = 255
        return e

    f1 = frame(13, 7)
    tail = L.orb_ring_place(buf.ctypes.data, 64, 32, f1.ctypes.data, f1.size)
    assert tail == 0
    out = np.zeros(64, dtype=np.uint8)
    internal = C.c_uint64(0)
    res = []
    for cap in (4, 4, 32):
        n = L.orb_ring_read(C.byref(ring), out.ctypes.data, cap, C.byref(internal))
        res.append((n, internal.value, ring.moving_head))
    assert res == [(4, 12, 44), (4, 4, 48), (5, 16, 0)]
    assert not buf.any()


@pytest.mark.skipif(not orlib.ref_available(debug=True), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("seed", range(12))
def test_oracle_matches_reference_random(oracle, seed):
    R = orlib.Ref(debug=True)
    rng = np.random.default_rng(seed)
    cap = [1024, 2048, 4096, 65536][seed % 4]
    ops = []
    for _ in range(120):
        k = rng.integers(0, 5)
        if k < 2:
            n = int(rng.integers(1, 40))
            style = rng.integers(0, 4)
            if style == 0:
                lens = [int(x) for x in rng.integers(1, 64, n)]
            elif style == 1:
                lens = [9 if i % 2 == 0 else int(rng.integers(1, min(16385, cap))) for i in range(n)]
            elif style == 2:
                lens = [int(x) for x in rng.integers(1, 2 * cap, max(1, n // 8))]
            else:
                lens = [int(x) for x in rng.integers(0, 20, n)]
            bidx = int(rng.integers(0, lens[0])) if lens[0] else 0
            ops.append(("send" if k == 0 else "send_all", lens, int(rng.integers(0, 1000)), bidx))
        elif k == 2:
            ops.append(("recv", int(rng.integers(1, cap))))
        else:
            ops.append(("recv_drain", int(rng.integers(1, 2 * cap))))
    a = trace.run_trace(oracle, cap, ops)
    b = trace.run_trace(R, cap, ops)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x == y, "seed %d op %d %s" % (seed, i, ops[i][:1])


def test_reference_status_and_close(oracle):
    """peer_exit half-close (pair.cc:330-337,354-356) behaves the same in port and reference: the statuses and bytes
    asserted here are the reference's, so the port is held to them also where oracle/_ref is not built."""
    engines = [oracle] + ([orlib.Ref(debug=True)] if orlib.ref_available(debug=True) else [])
    for eng in engines:
        a, b = eng.pair_pair(4096)
        assert eng.status(a) == 2 and eng.status(b) == 2
        buf = np.arange(100, dtype=np.uint8)
        assert eng.send(a, [buf]) == 100
        eng.disconnect(a)
        assert eng.status(b) == 3          # kHalfClosed seen by the peer
        assert np.array_equal(eng.recv(b, 1000), buf)   # data already in the ring still drains
        eng.destroy(b)
        if eng is oracle:
            eng.destroy(a)
        else:
            eng.L.ref_pair_destroy(a)
