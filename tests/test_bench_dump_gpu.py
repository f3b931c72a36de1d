"""GPU: `bench.py --dump-outputs DIR` saves what the last timed step delivered, and that is the payload bench.py
sent: per-connection byte counts plus a fixed sample of the delivered bytes, all float32 / float64."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_step(pkg, tmp_path):
    conns, msg, warmup, steps = 4, 65536, 3, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                          "--conns", str(conns), "--msg-bytes", str(msg), "--ring-kb", "1024", "--no-e2e", "--no-unary",
                          "--no-endpoint", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    d = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert sorted(d) == ["delivered_sample", "delivered_sample_index", "recv_bytes", "send_bytes"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    total = sum(pkg.chttp2_slice_lens(msg))
    assert d["send_bytes"].tolist() == [total] * conns and d["recv_bytes"].tolist() == [total] * conns
    # bench.py's payload: byte j of connection c is ((j * 2654435761) >> 11) + 131 c (mod 256); steps alternate it
    # with the same bytes XOR 0x5A, and the last timed step is step number W + steps - 1 (counted from 0), W being the
    # warm-up steps bench.py ran and reports (it runs at least 3 whatever --warmup asks for)
    f = d["delivered_sample_index"].astype(np.int64)
    c, j = f // total, f % total
    want = ((((j * 2654435761) >> 11) & 255) + 131 * c) & 255
    if (line["warmup"] + line["steps"] - 1) & 1:
        want ^= 0x5A
    assert f.size > 0 and np.array_equal(d["delivered_sample"], want.astype(np.float32))
