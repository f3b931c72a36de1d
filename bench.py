#!/usr/bin/env python
"""bench.py -- streaming throughput of the RDMA_BPEV endpoint hot path on B200.

Workload (BASELINE.json configs[1]): 256 connections, 16 MiB HBM ring per connection
(GRPC_RDMA_RING_BUFFER_SIZE_KB=16384), one 4 MiB gRPC message per connection per step,
handed to the endpoint the way chttp2 does (alternating 9-byte DATA-frame headers and
<=16384-byte payload slices, 5-byte gRPC prefix).  One step = every connection's message
gathered/encoded into the peer ring (k_send) and deframed/scattered/cleared out of it
(k_recv), loopback wire on one GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]
    torchrun ... bench.py --gpus N ...          (one rank per GPU, connections sharded, weak scaling)
    python bench.py --impl reference ...        (the reference's own CPU code on the host cores)
    python bench.py --dump-outputs DIR ...      (also save what the last timed step delivered, as .npy)

Prints ONE JSON line (see DESIGN.md "Measurement").
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the source tree, bytecode caches included

MSG_BYTES = 4 * 1024 * 1024
RING_KB = 16384
CONNS = 256


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--conns", type=int, default=CONNS)
    ap.add_argument("--msg-bytes", type=int, default=MSG_BYTES)
    ap.add_argument("--ring-kb", type=int, default=RING_KB)
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 8)")
    ap.add_argument("--e2e-mode", default="staged", choices=["auto", "zerocopy", "staged"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU-baseline sample length")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-unary", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--hugepages", action="store_true", help="e2e host buffers: THP + b200_mem_register_host instead of "
                    "b200_mem_alloc_host (measured at N=2: 76.6 vs 75.3 GB/s -- not the limiter)")
    ap.add_argument("--no-endpoint", action="store_true", help="skip the e2e_endpoint leg")
    ap.add_argument("--no-nvlink", action="store_true", help="skip the NVLink-wire integrity pass of N >= 2 runs")
    ap.add_argument("--endpoint-threads", type=int, default=8, help="client/server thread pairs of the endpoint leg")
    ap.add_argument("--endpoint-msgs", type=int, default=16)
    ap.add_argument("--endpoint-pool", type=int, default=128, help="pool CTAs of the service during the endpoint leg")
    ap.add_argument("--msgs-per-step", type=int, default=1, help="experiment: messages per connection per step")
    ap.add_argument("--unary-bytes", type=int, default=1024)
    ap.add_argument("--unary-iters", type=int, default=2000)
    ap.add_argument("--service-workers", type=int, default=16)
    ap.add_argument("--stagger", type=int, default=0, help="1 = de-correlate the connections' ring positions first")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step delivered (rank 0) to "
                    "DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm only")
    return args


# ----------------------------------------------------------------------------- clocks

class ClockSampler:
    """nvidia-smi sampled DURING the timed regions (B200_PROFILING.md clocks line).  The device-resident
    timed region of the default run lasts ~0.1 s, so the sampler runs at 20 ms from before the warm-up to
    after the e2e region and every row carries its own timestamp; `window(t0, t1)` reports the rows that
    fall inside one timed region (wall clock)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                ts = datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = time.time()
            self.rows.append((ts, r[1:]))

    def stop(self):
        if not self.proc:
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()

    def window(self, t0, t1, label):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if not (t0 - 0.02 <= ts <= t1 + 0.02):
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "region": label}


# ------------------------------------------------------------------------ CPU baseline

def cpu_engine():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orlib
    if orlib.ref_available(debug=False):
        return orlib.Ref(debug=False), "reference"
    return orlib.Oracle(), "port"


def usable_cpus():
    """Host threads this process may really use: the affinity mask, capped by a cgroup CPU quota if there is one
    (os.cpu_count() reports the machine, not the container)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_sample(eng, lens, conns, ring_bytes, threads, msgs, warm=1):
    t, delivered, _ = eng.bench_stream(conns, threads, warm, msgs, ring_bytes, lens)
    return t, delivered


def host_mem_gb():
    try:
        import psutil
        return psutil.virtual_memory().available / 2**30
    except Exception:
        return 32.0


def cpu_conns_that_fit(conns, ring_bytes, msg_total, kind):
    # per connection: 2 pairs x (ring + ring/2 staging [+ 1 KiB zero-copy buf]) + src + dst
    per = 2 * (ring_bytes + ring_bytes // 2) + 2 * msg_total + (1 << 20)
    fit = int(host_mem_gb() * 0.6 * 2**30 // per)
    return max(1, min(conns, fit))


def run_cpu_baseline(args, lens, payload_per_msg, seconds):
    eng, kind = cpu_engine()
    cores = usable_cpus()
    ring = args.ring_kb * 1024
    conns = cpu_conns_that_fit(args.conns, ring, sum(lens), kind)
    threads = min(cores, conns)
    t1, _ = cpu_sample(eng, lens, conns, ring, threads, 1)  # calibration pass (also warms the allocator)
    msgs = int(max(1, min(64, seconds / max(t1, 1e-3))))
    t, delivered = cpu_sample(eng, lens, conns, ring, threads, msgs)
    nmsg = conns * msgs
    gbs = nmsg * payload_per_msg / t / 1e9
    return {"value": gbs, "unit": "GB/s", "cores": threads, "kind": kind, "msgs_per_s": nmsg / t,
            "sample": "%d conns x %d msgs of %d B (chttp2-shaped, ring %d KiB), %.2f s, %d threads of %d cores"
                      % (conns, msgs, payload_per_msg, args.ring_kb, t, threads, cores)}


def bench_config(conns, msg_bytes, ring_kb):
    """The workload both arms are timed on, spelled identically in both JSON lines (BASELINE configs[1])."""
    return {"workload": "configs[1]: streaming, %d connections per GPU x %d-byte chttp2-shaped messages, ring %d KiB"
                        % (conns, msg_bytes, ring_kb),
            "connections": conns, "message_bytes": msg_bytes, "ring_kb": ring_kb,
            "l2": "inputs larger than the cache (every step streams %.2f GiB of slices through %.1f GiB of rings, "
                  "no reuse between steps)" % (conns * (msg_bytes + 4626) / 2**30, conns * ring_kb / 2**20)}


def reference_arm(args):
    """--impl reference: the reference's own CPU path (oracle/_ref when built, else the port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    pkg = ge.load_package()
    lens = pkg.chttp2_slice_lens(args.msg_bytes)
    eng, kind = cpu_engine()
    cores = usable_cpus()
    ring = args.ring_kb * 1024
    conns = cpu_conns_that_fit(args.conns, ring, sum(lens), kind)
    threads = min(cores, conns)
    # one "step" = one message on every connection, like the B200 arm; W untimed + K timed steps
    # in ONE run of the multi-threaded harness (pairs are set up once, outside the timed region)
    steps_done = args.steps
    t_total, _ = cpu_sample(eng, lens, conns, ring, threads, steps_done, warm=max(1, args.warmup))
    n_total = conns * steps_done
    gbs = n_total * args.msg_bytes / t_total / 1e9
    line = {
        "impl": "reference", "metric": "streaming_payload_GBps_256conns_4MiB", "value": gbs, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps_done, "warmup": max(1, args.warmup),
        "ms_per_step": t_total / steps_done * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "msgs_per_s": n_total / t_total,
        "config": bench_config(conns, args.msg_bytes, args.ring_kb),
        "config_details": {"arm": "reference CPU RDMA_BPEV path (PairPollable::Send/Recv, memcpy wire)",
                           "connections_timed": conns},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": kind,
                         "sample": "each step = 1 msg on each of %d conns; %d timed steps, %d threads of %d cores" % (conns, steps_done, threads, cores)},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ NUMA

def _parse_cpulist(txt):
    cpus = set()
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa(local):
    """Pin this rank (and every thread / pinned allocation it makes from now on: first touch) to the NUMA node
    its GPU hangs off.  SCALE_r01: GPUs 0-3 sit on node 0, 4-7 on node 1; unbound ranks put their pinned
    buffers wherever the launcher ran and half of the DMA traffic crossed the socket interconnect."""
    info = {"bound": False}
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        try:
            bdf = subprocess.check_output(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id",
                                           "--format=csv,noheader"], text=True).strip().lower()
            bdf = bdf[-12:]  # nvidia-smi prints an 8-digit domain
        except Exception as exc:
            info["why"] = repr(exc)
            return info
    info["pci"] = bdf
    try:
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            info["why"] = "no NUMA affinity reported"
            return info
        cpus = _parse_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            info["why"] = "node cpus outside the affinity mask"
            return info
        os.sched_setaffinity(0, allowed)
        info.update(bound=True, node=node, cpus=len(allowed))
    except Exception as exc:
        info["why"] = repr(exc)
    return info


# --------------------------------------------------------------------------- B200 arm

def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback")
    numa = bind_to_gpu_numa(local) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = ge.load_package()
    L = pkg.lib()
    pkg.init(local)
    pkg.config_set("GRPC_RDMA_RING_BUFFER_SIZE_KB", args.ring_kb)
    pkg.config_set("GRPC_RDMA_MAX_SGE", 30)

    conns, msg = args.conns, args.msg_bytes
    lens = pkg.chttp2_slice_lens(msg) * args.msgs_per_step
    total = sum(lens)                       # bytes the endpoint moves per message (payload + HTTP/2 framing)
    tx_alg, rx_alg = pkg.frame_hbm_bytes(lens)
    dev = torch.device("cuda", local)

    # connections are sharded: this rank owns `conns` of the N*conns connections of the job
    pairs = [pkg.connected_pair("c%d-%d-tx" % (rank, c), "c%d-%d-rx" % (rank, c)) for c in range(conns)]

    # synthetic payload resident in HBM: b[i] = f(i, connection), > L2 (1 GiB src, 4 GiB of rings)
    i = torch.arange(total, device=dev, dtype=torch.int64)
    row = (((i * 2654435761) >> 11) & 255).to(torch.uint8)                       # b[i]
    offs = ((torch.arange(conns, device=dev, dtype=torch.int64) + rank * conns) * 131 & 255).to(torch.uint8)
    src = (row[None, :] + offs[:, None]).reshape(-1)                             # + 131*c (mod 256), one kernel
    # a second, different payload: steps alternate between the two sources, so a step that delivered nothing
    # would leave the previous step's (different) bytes in dst and the comparison after the loop would fail
    src2 = src ^ 0x5A
    del i, row, offs
    dst = torch.zeros(conns * total, dtype=torch.uint8, device=dev)

    def build_batches(src_ptr, dst_ptr, extra_flags=0, dst_stride=None):
        dst_stride = dst_stride or total
        sops, rops, keep = [], [], []
        for c in range(conns):
            off, sl = 0, []
            for n in lens:
                sl.append((src_ptr + c * total + off, n))
                off += n
            arr = pkg.make_slices(sl)
            keep.append(arr)
            sops.append((pairs[c][0], arr, len(lens), 0))
            rops.append((pairs[c][1], dst_ptr + c * dst_stride, total))
        fl = pkg.UNTIL_BLOCKED | extra_flags
        return pkg.Batch("send", sops, fl), pkg.Batch("recv", rops, fl), keep

    bs, br, keep = build_batches(src.data_ptr(), dst.data_ptr())
    bs2, br2, keep_b = build_batches(src2.data_ptr(), dst.data_ptr())
    br2.destroy()                      # same destinations: one recv batch serves both sources
    sends, srcs = (bs, bs2), (src, src2)
    if args.stagger:
        # connections of a real server are at uncorrelated ring positions; without this every ring of the
        # job would sit at the same offset of its 16 MiB-aligned buffer on every step.  One preamble
        # message of a connection-specific size (8 KiB .. 4 MiB) moves each cursor before anything is timed.
        sops, rops, keep2 = [], [], []
        for c in range(conns):
            n = ((c * 40503 + 977 * rank) % 509 + 1) * 8192
            arr = pkg.make_slices([(src.data_ptr() + c * total, n)])
            keep2.append(arr)
            sops.append((pairs[c][0], arr, 1, 0))
            rops.append((pairs[c][1], dst.data_ptr() + c * total, n))
        ps, pr = pkg.Batch("send", sops, pkg.UNTIL_BLOCKED), pkg.Batch("recv", rops, pkg.UNTIL_BLOCKED)
        ps.launch(None)
        pr.launch(None)
        assert ps.results(None) == pr.results(None) == [((c * 40503 + 977 * rank) % 509 + 1) * 8192 for c in range(conns)]
        ps.destroy()
        pr.destroy()
    # an explicit stream: the library treats a NULL stream handle as "its own stream", and
    # torch.cuda.Event only sees the stream it is recorded on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sh = C.c_void_p(stream.cuda_stream)
    assert sh.value, "need a non-default stream handle"

    nstep = [0]

    def step():
        sends[nstep[0] & 1].launch(sh)
        br.launch(sh)
        nstep[0] += 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    last = sends[(nstep[0] - 1) & 1]
    assert last.results(sh) == [total] * conns and br.results(sh) == [total] * conns, "warm-up step incomplete"
    assert torch.equal(srcs[(nstep[0] - 1) & 1], dst), "delivered bytes differ from what was sent"

    # ---- timed region: device resident
    K = args.steps
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    launches0 = L.b200_launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    t_region0 = time.time()
    for k in range(K):
        ev[k][0].record(stream)
        sends[nstep[0] & 1].launch(sh)
        ev[k][1].record(stream)
        br.launch(sh)
        ev[k][2].record(stream)
        nstep[0] += 1
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    t_region1 = time.time()
    barrier()
    launches = L.b200_launch_count() - launches0
    t_dev_ms = ev[0][0].elapsed_time(ev[K - 1][2])
    send_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / K
    recv_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / K
    last = sends[(nstep[0] - 1) & 1]
    assert last.results(sh) == [total] * conns and br.results(sh) == [total] * conns
    # the LAST timed step's payload (the step before it carried the other one)
    assert torch.equal(srcs[(nstep[0] - 1) & 1], dst), "last timed step did not deliver its bytes"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dst, last.results(sh), br.results(sh))
    if world > 1:
        t = torch.tensor([t_dev_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev_ms = float(t.item())

    n_msgs = world * conns * K * args.msgs_per_step
    gbs = n_msgs * msg / (t_dev_ms * 1e-3) / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    recv_ach = conns * rx_alg / (recv_ms * 1e-3) / 1e9
    send_ach = conns * tx_alg / (send_ms * 1e-3) / 1e9
    dominant = ("k_recv", recv_ach, recv_ms) if recv_ms >= send_ms else ("k_send", send_ach, send_ms)
    traffic = None
    try:  # dram bytes per launch from the committed ncu --set full capture of this same workload
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if conns == CONNS and msg == MSG_BYTES:
            traffic = tj[dominant[0]]["dram_bytes"]
    except Exception:
        pass

    # ---- e2e: host buffers, through the same C-ABI calls, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, pkg, L, pairs, lens, total, conns, msg, world, dist if world > 1 else None, dev, stream, sh,
                      build_batches)

    t_e2e1 = time.time()
    sampler.stop()
    clocks = sampler.window(t_region0, t_region1, "device-resident timed region")
    if e2e is not None:
        w = e2e.pop("_wall", None) or (t_region1, t_e2e1)
        e2e["clocks"] = sampler.window(w[0], w[1], "e2e timed region")
    if not clocks.get("samples") and e2e is not None:
        # a very short timed region can fall between two 20 ms samples: say so and show the e2e window
        clocks = dict(e2e["clocks"], note="no sample fell inside the %.0f ms device-resident region; "
                                           "these are the samples of the e2e region that follows it" % ((t_region1 - t_region0) * 1e3))

    # ---- N >= 2: the CUDA-IPC / NVLink wire, exercised in every multi-GPU run (pytest -m gpu on one GPU skips it)
    nvlink = None
    if world > 1 and not args.no_nvlink:
        try:
            nvlink = run_nvlink_pass(pkg, L, dist, dev, stream, sh, rank, world, args.ring_kb, msg)
        except Exception as exc:
            nvlink = {"error": repr(exc)}

    unary = None
    if world > 1 and not args.no_unary:
        unary = {"note": "the unary leg runs in the N=1 line only (it is a one-GPU measurement; the other ranks would idle)"}
    if rank == 0 and world == 1 and not args.no_unary:
        for b in (bs, bs2, br):
            b.destroy()
        try:
            unary = run_unary(args, pkg, L, with_cpu=(world == 1 and not args.no_cpu_baseline))
        except Exception as exc:  # never take the streaming line down
            unary = {"error": repr(exc)}

    e2e_endpoint = None
    if rank == 0 and world == 1 and not args.no_endpoint:
        try:
            e2e_endpoint = run_e2e_endpoint(args, pkg, L, with_cpu=not args.no_cpu_baseline)
        except Exception as exc:
            e2e_endpoint = {"error": repr(exc)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = run_cpu_baseline(args, lens, msg, args.cpu_seconds)
        except Exception as exc:  # the baseline must never take the bench down
            cpu = {"value": None, "unit": "GB/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (exc,)}

    if rank == 0:
        line = {
            "metric": "streaming_payload_GBps_256conns_4MiB", "value": gbs, "unit": "GB/s", "n_gpus": world,
            "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": t_dev_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "msgs_per_s": n_msgs / (t_dev_ms * 1e-3),
            "config": bench_config(conns, msg, args.ring_kb),
            "config_details": {"arm": "B200: HBM rings, loopback wire (sender writes the peer ring in HBM), 1 message per "
                                      "connection per step; 514 slices per message: 9 B DATA headers + <=16384 B payload",
                               "connections_per_gpu": conns, "connections_total": conns * world,
                       "l2": "inputs larger than L2: %.2f GiB of slices + %.1f GiB of rings per GPU, no reuse "
                             "between steps" % (conns * total / 2**30, conns * args.ring_kb / 2**20),
                       "sharding": "connection c of rank r is independent; no data-path collective",
                       "ring_positions": "staggered by one untimed preamble message per connection" if args.stagger
                                         else "all connections at the same ring offset"},
            "roofline": {"bound": "hbm", "kernel": dominant[0], "achieved": dominant[1], "peak": peak,
                         "unit": "GB/s", "frac": dominant[1] / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": conns * (rx_alg if dominant[0] == "k_recv" else tx_alg),
                         "avg_launch_ms": dominant[2],
                         "kernels": {"k_send": {"ms": send_ms, "GBps": send_ach, "frac": send_ach / peak},
                                     "k_recv": {"ms": recv_ms, "GBps": recv_ach, "frac": recv_ach / peak}},
                         "step_frac": (conns * (tx_alg + rx_alg) / (t_dev_ms / K * 1e-3) / 1e9) / peak},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "e2e_endpoint": e2e_endpoint,
            "nvlink_wire": nvlink,
            "unary": unary,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "numa": numa,
            "wall_s_timed_region": t_wall,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_SAMPLES = 1 << 21
DUMP_SEED = 20250101


def dump_outputs(out_dir, dst, sent, received):
    """--dump-outputs: what a caller of the timed path receives from its last step -- the bytes each send batch
    consumed and each recv batch delivered per connection, and the delivered bytes themselves.  Those are 1 GiB at
    the default size, so a fixed sample of positions (same seed, same positions on every run) is stored with its
    indices: 24 MiB in all."""
    import numpy as np
    import torch
    n = dst.numel()
    idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, n, min(DUMP_SAMPLES, n)))
    sample = dst[torch.from_numpy(idx).to(dst.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("send_bytes", np.asarray(sent, dtype=np.float64)),
                    ("recv_bytes", np.asarray(received, dtype=np.float64)),
                    ("delivered_sample_index", idx.astype(np.float64)),
                    ("delivered_sample", sample.astype(np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_nvlink_pass(pkg, L, dist, dev, stream, sh, rank, world, ring_kb, msg, conns=64, steps=4):
    """Connections that CROSS GPUs: rank r's senders are connected to rank (r+1) % N's receivers over the CUDA-IPC
    wire, so k_send stores its frames into rings in the next GPU's HBM over NVLink and k_recv returns credit the
    other way.  A short pass with a full integrity check; time = max over ranks."""
    import torch
    pkg.config_set("GRPC_RDMA_RING_BUFFER_SIZE_KB", ring_kb)
    tx = [pkg.Pair("nv-tx-%d-%d" % (rank, c)) for c in range(conns)]
    rx = [pkg.Pair("nv-rx-%d-%d" % (rank, c)) for c in range(conns)]
    everyone = [None] * world
    dist.all_gather_object(everyone, {"tx": [p.address() for p in tx], "rx": [p.address() for p in rx]})
    nxt, prv = (rank + 1) % world, (rank - 1) % world
    for c in range(conns):
        if not tx[c].connect(everyone[nxt]["rx"][c]) or not rx[c].connect(everyone[prv]["tx"][c]):
            raise RuntimeError("nvlink wire connect failed: %s / %s" % (tx[c].error(), rx[c].error()))
    dist.barrier()
    lens = pkg.chttp2_slice_lens(msg)
    total = sum(lens)
    wire_bytes = sum(16 + (n + 7) // 8 * 8 for n in lens)
    i = torch.arange(total, device=dev, dtype=torch.int64)
    row = (((i * 2654435761) >> 11) & 255).to(torch.uint8)

    def payload(r, k):
        offs = (((torch.arange(conns, device=dev, dtype=torch.int64) + r * conns) * 131 + 29 * k) & 255).to(torch.uint8)
        return (row[None, :] + offs[:, None]).reshape(-1)

    srcs = [payload(rank, 0), payload(rank, 1)]
    dst = torch.zeros(conns * total, dtype=torch.uint8, device=dev)
    batches, keep = [], []
    for src in srcs:
        sops = []
        for c in range(conns):
            off, sl = 0, []
            for n in lens:
                sl.append((src.data_ptr() + c * total + off, n))
                off += n
            arr = pkg.make_slices(sl)
            keep.append(arr)
            sops.append((tx[c], arr, len(lens), 0))
        batches.append(pkg.Batch("send", sops, pkg.UNTIL_BLOCKED))
    br = pkg.Batch("recv", [(rx[c], dst.data_ptr() + c * total, total) for c in range(conns)], pkg.UNTIL_BLOCKED)
    send_ms, ok = [], True
    for k in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        e0.record(stream)
        batches[k & 1].launch(sh)
        e1.record(stream)
        stream.synchronize()
        dist.barrier()                                          # the neighbour's frames have landed in my rings
        br.launch(sh)
        stream.synchronize()
        ok = ok and batches[k & 1].results(sh) == [total] * conns and br.results(sh) == [total] * conns
        ok = ok and bool(torch.equal(dst, payload(prv, k & 1)))  # every step carries a different payload
        if k >= 1:
            send_ms.append(e0.elapsed_time(e1))
    t = torch.tensor([sum(send_ms) / max(1, len(send_ms)), 0.0 if ok else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    for b in batches + [br]:
        b.destroy()
    for p in tx + rx:
        p.disconnect()
    dist.barrier()
    s_ms, bad = t.tolist()
    return {"what": "k_send over the CUDA-IPC/NVLink wire into the next GPU's rings, k_recv credit back",
            "connections_per_gpu": conns, "message_bytes": msg, "steps": steps, "intact_all_ranks": bad == 0.0,
            "k_send_ms": s_ms, "payload_GBps_per_gpu": conns * msg / (s_ms * 1e-3) / 1e9 if s_ms else None,
            "nvlink_write_GBps_per_gpu": conns * wire_bytes / (s_ms * 1e-3) / 1e9 if s_ms else None}


def run_e2e_endpoint(args, pkg, L, with_cpu):
    """The same streaming workload THROUGH THE DROP-IN SURFACE: b200_endpoint_write / b200_endpoint_read +
    b200_engine_work (include/b200_endpoint.h = rdma_bp_posix.cc + the BPEV poll loop), 256 connections, one
    4 MiB chttp2-shaped message in flight per connection, 514 NON-ADJACENT host slices per message, every
    delivered byte compared on the reader (tools/native/ep_stream.cc).  The engine batches: one pass = one
    b200_pairs_submit of every ready rdma_flush / rdma_do_read loop, executed by the resident service kernels
    (no launch), slices and read buffers used in place over PCIe.  Beside it the same driver over the
    reference's own PairPollable on the host cores (tests/native/ref_pair_ops.cc, NDEBUG build)."""
    libdir = os.path.dirname(pkg.LIB_PATH)
    C.CDLL(pkg.ENDPOINT_LIB_PATH, mode=C.RTLD_GLOBAL)
    ES = C.CDLL(os.path.join(libdir, "libb200_epstream.so"))
    ES.ep_stream_run.restype = C.c_double
    ES.ep_stream_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]
    conns, threads, msgs = args.conns, args.endpoint_threads, args.endpoint_msgs
    pkg.config_set("GRPC_RDMA_RING_BUFFER_SIZE_KB", args.ring_kb)
    out = {"connections": conns, "message_bytes": args.msg_bytes, "msgs_per_connection": msgs, "unit": "GB/s",
           "thread_pairs": threads,
           "path": "b200_endpoint_write/read + b200_engine_work (batching engine -> b200_pairs_submit -> service kernels: "
                   "owner warps + %d pool CTAs), 514 non-adjacent pinned slices per message, every byte verified" % args.endpoint_pool}
    launches0 = L.b200_launch_count()
    if L.b200_service_start(args.endpoint_pool) != 0:
        return {"error": "b200_service_start: " + pkg.last_error()}
    try:
        o = (C.c_uint64 * 4)()
        t = ES.ep_stream_run(None, conns, threads, msgs, 2, args.msg_bytes, 0, o)
        if t <= 0:
            out["b200"] = {"error": "driver rc %s, bad bytes %d" % (t, o[1])}
        else:
            out["b200"] = {"value": o[0] / t / 1e9, "seconds": t, "msgs_per_s": conns * msgs / t, "bad_bytes": int(o[1]),
                           "submits_client": int(o[2]), "submits_server": int(o[3])}
            out["value"] = out["b200"]["value"]
    finally:
        L.b200_service_stop()
    out["kernel_launches"] = int(L.b200_launch_count() - launches0)   # the three resident kernels
    if with_cpu:
        relp = os.path.join(ROOT, "tests", "native", "libref_pair_ops_rel.so")
        if os.path.exists(relp):
            try:
                R = C.CDLL(relp)
                R.ref_pair_ops.restype = C.c_void_p
                R.ref_ops_config.argtypes = [C.c_uint32]
                R.ref_ops_config(args.ring_kb)
                cores = usable_cpus()
                ref = {"kind": "reference", "cores": cores}
                for label, th in (("same_threads", threads), ("all_cores", max(1, min(conns, cores // 2)))):
                    o = (C.c_uint64 * 4)()
                    t = ES.ep_stream_run(R.ref_pair_ops(), conns, th, max(2, msgs // 2), 1, args.msg_bytes, 0, o)
                    ref[label] = ({"value": o[0] / t / 1e9, "thread_pairs": th, "seconds": t, "bad_bytes": int(o[1])}
                                  if t > 0 else {"error": "driver rc %s" % t, "thread_pairs": th})
                out["cpu_reference"] = ref
            except Exception as exc:
                out["cpu_reference"] = {"error": repr(exc)}
        else:
            out["cpu_reference"] = {"error": "tests/native/libref_pair_ops_rel.so not built"}
    return out


def _pct(rtt_ns):
    import numpy as np
    r = np.sort(np.asarray(rtt_ns).reshape(-1)) / 1e3
    return {"p50_us": float(r[len(r) // 2]), "p99_us": float(r[int(len(r) * 0.99)]), "mean_us": float(r.mean())}


def run_unary(args, pkg, L, with_cpu):
    """BASELINE config 3 at the pair level: M-byte request + M-byte echo (default 1 KiB), round-trip time per
    call, 1 and 256 connections.  B200: through the C ABI with registered HOST buffers and the persistent
    service kernel (no launch per call; every request and echo crosses PCIe both ways).  Beside it the
    reference's own PairPollable ping-pong on the host cores (memcpy wire: no NIC, no PCIe in its path)."""
    import numpy as np
    PP = C.CDLL(os.path.join(os.path.dirname(pkg.LIB_PATH), "libb200_pingpong.so"))
    PP.b200_pp_run.restype = C.c_double
    PP.b200_pp_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_uint64)]
    m, iters = args.unary_bytes, args.unary_iters
    pkg.config_set("GRPC_RDMA_RING_BUFFER_SIZE_KB", 4096)   # the reference's default ring (config.cc:90-96)
    out = {"msg_bytes": m, "ring_kb": 4096, "b200": {}, "cpu_reference": None,
           "path": "b200_pair_send / has_message / recv on registered host buffers, persistent service kernel "
                   "(owner warps + %d pool CTAs + poller)" % args.service_workers}
    launches0 = L.b200_launch_count()
    if L.b200_service_start(args.service_workers) != 0:
        return {"error": "b200_service_start: " + pkg.last_error()}
    try:
        for conns, groups in ((1, 1), (256, 8)):
            it = iters if conns == 1 else max(50, iters // 20)
            rtt = np.zeros(conns * it, dtype=np.uint64)
            t = PP.b200_pp_run(conns, groups, it, max(10, it // 10), m, rtt.ctypes.data_as(C.POINTER(C.c_uint64)))
            if t < 0:
                out["b200"]["conns_%d" % conns] = {"error": "pingpong driver rc %d" % int(t)}
                continue
            d = _pct(rtt)
            d.update({"round_trips_per_s": conns * it / t, "client_threads": groups, "server_threads": groups,
                      "iters_per_conn": it})
            out["b200"]["conns_%d" % conns] = d
    finally:
        L.b200_service_stop()
    out["kernel_launches_during_unary"] = int(L.b200_launch_count() - launches0)   # 3 = the resident kernels themselves
    out["eager_recvs"] = int(L.b200_service_eager_hits())
    if with_cpu:
        try:
            eng, kind = cpu_engine()
            if hasattr(eng, "bench_pingpong"):
                ref = {"kind": kind}
                for conns, groups in ((1, 1), (256, 8)):
                    it = iters if conns == 1 else max(50, iters // 20)
                    t, rtt = eng.bench_pingpong(conns, groups, it, max(10, it // 10), m, 4096 * 1024)
                    d = _pct(rtt)
                    d.update({"round_trips_per_s": conns * it / t, "threads": 2 * groups})
                    ref["conns_%d" % conns] = d
                out["cpu_reference"] = ref
        except Exception as exc:
            out["cpu_reference"] = {"error": repr(exc)}
    return out


def run_e2e(args, pkg, L, pairs, lens, total, conns, msg, world, dist, dev, stream, sh, build_batches):
    """Same step through the public C-ABI with HOST buffers: slices live in pinned host memory and the
    delivered bytes must land in pinned host memory, every step, inside the timed region."""
    import torch
    nbytes = conns * total
    # Source slices sit wherever the application left them (here back to back: not even 16-byte aligned).
    # Destination windows are what the endpoint itself allocates for a read (rdma_bp_posix.cc:308-317):
    # one pinned slice per connection, 256-byte aligned like every b200_mem_alloc_host block.
    dstride = (total + 255) // 256 * 256
    # Host buffers: b200_mem_alloc_host (first touched from this rank's NUMA node).  --hugepages: anonymous memory
    # with transparent huge pages asked for, then registered (the ibv_reg_mr analogue).
    keep_maps, huge = [], args.hugepages

    def alloc_host(n):
        if huge:
            try:
                import mmap
                mm = mmap.mmap(-1, n + (4 << 20), flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
                base = C.addressof(C.c_char.from_buffer(mm))
                addr = (base + (2 << 20) - 1) & ~((2 << 20) - 1)
                if hasattr(mmap, "MADV_HUGEPAGE"):
                    mm.madvise(mmap.MADV_HUGEPAGE)
                C.memset(addr, 0, n)                                  # first touch: local node, huge pages
                if L.b200_mem_register_host(addr, (n + 4095) & ~4095) == 0:
                    keep_maps.append((mm, addr))
                    return addr
            except Exception:
                pass
        return L.b200_mem_alloc_host(n)

    def free_host(p):
        for mm, addr in keep_maps:
            if addr == p:
                L.b200_mem_unregister_host(addr)
                return
        L.b200_mem_free_host(p)

    hsrc = alloc_host(nbytes)
    hsrc2 = alloc_host(nbytes)
    hdst = alloc_host(conns * dstride)
    if not hsrc or not hsrc2 or not hdst:
        return {"value": None, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "pinned allocation failed: " + pkg.last_error()}
    import numpy as np
    hs = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(hsrc))
    hs2 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(hsrc2))
    hd = np.ctypeslib.as_array((C.c_uint8 * (conns * dstride)).from_address(hdst)).reshape(conns, dstride)
    i = np.arange(total, dtype=np.uint64)
    for c in range(conns):
        hs[c * total:(c + 1) * total] = ((i * np.uint64(40503) >> np.uint64(5)) + np.uint64(17 * c)).astype(np.uint8)
    np.bitwise_xor(hs, 0xA5, out=hs2)      # steps alternate between two different payloads (see main())
    hsv = (hs.reshape(conns, total), hs2.reshape(conns, total))
    K = args.e2e_steps or min(args.steps, 8)
    results = {}
    modes = ["zerocopy", "staged"] if args.e2e_mode == "auto" else [args.e2e_mode]
    for mode in modes:
        if mode == "zerocopy":
            # kernels address the pinned host slices / destinations directly: bytes cross PCIe once each way
            bs, br, keep = build_batches(hsrc, hdst, pkg.ZEROCOPY, dstride)
            bs2, br2, keep2 = build_batches(hsrc2, hdst, pkg.ZEROCOPY, dstride)
            lane_stream = sh
        else:
            # the library's host-staged path: per lane H2D -> k_send ... k_recv -> D2H on internal streams
            bs, br, keep = build_batches(hsrc, hdst, 0, dstride)
            bs2, br2, keep2 = build_batches(hsrc2, hdst, 0, dstride)
            lane_stream = None
        br2.destroy()
        sends = (bs, bs2)
        n = [0]

        def step():
            sends[n[0] & 1].launch(lane_stream)
            br.launch(lane_stream)
            n[0] += 1
        hd[:] = 0
        step()
        L.b200_lanes_join(None)
        torch.cuda.synchronize()
        ok = bool(np.array_equal(hsv[0], hd[:, :total]))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        tw0 = time.time()
        e0.record(stream)
        L.b200_lanes_fork(sh)        # lanes start after e0 ...
        for _ in range(K):
            step()
        L.b200_lanes_join(sh)        # ... and e1 waits for every lane
        e1.record(stream)
        torch.cuda.synchronize()
        tw1 = time.time()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        # after the timed loop: the host destination must hold the LAST step's payload, bit for bit
        ok = ok and bool(np.array_equal(hsv[(n[0] - 1) & 1], hd[:, :total]))
        ok = ok and sends[(n[0] - 1) & 1].results(sh) == [total] * conns and br.results(sh) == [total] * conns
        results[mode] = {"GBps": world * conns * K * msg / (ms * 1e-3) / 1e9, "ms_per_step": ms / K, "intact": ok,
                         "_wall": (tw0, tw1)}
        bs.destroy()
        bs2.destroy()
        br.destroy()
    del hs, hs2, hd, hsv
    free_host(hsrc)
    free_host(hsrc2)
    free_host(hdst)
    best = max((m for m in results if results[m]["intact"]), key=lambda m: results[m]["GBps"], default=None)
    if best is None:
        for m in results:
            results[m].pop("_wall", None)
        return {"value": None, "unit": "GB/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                "note": "e2e verification failed", "modes": results}
    wall = results[best].pop("_wall")
    for m in results:
        results[m].pop("_wall", None)
    return {"_wall": wall, "value": results[best]["GBps"], "unit": "GB/s", "h2d_bytes_per_step": nbytes,
            "d2h_bytes_per_step": nbytes, "mode": best, "steps": K, "ms_per_step": results[best]["ms_per_step"],
            "host_buffers": "THP + b200_mem_register_host" if keep_maps else "b200_mem_alloc_host",
            "modes": results,
            "note": "slices and destinations are pinned host memory; per step every payload byte crosses PCIe "
                    "once in each direction inside the timed region"}


if __name__ == "__main__":
    main()
