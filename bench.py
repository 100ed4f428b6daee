#!/usr/bin/env python
"""bench.py -- committed ops/s of the replication hot path (BASELINE.json metric:
"committed ops/s and p50/p99 commit latency, 64B reqs, 5 replicas").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic requests:
`--batch` SEND requests of `--payload` bytes are appended to the leader's log,
replicated to every follower, acked, and committed by majority.

  value      requests already resident in HBM (device submission ring, written there by the
             engine's fill kernel: apus_submit_synth) when the timed region starts; one fused
             kernel launch per GPU per step, a step = 2^20 requests (>= 2^24 per default run)
  e2e        the same metric through the C ABI with HOST buffers: apus_submit_uniform()
             from host memory + apus_wait_committed(); the kernels stay resident
  parity     outside every timed region: the same placement runs a bounded stream that the CPU
             oracle can follow; every replica's whole log is compared byte for byte (across
             ranks: hashes gathered over gloo) -- the cross-GPU parity evidence of the run
  roofline   algorithmic bytes (N-1)*(64+L) per committed op / CUDA-event time of the
             replica kernel, against MEASURED_PEAKS.json (HBM copy bandwidth: with all
             replicas on one GPU the "peer" stores land in local HBM; NVLink peer-copy
             figure when replicas sit on different GPUs)
  cpu_baseline  the reference's own software stack (oracle/_ref/libref_stack.so: its unmodified
             election / replication / commit code + proxy.c as N processes on a verbs shim
             NIC) on the host cores; `log_code_only` = its dare_log.h loop on threads with a
             memcpy transport (an upper bound on the log code alone)

N = 1: all `--replicas` replicas of ONE group live on GPU 0 (the 5-replica configuration
of the metric fits one GPU).  N > 1 (torchrun, one process per GPU): N groups, group g
led by GPU g, replica r of group g on GPU (g + r) % N, peers mapped with CUDA IPC; no
data-path collective (weak scaling: every GPU leads one group of the same size).

The log ring is the reference's LOG_SIZE (64 MiB); sustained runs wrap it many times,
kept alive by the device-side pruning rule (HEAD entries, APUS_F_AUTOPRUNE).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEND, CONNECT = 5, 4
UINT64_MAX = (1 << 64) - 1
NVLINK_PEER_GBS = 770.0     # measured peer copy per direction (B200_PROFILING.md)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--replicas", type=int, default=5)
    ap.add_argument("--payload", type=int, default=64)
    ap.add_argument("--batch", type=int, default=0, help="requests per step (0 = 2^20 for <= 256 B requests, else 16 MiB worth)")
    ap.add_argument("--log-size", type=int, default=0, help="bytes of entries[]; 0 = reference LOG_SIZE (64 MiB)")
    ap.add_argument("--lat-requests", type=int, default=20000, help="closed-loop requests for p50/p99")
    ap.add_argument("--failover", action="store_true",
                    help="BASELINE config 5: kill the leader process under load, report the recovery latency (reconf_bench.sh analogue)")
    ap.add_argument("--failover-trials", type=int, default=3)
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-proxy-leg", action="store_true", help="skip the 16-connection closed-loop leg through the reference's proxy.c")
    ap.add_argument("--profile-latency", action="store_true",
                    help="device timestamps inside the express path (adds ~0.6 us to every closed-loop request: diagnostic runs only)")
    ap.add_argument("--no-express", action="store_true", help="A/B: every publish fenced, no single-warp express path")
    ap.add_argument("--e2e-ring", default="mapped", choices=["mapped", "device"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-stats", action="store_true", help="value run without device-side profiling counters")
    ap.add_argument("--leader-ctas", type=int, default=16, help="leader worker CTAs (SMs building tiles in parallel)")
    ap.add_argument("--spread", action="store_true",
                    help="single process: place replica r on GPU r %% visible GPUs (NVLink path)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step committed as DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(n, payload, batch, ctas):
    """dram__bytes_read.sum + dram__bytes_write.sum of the replica kernel per launch, from the committed
    `ncu --set full` capture (profiles/r2_ncu.json); only valid for the configuration it was taken on."""
    p = os.path.join(ROOT, "profiles", "r2_ncu.json")
    try:
        d = json.load(open(p))
        c = d["config"]
        if (n, payload, batch, ctas) == (c["replicas"], c["payload_bytes"], c["batch"], c["leader_ctas"]):
            return float(d["traffic_bytes_per_launch"])
    except Exception:
        pass
    return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured HBM copy (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback HBM copy 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------
# CPU baseline / reference arm
# ------------------------------------------------------------------------------------
def cpu_library():
    import orc as O
    O.build_oracle()
    if O.have_ref():
        return O.Oracle("ref"), "reference"
    return O.Oracle("orc"), "port"


def cpu_run(oracle, n, payload, nreq, clients=64):
    secs = C.c_double()
    ops = oracle.bench_run(n, payload, nreq, clients, C.byref(secs))
    return float(ops), float(secs.value)


def default_batch(args):
    return args.batch or ((1 << 20) if args.payload <= 256 else max(4096, (16 << 20) // (64 + args.payload)))


def cpu_nreq(payload, batch):
    # stay inside one 64 MiB ring: the CPU run has no pruning
    return max(1, min(batch, (60 << 20) // (64 + payload)))


def log_code_baseline(n, payload, batch, budget_s=10.0):
    oracle, kind = cpu_library()
    nreq = cpu_nreq(payload, batch)
    best, total, runs = 0.0, 0.0, 0
    while total < budget_s and runs < 200:
        ops, s = cpu_run(oracle, n, payload, nreq)
        best = max(best, ops); total += s; runs += 1
    return {"value": round(best, 1), "unit": "ops/s", "cores": n, "kind": kind,
            "sample": f"best of {runs} runs x {nreq} requests of {payload} B; {n} replicas as threads of one process "
                      f"(leader + {n - 1} followers), closed loop with 64 outstanding requests, memcpy transport "
                      f"(zero latency), no BerkeleyDB put, fresh 64 MiB ring per run"}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


REFSTACK_CONNS = 16         # BASELINE.json configs[2]: 16 concurrent clients
TRANSPORT_TEXT = {"shm": "shm transport: the log is a shared mapping, an RDMA WRITE is a memcpy -- no wire latency, no system call",
                  "process_vm": "process_vm_writev transport: one or two system calls per RDMA operation, no wire latency"}


def refstack_leg(n, payload, nreq, steps, timeout=150, transport=None):
    """The reference's OWN software stack -- its unmodified election / replication / commit code (src/dare/*.c) and
    proxy.c, built by oracle/build_refapp.sh into oracle/_ref/libref_stack.so -- as n replica processes on this
    box's host cores, with oracle/verbs_shim standing in for the NIC (no wire latency; transport None: one or two
    process_vm_* system calls per RDMA operation, "shm": log writes are memcpys into a mapping the replicas share -- the
    zero-latency bound BASELINE.md s2 planned), driven by application threads through proxy_on_accept/read/close.
    Returns (per-step dicts, cores, threads, how the leader's RDMA operations travelled) or None when the stack cannot
    run here (library absent, or the box forbids process_vm_writev)."""
    import refstack as R
    if not R.available() or n < 2:        # a group of one never holds an election in the reference (it waits for joins)
        return None
    # The replicas are n worker processes that each load the reference stack; this process maps the same library too, so
    # that whoever records the native libraries of the bench process sees which build of the reference was timed.
    import ctypes
    ctypes.CDLL(R.STACK)
    cores = host_cores()
    threads = max(1, min(REFSTACK_CONNS, cores - n))
    try:
        # one attempt on the shm transport (the process_vm leg follows anyway), two on process_vm: a hung or disturbed
        # group must not stretch the arm beyond a few minutes
        rr = R.run(n, REFSTACK_CONNS, nreq, payload, attempts=1 if transport else 2, threads=threads, steps=steps,
                   images=False, timeout=timeout, transport=transport)
    except Exception as e:                                   # noqa: BLE001 - reported, and the caller falls back
        sys.stderr.write(f"[bench] reference stack ({transport or 'process_vm'} transport) could not run "
                         f"({type(e).__name__}: {str(e)[:300]})\n")
        return None
    lead = rr["results"][rr["leader"]]
    return lead["steps"], n + threads, threads, lead.get("rdma_ops")


def refstack_both(n, payload, nreq, steps, first):
    """The reference stack on both shim transports.  Returns (primary leg, {transport: summary}) -- primary = the shm
    transport when the leader's log writes really travelled as memcpys, else process_vm; None when neither ran."""
    legs, summary = {}, {}
    for tr in ("shm", None):
        leg = refstack_leg(n, payload, nreq, steps, transport=tr)
        name = tr or "process_vm"
        if leg is None:
            summary[name] = None
            continue
        st, cores, threads, ops = leg
        timed = st[first:]
        summary[name] = {"ops_per_s": round(sum(x["requests"] for x in timed) / sum(x["seconds"] for x in timed), 1),
                         "p50_us": round(statistics.median(x["p50_us"] for x in timed), 1),
                         "p99_us": round(max(x["p99_us"] for x in timed), 1), "leader_rdma_ops": ops}
        legs[name] = leg
    shm_real = "shm" in legs and (legs["shm"][3] or {}).get("memcpy", 0) > 0
    primary = "shm" if shm_real else ("process_vm" if "process_vm" in legs else ("shm" if "shm" in legs else None))
    return (legs[primary] if primary else None), primary, summary


def refstack_nreq(payload, steps_total):
    # the whole run stays inside ONE lap of the reference's 64 MiB ring: its wrap path has the H11 defects of
    # SURVEY.md s2 (an entry that ends exactly at len vanishes), so the reference arm is kept off it
    lap = (56 << 20) // (64 + payload + 8)
    return int(max(1000, min(50_000, lap // max(1, steps_total))))


def cpu_baseline(n, payload, batch, budget_s=10.0):
    """Reported beside our number: (1) the reference's full software stack on the shim NIC; (2) as an upper bound on
    what its log code alone could do, the dare_log.h append/replicate/commit loop on threads with a memcpy transport."""
    loop = log_code_baseline(n, payload, batch, budget_s=min(budget_s, 5.0))
    nreq = refstack_nreq(payload, 4)
    leg, primary, transports = refstack_both(n, payload, nreq, 4, first=1)
    if leg is None:
        return loop
    steps, cores, threads, _ = leg
    timed = steps[1:]
    ops = sum(s["requests"] for s in timed) / sum(s["seconds"] for s in timed)
    return {"value": round(ops, 1), "unit": "ops/s", "cores": cores, "kind": "reference",
            "sample": f"the reference's unmodified stack (src/dare/*.c, proxy.c; -O0 as it builds) as {n} replica "
                      f"processes + {threads} application threads on {host_cores()} host cores, {REFSTACK_CONNS} "
                      f"connections, closed loop, verbs shim NIC ({TRANSPORT_TEXT[primary]}), "
                      f"{len(timed)} x {nreq} requests of {payload} B after one warm-up pass",
            "p50_us": round(statistics.median(s["p50_us"] for s in timed), 1),
            "p99_us": round(max(s["p99_us"] for s in timed), 1),
            "shim_transport": primary, "shim_transports": transports,
            "log_code_only": loop}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, payload = args.replicas, args.payload
    total = args.steps + args.warmup
    nreq = refstack_nreq(payload, total)
    leg, primary, transports = refstack_both(n, payload, nreq, total, first=args.warmup)
    if leg is not None:
        steps, cores, threads, _ = leg
        timed = steps[args.warmup:]
        t = sum(s["seconds"] for s in timed)
        value = sum(s["requests"] for s in timed) / t
        kind = "reference"
        workload = (f"{n} replicas, {payload} B SEND requests, {nreq} requests per step over {REFSTACK_CONNS} connections; "
                    f"the reference's unmodified software stack (src/dare/*.c election/replication/commit, proxy.c, "
                    f"libev, BerkeleyDB) as {n} processes + {threads} application threads on the host cores, "
                    f"verbs shim NIC ({TRANSPORT_TEXT[primary]})")
        sample = (f"{len(timed)} timed steps x {nreq} requests after {args.warmup} warm-up steps, closed loop, "
                  f"{REFSTACK_CONNS} connections on {threads} application threads")
        extra = {"latency_us": {"p50": round(statistics.median(s["p50_us"] for s in timed), 1),
                                "p99": round(max(s["p99_us"] for s in timed), 1),
                                "clock": "host, around proxy_on_read (returns at commit)"},
                 "shim_transport": primary, "shim_transports": transports}
    else:
        oracle, kind = cpu_library()
        nreq = cpu_nreq(payload, default_batch(args))
        for _ in range(args.warmup):
            cpu_run(oracle, n, payload, nreq)
        t = 0.0
        for _ in range(args.steps):
            _, s = cpu_run(oracle, n, payload, nreq)
            t += s
        value = args.steps * nreq / t
        cores = n
        workload = (f"{n} replicas, {payload} B SEND requests, {nreq} requests per step; the reference's log code on host "
                    f"threads (memcpy transport), one fresh 64 MiB ring per step (the full reference stack could not run here)")
        sample = f"{args.steps} steps x {nreq} requests, closed loop, 64 outstanding"
        extra = {}
    out = {
        "impl": "reference", "metric": "committed ops/s", "value": round(value, 1), "unit": "ops/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * t / max(1, args.steps), 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload, "replicas": n, "payload_bytes": payload, "batch": nreq},
        "cpu_baseline": {"value": round(value, 1), "unit": "ops/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": round(value, 1), "unit": "ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    out.update(extra)
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------
class Cell:
    """The replicas this process hosts: in a single process all replicas of one group;
    under torchrun the leader of group `rank` plus the followers of the neighbouring
    groups that the placement (g + r) % N puts on this GPU."""

    def __init__(self, A, E, args, ring_mode, slots, ring_bytes, flags, dist=None, rank=0, world=1, local=0):
        self.A, self.E = A, E
        n, L = args.replicas, (args.log_size or A.LOG_SIZE)
        self.n, self.L = n, L
        self.local = []
        if world == 1:
            nd = A.lib().apus_device_count()
            devs = [r % nd for r in range(n)] if args.spread else [0] * n
            self.group = A.Group(n, devices=devs, log_size=L, ring_mode=ring_mode, ring_slots=slots,
                                 ring_bytes=ring_bytes, flags=flags, leader_ctas=args.leader_ctas)
            self.leader = self.group.leader
            self.local = list(self.group.replicas)
            self.devices = sorted(set(devs))
            self.placement = "all replicas on GPU 0" if not args.spread else f"replica r on GPU r % {nd}"
        else:
            from apus_b200 import placement as P
            self.group = None
            mine = {}
            for g, r in P.hosted(rank, world, n):
                mine[(g, r)] = E.Replica(local, r, n, 0, 1, L, ring_mode, slots if r == 0 else 0,
                                         ring_bytes if r == 0 else 0, flags, args.leader_ctas)
            merged = P.exchange(dist, {k: v.export() for k, v in mine.items()}, world)
            for g, r, p in P.connections(rank, world, n):
                mine[(g, r)].connect(p, merged[(g, p)])
            self.leader = mine[(rank, 0)]
            self.local = list(mine.values())
            self.devices = [local]
            self.placement = f"group g led by GPU g, replica r on GPU (g + r) % {world}, CUDA IPC"
        self.tickets = 0

    def launch(self, target):
        E, A = self.E, self.A
        by_dev = {}
        for r in self.local:
            by_dev.setdefault(r.device, []).append(r)
        for dev, rs in sorted(by_dev.items(), key=lambda kv: any(r.is_leader for r in kv[1])):
            arr = (C.c_void_p * len(rs))(*[r.h for r in rs])
            E._ck(A.lib().apus_replicas_launch(arr, len(rs), target), "apus_replicas_launch")

    def wait(self, timeout_ms=120_000):
        for r in self.local:
            r.wait(timeout_ms)

    def stop(self):
        arr = (C.c_void_p * len(self.local))(*[r.h for r in self.local])
        self.E._ck(self.A.lib().apus_replicas_stop(arr, len(self.local)), "apus_replicas_stop")

    def submit(self, typ, conn, req, payload=b""):
        self.tickets = self.leader.submit(typ, conn, req, payload)
        return self.tickets

    def submit_uniform(self, nreq, length, conn, first_req, payloads):
        types = np.full(nreq, SEND, dtype=np.uint8)
        conns = np.full(nreq, conn, dtype=np.uint16)
        reqs = np.arange(first_req, first_req + nreq, dtype=np.uint64)
        lens = np.full(nreq, length, dtype=np.uint16)
        t0 = self.leader.submit_batch(types, conns, reqs, lens, payloads, length)
        self.tickets = t0 + nreq - 1
        return self.tickets

    def close(self):
        for r in self.local:
            r.close()


def run_ours(args):
    import __graft_entry__ as ge
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    import apus_b200 as A
    from apus_b200 import engine as E

    if not torch.cuda.is_available() or A.lib().apus_device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    numa_node = E.pin_to_device_node(local)        # submitting / spinning threads and the pinned rings next to the leader's GPU

    n, payload = args.replicas, args.payload
    K, W = args.steps, args.warmup
    L = args.log_size or A.LOG_SIZE
    stride = 64 + payload
    batch = default_batch(args)
    inline = (2 + payload) <= 80                       # APUS_SLOT_INLINE: image rides in the 128 B slot
    img = 0 if inline else (2 + payload + 15) // 16 * 16
    total_req = (K + W) * batch + 64
    slots = 1 << max(16, (total_req - 1).bit_length())
    ring_bytes = ((total_req * img + (1 << 20)) + 4095) // 4096 * 4096
    if ring_bytes // 16 > 0xFFFFFF:
        raise SystemExit("steps*batch*payload too large for the device payload ring (256 MiB): lower --batch or --steps")
    xflag = (E.F_NO_EXPRESS if args.no_express else 0) | (E.F_PROFILE if args.profile_latency else 0)
    flags = E.F_DEVICE_STATS | E.F_AUTOPRUNE | xflag
    vflags = (E.F_AUTOPRUNE | xflag) if args.no_stats else flags
    SEED = 0xA5A50000 + payload

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    gloo = dist.new_group(backend="gloo") if world > 1 else None

    def host_barrier():
        # while the resident kernels run, nothing may synchronise the whole device
        if world > 1:
            dist.barrier(group=gloo)

    def log(msg):
        if rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)

    def max_over_ranks_host(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=gloo)
        return float(t.item())

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    conn = 0

    # =========================== parity: the placement of this run against the oracle =====
    parity = None
    if not args.no_parity:
        parity = parity_leg(A, E, args, dist, gloo, rank, world, local, log)
        if parity and not (parity["replicas_equal"] and parity["oracle_equal"]):
            if rank == 0:
                print(json.dumps({"metric": "committed ops/s", "value": 0, "parity": parity,
                                  "error": "PARITY MISMATCH: replica logs differ from the oracle"}), flush=True)
            raise SystemExit(3)

    # =========================== value: inputs resident in HBM ===========================
    cell = Cell(A, E, args, A.RING_DEVICE, slots, ring_bytes, vflags, dist, rank, world, local)
    cell.submit(E.CONFIG, 0, 0, E.cid_image(n)) if n > 1 else None
    cell.submit(CONNECT, conn, 1, b"")
    barrier()
    cell.launch(cell.tickets); cell.wait()
    req = 2
    targets = []
    cell.leader.defer(True)
    for s in range(W + K):
        t0 = cell.leader.submit_synth(batch, SEND, conn, req, payload, SEED)     # fill kernel: straight into the HBM ring
        cell.tickets = t0 + batch - 1
        req += batch
        targets.append(cell.tickets)
    cell.leader.flush()            # every step's requests are now in the HBM ring, doorbell rung
    cell.leader.defer(False)
    for s in range(W):
        barrier()
        cell.launch(targets[s]); cell.wait()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    kernel_ms = 0.0
    barrier()
    t0 = time.perf_counter()
    for s in range(W, W + K):
        cell.launch(targets[s]); cell.wait()
        kernel_ms += cell.leader.last_launch_ms()
    barrier()
    t1 = time.perf_counter()
    clocks = sampler.stop() if rank == 0 else None
    elapsed = max_over_ranks(t1 - t0)
    kernel_ms = max_over_ranks(kernel_ms)
    st = cell.leader.stats()
    assert st["tickets_committed"] == targets[-1], (st, targets[-1])
    value = world * K * batch / elapsed
    log(f"value: {value:.0f} ops/s, {1e3 * elapsed / K:.3f} ms/step, kernel {kernel_ms / K:.3f} ms/launch")
    launches = K * len(cell.devices) * world
    lat_dev = cell.leader.latency_ns()
    auto_heads = st["auto_heads"]
    log(f"leader phases (ns, cumulative): {st['phase_ns']}")
    log(f"worker-0 turns [claim-wait ns, place-wait ns, publish-wait ns, fast placements, slow placements, express, claims, place-hold ns]: {st['turn_ns'][:8]}")
    batches = st["batches"]
    off = cell.leader.offsets()
    # every replica this rank hosts holds the leader's live log (size-independent property of the timed run itself)
    live = live_log_check(cell, dist, gloo, rank, world, n, L) if not args.no_parity else None
    if args.dump_outputs and rank == 0:
        dump_outputs(cell, args.dump_outputs, req - 1, st["tickets_committed"], payload)
    cell.close()

    # =========================== e2e: host buffers through the C ABI =====================
    e2e = None
    lat_host = None
    if not args.no_e2e:
        payloads = np.random.default_rng(SEED).integers(0, 256, size=batch * max(payload, 1), dtype=np.uint8)
        mode = A.RING_HOST_MAPPED if args.e2e_ring == "mapped" else A.RING_DEVICE
        e_slots = 1 << max(16, (2 * batch - 1).bit_length())
        e_bytes = ((2 * batch * img + (1 << 20)) + 4095) // 4096 * 4096
        cell = Cell(A, E, args, mode, e_slots, e_bytes, flags, dist, rank, world, local)
        barrier()
        cell.launch(UINT64_MAX)     # resident kernels: from here on no device-wide synchronisation
        log("e2e: resident kernels launched")
        if n > 1:
            cell.submit(E.CONFIG, 0, 0, E.cid_image(n))
        t = cell.submit(CONNECT, conn, 1, b"")
        cell.leader.wait_committed(t, 20_000_000)
        req = 2

        def e2e_step():
            nonlocal req
            t0_ = cell.leader.submit_uniform(batch, SEND, conn, req, payload, payloads)
            req += batch
            cell.leader.wait_committed(t0_ + batch - 1, 120_000_000)

        for s in range(W):
            e2e_step()
        host_barrier()
        es0 = cell.leader.stats()
        t0 = time.perf_counter()
        for s in range(K):
            e2e_step()
        t1 = time.perf_counter()
        es1 = cell.leader.stats()
        host_barrier()
        log("e2e, worker-0 phase ns per tile [wait for requests, T1 fetch, T2 place, T3 prefill, T4 compose, T5 store, T6 publish]: "
            f"{[round((b - a) / max(1, es1['phase_ns'][7] - es0['phase_ns'][7])) for a, b in zip(es0['phase_ns'][:7], es1['phase_ns'][:7])]} "
            f"over {es1['phase_ns'][7] - es0['phase_ns'][7]} tiles")
        e_elapsed = max_over_ranks_host(t1 - t0)
        e2e = {"value": round(world * K * batch / e_elapsed, 1), "unit": "ops/s",
               "h2d_bytes_per_step": batch * (96 + img), "d2h_bytes_per_step": 16,
               "ms_per_step": round(1e3 * e_elapsed / K, 4),
               "submit_threads": int(os.environ.get("apus_submit_threads", "8")),
               "path": f"apus_submit_uniform(host numpy buffer, engine host threads) -> {args.e2e_ring} submission ring "
                       f"(pinned host memory read by the kernel over PCIe: 96 of the 128 slot bytes) -> resident kernels "
                       f"-> apus_wait_committed (16 B pinned commit record)"}
        # closed loop, one request in flight: host-view commit latency (proxy.c:160 spin)
        if rank == 0 and args.lat_requests > 0:
            st0 = cell.leader.stats()
            f0 = [r.stats()["phase_ns"] for r in cell.local if not r.is_leader]
            lats = cell.leader.closed_loop(args.lat_requests, payload, conn, req)
            st1 = cell.leader.stats()
            f1 = [r.stats()["phase_ns"] for r in cell.local if not r.is_leader]
            nx = max(1, st1["turn_ns"][5] - st0["turn_ns"][5])
            if args.profile_latency:
                log("closed loop, leader express ns per request [place, compose, push, publish turn, publish]: "
                    f"{[round((b - a) / nx) for a, b in zip(st0['phase_ns'][1:6], st1['phase_ns'][1:6])]} over {nx} requests")
                log("closed loop, followers [certificates verified, ns first sight -> verified (mean), verify retries]: "
                    f"{[(b[0] - a[0], round((b[1] - a[1]) / max(1, b[0] - a[0])), b[2] - a[2]) for a, b in zip(f0, f1)]}")
            req += args.lat_requests
            lats = np.sort(lats[args.lat_requests // 10:].astype(np.float64)) / 1e3
            lat_host = {"p50_us": round(float(lats[len(lats) // 2]), 2), "p99_us": round(float(lats[int(len(lats) * 0.99)]), 2),
                        "p999_us": round(float(lats[int(len(lats) * 0.999)]), 2), "min_us": round(float(lats[0]), 2),
                        "n": int(len(lats)), "express_requests": st1["turn_ns"][5] - st0["turn_ns"][5],
                        "what": "apus_closed_loop (C ABI): enqueue one request, spin on the pinned "
                                "commit word until it is committed; host clock, one request in flight"}
            d = cell.leader.latency_ns(args.lat_requests - args.lat_requests // 10)
            if len(d):
                d = np.sort(d.astype(np.float64)) / 1e3
                lat_host["device_p50_us"] = round(float(d[len(d) // 2]), 2)
                lat_host["device_p99_us"] = round(float(d[int(len(d) * 0.99)]), 2)
            log(f"closed loop: {lat_host}")
        host_barrier()
        cell.stop()
        cell.close()
        log(f"e2e done: {e2e}")

    # =========================== the reference's own proxy.c on the engine, 16 connections ==========
    proxy_leg = None
    if rank == 0 and world == 1 and not args.no_proxy_leg and not args.no_e2e:
        try:
            proxy_leg = proxy_closed_loop_leg(args, n, payload, log)
        except Exception as ex:                                   # noqa: BLE001 - reported in the JSON line
            proxy_leg = {"unavailable": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # =========================== CPU baseline, JSON line ==================================
    if rank != 0:
        return
    cpu = None if (args.no_cpu or world > 1) else cpu_baseline(n, payload, batch)
    alg_bytes_per_op = (n - 1) * (64 + payload)
    ach = alg_bytes_per_op * batch / (kernel_ms / K * 1e-3) / 1e9
    if world == 1 and not args.spread:
        peak, peak_src = hbm_peak()
        bound = "hbm"
    else:
        peak, peak_src = NVLINK_PEER_GBS, "measured NVLink peer copy per direction (B200_PROFILING.md)"
        bound = "nvlink"
    dl = np.sort(lat_dev.astype(np.float64)) / 1e3 if len(lat_dev) else None
    out = {
        "metric": "committed ops/s", "value": round(value, 1), "unit": "ops/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": round(1e3 * elapsed / K, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {
            "workload": f"{n}-replica Paxos group, {payload} B SEND requests, {batch} requests per step "
                        f"({K * batch} in the timed region), device-resident submission ring",
            "replicas": n, "payload_bytes": payload, "batch": batch, "groups": world,
            "placement": ("all replicas of the group on GPU 0" if world == 1 and not args.spread else
                          ("replica r on GPU r % visible GPUs, one process" if world == 1 else
                           f"group g led by GPU g, replica r on GPU (g + r) % {world}, one process per GPU, CUDA IPC")),
            "log_ring_bytes": L, "log_pruning": "device-side HEAD entries (APUS_F_AUTOPRUNE)",
            "host_numa_node": numa_node,
            "cache": f"inputs larger than L2: {(K + W) * batch * (128 + img) >> 20} MiB of requests stream through once; "
                     f"every step writes {batch * stride >> 20} MiB into each replica's {L >> 20} MiB log ring",
        },
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches,
        "parity": parity if parity is None else dict(parity, live_log=live),
        "roofline": {"bound": bound, "achieved": round(ach, 3), "peak": peak, "unit": "GB/s",
                     "frac": round(ach / peak, 6),
                     "traffic": (ncu_traffic(n, payload, batch, args.leader_ctas) if world == 1 and not args.spread else None),
                     "traffic_note": "bytes per launch (dram read+write), profiles/r2_ncu.json (ncu --set full of this configuration: above "
                                     "the algorithmic bytes because the leader's own copy, the slot reads and the hole-preserving "
                                     f"prefill read reach DRAM once the rings outgrow the L2); algorithmic bytes per launch = {alg_bytes_per_op * batch}",
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_op": alg_bytes_per_op,
                     "kernel": "apus_replica_kernel (one fused launch per step: leader CTAs + follower CTAs)",
                     "kernel_ms_per_launch": round(kernel_ms / K, 4)},
        "cpu_baseline": cpu,
        "latency": {"device_commit_us": (None if dl is None else
                                         {"p50": round(float(dl[len(dl) // 2]), 2), "p99": round(float(dl[int(len(dl) * 0.99)]), 2),
                                          "n": int(len(dl)), "what": "per replicate step: dequeue -> majority observed (%globaltimer), "
                                                                     "open-loop run (queueing included)"}),
                    "closed_loop": lat_host},
        "proxy_closed_loop": proxy_leg,
        "engine": {"replicate_steps": batches, "auto_head_entries": auto_heads, "final_offsets": off,
                   "leader_phase_ns": dict(zip(["wait", "T1_fetch", "T2_place", "T3_prefill", "T4_compose", "T5_store",
                                                "T6_publish", "tiles"], st["phase_ns"]))},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------
# parity legs (outside every timed region; the oracle is the checker, never the thing measured)
# ------------------------------------------------------------------------------------
PARITY_REQ = 1 << 16


def parity_stream(n, payload, leader_idx=0):
    import streams as S
    nreq = max(2048, min(PARITY_REQ, (24 << 20) // (64 + payload)))
    return S.uniform_stream(nreq, payload, conns=4, leader=leader_idx)


def parity_leg(A, E, args, dist, gloo, rank, world, local, log):
    """A bounded stream (prologue + 4 connections x up to 2^16 requests of the benchmark's size) through the SAME
    placement the timed run uses; every replica's log ring is compared byte for byte with the oracle's image of that
    replica (reply bytes included).  Under torchrun every rank checks the replicas it hosts and the verdicts are
    gathered over gloo -- followers of group g live on other GPUs than its leader, so equality here is equality
    across NVLink."""
    import hashlib
    import orc as O
    n, payload = args.replicas, args.payload
    Lp = 1 << 25                                           # 32 MiB ring: the stream stays inside one lap (no pruning)
    stream = parity_stream(n, payload)
    flags = E.F_DEVICE_STATS | (E.F_NO_EXPRESS if args.no_express else 0)
    pargs = argparse.Namespace(**vars(args))
    pargs.log_size = Lp
    cell = Cell(A, E, pargs, A.RING_HOST_MAPPED, 1 << 17, 64 << 20, flags, dist, rank, world, local)
    try:
        if n > 1:
            cell.submit(E.CONFIG, 0, 0, E.cid_image(n))
        lead = cell.leader
        lead.defer(True)
        for typ, clt, rid, pl in stream:
            cell.tickets = lead.submit(typ, clt, rid, pl)
        lead.flush(); lead.defer(False)
        import torch
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        cell.launch(cell.tickets); cell.wait()
        # the oracle's image of every replica index (the same stream in every group)
        O.build_oracle()
        orc = O.Oracle("orc")
        orc.set_rules(O.RULES_ENGINE)
        c = O.Cluster(orc, n, leader=0, term=1, length=Lp)
        if n > 1:
            c.prologue()
        for typ, clt, rid, pl in stream:
            assert c.submit(typ, clt, rid, O.cmd_image(pl))
        c.round(); c.round()
        mine = []
        for r in cell.local:
            img = r.image()
            oi = c.image(r.idx)
            oo, eo = c.offsets(r.idx), r.offsets()
            ok = bool(np.array_equal(img, oi)) and all(eo[k] == oo[k] for k in ("end", "commit", "apply", "head"))
            mine.append({"rank": rank, "device": r.device, "replica": r.idx, "oracle_equal": ok,
                         "sha": hashlib.sha256(img.tobytes()).hexdigest()[:16], "end": eo["end"]})
        c.close()
    finally:
        cell.close()
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine, group=gloo)
        allr = [x for part in gathered for x in part]
    else:
        allr = mine
    # replicas_equal: per replica index every group produced the same image (same stream), and all ends agree
    by_idx = {}
    for x in allr:
        by_idx.setdefault(x["replica"], set()).add(x["sha"])
    replicas_equal = all(len(v) == 1 for v in by_idx.values()) and len({x["end"] for x in allr}) == 1
    res = {"checked": True, "groups": world, "replicas_checked": len(allr),
           "gpus_holding_replicas": len({(x["rank"], x["device"]) for x in allr}),
           "replicas_equal": bool(replicas_equal), "oracle_equal": bool(all(x["oracle_equal"] for x in allr)),
           "stream": f"CONFIG prologue + 4 connections x {len(stream) - 4} SEND requests of {payload} B, {Lp >> 20} MiB ring, "
                     f"every byte of every replica's ring vs the CPU oracle (ENGINE rules), reply bytes included"}
    log(f"parity: {res}")
    return res


def live_log_check(cell, dist, gloo, rank, world, n, L):
    """After the timed (multi-lap, auto-pruned) run: hash of the live log [head, end) with reply bytes masked, per
    replica; every follower must hold exactly its leader's bytes and entries must parse with consecutive idx."""
    import hashlib
    import orc as O
    TAIL = 4096
    mine = []
    for r in cell.local:
        o = r.offsets()
        img = r.image()
        ents = O.walk_entries(img, o["head"], o["end"], L) if o["end"] != L else []
        first = int.from_bytes(img[ents[0][0]:ents[0][0] + 8].tobytes(), "little") if ents else 0
        last = int.from_bytes(img[ents[-1][0]:ents[-1][0] + 8].tobytes(), "little") if ents else 0
        consecutive = (not ents) or (last - first == len(ents) - 1)
        tail = ents[-TAIL:]
        m = O.mask_replies(img, tail)
        h = hashlib.sha256()
        for e, stride in tail:
            h.update(m[e:e + stride].tobytes())
        group = (rank - r.idx) % world if world > 1 else 0
        mine.append({"group": group, "replica": r.idx, "sha": h.hexdigest()[:16], "end": o["end"], "commit": o["commit"],
                     "last_idx": last, "tail_entries": len(tail), "entries": len(ents), "consecutive": bool(consecutive)})
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine, group=gloo)
        allr = [x for part in gathered for x in part]
    else:
        allr = mine
    ok = True
    for g in {x["group"] for x in allr}:
        grp = [x for x in allr if x["group"] == g]
        ok = (ok and len(grp) == n and all(x["consecutive"] for x in grp)
              and len({(x["sha"], x["end"], x["commit"], x["last_idx"], x["tail_entries"]) for x in grp}) == 1)
    return {"followers_equal_leader": bool(ok), "entries_compared_per_replica": int(allr[0]["tail_entries"]) if allr else 0,
            "what": "after the timed multi-lap run: the newest entries of every replica's live log (reply bytes masked), end, commit "
                    "and last idx equal within each group; entries parse with consecutive idx from head to end"}


def dump_outputs(cell, directory, last_req, committed, payload):
    """What the timed path hands its caller, for comparing two builds output for output: every hosted replica's copy of
    the newest requests of the last step (a step is larger than the log ring, so only its newest requests are still
    live; at most 4096 of them, and at most 64 MiB in all), and the number of committed tickets.

      requests.npy           float64 [replica, request, (term, req_id, connection, type, sender)]
      payloads.npy           float32 [replica, request, byte]
      tickets_committed.npy  float64 [1]

    Left out: the entry's idx, which counts the HEAD entries the pruning rule interleaves at timing-dependent places, the
    reply bytes (acks, also timing) and padding (whatever an earlier lap of the ring left there)."""
    import orc as O
    os.makedirs(directory, exist_ok=True)
    count = max(1, min(4096, (64 << 20) // ((4 * payload + 40) * len(cell.local))))
    reqs, pays = [], []
    for r in cell.local:
        o = r.offsets()
        img = r.image()
        ents = O.walk_entries(img, o["head"], o["end"], cell.L) if o["end"] != cell.L else []
        sends = [e for e, _ in ents if img[e + 26] == SEND][-count:]
        hdr = np.stack([img[e:e + 28] for e in sends]) if sends else np.zeros((0, 28), np.uint8)
        fields = np.stack([hdr[:, 8:16].copy().view("<u8")[:, 0], hdr[:, 16:24].copy().view("<u8")[:, 0],
                           hdr[:, 24:26].copy().view("<u2")[:, 0], hdr[:, 26], hdr[:, 27]], axis=1).astype(np.float64)
        if fields[:, 1].tolist() != list(range(last_req - count + 1, last_req + 1)):
            raise SystemExit(f"--dump-outputs: replica {r.idx} does not hold the newest {count} requests "
                             f"(found {len(sends)}, expected req_ids up to {last_req})")
        reqs.append(fields)
        pays.append(np.stack([img[e + 50:e + 50 + payload] for e in sends]).astype(np.float32))
    np.save(os.path.join(directory, "requests.npy"), np.stack(reqs))
    np.save(os.path.join(directory, "payloads.npy"), np.stack(pays))
    np.save(os.path.join(directory, "tickets_committed.npy"), np.array([committed], dtype=np.float64))


def proxy_closed_loop_leg(args, n, payload, log, conns=16, nreq=20000, steps=3):
    """The reference's UNMODIFIED proxy.c (oracle/_ref/libref_proxy.so) on libapus_dare.so/libapus_gpu.so, one process per
    replica, driven by the same multi-threaded closed-loop application driver the reference arm uses on its own stack
    (oracle/app_driver.inc): 16 connections, every proxy_on_read returns at commit.  This is the like-for-like
    counterpart of `bench.py --impl reference`."""
    import tempfile
    refproxy = os.path.join(ROOT, "oracle", "_ref", "libref_proxy.so")
    if not os.path.exists(refproxy):
        return {"unavailable": "oracle/_ref/libref_proxy.so absent"}
    import apus_b200 as A
    nd = max(1, A.lib().apus_device_count())
    cores = host_cores()
    threads = max(1, min(conns, cores - n))
    # one GPU cannot run the persistent kernels of several processes at once (contexts are time-sliced): with fewer GPUs than
    # replicas the followers' replicas live in the leader's process (kernels only, apus_colocate_followers)
    colocate = nd < n or not args.spread
    with tempfile.TemporaryDirectory() as d:
        env = dict(os.environ, apus_rendezvous=os.path.join(d, "rdv"), PROXY_RUN_TIMEOUT="120", APUS_NO_BUILD="1")
        procs = []
        for i in range(1 if colocate else n):
            e = dict(env, apus_gpu=("0" if colocate else str(i % nd)))
            if colocate:
                e["apus_colocate_followers"] = "1"
            procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "proxy_worker.py"), str(i), str(1 if colocate else n),
                                           str(conns), str(nreq), str(payload), d, str(threads), str(steps)] + ([str(n)] if colocate else []),
                                          env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
        outs = []
        try:
            for p in procs:
                outs.append(p.communicate(timeout=300)[0].decode(errors="replace"))
        finally:
            for p in procs:
                if p.poll() is None:
                    p.kill()
        path = os.path.join(d, "result0.json")
        if not os.path.exists(path):
            return {"unavailable": "leader process produced no result: " + outs[0][-300:]}
        r0 = json.load(open(path))
        followers_ok = 0
        for i in range(1, 1 if colocate else n):
            fp = os.path.join(d, f"result{i}.json")
            if os.path.exists(fp) and json.load(open(fp)).get("bytes") == nreq * payload * steps:
                followers_ok += 1
    timed = r0["steps"][1:]
    ops = sum(s_["requests"] + 2 * conns for s_ in timed) / sum(s_["seconds"] for s_ in timed)
    res = {"value": round(ops, 1), "unit": "ops/s", "connections": conns, "app_threads": threads, "replica_processes": n,
           "p50_us": round(statistics.median(s_["p50_us"] for s_ in timed), 2), "p99_us": round(max(s_["p99_us"] for s_ in timed), 2),
           "followers_replayed_everything": (None if colocate else followers_ok == n - 1),
           "what": f"unmodified src/proxy/proxy.c on the engine, " + (f"{n} replicas on GPU 0, the followers' replicas hosted by the leader's process "
                   f"(kernels only: one GPU cannot run kernels of several processes concurrently), " if colocate else f"{n} replica processes, one GPU each, ") +
                   f"{conns} connections closed loop on {threads} application threads, {len(timed)} x {nreq} requests of {payload} B "
                   f"after one warm-up session; latency = proxy_on_read call (returns at commit); same driver and shape as --impl reference"}
    log(f"proxy leg: {res}")
    return res


def run_failover(args):
    """Leader failover mid-run (BASELINE config 5): tools/failover_drill.py, twice -- with the timeouts the reference ships in
    target/nodes.local.cfg (hb 10 ms, detection after 10 missed beats, election timeout 100-300 ms; its own stack needs
    ~0.35 s with these, profiles/r1_refstack_failover_buildbox.txt) and with timeouts sized for heartbeats that are
    written by a GPU kernel every 200 us."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import __graft_entry__ as ge
    ge.build()
    import apus_b200 as A
    import failover_drill as FD
    nd = max(1, A.lib().apus_device_count())
    n = args.replicas
    out = {"metric": "leader failover: kill -> new leader serving", "unit": "ms", "higher_is_better": False, "n_gpus": min(nd, n),
           "data": "synthetic", "dtype": "u8", "config": {"workload": f"{n} replica processes (unmodified proxy.c on the engine), closed-loop "
                                                                      f"{args.payload} B requests, leader killed with SIGKILL after 1 s",
                                                          "replicas": n, "placement": "all replica processes on GPU 0 (time-sliced contexts: the latencies are "
                                                                                      "dominated by the driver's time slices, see tools/failover_drill.py)"}}
    trials = []
    for _ in range(args.failover_trials):
        r = FD.run(n=n, plen=args.payload, spread=False, ndev=nd, kill_after_s=1.0)
        trials.append({"new_leader": r["new_leader"], "term": r["term"], "kill_to_leader_line_ms": r["recovery_ms_kill_to_leader_line"],
                       "kill_to_first_commit_ms": r["recovery_ms_kill_to_first_commit"], "requests_before_kill": r["requests_before_kill"],
                       "hb_period_us": r["hb_period_us"], "hb_timeout_us": r["hb_timeout_us"], "election_timeout_us": r["elec_timeout_us"]})
    out["trials"] = trials
    out["value"] = statistics.median(t["kill_to_first_commit_ms"] for t in trials)
    out["note"] = ("replica processes share one GPU (their contexts are time-sliced), so the failure detector runs with a 400 ms heartbeat "
                   "timeout and the reference's 100-300 ms election timeouts; the reference's own stack needs ~350 ms with its shipped "
                   "timeouts (profiles/r1_refstack_failover_buildbox.txt)")
    print(json.dumps(out), flush=True)


def main():
    args = parse()
    if args.failover:
        run_failover(args)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
