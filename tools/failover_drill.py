#!/usr/bin/env python
"""Leader-failover drill on the GPU engine (BASELINE config 5; the analogue of benchmarks/reconf_bench.sh:249-343, which
starts the replicas, loads the leader, `kill`s it and greps the survivors' logs for the next "] LEADER" line).

n replica processes (tests/failover_worker.py: the reference's unmodified proxy.c on libapus_dare.so / libapus_gpu.so);
replica 0 leads and is loaded in a closed loop; after `kill_after_s` it is killed with SIGKILL.  The survivors' failure
detector (heartbeat words written by the leader KERNEL) fires, they elect, the winner adjusts the others' logs and goes on
serving.  Reported: kill -> "] LEADER" (what reconf_bench.sh measures) and kill -> first commit of the new leader.

    python tools/failover_drill.py [--replicas 5] [--spread] [--hb-us 200] [--hb-timeout-us 4000] [--elec-us 2000,6000]
"""
import argparse
import json
import os
import signal
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(n=5, nconn=4, nreq2=2000, plen=64, kill_after_s=1.0, spread=False, hb_us=200, hb_timeout_us=4000, elec_us="2000,6000",
        log_size=1 << 24, keep=None, ndev=1, config_timeouts=False):
    ndev = 1                      # (see the placement note below)
    if ndev < n and not config_timeouts:
        # fewer GPUs than replica processes: the contexts are time-sliced (milliseconds), a heartbeat timeout sized for
        # a resident kernel would fire spuriously -- functional run only, the latencies mean nothing here
        hb_us, hb_timeout_us, elec_us = max(hb_us, 2000), max(hb_timeout_us, 400000), "100000,300000"
    d = keep or tempfile.mkdtemp(prefix="apus-failover-")
    os.makedirs(d, exist_ok=True)
    env = dict(os.environ, apus_rendezvous=os.path.join(d, "rdv"), apus_log_size=str(log_size), APUS_NO_BUILD="1")
    if not config_timeouts:
        env.update(apus_hb_period_us=str(hb_us), apus_hb_timeout_us=str(hb_timeout_us), apus_elec_timeout_us=elec_us)
    procs = []
    for i in range(n):
        # All replica processes share GPU 0 for now.  With one GPU per process the survivors' kernels keep storing acks into
        # the killed leader's region for a heartbeat timeout, and a cudaIpc mapping of memory whose exporter died is not
        # kept alive across GPUs (observed on the 8-GPU box: the drill hangs); the fix is regions allocated with
        # cuMemCreate and imported by file descriptor -- the importer then holds its own reference (DESIGN.md section 7).
        e = dict(env, apus_gpu="0")
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "failover_worker.py"), str(i), str(n), str(nconn),
                                       str(nreq2), str(plen), d], env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    out = {"dir": d}
    try:
        t0 = time.time()
        while not os.path.exists(os.path.join(d, "phase1_started")):
            if time.time() - t0 > 90 or procs[0].poll() is not None:
                raise RuntimeError("the first leader never started:\n" + (procs[0].communicate()[0] or b"").decode(errors="replace")[-2000:])
            time.sleep(0.01)
        time.sleep(kill_after_s)
        pfile = os.path.join(d, "progress_p1.txt")
        before = int(open(pfile).read().split()[0]) if os.path.exists(pfile) else 0
        t_kill = time.time()
        os.kill(procs[0].pid, signal.SIGKILL)                     # reconf_bench.sh:265-289
        nl = os.path.join(d, "new_leader.json")
        while not os.path.exists(nl):
            if time.time() - t_kill > 60:
                raise RuntimeError("no new leader within 60 s:\n" + "\n".join(
                    open(os.path.join(d, f"dare{i}.log")).read()[-1500:] for i in range(1, n) if os.path.exists(os.path.join(d, f"dare{i}.log"))))
            time.sleep(0.0005)
        lead = json.load(open(nl))
        p2 = os.path.join(d, "progress_p2.txt")
        t_first = None
        while t_first is None and time.time() - t_kill < 60:
            if os.path.exists(p2):
                try:
                    t_first = float(open(p2).read().split()[1])
                except (IndexError, ValueError):
                    pass
            time.sleep(0.0005)
        # A survivor that answered too late for the winner's grace period is treated as failed and removed from the
        # configuration by the new leader (check_failure_count, dare_server.c:1189-1228): it keeps standing for election
        # without ever getting a vote and reports nothing.  The drill collects whoever reports within the deadline.
        res, missing = {}, []
        deadline = time.time() + 90
        for i in range(1, n):
            path = os.path.join(d, f"result{i}.json")
            while not os.path.exists(path) and time.time() < deadline and procs[i].poll() is None:
                time.sleep(0.05)
            time.sleep(0.05)
            if os.path.exists(path):
                res[i] = json.load(open(path))
            else:
                missing.append(i)
        if lead["idx"] not in res:
            p = procs[lead["idx"]]
            state = "still running" if p.poll() is None else f"exit code {p.returncode}"
            if p.poll() is None:
                p.kill()
            log = os.path.join(d, f"dare{lead['idx']}.log")
            raise RuntimeError(f"the new leader p{lead['idx']} produced no result ({state}; progress "
                               f"{open(p2).read().strip() if os.path.exists(p2) else 'none'}); its output:\n"
                               + (p.communicate()[0] or b"").decode(errors="replace")[-2000:]
                               + "\nits log:\n" + (open(log).read()[-3000:] if os.path.exists(log) else "absent"))
        logs = {i: open(os.path.join(d, f"dare{i}.log")).read() for i in range(n) if os.path.exists(os.path.join(d, f"dare{i}.log"))}
        out.update(new_leader=lead["idx"], term=lead["term"], requests_before_kill=before,
                   recovery_ms_kill_to_leader_line=round((lead["t_leader"] - t_kill) * 1e3, 2),
                   recovery_ms_kill_to_first_commit=(round((t_first - t_kill) * 1e3, 2) if t_first else None),
                   results=res, missing=missing, logs=logs, hb_period_us=hb_us, hb_timeout_us=hb_timeout_us, elec_timeout_us=elec_us)
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
        if keep is None:
            subprocess.run(["rm", "-rf", d])
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicas", type=int, default=5)
    ap.add_argument("--spread", action="store_true")
    ap.add_argument("--hb-us", type=int, default=200)
    ap.add_argument("--hb-timeout-us", type=int, default=4000)
    ap.add_argument("--elec-us", default="2000,6000")
    ap.add_argument("--reference-timeouts", action="store_true", help="hb 10 ms / timeout 100 ms / election 100-300 ms (target/nodes.local.cfg)")
    ap.add_argument("--trials", type=int, default=3)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    import apus_b200
    nd = max(1, apus_b200.lib().apus_device_count())
    kw = dict(hb_us=10000, hb_timeout_us=100000, elec_us="100000,300000") if a.reference_timeouts else dict(hb_us=a.hb_us, hb_timeout_us=a.hb_timeout_us, elec_us=a.elec_us)
    for t in range(a.trials):
        r = run(n=a.replicas, spread=a.spread, ndev=nd, **kw)
        print(f"trial {t}: leader p0 killed after {r['requests_before_kill']} requests -> p{r['new_leader']} is LEADER of term {r['term']} after "
              f"{r['recovery_ms_kill_to_leader_line']} ms; first commit of the new leader after {r['recovery_ms_kill_to_first_commit']} ms "
              f"(hb {kw['hb_us']} us, timeout {kw['hb_timeout_us']} us, election {kw['elec_us']} us)", flush=True)
