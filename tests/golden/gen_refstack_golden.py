#!/usr/bin/env python
"""Generate tests/golden/refstack_golden.json and refstack_runs_golden.json from the RUNNING REFERENCE: the reference's unmodified election /
replication / commit code and proxy.c (oracle/_ref/libref_stack.so on oracle/verbs_shim, built from /root/reference
by oracle/build_refapp.sh) execute each scenario as N processes; the fixture records, per replica, the offsets and
the SHA-256 of the log it left behind (leader: all bytes; followers: reply[0..12] masked, the H5 rule of SURVEY.md
s8c), with the leader index and term the election produced.  Run where /root/reference exists:

    python tests/golden/gen_refstack_golden.py

tests/test_golden.py replays the same streams through the oracle (anywhere) and tests/test_gpu_parity.py through the
CUDA engine and compares against these hashes; tests/test_oracle_vs_refstack.py compares the oracle with the runs
recorded in refstack_runs_golden.json."""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

import orc as O                          # noqa: E402
import refgold                           # noqa: E402
import refstack as R                     # noqa: E402
import test_oracle_vs_refstack as TVS    # noqa: E402

SCENARIOS = [dict(name="ref3_2conn_300x64", n=3, nconn=2, nreq=300, plen=64),
             dict(name="ref5_3conn_200x128", n=5, nconn=3, nreq=200, plen=128),
             dict(name="ref3_ragged_120_upto3000", n=3, nconn=1, nreq=120, plen=-3000),
             dict(name="ref7_4conn_400x64", n=7, nconn=4, nreq=400, plen=64)]


def digest(img, ents, mask):
    return hashlib.sha256((O.mask_replies(img, ents) if mask else img).tobytes()).hexdigest()


if __name__ == "__main__":
    assert R.available(), "needs oracle/_ref/libref_stack.so (oracle/build_refapp.sh, /root/reference)"
    out = []
    for sc in SCENARIOS:
        rr = R.run(sc["n"], sc["nconn"], sc["nreq"], sc["plen"], prune=1000.0)
        lead = rr["leader"]
        end = rr["results"][lead]["offsets"]["end"]
        ents = O.walk_entries(rr["images"][lead], 0, end, O.LOG_SIZE)
        out.append(dict(sc, leader=lead, term=rr["term"], end=end, entries=len(ents),
                        offsets=[{k: r["offsets"][k] for k in ("head", "apply", "commit", "end")} for r in rr["results"]],
                        sha256=[digest(rr["images"][i], ents, mask=(i != lead)) for i in range(sc["n"])],
                        replay_sha256=sorted(rr["results"][(lead + 1) % sc["n"]]["replay"]["sha"])))
        print(sc["name"], "leader", lead, "term", rr["term"], "end", end)
    path = os.path.join(HERE, "refstack_golden.json")
    with open(path, "w") as f:
        json.dump(dict(source="oracle/_ref/libref_stack.so: reference src/dare/*.c + proxy.c, unmodified, on oracle/verbs_shim",
                       scenarios=out), f, indent=1, sort_keys=True)
    print("wrote", path)
    refgold.write("refstack_runs_golden.json", "oracle/_ref/libref_stack.so: reference src/dare/*.c + proxy.c, unmodified "
                  "(commit 896959f), on oracle/verbs_shim", TVS.record())
    print("wrote refstack_runs_golden.json")
