"""Pins the oracle's CLUSTER restatement (oracle/cluster_sim.inc: submit, replicate, ack, commit scan, apply,
HEAD-entry pruning) against the reference ITSELF: the reference's unmodified election / replication / commit code
(src/dare/dare_server.c, dare_ibv_rc.c, dare_ibv_ud.c, dare_ibv.c) and proxy.c run here as N processes on the
verbs shim (oracle/verbs_shim; build recipe oracle/build_refapp.sh), an application driver issues a deterministic
request stream through proxy_on_accept/read/close, and the log the reference leaves behind is compared with the
log the oracle computes for the same stream -- every byte, reply bytes included.

What each run of the reference left behind is recorded in tests/golden/refstack_runs_golden.json
(tests/golden/gen_refstack_golden.py re-records it where the reference's sources exist): the leader index and term its
election produced, every replica's offsets, proxy counters and replayed streams, and of every replica's log the
SHA-256 of its bytes, the SHA-256 with reply bytes masked, and the distinct (sender, reply[0..12]) stamps its entries
carry.  The tests below compare the oracle with these recordings, so they run anywhere."""
import hashlib

import numpy as np
import pytest

import orc as O
import refstack as R
import streams as S
from refgold import recorded, sha

GOLD = "refstack_runs_golden.json"


def reference(key):
    return recorded(GOLD)[key]


def summarize_run(rr, entries=False):
    """A run of the reference stack (refstack.run) in the stored form, with the number of entries in the leader's log and
    the position and value of every HEAD entry in it; `entries`: also every request entry's position, type, connection,
    req_id, length and first payload byte."""
    lead = rr["leader"]
    limg = rr["images"][lead]
    end = rr["results"][lead]["offsets"]["end"]
    ents = O.walk_entries(limg, 0, end, O.LOG_SIZE)
    images = []
    for img in rr["images"]:
        stamps = {}
        for off, _ in ents:
            k = img[off + 27: off + 41].tobytes().hex()
            stamps[k] = stamps.get(k, 0) + 1
        images.append(dict(len=len(img), sha=sha(img), masked_sha=sha(O.mask_replies(img, ents)), stamps=stamps))
    out = dict(leader=lead, term=rr["term"], images=images,
               results=[{k: r[k] for k in ("leader", "offsets", "proxy", "replay")} for r in rr["results"]])
    seq, payloads = [], hashlib.sha256()
    for k, (off, _) in enumerate(ents):
        typ = int(limg[off + 26])
        if typ == O.HEAD:
            out.setdefault("heads", []).append([k, int(np.frombuffer(limg[off + 48: off + 56].tobytes(), dtype="<u8")[0])])
        elif entries and typ != O.NOOP and typ != O.CONFIG:
            ln = int(limg[off + 48]) | (int(limg[off + 49]) << 8)
            rid = int(np.frombuffer(limg[off + 16: off + 24].tobytes(), dtype="<u8")[0])
            clt = int(limg[off + 24]) | (int(limg[off + 25]) << 8)
            seq.append([k, typ, clt, rid, ln, int(limg[off + 50]) if ln else 0])
            payloads.update(limg[off + 50: off + 50 + ln].tobytes())
    out["entries"] = len(ents)
    if entries:
        out["requests"] = seq
        out["payloads_sha"] = payloads.hexdigest()
    return out


def pattern_payload(first, ln):
    """The driver's payloads: byte k of request i is (i * 31 + k) & 0xFF (refstack.expected_stream), so the first byte
    determines the rest; the recording's SHA-256 of all payloads checks that."""
    return bytes(((first + k) & 0xFF) for k in range(ln))



def oracle_for(orc, rr, n, nconn, nreq, plen):
    orc.set_rules(O.RULES_REFERENCE)
    c = O.Cluster(orc, n, leader=rr["leader"], term=rr["term"], length=O.LOG_SIZE)
    c.prologue()
    for typ, clt, rid, payload in R.expected_stream(rr["leader"], nconn, nreq, plen):
        assert c.submit(typ, clt, rid, O.cmd_image(payload))
    for _ in range(2):
        c.round()
    return c


def check_replay(rr, nconn, nreq, plen):
    """followers replayed every connection's byte stream, in order, into their local application"""
    want = []
    for c in range(nconn):
        h = hashlib.sha256()
        for typ, clt, rid, payload in R.expected_stream(rr["leader"], nconn, nreq, plen):
            if typ == S.SEND and (clt & 0xFF) == c:
                h.update(payload)
        want.append(h.hexdigest())
    for r in rr["results"]:
        if not r["leader"]:
            assert r["replay"]["conns"] == nconn
            assert sorted(r["replay"]["sha"]) == sorted(want)


def check_follower_stamps(img, ents, i, lead, n):
    """A follower's copy of an entry carries whatever reply bytes the LEADER's copy held at the instant it was
    replicated (acks of faster followers; timing, the H5 mask of SURVEY.md s8c) plus its own ack (I7)."""
    assert sum(img["stamps"].values()) == len(ents)
    for k in img["stamps"]:
        rep = bytes.fromhex(k)[1:]
        assert rep[i] == 1 and rep[lead] == 0 and not any(rep[n:]), (i, k)


LOG_EQUALS = [(3, 2, 300, 64), (5, 3, 200, 128), (3, 1, 120, -3000), (7, 4, 400, 64)]
LOG_EQUALS_SHM = [(5, 3, 200, 128), (3, 1, 120, -3000)]


@pytest.mark.parametrize("n,nconn,nreq,plen", LOG_EQUALS)
def test_reference_log_equals_oracle_log(orc, n, nconn, nreq, plen):
    """log_pruning_period is set out of reach, so the log holds exactly CONFIG + the stream."""
    _log_equals_oracle(orc, reference(f"log_equals/{n}/{nconn}/{nreq}/{plen}"), n, nconn, nreq, plen)


@pytest.mark.parametrize("n,nconn,nreq,plen", LOG_EQUALS_SHM)
def test_reference_log_equals_oracle_log_shm_transport(orc, n, nconn, nreq, plen):
    """The shim's shm transport (the log re-backed by a shared mapping, RDMA WRITE = memcpy: what bench.py's reference arm
    also times) leaves the same logs as the process_vm transport."""
    _log_equals_oracle(orc, reference(f"log_equals_shm/{n}/{nconn}/{nreq}/{plen}"), n, nconn, nreq, plen)


def _log_equals_oracle(orc, rr, n, nconn, nreq, plen):
    c = oracle_for(orc, rr, n, nconn, nreq, plen)
    lead = rr["leader"]
    oo = c.offsets(lead)
    for i in range(n):
        ro = rr["results"][i]["offsets"]
        assert ro["end"] == oo["end"] and ro["head"] == 0 and ro["len"] == O.LOG_SIZE, (i, ro, oo, rr["term"], lead)
        assert ro["commit"] == ro["end"] == ro["apply"], ro
        if i == lead:
            assert ro["tail"] == oo["tail"]
        img, want = rr["images"][i], c.image(i, 0, oo["end"])
        assert img["len"] == oo["end"]
        ents = O.walk_entries(want, 0, oo["end"], O.LOG_SIZE)
        if i != lead:
            check_follower_stamps(img, ents, i, lead, n)
            assert img["masked_sha"] == sha(O.mask_replies(want, ents)), f"replica {i} (leader {lead}, term {rr['term']})"
        else:                                             # the leader's copy: every byte, reply bytes included
            assert img["sha"] == sha(want), f"replica {i} (leader {lead}, term {rr['term']})"
    if n > 1:
        check_replay(rr, nconn, nreq, plen)
    # what proxy.c / db-interface.c counted (the callbacks the engine entry must reproduce, SURVEY.md H4):
    # store_cmd once per entry on every replica -- 4 B records for CONNECT/CLOSE, 24 B for SEND whatever its payload;
    # update_state once per committed request on the leader
    for r in rr["results"]:
        assert r["proxy"]["records_len"] == 8 * nconn + 24 * nreq, r["proxy"]
        if r["leader"]:
            assert r["proxy"]["highest_rec"] == r["proxy"]["cur_rec"] == 2 * nconn + nreq
    c.close()


PRUNING = (3, 2, 6000, 64)


def test_reference_pruning_matches_oracle_rules(orc):
    """With the stock log_pruning_period (0.05 s) the reference leader interleaves HEAD entries at timer-dependent
    places.  Their PLACEMENT is timing; their content and consequences are rules the oracle restates:
    a HEAD entry carries the new head, which is an earlier entry boundary, larger than the previous head, never two
    HEAD entries in a row (dare_server.c:1996-2067, dare_log.h:472-478); followers adopt it (dare_server.c:2163-2186).
    Rebuilding the log with the oracle's append -- the stream plus HEAD entries where the reference put them --
    must reproduce the reference's bytes."""
    n, nconn, nreq, plen = PRUNING
    rr = reference("pruning")
    lead = rr["leader"]
    end = rr["results"][lead]["offsets"]["end"]
    stream = iter(R.expected_stream(lead, nconn, nreq, plen))
    orc.set_rules(O.RULES_REFERENCE)
    log = O.Log(orc, O.LOG_SIZE)
    heads, prev_head, prev_was_head = [], 0, False
    head_at = dict(rr.get("heads", []))
    for k in range(rr["entries"]):
        if k == 0:
            assert k not in head_at
            assert log.append(rr["term"], 0, 0, O.CONFIG, O.cid_image(n)) == 1
            typ = O.CONFIG
        elif k in head_at:
            h = head_at[k]
            assert h > prev_head and not prev_was_head
            heads.append((k, h))
            prev_head = h
            assert log.append(rr["term"], 0, 0, O.HEAD, h.to_bytes(8, "little")) == k + 1
            typ = O.HEAD
        else:
            typ, clt, rid, payload = next(stream)
            assert log.append(rr["term"], rid, clt, typ, O.cmd_image(payload)) == k + 1
        prev_was_head = typ == O.HEAD
    assert next(stream, None) is None, "every request is in the log"
    assert len(heads) >= 2, "the run was long enough to prune"
    want = log.image(0, end)
    ents = O.walk_entries(want, 0, end, O.LOG_SIZE)
    assert len(ents) == rr["entries"]
    bounds = {off for off, _ in ents}
    for k, h in heads:
        assert h in bounds and h < ents[k][0], "the new head is an earlier entry boundary"
    for off, _ in ents:                       # the single-log oracle has no followers and no leader stamp
        want[off + 27] = lead
    got = rr["images"][lead]["masked_sha"]
    assert got == sha(O.mask_replies(want, ents))
    last_heads = [h for _, h in heads[-2:]]
    for i in range(n):
        ro = rr["results"][i]["offsets"]
        assert ro["end"] == end and ro["commit"] == end
        assert ro["head"] in last_heads, "every replica adopted one of the last heads"
        assert rr["images"][i]["masked_sha"] == got
    log.close()
    check_replay(rr, nconn, nreq, plen)


I7 = (3, 1, 100, 64)


def test_reference_reply_bytes_invariant_I7(orc):
    """At quiescence the leader's copy of an entry holds reply[f] == 1 for every follower f and follower f's own copy
    holds reply[f] == 1 (dare_ibv_rc.c:1838-1839) -- the bytes the GPU engine also deposits."""
    n, nconn, nreq, plen = I7
    rr = reference("I7")
    lead = rr["leader"]
    c = oracle_for(orc, rr, n, nconn, nreq, plen)
    end = c.offsets(lead)["end"]
    ents = O.walk_entries(c.image(lead, 0, end), 0, end, O.LOG_SIZE)
    c.close()
    for i in range(n):
        img = rr["images"][i]
        assert sum(img["stamps"].values()) == len(ents)
        for k in img["stamps"]:
            sender, rep = bytes.fromhex(k)[0], bytes.fromhex(k)[1:]
            if i == lead:
                assert all(rep[f] == 1 for f in range(n) if f != lead) and rep[lead] == 0 and not any(rep[n:])
            else:
                assert rep[i] == 1 and rep[lead] == 0
            assert sender == lead          # sender stamped before replication (dare_server.c:1803)


def random_shape(seed):
    """Group size, connection count, request count and payload regime drawn from a seeded generator."""
    rng = np.random.default_rng(0xA5A5 + seed)
    n = int(rng.choice([3, 5]))
    nconn = int(rng.integers(1, 7))
    nreq = int(rng.integers(50, 500))
    plen = int(rng.choice([1, 17, 64, 255, 1024, -200, -1500, -9000]))
    return n, nconn, nreq, plen


RANDOM_SEEDS = [1, 2, 3]


@pytest.mark.parametrize("seed", RANDOM_SEEDS)
def test_reference_log_equals_oracle_log_random_shapes(orc, seed):
    n, nconn, nreq, plen = random_shape(seed)
    rr = reference(f"random_shape/{seed}")
    c = oracle_for(orc, rr, n, nconn, nreq, plen)
    lead = rr["leader"]
    end = c.offsets(lead)["end"]
    ents = O.walk_entries(c.image(lead, 0, end), 0, end, O.LOG_SIZE)
    assert len(ents) == 1 + 2 * nconn + nreq
    for i in range(n):
        assert rr["results"][i]["offsets"]["end"] == end, (n, nconn, nreq, plen)
        img, want = rr["images"][i], c.image(i, 0, end)
        if i != lead:
            assert img["masked_sha"] == sha(O.mask_replies(want, ents)), (i, lead, n, nconn, nreq, plen)
        else:
            assert img["sha"] == sha(want), (i, lead, n, nconn, nreq, plen)
    check_replay(rr, nconn, nreq, plen)
    c.close()


THREADS = (3, 8, 800, 96, 4)


def test_reference_log_with_concurrent_application_threads(orc):
    """Four application threads (memcached-style) race into proxy.c's admission lock, so the global order is whatever
    the lock produced.  The order is read back from the reference's log, the oracle replays exactly that order and
    must produce the same bytes; per connection the requests are all there, in order, with consecutive req_ids
    (proxy.c:121-133), and followers replay each connection's stream in order."""
    n, nconn, nreq, plen, threads = THREADS
    rr = reference("threads")
    lead = rr["leader"]
    end = rr["results"][lead]["offsets"]["end"]
    assert rr["entries"] == 1 + 2 * nconn + nreq and len(rr["requests"]) == 2 * nconn + nreq
    orc.set_rules(O.RULES_REFERENCE)
    c = O.Cluster(orc, n, leader=lead, term=rr["term"], length=O.LOG_SIZE)
    c.prologue()
    seen, payloads, want_sha = {}, hashlib.sha256(), {}
    for k, (pos, typ, clt, rid, ln, first) in enumerate(rr["requests"]):
        assert pos == k + 1
        payload = pattern_payload(first, ln)
        payloads.update(payload)
        assert (clt >> 8) == lead
        assert rid == seen.get(clt, 0) + 1, "req_ids of one connection are consecutive, in log order"
        seen[clt] = rid
        if typ == S.SEND:
            assert ln == plen
            want_sha.setdefault(clt, hashlib.sha256()).update(payload)
        assert c.submit(typ, clt, rid, O.cmd_image(payload))
    assert payloads.hexdigest() == rr["payloads_sha"]
    c.round(); c.round()
    assert len(seen) == nconn and sum(seen.values()) == 2 * nconn + nreq
    ents = O.walk_entries(c.image(lead, 0, end), 0, end, O.LOG_SIZE)
    for i in range(n):
        img, want = rr["images"][i], c.image(i, 0, end)
        if i != lead:
            assert img["masked_sha"] == sha(O.mask_replies(want, ents)), i
        else:
            assert img["sha"] == sha(want), i
    # followers: every connection's byte stream arrived in order
    for r in rr["results"]:
        if not r["leader"]:
            assert sorted(r["replay"]["sha"]) == sorted(h.hexdigest() for h in want_sha.values())
    c.close()


def record():
    """Run every scenario above on the reference's own stack (tests/golden/gen_refstack_golden.py)."""
    out = {}
    for n, nconn, nreq, plen in LOG_EQUALS:
        out[f"log_equals/{n}/{nconn}/{nreq}/{plen}"] = summarize_run(R.run(n, nconn, nreq, plen, prune=1000.0))
    for n, nconn, nreq, plen in LOG_EQUALS_SHM:
        out[f"log_equals_shm/{n}/{nconn}/{nreq}/{plen}"] = summarize_run(
            R.run(n, nconn, nreq, plen, prune=1000.0, transport="shm"))
    for attempt in range(3):
        rr = R.run(*PRUNING, prune=0.005)
        out["pruning"] = summarize_run(rr)
        # whether the timer finds something to prune is timing (it needs every follower's apply offset to have moved since
        # the last HEAD entry): a run without two HEAD entries says nothing about the rules, take another one
        if len(out["pruning"].get("heads", [])) >= 2:
            break
    out["I7"] = summarize_run(R.run(*I7, prune=1000.0))
    for seed in RANDOM_SEEDS:
        out[f"random_shape/{seed}"] = summarize_run(R.run(*random_shape(seed), prune=1000.0))
    n, nconn, nreq, plen, threads = THREADS
    out["threads"] = summarize_run(R.run(n, nconn, nreq, plen, threads=threads, prune=1000.0), entries=True)
    return out
