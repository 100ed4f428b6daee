"""The restated oracle (oracle/orc_log.h, cluster_sim.inc) against the compiled reference header (dare_log.h,
unmodified, built into oracle/_ref by oracle/Makefile).

What the reference produced for every scenario below is recorded in tests/golden/ref_log_golden.json
(tests/golden/gen_golden.py re-records it where the reference's sources exist), so these tests run anywhere.
Each `observe_*` function is run on the reference by the generator and on the oracle by the test.
"""
import numpy as np
import pytest

import orc as O
import streams as S
from refgold import digest, recorded

GOLD = "ref_log_golden.json"


def reference(key):
    return recorded(GOLD)[key]


def observe_layout(ref):
    return dict(sizeof_entry=int(ref.sizeof_entry()), sizeof_log=int(ref.lib.ref_sizeof_log()),
                log_size=int(ref.lib.ref_log_size()))


def test_layout_constants(orc):
    g = reference("layout")
    assert g == dict(sizeof_entry=64, sizeof_log=319656, log_size=O.LOG_SIZE)
    assert orc.sizeof_entry() == g["sizeof_entry"]


KAT = [(1, 0, 128), (2, 128, 256), (3, 256, 384), (4, 384, 548), (5, 548, 4708), (6, 4708, 4772), (7, 4772, 4836)]


def observe_kat(oracle):
    oracle.set_rules(O.RULES_REFERENCE)
    lens = [64, 64, 64, 100, 4096]
    log = O.Log(oracle)
    off = log.offsets()
    first = [off[k] for k in ("head", "apply", "commit", "end", "tail", "len")]
    got = []
    for i, ln in enumerate(lens):
        idx = log.append(1, i + 1, 0x0100, O.SEND, O.cmd_image(S.payload_kat(i, ln)))
        o = log.offsets()
        got.append((idx, o["tail"], o["end"]))
    idx = log.append(1, 6, 0x0100, O.CONNECT, O.cmd_image(b""))
    o = log.offsets(); got.append((idx, o["tail"], o["end"]))
    idx = log.append(1, 7, 0x0100, O.NOOP, b"")
    o = log.offsets(); got.append((idx, o["tail"], o["end"]))
    fnv = O.fnv1a(log.image(0, 4836))
    log.close()
    return dict(first=first, got=got, fnv=f"{fnv:016x}")


def test_kat_from_survey(orc):
    """SURVEY.md s8c known-answer vector, as the compiled reference produced it."""
    g = reference("kat")
    # (idx, tail, end) are the triples quoted in SURVEY.md s8c.  The FNV-1a-64 quoted there came from a probe harness
    # that was never committed and cannot be reproduced byte for byte; this checksum is the compiled reference's.
    assert g == dict(first=[0, 0, 0, 67108864, 67108864, 67108864], got=[list(t) for t in KAT], fnv="6ef37439cde8f856")
    assert digest(observe_kat(orc)) == g


def observe_random_stream(oracle, seed, length):
    oracle.set_rules(O.RULES_REFERENCE)
    stream = S.ragged_stream(600, 300, conns=3, seed=seed, close_every=50)
    log = O.Log(oracle, length)
    rets = []
    r = np.random.default_rng(seed + 99)
    for k, (typ, clt, rid, payload) in enumerate(stream):
        rets.append(log.append(1 + k // 200, rid, clt, typ, O.cmd_image(payload)))
        # advance head now and then so the ring keeps accepting entries
        if k % 7 == 0:
            o = log.offsets()
            if o["end"] != o["len"]:
                log.set_offsets(head=o["tail"], apply=o["tail"], commit=o["tail"])
        if r.random() < 0.05:
            rets.append(log.append(1, 0, 0, O.NOOP, b""))
        if r.random() < 0.03:
            rets.append(log.append(1, 0, 0, O.CONFIG, O.cid_image(3)))
        if r.random() < 0.03:
            rets.append(log.append(1, 0, 0, O.HEAD, (12345).to_bytes(8, "little")))
    out = dict(rets=rets, offsets=log.offsets(), image=log.image())
    log.close()
    return out


RANDOM_STREAMS = [(seed, length) for length in (4096, 1 << 16) for seed in (1, 2, 3)]


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("length", [4096, 1 << 16])
def test_random_streams_with_wraps(orc, seed, length):
    """Small rings force every wrap rule of log_append_entry (ghost header, header
    does not fit, exact fit, full) -- reference rules must match bit for bit."""
    assert digest(observe_random_stream(orc, seed, length)) == reference(f"random_stream/{seed}/{length}")


def observe_wrap_edge(oracle, left, typ):
    """Place `end` exactly `left` bytes before len and append one entry (64 B payload)."""
    oracle.set_rules(O.RULES_REFERENCE)
    length = 8192
    log = O.Log(oracle, length)
    # fill with 64 B NOOP-size strides up to the desired position, head moved away
    log.append(1, 1, 7, O.SEND, O.cmd_image(b"x" * 64))
    pos = length - left
    log.poke(0, bytes(range(256)) * (length // 256))      # stale bytes everywhere
    # fabricate a log whose last entry ends at pos: tail entry must parse
    tail = pos - 64
    hdr = (41).to_bytes(8, "little") + (1).to_bytes(8, "little") + bytes(8) + bytes([7, 0, O.NOOP, 0]) + bytes(36)
    log.poke(tail, hdr)
    log.set_offsets(head=256, apply=256, commit=256, end=pos, tail=tail, old_end=pos)
    data = {O.SEND: O.cmd_image(bytes(range(64))), O.NOOP: b"", O.HEAD: (77).to_bytes(8, "little"),
            O.CONFIG: O.cid_image(5)}[typ]
    idx = log.append(2, 9, 0x0203, typ, data)
    out = dict(idx=idx, offsets=log.offsets(), image=log.image())
    log.close()
    return out


WRAP_LEFT = [0, 1, 40, 63, 64, 65, 100, 127, 128, 129, 200]
WRAP_TYPES = [O.SEND, O.NOOP, O.HEAD, O.CONFIG]


@pytest.mark.parametrize("left", WRAP_LEFT)
@pytest.mark.parametrize("typ", WRAP_TYPES)
def test_wrap_edges(orc, left, typ):
    assert digest(observe_wrap_edge(orc, left, typ)) == reference(f"wrap_edge/{left}/{typ}")


def observe_wrap_into_head_zero(oracle):
    oracle.set_rules(O.RULES_REFERENCE)
    log = O.Log(oracle, 4096)
    rets = [log.append(1, i + 1, 1, O.SEND, O.cmd_image(b"a" * 70)) for i in range(40)]
    out = dict(rets=rets, offsets=log.offsets(), image=log.image())
    log.close()
    return out


def test_wrap_into_head_zero_is_full(orc):
    """H11(iii): wrapping while head == 0 reports full and leaves end = 0."""
    got = observe_wrap_into_head_zero(orc)
    assert digest(got) == reference("wrap_into_head_zero")
    assert 0 in got["rets"]


def cluster_script(oracle, n, stream, length, schedule_seed):
    """Drive the cluster with a randomised (but seeded) interleaving of follower
    replication / ack steps; return everything observable."""
    c = O.Cluster(oracle, n, leader=0, term=1, length=length)
    rng = np.random.default_rng(schedule_seed)
    c.prologue()
    commits = []
    for k, (typ, clt, rid, payload) in enumerate(stream):
        c.submit(typ, clt, rid, O.cmd_image(payload))
        if rng.random() < 0.6:
            c.leader_persist()
            order = rng.permutation(n)
            for i in order:
                if rng.random() < 0.8:
                    c.replicate(int(i))
                if rng.random() < 0.7:
                    c.follower_persist(int(i))
            if c.commit_scan():
                commits.append(c.offsets(0)["commit"])
            for i in range(n):
                if rng.random() < 0.5:
                    c.push_commit(i)
                    c.apply(i)
    for _ in range(3):
        c.round()
    commits.append(c.offsets(0)["commit"])
    obs = dict(
        offsets=[c.offsets(i) for i in range(n)],
        images=[c.image(i) for i in range(n)],
        applied=[c.applied(i) for i in range(n)],
        commits=commits,
        store=[c.store_cmd_calls(i) for i in range(n)],
        update_state=c.update_state_calls(),
        bytes_rep=c.bytes_replicated(),
    )
    c.close()
    return obs


def observe_cluster_steps(oracle, n):
    oracle.set_rules(O.RULES_REFERENCE)
    stream = S.ragged_stream(400, 200, conns=4, seed=n, close_every=40)
    return cluster_script(oracle, n, stream, 1 << 20, 5)


CLUSTER_SIZES = [1, 3, 5, 7]


@pytest.mark.parametrize("n", CLUSTER_SIZES)
def test_cluster_steps_match(orc, n):
    b = observe_cluster_steps(orc, n)
    assert digest(b) == reference(f"cluster_steps/{n}")
    # invariants of SURVEY.md s8a: commit == end on the leader at quiescence,
    # apply order == log order, every follower applied the same sequence
    assert b["offsets"][0]["commit"] == b["offsets"][0]["end"]
    idxs = [t[0] for t in b["applied"][0]]
    assert idxs == sorted(idxs)
    for i in range(1, n):
        assert b["applied"][i] == b["applied"][0]


def observe_cluster_wrap_and_prune(oracle):
    """Ring of 16 KiB, pruning by HEAD entries between rounds, several laps."""
    oracle.set_rules(O.RULES_REFERENCE)
    stream = S.ragged_stream(900, 150, conns=2, seed=77)
    c = O.Cluster(oracle, 3, leader=0, term=1, length=16384)
    c.prologue()
    heads = []
    cido = [(O.u64)(0) for _ in range(3)]
    for k, (typ, clt, rid, payload) in enumerate(stream):
        c.submit(typ, clt, rid, O.cmd_image(payload))
        if k % 5 == 4:
            c.round()
            heads.append(c.prune())
            c.round()
            for i in (1, 2):
                c.poll_head(i, cido[i])
    c.round()
    obs = dict(offsets=[c.offsets(i) for i in range(3)], images=[c.image(i) for i in range(3)],
               applied=[c.applied(i) for i in range(3)], heads=heads)
    c.close()
    return obs


def test_cluster_wrap_and_prune_match(orc):
    b = observe_cluster_wrap_and_prune(orc)
    assert digest(b) == reference("cluster_wrap_and_prune")
    assert any(h for h in b["heads"])


def record(ref):
    """Every observation above, made on the compiled reference (tests/golden/gen_golden.py)."""
    out = {"layout": observe_layout(ref), "kat": observe_kat(ref),
           "wrap_into_head_zero": observe_wrap_into_head_zero(ref),
           "cluster_wrap_and_prune": observe_cluster_wrap_and_prune(ref)}
    for seed, length in RANDOM_STREAMS:
        out[f"random_stream/{seed}/{length}"] = observe_random_stream(ref, seed, length)
    for left in WRAP_LEFT:
        for typ in WRAP_TYPES:
            out[f"wrap_edge/{left}/{typ}"] = observe_wrap_edge(ref, left, typ)
    for n in CLUSTER_SIZES:
        out[f"cluster_steps/{n}"] = observe_cluster_steps(ref, n)
    return digest(out)
