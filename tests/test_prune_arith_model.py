"""The leader's space / pruning rules -- apus_b200/csrc/apus_place.h, the functions the kernels use (ring offsets, head :=
the furthest-behind apply offset, free-space rule E2, the wrap rule), compiled as C (tests/hostlogic/place_rules.c) and
driven through ctypes by a model of the tile machine -- checked against ground truth kept in ABSOLUTE byte positions.

It documents the round-2 finding behind DESIGN.md section 3a: apply offsets are ring offsets, so a SNAPSHOT of them that is
used after other workers have pruned can alias into the used region of the next lap ("almost caught up") and let the head
overtake an application that is a lap behind -- the model reproduces that within a few dozen tiles -- while offsets read
at the time of use (what the kernel does now: under the place turn) never do.  No GPU."""
import ctypes
import os
import random
import subprocess

import pytest

L = 1 << 20
ES, TILE = 264, 256
HERE = os.path.dirname(os.path.abspath(__file__))
U64 = ctypes.c_uint64


@pytest.fixture(scope="module")
def P(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("place_rules") / "place_rules.so")
    subprocess.run(["gcc", "-O2", "-std=gnu99", "-Wall", "-shared", "-fPIC", "-o", so,
                    os.path.join(HERE, "hostlogic", "place_rules.c")], check=True)
    lib = ctypes.CDLL(so)
    for name, res, args in (("pr_ring_dist", U64, [U64] * 3), ("pr_place_limit", U64, [U64] * 4),
                            ("pr_wrap_rule", ctypes.c_int, [U64, U64, U64, ctypes.c_int, U64, U64]),
                            ("pr_prune_considered", ctypes.c_int, [U64, U64, ctypes.c_int, U64]),
                            ("pr_prune_dist", U64, [U64] * 4),
                            ("pr_prune_decide", ctypes.c_int, [U64] * 4 + [ctypes.POINTER(U64)] * 2),
                            ("pr_blocked", ctypes.c_int, [])):
        getattr(lib, name).restype, getattr(lib, name).argtypes = res, args
    return lib


def run(P, seed, stale_snapshots, n_tiles=300):
    rnd = random.Random(seed)
    pos_of = {0: 0}                                   # absolute entry boundary -> ring offset
    end_abs = head_abs = 0
    end, head, tail, prev_head, was_blocked = L, 0, 0, False, False
    true_ap = [0, 0]                                  # the followers' applications, absolute (ground truth)
    hist = [[(0, 0)], [(0, 0)]]                       # what they forwarded to the leader: (absolute, ring offset)
    tiles = guard = 0
    while tiles < n_tiles:
        guard += 1
        assert guard < 200000
        for f in range(2):
            if rnd.random() < 0.7:
                true_ap[f] = min(end_abs, true_ap[f] + rnd.randrange(0, 200000))
            if rnd.random() < 0.5 and true_ap[f] in pos_of:
                hist[f].append((true_ap[f], pos_of[true_ap[f]]))
        aps = [(end_abs, 0 if end == L else end)]     # the leader's own apply == its commit
        for f in range(2):
            k = rnd.randrange(0, 3) if stale_snapshots else 0
            aps.append(hist[f][max(0, len(hist[f]) - 1 - k)])
        pos0 = 0 if end == L else end
        used = 0 if end == L else P.pr_ring_dist(head, end, L)
        autoh = False
        if P.pr_prune_considered(end, used, not prev_head or was_blocked, L):
            d = max(P.pr_prune_dist(ring, end, used, L) for _, ring in aps)
            h, u = U64(head), U64(used)
            if P.pr_prune_decide(d, tail, end, L, ctypes.byref(h), ctypes.byref(u)):
                autoh, head, used = True, h.value, u.value
                old_head_abs, head_abs = head_abs, end_abs - used
                # pruning starts at a quarter of the ring used, and only to gain an eighth of it
                assert end_abs - old_head_abs >= L >> 2 and head_abs - old_head_abs >= L >> 3
                for f in range(2):
                    if head_abs > true_ap[f]:
                        return f"head passed follower {f}'s application by {head_abs - true_ap[f]} bytes after {tiles} tiles"
        hbytes = 64 if autoh else 0
        limit = P.pr_place_limit(pos0, used, 64, L)
        m = 0
        while m < TILE and hbytes + (m + 1) * ES <= limit:
            m += 1
        if m == 0 and not autoh:
            if P.pr_wrap_rule(pos0, used, ES, 1, 64, L) != P.pr_blocked():
                end_abs += L - pos0
                end = 0
                continue
            was_blocked = True
            continue
        was_blocked = False
        p_abs, p = end_abs, pos0
        if autoh:
            pos_of[p_abs] = p; p_abs += 64; p += 64
        for _ in range(m):
            pos_of[p_abs] = p; p_abs += ES; p += ES
        pos_of[p_abs] = 0 if p == L else p
        tail = p - (ES if m else 64)
        end_abs, end = p_abs, (0 if p == L else p)
        prev_head = autoh and m == 0
        assert end_abs - head_abs < L, "ring overfull"
        tiles += 1
    return None


def test_stale_apply_snapshots_alias_and_overtake_an_application(P):
    hits = [run(P, seed, stale_snapshots=True) for seed in range(40)]
    assert any(hits), "the model no longer reproduces the aliasing it documents"


@pytest.mark.parametrize("block", range(4))
def test_apply_offsets_read_at_time_of_use_never_overtake(P, block):
    for seed in range(block * 150, (block + 1) * 150):
        assert run(P, seed, stale_snapshots=False) is None
