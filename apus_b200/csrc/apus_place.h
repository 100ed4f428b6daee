/*
 * apus_place.h -- the leader's placement rules on the ring (DESIGN.md section 3a), shared by the kernels (apus_kernels.cu)
 * and by the CPU model of the pruning rule (tests/hostlogic/place_rules.c), which is why it compiles as plain C as well.
 * Offsets are ring offsets in [0, L); an end offset of L stands for the empty log.
 */
#ifndef APUS_PLACE_H
#define APUS_PLACE_H
#include <stdint.h>
#include "apus_layout.h"
#ifndef APUS_HD
#ifdef __CUDACC__
#define APUS_HD __host__ __device__ __forceinline__
#else
#define APUS_HD static inline
#endif
#endif

APUS_HD uint64_t ring_dist(uint64_t from, uint64_t to, uint64_t L) { return to >= from ? to - from : L - (from - to); }
/* rule E1: an entry that ends exactly at len leaves end at 0; an empty log (end == len) starts at 0 (dare_log.h:216-219) */
APUS_HD uint64_t ring_pos(uint64_t off, uint64_t L) { return off == L ? 0 : off; }
/* bytes between head and end */
APUS_HD uint64_t ring_used(uint64_t head, uint64_t end, uint64_t L) { return end == L ? 0 : ring_dist(head, end, L); }

/* A host control plane moves the head the way the reference's log_pruning does (dare_server.c:2041-2046): it appends a
 * HEAD entry that CARRIES the new head offset.  The leader adopts the offset when it places that entry -- never by
 * re-reading the log header: a ring offset read "a while ago" cannot be told from a new one (the reader may have waited
 * for its turn while almost a whole ring was appended), and a stale head taken for an advance unprotects entries the
 * followers' applications have not replayed yet. */
APUS_HD uint64_t adopt_head(uint64_t head, uint64_t carried, uint64_t new_end, uint64_t L)
{
    if (carried >= L) return head;
    return (ring_dist(head, carried, L) <= ring_dist(head, ring_pos(new_end, L), L)) ? carried : head;   /* only forward, only inside the used region */
}

/* rule E2: bytes that may be appended before head (strictly: a full ring cannot be told from an empty one), keeping
 * `reserve` bytes for the HEAD entry of the device-side pruning rule (APUS_HDR_BYTES when it is on, else 0) */
APUS_HD uint64_t e2_room(uint64_t used, uint64_t reserve, uint64_t L) { return (L - used > 1 + reserve) ? L - used - 1 - reserve : 0; }
/* bytes that fit contiguously at pos0: no entry crosses len, rule E2 */
APUS_HD uint64_t place_limit(uint64_t pos0, uint64_t used, uint64_t reserve, uint64_t L)
{
    const uint64_t room = e2_room(used, reserve, L);
    return L - pos0 < room ? L - pos0 : room;
}

/* An entry of es bytes that does not fit at pos0 (dare_log.h:502-504, 526-538): it wraps to 0 when it does not fit
 * before len and the bytes up to len plus the entry fit under rule E2 -- leaving its header behind as a ghost when the
 * header fits and the entry carries a command -- else the placement is blocked until the head advances. */
enum { PLACE_WRAP_GAP = 0, PLACE_WRAP_GHOST = 1, PLACE_BLOCKED = 2 };
APUS_HD int wrap_rule(uint64_t pos0, uint64_t used, uint64_t es, int has_cmd, uint64_t reserve, uint64_t L)
{
    const uint64_t left = L - pos0;
    if (es > left && left + es <= e2_room(used, reserve, L))
        return (left >= APUS_HDR_BYTES && has_cmd) ? PLACE_WRAP_GHOST : PLACE_WRAP_GAP;
    return PLACE_BLOCKED;
}

/* Device-side log pruning (log_pruning / force_log_pruning, dare_server.c:1996-2122): head := the furthest-behind apply
 * offset in the group, published through a HEAD entry; the callers take the maximum of prune_dist over the replicas
 * (warp shuffles in leader_place, a loop in the fast path).  The rule is considered once a quarter of the ring is used,
 * when the HEAD entry fits before len, and when prev_ok: the last placed entry is not a HEAD entry of this rule ("never
 * two HEAD entries in a row", dare_server.c:2042, keeps an idle log from filling with them) -- or the placement is
 * blocked on space right behind one, else a slow follower host deadlocks the leader (back-pressure, rule E2). */
APUS_HD int prune_considered(uint64_t end, uint64_t used, int prev_ok, uint64_t L)
{
    return end != L && used >= (L >> 2) && prev_ok && L - end >= APUS_HDR_BYTES;
}
/* distance from a replica's apply offset to end, never behind the current head (a stale read cannot move it back) */
APUS_HD uint64_t prune_dist(uint64_t apply, uint64_t end, uint64_t used, uint64_t L)
{
    const uint64_t d = ring_dist(apply, end, L);
    return d > used ? used : d;
}
/* from dmax, the largest prune_dist over the replicas: whether a HEAD entry is due (it must gain L/8); if so the head
 * moves to *head and *used shrinks to what stays, before the append (dare_server.c:2041) */
APUS_HD int prune_decide(uint64_t dmax, uint64_t tail, uint64_t end, uint64_t L, uint64_t *head, uint64_t *used)
{
    if (dmax == 0) dmax = ring_dist(tail, end, L);          /* leave one entry (dare_server.c:2031-2034) */
    if (dmax > *used || *used - dmax < (L >> 3)) return 0;
    *head = end >= dmax ? end - dmax : L - (dmax - end);
    *used = dmax;
    return 1;
}

/* the tail word of the placement record: tail offset | APUS_REC_WRAPPED | APUS_REC_PREV_HEAD */
APUS_HD uint64_t rec_tail_pack(uint64_t tail, int wrapped, int prev_head) { return tail | (wrapped ? APUS_REC_WRAPPED : 0ull) | (prev_head ? APUS_REC_PREV_HEAD : 0ull); }
APUS_HD uint64_t rec_tail_off(uint64_t tw) { return tw & ~(APUS_REC_WRAPPED | APUS_REC_PREV_HEAD); }
#endif
