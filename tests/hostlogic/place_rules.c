/*
 * tests/hostlogic/place_rules.c -- the leader's placement rules (apus_b200/csrc/apus_place.h, the functions the kernels
 * use) exported from a shared library for tests/test_prune_arith_model.py, which drives them through ctypes.
 */
#include "../../apus_b200/csrc/apus_place.h"

uint64_t pr_ring_dist(uint64_t from, uint64_t to, uint64_t L) { return ring_dist(from, to, L); }
uint64_t pr_place_limit(uint64_t pos0, uint64_t used, uint64_t reserve, uint64_t L) { return place_limit(pos0, used, reserve, L); }
int pr_wrap_rule(uint64_t pos0, uint64_t used, uint64_t es, int has_cmd, uint64_t reserve, uint64_t L)
{
    return wrap_rule(pos0, used, es, has_cmd, reserve, L);
}
int pr_prune_considered(uint64_t end, uint64_t used, int prev_ok, uint64_t L) { return prune_considered(end, used, prev_ok, L); }
uint64_t pr_prune_dist(uint64_t apply, uint64_t end, uint64_t used, uint64_t L) { return prune_dist(apply, end, used, L); }
int pr_prune_decide(uint64_t dmax, uint64_t tail, uint64_t end, uint64_t L, uint64_t *head, uint64_t *used)
{
    return prune_decide(dmax, tail, end, L, head, used);
}
int pr_blocked(void) { return PLACE_BLOCKED; }
