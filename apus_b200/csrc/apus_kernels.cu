/*
 * apus_kernels.cu -- the persistent sm_100a kernels of the replication engine.
 *
 * One kernel, `apus_replica_kernel`, launched with one CTA per replica ROLE that
 * lives on the launching GPU (apus_role_t table).  Two roles:
 *
 *   LEADER   the hot loop of the reference's leader, fused:
 *            get_tailq_message (dare_ibv_ud.c:780-790) + log_append_entry
 *            (dare_log.h:466-558) + persist_new_entries' sender stamp
 *            (dare_server.c:1803-1804) + update_remote_logs step I/II
 *            (dare_ibv_rc.c:1526-1573: byte range then tail) + the commit rule
 *            (dare_ibv_rc.c:1725-1758) + the commit publish (:1760-1822) +
 *            log pruning (dare_server.c:1996-2122).
 *            15 producer warps build a TILE of entries in shared memory and push
 *            it with 16 B vector stores into the local log and into every
 *            follower's log over NVLink; warp 15 is the commit warp: lane i
 *            polls follower i's ack word and a shuffle ranking of the acks finds
 *            the count a majority holds.
 *   FOLLOWER persist_new_entries' follower branch (dare_server.c:1792-1810) +
 *            rc_send_entries_reply (dare_ibv_rc.c:1828-1863): poll the tail
 *            publish, walk the new entries, set reply[me] locally and in the
 *            leader's copy, publish the ack word, follow `commit`, adopt `head`
 *            from committed HEAD entries (dare_server.c:2163-2186).
 *
 * Ordering (invariant I1, "data before tail"): all data stores of a tile ->
 * bar.sync -> fence.acq_rel.sys -> 16 B st.relaxed.sys of {end, count}.  The
 * follower reads the pair, fences, and reads the entry bytes with ld.relaxed.sys
 * (never through a stale L1 line).  Acks mirror this in the other direction.
 *
 * Pure integer / byte work: no tensor cores, bound by NVLink store bandwidth and
 * by launch-free round-trip latency.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "apus_layout.h"
#include "apus_cert.h"
#include "apus_place.h"

// ---------------------------------------------------------------------------------
// memory-model helpers (system scope: peers and the host observe these)
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t ld_relaxed_sys(const volatile void *p)
{
    uint64_t v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t ld_acquire_sys(const volatile void *p)
{
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_sys_u32(const volatile void *p)
{
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_acquire_sys_2x64(const volatile void *p, uint64_t &a, uint64_t &b)
{
    // an acquire LOAD costs ~0.26 us here, a system fence ~1.5 us (profiles/r1_ubench_2gpu.txt)
    asm volatile("ld.acquire.sys.global.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void ld_relaxed_sys_2x64(const volatile void *p, uint64_t &a, uint64_t &b)
{
    asm volatile("ld.relaxed.sys.global.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(volatile void *p, uint64_t v)
{
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_2x64(volatile void *p, uint64_t a, uint64_t b)
{
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys_u8(volatile void *p, uint8_t v)
{
    asm volatile("st.relaxed.sys.global.u8 [%0], %1;" ::"l"(p), "r"((uint32_t)v) : "memory");
}
__device__ __forceinline__ uint4 ld_relaxed_sys_v4(const void *p)
{
    uint4 v;
    asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p)
                 : "memory");
    return v;
}
__device__ __forceinline__ void st_v4(void *p, uint4 v)
{
    asm volatile("st.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}
// NVSwitch multicast stores: ONE store, every replica of the group (the issuing GPU's own copy included) receives it
__device__ __forceinline__ void mst_v4(void *p, uint4 v)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(__uint_as_float(v.x)),
                 "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w))
                 : "memory");
}
__device__ __forceinline__ void mst_u32(void *p, uint32_t v)
{
    asm volatile("multimem.st.relaxed.sys.global.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_u8(void *p, uint32_t v)
{
    asm volatile("st.global.u8 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t globaltimer_ns()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// named barrier for a subset of the CTA's warps
__device__ __forceinline__ void bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ bool has_cmd(uint32_t type)
{
    return !(type == T_NOOP || type == T_CONFIG || type == T_HEAD);
}
// bytes placed at entry+48 (sm_cmd_t image {u16 len; cmd}, dare_cid_t, or head offset)
__device__ __forceinline__ uint32_t data_bytes(uint32_t type, uint32_t len)
{
    if (type == T_NOOP) return 0;
    if (type == T_CONFIG) return 16;
    if (type == T_HEAD) return 8;
    return 2u + len;
}
__device__ __forceinline__ uint32_t entry_stride(uint32_t type, uint32_t len)
{
    return has_cmd(type) ? APUS_HDR_BYTES + len : APUS_HDR_BYTES;   // dare_log.h:228-234
}
__device__ __forceinline__ uint64_t slot_head_value(const apus_cslot_t *sl)
{
    uint64_t v = 0;
#pragma unroll
    for (int q = 7; q >= 0; q--) v = (v << 8) | sl->inl[q];
    return v;
}

#define WATCHDOG_NS (20ull * 1000ull * 1000ull * 1000ull)

// error codes reported through hostwords.error
#define APUS_KERR_WATCHDOG_LEADER   1
#define APUS_KERR_WATCHDOG_FOLLOWER 2
#define APUS_KERR_WATCHDOG_COMMIT   3
#define APUS_KERR_BAD_ENTRY         4
#define APUS_KERR_COUNT_MISMATCH    5

// ---------------------------------------------------------------------------------
// shared memory
// ---------------------------------------------------------------------------------
#define N_PRODUCER_WARPS 15
#define NT (N_PRODUCER_WARPS * 32)      // producer threads
#define MAXB APUS_MAX_TILE_ENTRIES
#define PUBMASK (APUS_PUBRING_RECORDS - 1)

struct LeaderShared {
    // per fetched slot (filled while fetching: no strided re-reads of the 128 B slots)
    uint32_t es[MAXB];         // log stride of the entry (64 + len, or 64)
    uint32_t xb[MAXB];         // payload-ring bytes to stage for it (0 when inline)
    uint32_t cum_es[MAXB];     // inclusive prefix sum of es over the fetched batch (state independent)
    uint32_t cum_xb[MAXB];     // inclusive prefix sum of xb
    uint32_t rel[MAXB];        // entry start - sub-tile start (bytes)
    uint32_t xoff[MAXB];       // offset of the entry's image in the ext staging
    uint32_t static_cut;       // first k > 0 whose payload image restarted the payload ring (else n_fetch)
    uint32_t first_ext_all;    // first entry with an external payload image (else 0xffffffff)
    uint32_t host_head_k;      // last HEAD entry submitted by the host in this batch (else 0xffffffff): it carries the new head
    uint64_t idx_base;         // idx of an entry = idx_base + its 1-based position in the placement order
    uint8_t  ty[MAXB];
    uint8_t  flg[MAXB];        // bit0 EXT, bit1 WRAP
    // claim
    uint32_t n_fetch, finish, abort, was_blocked;
    uint32_t avg_es, avg_xb;   // log / staged bytes per entry seen in this worker's last claim (sizes the next one)
    uint64_t slot0, my_seq, t_dequeue, st_head, t_place_acq, pub_h, pub_tail_seen;
    // placement state while this CTA holds the place turn (mirrors apus_seq_t.p_*)
    uint64_t st_end, st_tail, st_next_idx, st_hwm, st_placed;
    uint32_t st_prev_head, pad0;
    // current sub-tile
    uint32_t kbase, m, gap, ghost, fresh, auto_head, ext_bytes, last, blocked, hbytes;
    uint32_t base_es, base_xb;
    uint64_t ext_base, auto_head_val, a, b, idx0, cum_after, new_end, tail_after, hwm_after;
    uint8_t  *peer_entries[APUS_MAX_SERVERS];
    uint32_t *peer_index[APUS_MAX_SERVERS];
};

#define LS_BYTES ((sizeof(LeaderShared) + 127u) & ~127u)
#define L_SLOTS_OFF LS_BYTES
#define L_EXT_OFF   (L_SLOTS_OFF + MAXB * APUS_CSLOT_BYTES)
#define L_IMG_OFF   (L_EXT_OFF + APUS_LEADER_EXT_BYTES)
#define L_TOTAL     (L_IMG_OFF + APUS_LEADER_IMG_BYTES + 16)

struct FollowerShared {
    uint32_t off[APUS_FOLLOWER_WIN_BYTES / 64 + 8];   // entry offsets found in the window (relative to win_lo)
    uint32_t n;
    uint32_t done;
    uint64_t win_lo, win_hi, next;           // window bounds in the log, next walk offset
    uint64_t head_val, head_end;             // last HEAD entry of the window (head_end == len: none)
    uint64_t end_seen, cum_seen, commit_seen;
    uint32_t head_j;                         // index mode: 1 + position of the last HEAD entry of the batch
    uint32_t cert;                           // the publish being processed was self-certifying: ONE entry at cert_start
    uint64_t cert_start;
};
#define FS_BYTES ((sizeof(FollowerShared) + 127u) & ~127u)
#define F_TOTAL (FS_BYTES + APUS_FOLLOWER_WIN_BYTES + 16)

extern __shared__ __align__(16) uint8_t smem_raw[];

// gpu-scope handoffs between the leader's worker CTAs
__device__ __forceinline__ uint64_t ld_acquire_gpu(const volatile void *p)
{
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_acquire_gpu_2x64(const volatile void *p, uint64_t &a, uint64_t &b)
{
    asm volatile("ld.acquire.gpu.global.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_release_gpu(volatile void *p, uint64_t v)
{
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// ---------------------------------------------------------------------------------
// Self-certifying publishes: the checksum (cs_weight / cs_mask / cs_chunk_words / cs_key) lives in apus_cert.h, which
// the CPU property test compiles too.
// ---------------------------------------------------------------------------------
// contribution of the 16 B chunk at log offset lo (16 B aligned), restricted to the bytes inside [a, b)
__device__ __forceinline__ uint64_t cs_chunk(const uint4 v, uint64_t lo, uint64_t a, uint64_t b)
{
    return cs_chunk_words((uint64_t)v.x | ((uint64_t)v.y << 32), (uint64_t)v.z | ((uint64_t)v.w << 32), lo, a, b);
}
// first n bytes of a 16 B chunk from `nw`, the rest from `old`
__device__ __forceinline__ uint4 chunk_select(const uint4 nw, const uint4 old, int n)
{
    uint32_t a[4] = {nw.x, nw.y, nw.z, nw.w}, o[4] = {old.x, old.y, old.z, old.w}, r[4];
#pragma unroll
    for (int w = 0; w < 4; w++) {
        const int k = n - 4 * w;                      // bytes of this word that come from `nw`
        const uint32_t m = k >= 4 ? 0xffffffffu : (k <= 0 ? 0u : ((1u << (8 * k)) - 1u));
        r[w] = (a[w] & m) | (o[w] & ~m);
    }
    return make_uint4(r[0], r[1], r[2], r[3]);
}


// ---------------------------------------------------------------------------------
// LEADER
// ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hdr_byte(uint32_t j, uint64_t idx, uint64_t term, uint64_t req_id,
                                             uint32_t clt, uint32_t type, uint32_t sender)
{
    // dare_log_entry_t bytes 0..40 (dare_log.h:33-48)
    if (j < 8) return (uint32_t)(idx >> (8 * j)) & 0xFF;
    if (j < 16) return (uint32_t)(term >> (8 * (j - 8))) & 0xFF;
    if (j < 24) return (uint32_t)(req_id >> (8 * (j - 16))) & 0xFF;
    if (j == 24) return clt & 0xFF;
    if (j == 25) return (clt >> 8) & 0xFF;
    if (j == 26) return type;
    if (j == 27) return sender;
    return 0;   // reply[13]
}

// bytes 0..40 of an entry header into shared memory at any alignment, by `gl` lanes (sub = lane in group)
__device__ __noinline__ void group_write_header(uint8_t *e, int sub, int gl, uint64_t idx, uint64_t term, uint64_t req_id,
                                                   uint32_t clt, uint32_t type, uint32_t sender, bool skip_sender)
{
    if ((((uint32_t)(uintptr_t)e) & 15u) == 0 && !skip_sender) {
        // 16 B aligned entry: two 16 B stores, one 8 B store, one byte; bytes 41..47 stay (hole)
        if (sub == 0) *reinterpret_cast<uint4 *>(e + 0) = make_uint4((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)term, (uint32_t)(term >> 32));
        else if (sub == 1) *reinterpret_cast<uint4 *>(e + 16) = make_uint4((uint32_t)req_id, (uint32_t)(req_id >> 32),
                                                                         (clt & 0xffffu) | (type << 16) | (sender << 24), 0u);
        else if (sub == 2) *reinterpret_cast<uint64_t *>(e + 32) = 0;
        else if (sub == 3) e[40] = 0;
    } else if ((((uint32_t)(uintptr_t)e) & 7u) == 0) {
        // aligned entry: 8-byte stores for bytes 0..39, byte 40 separately; bytes 41..47 stay (hole)
        if (sub == 0) *reinterpret_cast<uint64_t *>(e + 0) = idx;
        else if (sub == 1) *reinterpret_cast<uint64_t *>(e + 8) = term;
        else if (sub == 2) *reinterpret_cast<uint64_t *>(e + 16) = req_id;
        else if (sub == 3) {
            if (skip_sender) {
                e[24] = (uint8_t)clt; e[25] = (uint8_t)(clt >> 8); e[26] = (uint8_t)type;
                e[28] = 0; e[29] = 0; e[30] = 0; e[31] = 0;
            } else {
                *reinterpret_cast<uint64_t *>(e + 24) =
                    (uint64_t)(clt & 0xffffu) | ((uint64_t)type << 16) | ((uint64_t)sender << 24);
            }
        } else if (sub == 4) *reinterpret_cast<uint64_t *>(e + 32) = 0;
        else if (sub == 5) e[40] = 0;
    } else {
        for (uint32_t j = sub; j < 41; j += gl)
            if (!(skip_sender && j == E_SENDER)) e[j] = (uint8_t)hdr_byte(j, idx, term, req_id, clt, type, sender);
    }
}

// copy nbytes from a 16 B-aligned shared source to an arbitrarily aligned shared destination
__device__ __noinline__ void group_copy_smem(uint8_t *dst, const uint8_t *src, uint32_t nbytes, int sub, int gl)
{
    const uint32_t nchunks = (nbytes + 15u) >> 4;
    const uint32_t dalign = (uint32_t)(uintptr_t)dst & 15u;
    for (uint32_t c = sub; c < nchunks; c += gl) {
        const uint4 v = *reinterpret_cast<const uint4 *>(src + 16u * c);
        uint8_t *d = dst + 16u * c;
        const uint32_t left = nbytes - 16u * c;
        if (dalign == 0 && left >= 16) {
            *reinterpret_cast<uint4 *>(d) = v;
        } else if ((dalign & 3u) == 0 && left >= 16) {
            uint32_t *d4 = reinterpret_cast<uint32_t *>(d);
            d4[0] = v.x; d4[1] = v.y; d4[2] = v.z; d4[3] = v.w;
        } else if ((dalign & 1u) == 0 && left >= 16) {
            uint16_t *d2 = reinterpret_cast<uint16_t *>(d);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 8; k++) d2[k] = (uint16_t)(w[k >> 1] >> (16 * (k & 1)));
        } else {
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            const uint32_t nb = left < 16 ? left : 16;
#pragma unroll
            for (uint32_t k = 0; k < 16; k++)
                if (k < nb) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        }
    }
}

// global (16 B aligned) -> shared, nchunks 16 B chunks, by all producer threads, 4 loads in flight each
__device__ __noinline__ void cta_fetch_chunks(uint8_t *dst, const uint8_t *src, uint32_t nchunks, int tid)
{
    uint32_t c = tid;
    for (; c + 3u * NT < nchunks; c += 4u * NT) {
        const uint4 v0 = ld_relaxed_sys_v4(src + 16ull * c);
        const uint4 v1 = ld_relaxed_sys_v4(src + 16ull * (c + NT));
        const uint4 v2 = ld_relaxed_sys_v4(src + 16ull * (c + 2u * NT));
        const uint4 v3 = ld_relaxed_sys_v4(src + 16ull * (c + 3u * NT));
        reinterpret_cast<uint4 *>(dst)[c] = v0;
        reinterpret_cast<uint4 *>(dst)[c + NT] = v1;
        reinterpret_cast<uint4 *>(dst)[c + 2u * NT] = v2;
        reinterpret_cast<uint4 *>(dst)[c + 3u * NT] = v3;
    }
    for (; c < nchunks; c += NT) reinterpret_cast<uint4 *>(dst)[c] = ld_relaxed_sys_v4(src + 16ull * c);
}

// the descriptor chunk of a slot -> compact per-entry arrays
__device__ __forceinline__ void note_desc(LeaderShared *S, uint32_t k, const uint4 v)
{
    const uint32_t to = v.z, ty = (to >> APUS_SLOT_TYPE_SHIFT) & APUS_SLOT_TYPE_MASK, len = v.w & 0xffffu;
    S->ty[k] = (uint8_t)ty;
    S->flg[k] = (uint8_t)(((to & APUS_SLOT_EXT) ? 1u : 0u) | ((to & APUS_SLOT_WRAP) ? 2u : 0u));
    S->es[k] = entry_stride(ty, len);
    S->xb[k] = (to & APUS_SLOT_EXT) ? ((data_bytes(ty, len) + 15u) & ~15u) : 0u;
}

// fetch `cnt` slots starting at ring slot `s` into shared slot `k0` onward.  A 128 B ring slot is kept as a
// 96 B compact slot: its two stamp chunks (3 and 7) are neither loaded nor stored, so that the inline image
// is contiguous in shared memory (and a quarter of the PCIe / HBM read traffic is saved).
__device__ __noinline__ void cta_fetch_slots(LeaderShared *S, uint8_t *slots, const apus_slot_t *ring, uint64_t s, uint32_t k0,
                                                uint32_t cnt, int tid)
{
    const uint8_t *src = reinterpret_cast<const uint8_t *>(ring + s);
    uint8_t *dst = slots + (size_t)k0 * APUS_CSLOT_BYTES;
    const uint32_t nq = cnt * 6u;                                  // compact chunks
    uint32_t q = (tid >= 32) ? tid - 32 : tid + NT - 32;           // warp 1 takes the first chunks (warp 0 is busy with the turns)
#define SRC_OF(qq, kk, rr) const uint32_t kk = (qq) / 6u, rr = (qq) - 6u * kk; const uint8_t *p_##qq = src + (size_t)kk * APUS_SLOT_BYTES + 16u * (rr < 3u ? rr : rr + 1u)
    for (; q + 3u * NT < nq; q += 4u * NT) {
        const uint32_t q0 = q, q1 = q + NT, q2 = q + 2u * NT, q3 = q + 3u * NT;
        SRC_OF(q0, ka, ra); SRC_OF(q1, kb, rb); SRC_OF(q2, kc, rc); SRC_OF(q3, kd, rd);
        const uint4 v0 = ld_relaxed_sys_v4(p_q0);
        const uint4 v1 = ld_relaxed_sys_v4(p_q1);
        const uint4 v2 = ld_relaxed_sys_v4(p_q2);
        const uint4 v3 = ld_relaxed_sys_v4(p_q3);
        reinterpret_cast<uint4 *>(dst)[q0] = v0;
        reinterpret_cast<uint4 *>(dst)[q1] = v1;
        reinterpret_cast<uint4 *>(dst)[q2] = v2;
        reinterpret_cast<uint4 *>(dst)[q3] = v3;
        if (ra == 0) note_desc(S, k0 + ka, v0);
        if (rb == 0) note_desc(S, k0 + kb, v1);
        if (rc == 0) note_desc(S, k0 + kc, v2);
        if (rd == 0) note_desc(S, k0 + kd, v3);
    }
    for (; q < nq; q += NT) {
        const uint32_t q0 = q;
        SRC_OF(q0, ka, ra);
        const uint4 v = ld_relaxed_sys_v4(p_q0);
        reinterpret_cast<uint4 *>(dst)[q0] = v;
        if (ra == 0) note_desc(S, k0 + ka, v);
    }
#undef SRC_OF
}

__device__ void leader_commit_warp(const apus_devctx_t *__restrict__ cx)
{
    const int lane = threadIdx.x & 31;
    const int N = cx->group_size, me = cx->idx, quorum = cx->quorum;
    apus_ctrl_t *ctrl = reinterpret_cast<apus_ctrl_t *>(cx->region);
    apus_seq_t *seq = reinterpret_cast<apus_seq_t *>(cx->region + APUS_SEQ_OFF);
    const apus_pubrec_t *ring = reinterpret_cast<const apus_pubrec_t *>(cx->region + APUS_PUBRING_OFF);
    apus_loghdr_t *hdr = reinterpret_cast<apus_loghdr_t *>(cx->region + APUS_HDR_OFF);
    apus_hostwords_t *hw = cx->hw;
    uint64_t committed = ctrl->committed;
    uint64_t committed_tickets = ctrl->committed_tickets;
    uint64_t lat_count = ctrl->lat_count;
    uint64_t bytes_rep = ctrl->bytes_replicated, batches = ctrl->batches;
    uint64_t tail = 0;                       // next record to commit
    uint64_t seen = 0;                       // records [tail, seen) are valid and not committed yet
    uint64_t published = ctrl->published;    // entries published = cum of the newest valid record
    uint64_t last_progress = globaltimer_ns();
    uint32_t spins = 0, hb_spins = 0;
    uint64_t last_hb = 0, hb_beat = globaltimer_ns() >> 10;   // beats keep growing across launches
    bool S_rec_ok = false;
    volatile uint64_t *peer_commit = nullptr;
    if (lane < N && lane != me && cx->peer[lane])
        peer_commit = &reinterpret_cast<apus_loghdr_t *>(cx->peer[lane] + APUS_HDR_OFF)->commit;

    for (;;) {
        // every lane looks at one 16 B pair of the next four publish records (lane>>3 = record, lane&7 = pair)
        // while lanes 0..N-1 also poll the acks
        uint64_t st = 0, rv = 0, v = 0;
        const uint64_t seen_before = seen;
        {
            const uint64_t rn = seen + (uint64_t)(lane >> 3);
            ld_relaxed_sys_2x64(&ring[rn & PUBMASK].w[2 * (lane & 7)], st, rv);
            const uint32_t okm = __ballot_sync(0xffffffffu, st == rn + 1);
            // records are valid only in order: count the leading records whose eight pairs all match
            uint32_t nvalid = 0;
            while (nvalid < 4 && ((okm >> (8 * nvalid)) & 0xffu) == 0xffu) nvalid++;
            if (nvalid) {
                published = __shfl_sync(0xffffffffu, rv, 8 * (nvalid - 1) + PR_CUM);
                seen += nvalid;
            }
            S_rec_ok = nvalid != 0;
        }
        if (lane < N && lane != me) v = ld_relaxed_sys(&ctrl->ack[lane]);
        // lane i holds what replica i has acked (entries, monotone); the leader's own vote is
        // everything it has published (dare_ibv_rc.c:1736 "i == idx")
        if (lane == me) v = published;
        // rank: how many replicas hold at least what I hold
        int cnt = 0;
        for (int j = 0; j < N; j++) {
            uint64_t vj = __shfl_sync(0xffffffffu, v, j);
            cnt += (vj >= v) ? 1 : 0;
        }
        uint64_t cand = (lane < N && cnt >= quorum) ? v : 0;
        // the largest count a majority holds (size/2+1, dare_ibv_rc.c:1741)
        for (int s = 16; s > 0; s >>= 1) {
            uint64_t o = __shfl_xor_sync(0xffffffffu, cand, s);
            cand = o > cand ? o : cand;
        }
        const uint64_t Q = cand;
        if (Q > committed && tail != seen) {
            // map the entry count to the log offset recorded at publish time; the commit is a
            // prefix and an entry boundary (invariant I3).  Four records per step.
            uint64_t off = 0, tickets = committed_tickets, r_tail = 0, r_hwm = 0, r_next = 0;
            bool any = false;
            bool reuse = (tail == seen_before);          // the pending records are exactly the ones this iteration loaded
            while (tail != seen) {
                const uint64_t rn = tail + (uint64_t)(lane >> 3);
                uint64_t st2 = 0, val = 0;
                if (reuse) { val = rv; reuse = false; }
                else if (rn < seen) ld_relaxed_sys_2x64(&ring[rn & PUBMASK].w[2 * (lane & 7)], st2, val);
                // how many of these (up to four, in order) are covered by the quorum count
                const uint32_t cm = __ballot_sync(0xffffffffu, (lane & 7) == PR_CUM && rn < seen && val <= Q);
                uint32_t nc = 0;
                while (nc < 4 && ((cm >> (8 * nc)) & 1u)) nc++;
                if (nc == 0) break;
                const int base = 8 * (int)(nc - 1);
                committed = __shfl_sync(0xffffffffu, val, base + PR_CUM);
                off = __shfl_sync(0xffffffffu, val, base + PR_END);
                tickets = __shfl_sync(0xffffffffu, val, base + PR_TICKETS);
                r_tail = __shfl_sync(0xffffffffu, val, base + PR_TAIL);
                r_hwm = __shfl_sync(0xffffffffu, val, base + PR_HWM);
                r_next = __shfl_sync(0xffffffffu, val, base + PR_NEXTIDX);
                for (uint32_t q = 0; q < nc; q++) {
                    bytes_rep += __shfl_sync(0xffffffffu, val, 8 * q + PR_BYTES);
                    const uint64_t t0 = __shfl_sync(0xffffffffu, val, 8 * q + PR_T0);
                    if ((cx->flags & APUS_FLAG_STATS) && cx->lat_ns && lane == 0) {
                        const uint64_t d = globaltimer_ns() - t0;
                        cx->lat_ns[(lat_count + q) & (APUS_LAT_RING - 1)] = d > 0xffffffffull ? 0xffffffffu : (uint32_t)d;
                    }
                }
                lat_count += nc; batches += nc;
                tail += nc;
                any = true;
                if (nc < 4) break;
            }
            if (any) {
                if (peer_commit) st_relaxed_sys(peer_commit, off);          // dare_ibv_rc.c:1810
                if (lane == 0) {
                    // {commit offset, committed tickets}: ONE 16 B store into pinned host memory -- this is what
                    // releases the proxy.c:160 spinners; a 16 B host load sees a consistent pair
                    st_relaxed_sys_2x64(&hw->commit_off, off, tickets);
                    st_relaxed_sys(&hw->consumed, tickets);                 // submission-ring space
                    st_relaxed_sys(&hw->last_commit_ns, globaltimer_ns());
                    st_relaxed_sys(&seq->pub_tail, tail);                   // publish-ring space
                    // the leader's bookkeeping, in publish order (single writer)
                    hdr->commit = off;
                    st_relaxed_sys(&hdr->apply, off);                       // leader applies = update_state
                    hdr->end = off; hdr->tail = r_tail; hdr->old_end = off;
                    ctrl->committed = committed; ctrl->committed_tickets = tickets; ctrl->lat_count = lat_count;
                    ctrl->published = committed; ctrl->consumed = tickets; ctrl->next_idx = r_next; ctrl->hwm = r_hwm;
                    ctrl->bytes_replicated = bytes_rep; ctrl->batches = batches;
                }
                committed_tickets = tickets;
                last_progress = globaltimer_ns();
                __syncwarp();
            }
        }
        // heartbeat (dare_ibv_rc.c:868-958: the leader writes its SID into every follower's ctrl_data.hb[]): the
        // commit warp is the leader's liveness -- when the hosting process dies the context goes with it and the beats stop
        if (cx->hb_period_ns && (++hb_spins & 0x1fu) == 0) {
            const uint64_t now = globaltimer_ns();
            if (now - last_hb >= cx->hb_period_ns) {
                last_hb = now; hb_beat++;
                if (lane < N && lane != me && cx->peer[lane])
                    st_relaxed_sys(&reinterpret_cast<apus_ctrl_t *>(cx->peer[lane])->hb,
                                   ((cx->term & 0xffffull) << APUS_PUB_TERM_SHIFT) | (hb_beat & APUS_PUB_CUM_MASK));
            }
        }
        const bool rec_ok = S_rec_ok;
        // exit: every worker finished and nothing is in flight
        int ex = 0;
        if (lane == 0) {
            if (!rec_ok && tail == seen && committed == published && ld_acquire_gpu(&seq->workers_done) == cx->n_workers) {
                // one more look at the ring after the workers are known to be done
                ex = 3;
            } else if ((++spins & 0x3ffu) == 0) {
                if (ld_relaxed_sys(&seq->abort_flag)) ex = 2;
                else if (globaltimer_ns() - last_progress > WATCHDOG_NS && (tail != seen || committed != published) &&
                         (cx->target != ~0ull || ld_relaxed_sys_u32(&hw->stop))) {
                    st_relaxed_sys(&hw->error, APUS_KERR_WATCHDOG_COMMIT);
                    st_relaxed_sys(&seq->abort_flag, 1);
                    ex = 2;
                }
            }
        }
        ex = __shfl_sync(0xffffffffu, ex, 0);
        if (ex == 3) {
            // workers are done (acquire above): any record they wrote is visible now; re-check once
            uint64_t st3 = 0, v3 = 0;
            if (lane >= 16 && lane < 24) ld_relaxed_sys_2x64(&ring[seen & PUBMASK].w[2 * (lane - 16)], st3, v3);
            const bool more = __ballot_sync(0xffffffffu, lane >= 16 && lane < 24 && st3 == seen + 1) == 0x00ff0000u;
            ex = more ? 0 : 1;
        }
        if (ex) {
            // clean end of a bounded launch: tell every follower how many entries exist, so
            // that it can leave once it has acked and applied all of them
            if (ex == 1 && cx->target != ~0ull && lane < N && lane != me && cx->peer[lane]) {
                apus_ctrl_t *pc = reinterpret_cast<apus_ctrl_t *>(cx->peer[lane]);
                st_relaxed_sys(&pc->fin_entries, committed);
                __threadfence_system();
                st_relaxed_sys(&pc->fin_target, cx->target);
            }
            break;
        }
    }
}

// The protocol steps of both producers of log entries (the tile machine, leader_express).  The waits run on one lane and
// return true when the abort flag was seen instead of the turn: the caller then holds no valid state.
// The placement state travels from claim to claim as four {stamp, value} pairs of apus_seq_t (DESIGN.md 3a).
struct PlaceRec { uint64_t placed, end, tw, head; };   // tw: rec_tail_pack(tail, wrapped, prev_head)
__device__ __forceinline__ bool place_turn_wait(apus_seq_t *seq, uint64_t stamp, PlaceRec &r)
{
    uint64_t s0, s1, s2, s3;
    uint32_t spins = 0;
    for (;;) {
        ld_relaxed_sys_2x64(seq->rec_placed, s0, r.placed);
        ld_relaxed_sys_2x64(seq->rec_end, s1, r.end);
        ld_relaxed_sys_2x64(seq->rec_tail, s2, r.tw);
        ld_relaxed_sys_2x64(seq->rec_head, s3, r.head);
        if (s0 == stamp && s1 == stamp && s2 == stamp && s3 == stamp) return false;
        if ((++spins & 0x3ffu) == 0 && ld_relaxed_sys(&seq->abort_flag)) return true;
    }
}
// hand the place turn to the claim that starts at slot `stamp`: four 16 B stores, no fence
__device__ __forceinline__ void place_turn_pass(apus_seq_t *seq, uint64_t stamp, const PlaceRec &r)
{
    st_relaxed_sys_2x64(seq->rec_placed, stamp, r.placed);
    st_relaxed_sys_2x64(seq->rec_end, stamp, r.end);
    st_relaxed_sys_2x64(seq->rec_tail, stamp, r.tw);
    st_relaxed_sys_2x64(seq->rec_head, stamp, r.head);
}
// the publish turn {slot number, record number}; acquire: a predecessor that published self-certified data fenced it
// before it handed the turn over
__device__ __forceinline__ bool pub_turn_wait(apus_seq_t *seq, uint64_t stamp, uint64_t &h)
{
    uint64_t sq;
    uint32_t spins = 0;
    for (;;) {
        ld_acquire_gpu_2x64(seq->pub_turn, sq, h);
        if (sq == stamp) return false;
        if ((++spins & 0x3ffu) == 0 && ld_relaxed_sys(&seq->abort_flag)) return true;
    }
}
// room for record h in the publish ring (the commit warp drains it); the tail is re-read only when the last value
// seen would not leave room
__device__ __forceinline__ bool pub_room_wait(apus_seq_t *seq, uint64_t h, uint64_t &tail_seen)
{
    uint32_t spins = 0;
    while (h - tail_seen >= APUS_PUBRING_RECORDS - 2) {
        tail_seen = ld_relaxed_sys(&seq->pub_tail);
        if ((++spins & 0x3ffu) == 0 && ld_relaxed_sys(&seq->abort_flag)) return true;
    }
    return false;
}
__device__ __forceinline__ void pub_turn_pass(apus_seq_t *seq, uint64_t stamp, uint64_t h) { st_relaxed_sys_2x64(seq->pub_turn, stamp, h); }
// publish record h: lanes 16..23 store one {h + 1, value} pair each (the stamp makes the pair valid)
__device__ __forceinline__ void pub_record_write(apus_pubrec_t *ring, uint64_t h, int lane, uint64_t cum, uint64_t end, uint64_t tickets,
                                                 uint64_t t0, uint64_t tail, uint64_t hwm, uint64_t next_idx, uint64_t bytes)
{
    if (lane >= 16 && lane < 24) {
        const int q = lane - 16;
        const uint64_t val = q == PR_CUM ? cum : q == PR_END ? end : q == PR_TICKETS ? tickets : q == PR_T0 ? t0
                           : q == PR_TAIL ? tail : q == PR_HWM ? hwm : q == PR_NEXTIDX ? next_idx : bytes;
        st_relaxed_sys_2x64(&ring[h & PUBMASK].w[2 * q], h + 1, val);
    }
}
// push the 16 B chunk v at log offset lo of the byte range [a, b) to the local log and to every follower: one 16 B store
// per replica (or ONE multicast store, the switch fans it out: leader egress 1x instead of (N-1)x), byte stores at the edges
__device__ __forceinline__ void push_chunk(const apus_devctx_t *__restrict__ cx, const LeaderShared *S, uint64_t lo,
                                           const uint4 v, uint64_t a, uint64_t b)
{
    const int N = cx->group_size;
    uint8_t *entries = cx->region + cx->entries_off;
    if (lo >= a && lo + 16 <= b) {
        if (cx->mc_region) {
            mst_v4(cx->mc_region + cx->entries_off + lo, v);
        } else {
            st_v4(entries + lo, v);
#pragma unroll 1
            for (int f = 0; f < N; f++)
                if (S->peer_entries[f]) st_v4(S->peer_entries[f] + lo, v);
        }
    } else {
#pragma unroll 1
        for (uint32_t j = 0; j < 16; j++) {
            const uint64_t o = lo + j;
            if (o < a || o >= b) continue;
            const uint32_t w = (j < 4) ? v.x : (j < 8) ? v.y : (j < 12) ? v.z : v.w;
            const uint32_t byte = (w >> (8 * (j & 3))) & 0xff;
            st_u8(entries + o, byte);
#pragma unroll 1
            for (int f = 0; f < N; f++)
                if (S->peer_entries[f]) st_u8(S->peer_entries[f] + o, byte);
        }
    }
}
// replica i's apply offset (the leader's own: its log header), what the pruning rule may move the head up to.  Read while
// holding the place turn, at the time of use: it is a ring offset, and a snapshot taken earlier can be so old by then --
// other workers may have pruned meanwhile -- that it falls into the used region of the NEXT lap, "almost caught up"
__device__ __forceinline__ uint64_t apply_off(const apus_devctx_t *__restrict__ cx, int i)
{
    return (i == cx->idx) ? ld_relaxed_sys(&reinterpret_cast<const apus_loghdr_t *>(cx->region + APUS_HDR_OFF)->apply)
                          : ld_relaxed_sys(&reinterpret_cast<const apus_ctrl_t *>(cx->region)->apply_off[i]);
}

// T2a (outside the place turn): state-independent part of the placement -- inclusive prefix sums
// of the log strides and of the staged payload bytes of the fetched batch; apply offsets read ahead
__device__ __noinline__ void leader_prescan(const apus_devctx_t *__restrict__ cx, LeaderShared *S, int lane)
{
    const uint32_t nf = S->n_fetch;
    uint32_t carry = 0, xcarry = 0, scut = nf, fext = 0xffffffffu, hhk = 0xffffffffu;
    // a batch of ONE request shape (the benchmark's, and most applications' bursts) needs no scan: cum[k] = (k+1) * stride
    const uint32_t es0 = S->es[0], xb0 = S->xb[0];
    bool uniform = true;
    for (uint32_t r = 0; r < nf; r += 32) {
        const uint32_t k = r + lane;
        if (__ballot_sync(0xffffffffu, k < nf && (S->es[k] != es0 || S->xb[k] != xb0))) { uniform = false; break; }
    }
    for (uint32_t r = 0; r < nf; r += 32) {
        const uint32_t k = r + lane;
        const bool in = k < nf;
        uint32_t inc = in ? S->es[k] : 0u, xinc = in ? S->xb[k] : 0u;
        if (uniform) {
            if (in) { S->cum_es[k] = (k + 1u) * es0; S->cum_xb[k] = (k + 1u) * xb0; }
        } else {
#pragma unroll
            for (int sft = 1; sft < 32; sft <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, inc, sft);
                const uint32_t xo = __shfl_up_sync(0xffffffffu, xinc, sft);
                if (lane >= sft) { inc += o; xinc += xo; }
            }
            if (in) { S->cum_es[k] = carry + inc; S->cum_xb[k] = xcarry + xinc; }
            carry += __shfl_sync(0xffffffffu, inc, 31);
            xcarry += __shfl_sync(0xffffffffu, xinc, 31);
        }
        const uint32_t hm = __ballot_sync(0xffffffffu, in && S->ty[k] == T_HEAD);
        if (hm) hhk = r + (31u - (uint32_t)__clz(hm));                 // the LAST host HEAD entry of the batch
        const uint32_t wm = __ballot_sync(0xffffffffu, in && k > 0 && (S->flg[k] & 2u));
        const uint32_t em = __ballot_sync(0xffffffffu, in && (S->flg[k] & 1u));
        if (wm && scut == nf) scut = r + (uint32_t)(__ffs(wm) - 1);
        if (em && fext == 0xffffffffu) fext = r + (uint32_t)(__ffs(em) - 1);
    }
    if (lane == 0) { S->static_cut = scut; S->first_ext_all = fext; S->host_head_k = hhk; }
}

// T2b (inside the place turn): place the next sub-tile of the fetched batch (entries kbase..nf) --
// log_append_entry's offset rules, free-space rule E2 and the pruning rule, on the placement
// state this CTA holds.  Kept short: everything state independent was done by leader_prescan.
__device__ __noinline__ void leader_place(const apus_devctx_t *__restrict__ cx, LeaderShared *S, const apus_cslot_t *sl, int lane)
{
    const int N = cx->group_size;
    apus_loghdr_t *hdr = reinterpret_cast<apus_loghdr_t *>(cx->region + APUS_HDR_OFF);
    const uint64_t L = cx->log_len;
    const bool autoprune = (cx->flags & APUS_FLAG_AUTOPRUNE) != 0;
    const uint32_t kbase = S->kbase, nf = S->n_fetch;
    const uint64_t end = S->st_end;

    const uint64_t pos0 = ring_pos(end, L);
    uint64_t used = ring_used(S->st_head, end, L);            // st_head: refreshed by the caller while blocked
    // ---- device-side log pruning (apus_place.h): the furthest-behind apply offset, one replica per lane
    uint32_t autoh = 0;
    uint64_t new_head = 0;
    if (autoprune && prune_considered(end, used, !S->st_prev_head || S->was_blocked, L)) {
        uint64_t d = lane < N ? prune_dist(apply_off(cx, lane), end, used, L) : 0;
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) {
            const uint64_t o = __shfl_xor_sync(0xffffffffu, d, sft);
            d = o > d ? o : d;
        }
        autoh = prune_decide(d, S->st_tail, end, L, &new_head, &used);
    }
    const uint32_t hbytes = autoh ? APUS_HDR_BYTES : 0;
    // limits for a contiguous sub-tile starting at pos0: before len, rule E2, the tile image
    const uint64_t reserve = autoprune ? APUS_HDR_BYTES : 0;
    uint64_t limit = place_limit(pos0, used, reserve, L);
    const uint64_t imgcap = APUS_LEADER_IMG_BYTES - 16u - (pos0 & 15u);
    if (limit > imgcap) limit = imgcap;
    const uint32_t base_es = kbase ? S->cum_es[kbase - 1] : 0u, base_xb = kbase ? S->cum_xb[kbase - 1] : 0u;

    // how many entries from kbase fit: the prefix sums are monotone, one compare + ballot per 32 entries
    uint32_t m = nf - kbase, first_ext = 0xffffffffu;
    for (uint32_t r = kbase; r < nf; r += 32) {
        const uint32_t k = r + lane;
        const bool in = k < nf;
        const bool bad = in && ((uint64_t)hbytes + (S->cum_es[k] - base_es) > limit ||
                                S->cum_xb[k] - base_xb > APUS_LEADER_EXT_BYTES || (k > kbase && (S->flg[k] & 2u)));
        const uint32_t badmask = __ballot_sync(0xffffffffu, bad);
        const uint32_t good = badmask ? (uint32_t)(__ffs(badmask) - 1) : 32u;
        if (first_ext == 0xffffffffu) {
            const uint32_t extmask = __ballot_sync(0xffffffffu, in && (uint32_t)lane < good && (S->flg[k] & 1u));
            if (extmask) first_ext = r + (uint32_t)(__ffs(extmask) - 1);
        }
        if (badmask) { m = r + good - kbase; break; }
    }
    if (lane == 0) {
        const uint32_t carry = hbytes + (m ? S->cum_es[kbase + m - 1] - base_es : 0u);      // log bytes of the sub-tile
        const uint32_t xcarry = m ? S->cum_xb[kbase + m - 1] - base_xb : 0u;               // staged payload bytes
        S->gap = 0; S->ghost = 0; S->blocked = 0; S->last = 0;
        uint64_t a = pos0, b = pos0;
        if (m == 0 && !autoh) {
            // entry kbase does not fit at pos0: wrap or no space
            const int w = wrap_rule(pos0, used, S->es[kbase], has_cmd(S->ty[kbase]), reserve, L);
            if (w != PLACE_BLOCKED) {
                S->gap = 1;
                S->ghost = w == PLACE_WRAP_GHOST ? 1u : 0u;
                b = L;
            } else {
                S->blocked = 1;        // back-pressure: wait for head to advance
            }
        } else {
            b = pos0 + carry;
        }
        S->a = a; S->b = b; S->m = m;
        S->hbytes = hbytes; S->base_es = base_es; S->base_xb = base_xb;
        S->ext_bytes = (m && first_ext != 0xffffffffu) ? xcarry : 0u;
        S->ext_base = (first_ext != 0xffffffffu) ? (uint64_t)(sl[first_ext].type_off & APUS_SLOT_OFF_MASK) * 16ull : 0ull;
        S->auto_head = autoh; S->auto_head_val = new_head;
        S->idx0 = S->st_next_idx;
        S->fresh = (a >= S->st_hwm) ? 1u : 0u;
        if (S->blocked) S->was_blocked = 1;
        if (!S->blocked) {
            S->was_blocked = 0;
            // commit the placement to the state this CTA carries
            if (autoh) { st_relaxed_sys(&hdr->head, new_head); S->st_head = new_head; }
            if (S->host_head_k != 0xffffffffu && S->host_head_k >= kbase && S->host_head_k < kbase + m) {
                const uint64_t nh = adopt_head(S->st_head, slot_head_value(&sl[S->host_head_k]), b, L);
                if (nh != S->st_head) { S->st_head = nh; st_relaxed_sys(&hdr->head, nh); }
            }
            if (S->gap) {
                S->st_end = 0; S->st_hwm = L;
            } else {
                const uint64_t ne = ring_pos(b, L);                     // rule E1
                S->new_end = ne;
                S->st_end = ne;
                S->st_tail = m ? a + hbytes + (S->cum_es[kbase + m - 1] - base_es) - S->es[kbase + m - 1] : a;
                S->tail_after = S->st_tail;
                S->st_next_idx += m + autoh;
                S->st_placed += m + autoh;
                S->cum_after = S->st_placed;
                if (autoh) atomicAdd(reinterpret_cast<unsigned long long *>(&reinterpret_cast<apus_ctrl_t *>(cx->region)->auto_heads), 1ull);
                S->st_prev_head = (autoh && m == 0) ? 1u : 0u;         // never two HEAD entries in a row (dare_log.h:477-480)
                if (b > S->st_hwm) S->st_hwm = b;
                S->last = (kbase + m == nf) ? 1u : 0u;
            }
            S->hwm_after = S->st_hwm;
        }
    }
}


// ---------------------------------------------------------------------------------
// Express path: ONE request, handled by warp 0 alone while the rest of the CTA stays parked at its barrier.
// This is the closed-loop commit-latency path (proxy.c:108-161: an application thread enqueues one request and
// spins until it is committed): slot already in registers (worker 0 polls the slot itself), placement state
// cached from the previous request, the 64+len bytes composed in a 256 B scratch, pushed with one 16 B store per
// chunk and follower, and published with a SELF-CERTIFYING record -- no system fence anywhere on the way.
// The publish turn is then HELD (nobody is waiting for it) and handed on, after a fence, when somebody else claims.
// Anything unusual (wrap, pruning due, payload in the byte ring, no room) returns 1: the tile machine takes the claim.
// ---------------------------------------------------------------------------------
struct Express {
    uint64_t next_seq;                 // slot number right after my latest claim
    PlaceRec rec;                      // placement state I handed on under stamp next_seq
    uint64_t pub_h;                    // publish-ring record number that goes with publish turn next_seq
    uint32_t have_place;               // rec is what the sequencer records hold
    uint32_t hold;                     // I still hold publish turn next_seq (self-certified data, not fenced yet)
    uint64_t pub_tail_seen;            // publish-ring tail as last read (lane 0)
    uint64_t dt[5];                    // ns of the latest request: place, compose, push, publish turn, publish (profiling)
};

__device__ __forceinline__ void express_release(apus_seq_t *seq, Express &X, int lane)
{
    // the data of my self-certified publishes becomes ordinary fenced data before anybody else may publish behind it
    __syncwarp();
    if (lane == 0) {
        __threadfence_system();
        pub_turn_pass(seq, X.next_seq, X.pub_h);
    }
    X.hold = 0;
    __syncwarp();
}

__device__ __noinline__ int leader_express(const apus_devctx_t *__restrict__ cx, const LeaderShared *S, Express &X,
                                              const uint64_t claimed, uint4 sv, const bool have_slot, uint8_t *scratch,
                                              const int lane, const uint4 pf, const uint64_t pf_pos)
{
    const int N = cx->group_size, me = cx->idx;
    const uint64_t L = cx->log_len;
    apus_ctrl_t *ctrl = reinterpret_cast<apus_ctrl_t *>(cx->region);
    apus_seq_t *seq = reinterpret_cast<apus_seq_t *>(cx->region + APUS_SEQ_OFF);
    apus_pubrec_t *pubring = reinterpret_cast<apus_pubrec_t *>(cx->region + APUS_PUBRING_OFF);
    uint8_t *entries = cx->region + cx->entries_off;
    uint32_t *lindex = reinterpret_cast<uint32_t *>(cx->region + APUS_INDEX_OFF);
    const uint64_t t_deq = (cx->flags & (APUS_FLAG_STATS | APUS_FLAG_PROFILE)) ? globaltimer_ns() : 0;

    if (!have_slot && lane < 8)
        sv = ld_relaxed_sys_v4(reinterpret_cast<const uint8_t *>(cx->sub_slots + (claimed & cx->sub_mask)) + 16u * lane);
    const uint32_t to = __shfl_sync(0xffffffffu, sv.z, 0), lw = __shfl_sync(0xffffffffu, sv.w, 0);
    const uint32_t ty = (to >> APUS_SLOT_TYPE_SHIFT) & APUS_SLOT_TYPE_MASK, len = lw & 0xffffu, clt = lw >> 16;
    const uint64_t req_id = (uint64_t)__shfl_sync(0xffffffffu, sv.x, 0) | ((uint64_t)__shfl_sync(0xffffffffu, sv.y, 0) << 32);
    if (!has_cmd(ty) || (to & APUS_SLOT_EXT)) return 1;
    const uint32_t es = APUS_HDR_BYTES + len, nb = 2u + len;

    // the followers' ack counts (is everybody caught up?) are needed only when the entry is published: in flight meanwhile
    const bool isf = lane < N && lane != me && cx->peer[lane];
    uint64_t ackv = 0;
    if (isf) ackv = ld_relaxed_sys(&ctrl->ack[lane]);

    // ---- place turn ----
    PlaceRec r = X.rec;
    if (!(X.have_place && X.next_seq == claimed)) {
        if (__shfl_sync(0xffffffffu, lane == 0 && place_turn_wait(seq, claimed, r), 0)) return 2;
        r.placed = __shfl_sync(0xffffffffu, r.placed, 0); r.end = __shfl_sync(0xffffffffu, r.end, 0);
        r.tw = __shfl_sync(0xffffffffu, r.tw, 0); r.head = __shfl_sync(0xffffffffu, r.head, 0);
        X.rec = r; X.have_place = 1; X.next_seq = claimed;
    }
    const uint64_t placed = r.placed, end = r.end, pos0 = ring_pos(end, L), used = ring_used(r.head, end, L);
    const bool wrapped = (r.tw & APUS_REC_WRAPPED) != 0;
    const bool autoprune = (cx->flags & APUS_FLAG_AUTOPRUNE) != 0;
    // Pruning is the tile machine's business (it appends the HEAD entry): once the ring is half used every request is
    // handed over until a HEAD entry has made room.  Below that the express path does not even look at the apply offsets.
    if (autoprune && used >= (L >> 1)) return 1;
    if (es > place_limit(pos0, used, autoprune ? APUS_HDR_BYTES : 0, L)) return 1;   // wrap / no room: general placement

    const uint64_t a = pos0, b = pos0 + es;
    const uint64_t ne = ring_pos(b, L);                               // rule E1
    const bool nw = wrapped || b == L;
    const uint64_t cum = placed + 1;
    // hand the place turn on at once (stamp = next slot number) and remember what I wrote
    X.rec = PlaceRec{cum, ne, rec_tail_pack(a, nw, 0), r.head};
    if (lane == 0) place_turn_pass(seq, claimed + 1, X.rec);
    const uint64_t idx = S->idx_base + placed + 1;
    const bool xprof = (cx->flags & APUS_FLAG_PROFILE) != 0;
    const uint64_t t_place = xprof ? globaltimer_ns() : 0;

    // ---- compose: lane c builds the 16 B chunk c of the entry.  Everything except two HOLES (bytes 41..47 and the
    //      slack behind the data image) is new; the holes keep what the log held (dare_log.h:507-529 never writes them) --
    //      those bytes were PREFETCHED while this warp was idle (pf, taken at the offset the next entry was going to get) ----
    const uint64_t a16 = a & ~15ull;
    const uint32_t nch = (uint32_t)(((b + 15ull) & ~15ull) - a16) >> 4;          // <= 11
    const uint64_t lo = a16 + 16ull * lane;
    uint4 v = make_uint4(0, 0, 0, 0);
    if ((a & 15ull) == 0) {
        uint4 oldv = make_uint4(0, 0, 0, 0);
        if (wrapped) {
            if (pf_pos == a) oldv = pf;
            else if (lane < (int)nch) oldv = ld_relaxed_sys_v4(entries + lo);
        }
        const int j = lane - 3;                                       // data image chunk of this lane
        const int srcl = (j < 0) ? 0 : ((j < 2) ? j + 1 : ((j + 2) & 31));   // slot chunk holding image bytes [16j, 16j+16)
        uint4 dv;
        dv.x = __shfl_sync(0xffffffffu, sv.x, srcl); dv.y = __shfl_sync(0xffffffffu, sv.y, srcl);
        dv.z = __shfl_sync(0xffffffffu, sv.z, srcl); dv.w = __shfl_sync(0xffffffffu, sv.w, srcl);
        if (lane == 0) v = make_uint4((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)cx->term, (uint32_t)(cx->term >> 32));
        else if (lane == 1) v = make_uint4((uint32_t)req_id, (uint32_t)(req_id >> 32), (clt & 0xffffu) | (ty << 16) | ((uint32_t)me << 24), 0u);
        else if (lane == 2) v = make_uint4(0u, 0u, oldv.z & 0xffffff00u, oldv.w);           // reply[4..12] = 0, bytes 41..47 stay
        else v = chunk_select(dv, oldv, (int)nb - 16 * j);
    } else {
        // entry at an odd offset (ragged payloads): byte-granular composition in shared memory
        uint8_t *img = scratch, *xsl = scratch + 256;
        if (lane < (int)nch)
            reinterpret_cast<uint4 *>(img)[lane] = wrapped ? ld_relaxed_sys_v4(entries + lo) : make_uint4(0, 0, 0, 0);
        if (lane == 1 || lane == 2) reinterpret_cast<uint4 *>(xsl)[lane - 1] = sv;   // inline image bytes 0..31
        if (lane >= 4 && lane <= 6) reinterpret_cast<uint4 *>(xsl)[lane - 2] = sv;   // ... 32..79
        __syncwarp();
        uint8_t *e = img + (a - a16);
        group_write_header(e, lane, 32, idx, cx->term, req_id, clt, ty, me, false);
        group_copy_smem(e + E_DATA, xsl, nb, lane, 32);
        __syncwarp();
        if (lane < (int)nch) v = reinterpret_cast<const uint4 *>(img)[lane];
    }
    const uint64_t t_compose = xprof ? globaltimer_ns() : 0;

    // ---- push: local log first, then every follower; checksum of exactly the bytes [a, b) ----
    uint64_t cs = 0;
    if (lane < (int)nch) {
        cs = cs_chunk(v, lo, a, b);
        push_chunk(cx, S, lo, v, a, b);
    }
    {   // offset index: lane f writes replica f's word (lane `me` the local one)
        const uint32_t at = (uint32_t)cum & cx->idx_mask;
        uint32_t *ip = (lane == me) ? lindex : (lane < N ? S->peer_index[lane] : nullptr);
        if (ip) ip[at] = (uint32_t)a;
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) cs += __shfl_xor_sync(0xffffffffu, cs, sft);
    // self-certify only when every follower has acked everything before this entry: each of them is then at
    // exactly `a` and can verify the one entry; a follower that lags is served by a fenced publish (it may skip records)
    const bool caught = __ballot_sync(0xffffffffu, isf && ackv != placed) == 0;

    const uint64_t t_push = xprof ? globaltimer_ns() : 0;
    // ---- publish turn (mine already when I held it) ----
    uint64_t h = X.pub_h;
    const bool ab = lane == 0 && ((!X.hold && pub_turn_wait(seq, claimed, h)) || pub_room_wait(seq, h, X.pub_tail_seen));
    if (__shfl_sync(0xffffffffu, ab, 0)) return 2;
    h = __shfl_sync(0xffffffffu, h, 0);
    const uint64_t t_turn = xprof ? globaltimer_ns() : 0;
    const uint64_t cumt = cum | ((cx->term & 0xffffull) << APUS_PUB_TERM_SHIFT);
    const bool cert = caught && !(cx->flags & APUS_FLAG_NO_EXPRESS);
    if (isf) {
        apus_ctrl_t *pc = reinterpret_cast<apus_ctrl_t *>(cx->peer[lane]);
        if (cert) {
            st_relaxed_sys_2x64(&pc->pub_csum, cs + cs_key(cumt), a);
            st_relaxed_sys_2x64(&pc->pub_end, ne | APUS_PUB_CERT, cumt);
        } else {
            __threadfence_system();                                  // data before tail (I1), the classic way
            st_relaxed_sys_2x64(&pc->pub_end, ne, cumt);
        }
    }
    pub_record_write(pubring, h, lane, cum, ne, claimed + 1, t_deq, a, nw ? L : b, idx + 1, (uint64_t)es * (uint64_t)(N - 1));
    X.next_seq = claimed + 1; X.pub_h = h + 1;
    if (xprof) {
        const uint64_t t_end = globaltimer_ns();
        X.dt[0] = t_place - t_deq; X.dt[1] = t_compose - t_place; X.dt[2] = t_push - t_compose; X.dt[3] = t_turn - t_push; X.dt[4] = t_end - t_turn;
    }
    if (cert) {
        X.hold = 1;                    // nobody is waiting: keep the turn, skip the fence
    } else {
        X.hold = 0;
        __syncwarp();
        if (lane == 0) pub_turn_pass(seq, claimed + 1, h + 1);
    }
    return 0;
}

// T2 at the start of a claim (lane 0 of warp 0): wait for the place turn, then place the whole claim when it fits
// contiguously and no pruning is due.  The turn is held for the state-dependent offset arithmetic alone (not the fetch,
// not the prefix sums), in this common case for a dozen integer operations: it is handed on before the tile is written
// down for the other warps.  Otherwise the placement state is left in S->st_* for leader_place.
enum { CLAIM_FAST, CLAIM_SLOW, CLAIM_ABORTED };
__device__ __forceinline__ int place_claim(const apus_devctx_t *__restrict__ cx, LeaderShared *S, const apus_cslot_t *sl,
                                           const bool prof, uint64_t *tn)
{
    apus_seq_t *seq = reinterpret_cast<apus_seq_t *>(cx->region + APUS_SEQ_OFF);
    apus_loghdr_t *hdr = reinterpret_cast<apus_loghdr_t *>(cx->region + APUS_HDR_OFF);
    const uint64_t L = cx->log_len;
    const uint32_t nf = S->n_fetch;
    const uint64_t tw0 = prof ? globaltimer_ns() : 0;
    PlaceRec r;
    const bool ab = place_turn_wait(seq, S->my_seq, r);
    if (prof) { tn[1] += globaltimer_ns() - tw0; S->t_place_acq = globaltimer_ns(); }
    if (ab) return CLAIM_ABORTED;                       // no stamp: nothing may be placed
    const bool wrapped = (r.tw & APUS_REC_WRAPPED) != 0, prevh = (r.tw & APUS_REC_PREV_HEAD) != 0;
    const uint64_t end = r.end, tail = rec_tail_off(r.tw);
    S->st_head = r.head;
    const uint64_t pos0 = ring_pos(end, L), used = ring_used(r.head, end, L);
    const uint64_t total = S->cum_es[nf - 1];
    const bool autoprune = (cx->flags & APUS_FLAG_AUTOPRUNE) != 0;
    bool prune_due = false;
    if (autoprune && prune_considered(end, used, !prevh || S->was_blocked, L)) {
        uint64_t d = 0;
        for (int i = 0; i < cx->group_size; i++) {
            const uint64_t di = prune_dist(apply_off(cx, i), end, used, L);
            d = di > d ? di : d;
        }
        uint64_t nh = r.head, nu = used;
        prune_due = prune_decide(d, tail, end, L, &nh, &nu);
    }
    if (prune_due || total > place_limit(pos0, used, autoprune ? APUS_HDR_BYTES : 0, L) ||
        total > APUS_LEADER_IMG_BYTES - 16u - (pos0 & 15u) || S->cum_xb[nf - 1] > APUS_LEADER_EXT_BYTES || S->static_cut != nf) {
        S->st_end = end; S->st_tail = tail; S->st_placed = r.placed;
        S->st_next_idx = S->idx_base + r.placed + 1;
        S->st_hwm = wrapped ? L : pos0; S->st_prev_head = prevh ? 1u : 0u;
        if (prof) tn[4]++;
        return CLAIM_SLOW;
    }
    const uint64_t b = pos0 + total, ne = ring_pos(b, L), nt = b - S->es[nf - 1];
    const bool nw = wrapped || b == L;
    // a HEAD entry submitted by the host carries the new head
    const uint64_t headv = S->host_head_k != 0xffffffffu ? adopt_head(r.head, slot_head_value(&sl[S->host_head_k]), ne, L) : r.head;
    if (headv != r.head) st_relaxed_sys(&hdr->head, headv);
    place_turn_pass(seq, S->my_seq + nf, PlaceRec{r.placed + nf, ne, rec_tail_pack(nt, nw, 0), headv});
    if (prof) { tn[7] += globaltimer_ns() - S->t_place_acq; tn[3]++; }
    // ... and only then write down the tile for the other warps
    S->gap = 0; S->ghost = 0; S->blocked = 0; S->last = 1;
    S->a = pos0; S->b = b; S->m = nf;
    S->hbytes = 0; S->base_es = 0; S->base_xb = 0;
    S->ext_bytes = (S->first_ext_all != 0xffffffffu) ? S->cum_xb[nf - 1] : 0u;
    S->ext_base = (S->first_ext_all != 0xffffffffu) ? (uint64_t)(sl[S->first_ext_all].type_off & APUS_SLOT_OFF_MASK) * 16ull : 0ull;
    S->auto_head = 0; S->auto_head_val = 0;
    S->idx0 = S->idx_base + r.placed + 1;
    S->fresh = wrapped ? 0u : 1u;
    S->new_end = ne; S->tail_after = nt; S->cum_after = r.placed + nf;
    S->hwm_after = nw ? L : b;
    return CLAIM_FAST;
}

__device__ void leader_main(const apus_devctx_t *__restrict__ cx, const uint32_t wid)
{
    LeaderShared *S = reinterpret_cast<LeaderShared *>(smem_raw);
    uint8_t *slots = smem_raw + L_SLOTS_OFF;
    uint8_t *ext = smem_raw + L_EXT_OFF;
    uint8_t *img = smem_raw + L_IMG_OFF;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = cx->group_size, me = cx->idx;
    apus_ctrl_t *ctrl = reinterpret_cast<apus_ctrl_t *>(cx->region);
    apus_seq_t *seq = reinterpret_cast<apus_seq_t *>(cx->region + APUS_SEQ_OFF);
    apus_pubrec_t *pubring = reinterpret_cast<apus_pubrec_t *>(cx->region + APUS_PUBRING_OFF);
    apus_loghdr_t *hdr = reinterpret_cast<apus_loghdr_t *>(cx->region + APUS_HDR_OFF);
    uint8_t *entries = cx->region + cx->entries_off;
    uint32_t *lindex = reinterpret_cast<uint32_t *>(cx->region + APUS_INDEX_OFF);
    apus_hostwords_t *hw = cx->hw;

    // ---- sequencer reset handshake: worker 0 prepares the shared words of this launch ----
    if (tid == 0) {
        if (wid == 0) {
            seq->claimed_slots = ctrl->consumed;
            seq->doorbell = ctrl->consumed;
            seq->place_seq = 0; seq->workers_done = 0; seq->abort_flag = 0; seq->w0_idle = 0;
            for (uint32_t i = 0; i < APUS_PUBRING_RECORDS; i++)
                for (int q = 0; q < 8; q++) pubring[i].w[2 * q] = 0;          // no valid record
            // the turns are stamped with slot numbers: the first claim of this launch starts at ctrl->consumed
            place_turn_pass(seq, ctrl->consumed, PlaceRec{ctrl->published, hdr->end,
                                                          rec_tail_pack(hdr->tail, ctrl->hwm == cx->log_len, 0), hdr->head});
            // entries published by an earlier launch but not yet committed come back as one record
            seq->pub_head = 0; seq->pub_tail = 0;
            pub_turn_pass(seq, ctrl->consumed, 0);
            // (the commit warp keeps ctrl/hdr in step with what is COMMITTED; a clean launch ends with
            //  everything committed, so there is nothing published-but-uncommitted to carry over)
            __threadfence();
            st_release_gpu(&seq->ready_epoch, cx->epoch);
        } else {
            while (ld_acquire_gpu(&seq->ready_epoch) != cx->epoch) { }
        }
        S->finish = 0; S->abort = 0; S->was_blocked = 0; S->avg_es = 128; S->avg_xb = 0; S->pub_tail_seen = 0;
        S->idx_base = ctrl->next_idx - 1 - ctrl->published;
        for (int i = 0; i < APUS_MAX_SERVERS; i++) {
            S->peer_entries[i] = (i < N && i != me && cx->peer[i]) ? cx->peer[i] + cx->entries_off : nullptr;
            S->peer_index[i] = (i < N && i != me && cx->peer[i]) ? reinterpret_cast<uint32_t *>(cx->peer[i] + APUS_INDEX_OFF) : nullptr;
        }
    }
    __syncthreads();

    if (warp == N_PRODUCER_WARPS) {   // warp 15: the commit warp lives in worker 0
        if (wid == 0) leader_commit_warp(cx);
        else if (wid == 1 && cx->doorbell_relay && lane == 0) {
            // doorbell relay: the only poller of the host-mapped doorbell (one PCIe read in flight instead
            // of one per idle worker -- those reads also slow every system fence down); workers poll the mirror
            uint64_t last = ld_relaxed_sys(&seq->doorbell);
            uint32_t spins = 0;
            for (;;) {
                const uint64_t t = ld_acquire_sys(cx->sub_tail);
                if (t != last) { st_release_gpu(&seq->doorbell, t); last = t; }   // slots were written before the doorbell
                if ((++spins & 0x3fu) == 0 &&
                    (ld_relaxed_sys(&seq->abort_flag) || ld_relaxed_sys(&seq->workers_done) >= cx->n_workers)) break;
            }
        }
        return;
    }

    // ---- producer warps 0..14 ------------------------------------------------------
    uint64_t last_progress = globaltimer_ns();
    const bool prof = (cx->flags & APUS_FLAG_STATS) != 0 && tid == 0 && wid == 0;
    uint64_t ph[8], tn[8], tprev = globaltimer_ns();
    for (int i = 0; i < 8; i++) { ph[i] = ctrl->phase_ns[i]; tn[i] = ctrl->turn_ns[i]; }
#define PHASE(i) do { if (prof) { const uint64_t _t = globaltimer_ns(); ph[i] += _t - tprev; tprev = _t; } } while (0)
    Express X{};
    uint64_t xguess = ctrl->consumed;          // worker 0: the slot it expects to be claimed next
    uint4 pf = make_uint4(0, 0, 0, 0);         // express: prefetched log bytes at offset pf_pos (lane c: chunk c)
    uint64_t pf_pos = ~0ull;

    for (;;) {
        // ---- T0: claim the next slots of the submission ring: lock-free, one compare-and-swap on the
        //      claimed-slots counter.  The claimed range [slot0, slot0+n) is also the worker's place in
        //      the order: the place and publish turns are stamped with slot numbers ----
        if (warp == 0) {
            uint32_t n = 0, fin = 0, spins = 0, lone_waits = 0;
            const uint64_t tw0 = prof ? globaltimer_ns() : 0;
            uint64_t claimed = 0;
            const bool poll_slot = cx->slot_poll != 0 && wid == 0;
            const bool express_on = (cx->flags & APUS_FLAG_NO_EXPRESS) == 0;
            if (wid == 0 && lane == 0) st_relaxed_sys(&seq->w0_idle, 1);
            for (;;) {
                // worker 0 polls the NEXT SLOT itself (lanes 0..7, one 128 B read over PCIe) while lane 0 looks at the
                // claim counter and the doorbell: a lone request is in registers one PCIe round trip after the host wrote it
                uint4 sv = make_uint4(0, 0, 0, 0);
                const uint64_t sv_for = xguess;
                if (poll_slot && lane < 8)
                    sv = ld_relaxed_sys_v4(reinterpret_cast<const uint8_t *>(cx->sub_slots + (xguess & cx->sub_mask)) + 16u * lane);
                // (a second poll in flight does not help: two loads of one line from one SM are merged, the younger one
                //  returns the older one's sample -- measured: host-clock latency got worse by ~1.5 us)
                // idle-time prefetch: the bytes the log holds where the NEXT entry will go (its holes keep them); the offset
                // is known as long as this warp placed the latest entry
                if (express_on && X.have_place && X.rec.end != cx->log_len && (X.rec.tw & APUS_REC_WRAPPED) &&
                    pf_pos != X.rec.end && (X.rec.end & 15ull) == 0 && X.rec.end + 16ull * 12 <= cx->log_len) {
                    if (lane < 12) pf = ld_relaxed_sys_v4(entries + X.rec.end + 16ull * lane);
                    pf_pos = X.rec.end;
                }
                uint32_t ctl = 0;
                uint64_t t = 0, w0i = 0;
                if (lane == 0) {
                    if ((spins & 0x3fu) == 0 && ld_relaxed_sys(&seq->abort_flag)) ctl = 1;
                    // (relaxed: a doorbell that shows requests is re-read with acquire before anything is fetched)
                    t = cx->doorbell_relay ? ld_relaxed_sys(&seq->doorbell) : ld_relaxed_sys(cx->sub_tail);
                    claimed = ld_relaxed_sys(&seq->claimed_slots);
                    if (claimed >= cx->target) ctl = 1;
                    if (wid != 0) w0i = ld_relaxed_sys(&seq->w0_idle);
                    if (t > claimed) t = cx->doorbell_relay ? ld_acquire_gpu(&seq->doorbell) : ld_acquire_sys(cx->sub_tail);
                }
                ctl = __shfl_sync(0xffffffffu, ctl, 0);
                claimed = __shfl_sync(0xffffffffu, claimed, 0);
                t = __shfl_sync(0xffffffffu, t, 0);
                w0i = __shfl_sync(0xffffffffu, w0i, 0);
                // a held publish turn is passed on as soon as anybody else has claimed slots (or I am leaving)
                if (X.hold && (ctl || claimed != X.next_seq)) express_release(seq, X, lane);
                if (ctl) { fin = 1; break; }
                bool slot_ok = false;
                if (poll_slot) {
                    const uint64_t stamp = (uint64_t)sv.x | ((uint64_t)sv.y << 32);
                    slot_ok = (__ballot_sync(0xffffffffu, (lane == 3 || lane == 7) && stamp == sv_for + 1) == 0x88u) && sv_for == claimed;
                    xguess = claimed;
                }
                uint64_t avail = t > claimed ? t - claimed : 0;
                if (slot_ok && avail == 0) avail = 1;
                // the doorbell may show a lone request before the slot poll in flight does: wait for the poll (next
                // iteration) instead of claiming now and fetching the slot with one more PCIe round trip
                if (poll_slot && express_on && avail == 1 && !slot_ok && ++lone_waits < 8) avail = 0; else lone_waits = 0;
                // lone requests belong to worker 0 while it is polling (express path)
                if (avail == 1 && wid != 0 && w0i) avail = 0;
                if (avail) {
                    const uint64_t room = cx->target - claimed;
                    if (avail > room) avail = room;
                    uint32_t nn = 0, won = 0;
                    if (lane == 0) {
                        // share a shallow queue between the workers instead of one big tile
                        uint64_t want = (avail + cx->n_workers - 1) / cx->n_workers;
                        if (want < 32) want = avail < 32 ? avail : 32;
                        // a claim should fit ONE tile image / staging buffer (else it is placed in pieces
                        // while holding the place turn, which serializes the workers)
                        uint64_t aes = ld_relaxed_sys(&seq->avg_es), axb = ld_relaxed_sys(&seq->avg_xb);
                        if (aes < 64) aes = 128;
                        uint64_t fit = (APUS_LEADER_IMG_BYTES - 256u) / aes;
                        if (axb) { const uint64_t xf = APUS_LEADER_EXT_BYTES / axb; if (xf < fit) fit = xf; }
                        if (fit < 1) fit = 1;
                        if (want > fit) want = fit;
                        nn = want > MAXB ? MAXB : (uint32_t)want;
                        won = atomicCAS(reinterpret_cast<unsigned long long *>(&seq->claimed_slots), (unsigned long long)claimed,
                                        (unsigned long long)(claimed + nn)) == (unsigned long long)claimed;
                    }
                    nn = __shfl_sync(0xffffffffu, nn, 0);
                    won = __shfl_sync(0xffffffffu, won, 0);
                    if (!won) continue;                   // somebody else took these slots: look again
                    if (nn == 1 && express_on) {
                        const int rc = leader_express(cx, S, X, claimed, sv, slot_ok, img, lane, pf, pf_pos);
                        if (rc == 0) {
                            xguess = claimed + 1; last_progress = globaltimer_ns();
                            if (prof) { tn[5]++; ph[7]++; for (int q = 0; q < 5; q++) ph[1 + q] += X.dt[q]; }
                            continue;
                        }
                        if (rc == 2) { fin = 1; break; }
                        // rc == 1: the tile machine places this claim; the cached placement state is still what the records hold
                    }
                    n = nn;
                    break;
                }
                if ((++spins & 0x1ffu) == 0) {
                    uint32_t stopf = 0;
                    if (lane == 0) {
                        if (ld_relaxed_sys_u32(&hw->stop)) stopf = 1;
                        else if (cx->target != ~0ull && globaltimer_ns() - last_progress > WATCHDOG_NS) {
                            st_relaxed_sys(&hw->error, APUS_KERR_WATCHDOG_LEADER);
                            st_relaxed_sys(&seq->abort_flag, 1); stopf = 1;
                        }
                        if (prof) for (int i = 0; i < 8; i++) { ctrl->phase_ns[i] = ph[i]; ctrl->turn_ns[i] = tn[i]; }
                    }
                    stopf = __shfl_sync(0xffffffffu, stopf, 0);
                    if (stopf) { fin = 1; break; }
                }
            }
            if (X.hold) express_release(seq, X, lane);
            X.have_place = 0; pf_pos = ~0ull;                  // other workers may place in between
            if (lane == 0) {
                if (wid == 0) st_relaxed_sys(&seq->w0_idle, 0);
                if (prof) { tn[0] += globaltimer_ns() - tw0; tn[6]++; }
                if (n) { S->slot0 = claimed; S->my_seq = claimed; }
                S->n_fetch = n; S->finish = fin;
                S->t_dequeue = globaltimer_ns();
            }
        }
        bar_sync(1, NT);
        if (S->finish) break;
        const uint32_t nf = S->n_fetch;
        PHASE(0);

        // ---- T1: fetch the slots (descriptor + inline payload), coalesced 16 B loads --------
        {
            const uint64_t s0 = S->slot0 & cx->sub_mask;
            const uint64_t nslots = (uint64_t)cx->sub_mask + 1;
            const uint32_t first = (s0 + nf <= nslots) ? nf : (uint32_t)(nslots - s0);   // ring wrap: two runs
            cta_fetch_slots(S, slots, cx->sub_slots, s0, 0, first, tid);
            if (first < nf) cta_fetch_slots(S, slots, cx->sub_slots, 0, first, nf - first, tid);
        }
        if (tid == 0) S->kbase = 0;
        bar_sync(1, NT);
        PHASE(1);
        if (warp == 1) {
            // entry-size statistics of this claim (sizes the next one)
            uint32_t se = 0, sx = 0;
            for (uint32_t k = lane; k < nf; k += 32) { se += S->es[k]; sx += S->xb[k]; }
            for (int sft = 16; sft > 0; sft >>= 1) { se += __shfl_xor_sync(0xffffffffu, se, sft); sx += __shfl_xor_sync(0xffffffffu, sx, sft); }
            if (lane == 0) { st_relaxed_sys(&seq->avg_es, (se + nf - 1) / nf); st_relaxed_sys(&seq->avg_xb, (sx + nf - 1) / nf); }
        }
        const apus_cslot_t *sl = reinterpret_cast<const apus_cslot_t *>(slots);
        bool have_pub_turn = false, have_place_turn = false, aborted = false;
        uint64_t gap_bytes = 0;      // bytes of a wrap gap replicated ahead of the next publish

        while (S->kbase < nf) {
            // ---- T2: placement of the next sub-tile (warp 0) ----
            if (warp == 0) {
                int rc = CLAIM_SLOW;                      // the sub-tiles after the first: leader_place
                if (!have_place_turn) {
                    if (nf == 1) {
                        // one request in flight (closed-loop latency path): nothing to scan
                        if (lane == 0) {
                            S->cum_es[0] = S->es[0]; S->cum_xb[0] = S->xb[0];
                            S->static_cut = 1; S->first_ext_all = (S->flg[0] & 1u) ? 0u : 0xffffffffu;
                            S->host_head_k = (S->ty[0] == T_HEAD) ? 0u : 0xffffffffu;
                        }
                    } else {
                        leader_prescan(cx, S, lane);
                    }
                    __syncwarp();
                    if (lane == 0) { rc = place_claim(cx, S, sl, prof, tn); S->abort = rc == CLAIM_ABORTED; }
                    __syncwarp();
                    rc = __shfl_sync(0xffffffffu, rc, 0);
                }
                if (rc == CLAIM_SLOW) {
                    leader_place(cx, S, sl, lane);
                    if (lane == 0 && S->last) {
                        // all my slots are placed: hand the placement state to the next claim
                        place_turn_pass(seq, S->my_seq + S->n_fetch,
                                        PlaceRec{S->st_placed, S->st_end,
                                                 rec_tail_pack(S->st_tail, S->st_hwm == cx->log_len, S->st_prev_head), S->st_head});
                        if (prof) tn[7] += globaltimer_ns() - S->t_place_acq;
                    }
                }
            }
            have_place_turn = true;
            bar_sync(1, NT);
            PHASE(2);
            // stop / watchdog while waiting for a turn: this worker holds no valid placement -- it must not hand a turn
            // on, store a byte or publish (a stale placement would overwrite entries that are already acked)
            if (S->abort) { aborted = true; break; }
            if (S->blocked) {   // no space before head: poll again
                if (tid == 0) {
                    if (ld_relaxed_sys_u32(&hw->stop) || ld_relaxed_sys(&seq->abort_flag)) { st_relaxed_sys(&seq->abort_flag, 1); S->finish = 1; }
                    else if (cx->target != ~0ull && globaltimer_ns() - last_progress > WATCHDOG_NS) {
                        st_relaxed_sys(&hw->error, APUS_KERR_WATCHDOG_LEADER);
                        st_relaxed_sys(&seq->abort_flag, 1); S->finish = 1;
                    }
                }
                bar_sync(1, NT);
                if (S->finish) { aborted = true; break; }
                continue;
            }
            const uint32_t kbase = S->kbase, m = S->m, gap = S->gap, autoh = S->auto_head;
            const uint64_t a = S->a, b = S->b;
            const uint64_t a16 = a & ~15ull;
            const uint32_t nchunks = (uint32_t)(((b + 15ull) & ~15ull) - a16) >> 4;

            // ---- T3: prefill the image (zeros when the range is fresh, else the bytes the local
            //      log holds: holes of an entry keep what was there, like the reference) and
            //      stage the payload-ring range of the sub-tile; all loads in flight together
            // A composed entry overwrites all of its bytes except two HOLES -- bytes 41..47 of the header and the slack
            // behind the data image ([48 + nb, stride): 14 bytes for a request) -- which keep what the log held
            // (dare_log.h:507-529 never writes them).  For tiles of large entries only the chunks that overlap a hole are
            // brought in; small entries are mostly holes' neighbours, the whole range is read in one coalesced sweep.
            const bool holes_only = !gap && (b - a) >= (uint64_t)(m + autoh) * 512ull;
            if (holes_only) {
                for (uint32_t j = tid; j < m + autoh; j += NT) {
                    uint32_t rel, es_, nb_;
                    if (autoh && j == 0) { rel = 0; es_ = APUS_HDR_BYTES; nb_ = 8; }
                    else {
                        const uint32_t k = kbase + j - autoh;
                        rel = S->hbytes + (S->cum_es[k] - S->base_es) - S->es[k];
                        es_ = S->es[k]; nb_ = data_bytes(S->ty[k], sl[k].len);
                    }
                    const uint64_t eo = a + rel;
                    const uint64_t h0 = eo + 41, h1 = eo + 47, g0 = eo + 48 + nb_, g1 = eo + es_ - 1;   // hole byte ranges (inclusive)
                    const uint64_t cs[4] = { h0 >> 4, h1 >> 4, g0 >> 4, g1 >> 4 };
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        if (q == 3 && g1 < g0) continue;
                        if (q == 2 && g1 < g0) continue;
                        if (q > 0 && cs[q] == cs[q - 1]) continue;
                        const uint64_t lo = cs[q] << 4;
                        if (lo < a16 || lo >= a16 + 16ull * nchunks) continue;
                        reinterpret_cast<uint4 *>(img)[(lo - a16) >> 4] =
                            S->fresh ? make_uint4(0, 0, 0, 0) : ld_relaxed_sys_v4(entries + lo);
                    }
                }
            } else if (S->fresh) {
                for (uint32_t c = tid; c < nchunks; c += NT) reinterpret_cast<uint4 *>(img)[c] = make_uint4(0, 0, 0, 0);
            } else {
                cta_fetch_chunks(img, entries + a16, nchunks, tid);
            }
            if (!gap && S->ext_bytes) cta_fetch_chunks(ext, cx->sub_pay + S->ext_base, S->ext_bytes >> 4, tid);
            for (uint32_t j = tid; j < m; j += NT) {
                const uint32_t k = kbase + j;
                S->rel[k] = S->hbytes + (S->cum_es[k] - S->base_es) - S->es[k];
                S->xoff[k] = (S->cum_xb[k] - S->base_xb) - S->xb[k];
            }
            bar_sync(1, NT);
            PHASE(3);

            // ---- T4: compose entries into the image ----
            if (gap) {
                if (S->ghost && warp == 0) {
                    // header of the wrapping entry without payload, sender untouched (dare_log.h:496-503, 521)
                    uint8_t *e = img + (a - a16);
                    group_write_header(e, lane, 32, S->idx0, cx->term, sl[kbase].req_id, sl[kbase].clt_id, S->ty[kbase], 0, true);
                    if (lane == 8) { e[E_DATA] = (uint8_t)(sl[kbase].len & 0xff); e[E_DATA + 1] = (uint8_t)(sl[kbase].len >> 8); }
                }
            } else {
                if (autoh && warp == N_PRODUCER_WARPS - 1) {
                    // <HEAD, head_offset> entry (dare_log.h:29-32, dare_server.c:2043-2046)
                    uint8_t *e = img + (a - a16);
                    group_write_header(e, lane, 32, S->idx0, cx->term, 0, 0, T_HEAD, me, false);
                    if (lane >= 8 && lane < 16) e[E_DATA + lane - 8] = (uint8_t)(S->auto_head_val >> (8 * (lane - 8)));
                }
                // small entries: 8 lanes per entry (4 entries per warp step); large ones: the whole warp
                const bool small = (b - a) <= (uint64_t)(m + autoh) * 256ull;
                const int gl = small ? 8 : 32;
                const int grp = small ? (lane >> 3) : 0, sub = small ? (lane & 7) : lane;
                const uint32_t per_step = small ? 4u * N_PRODUCER_WARPS : N_PRODUCER_WARPS;
                for (uint32_t j = (small ? warp * 4u + grp : warp); j < m; j += per_step) {
                    const uint32_t k = kbase + j;
                    uint8_t *e = img + (a - a16) + S->rel[k];
                    const uint32_t ty = S->ty[k];
                    const uint32_t nb = data_bytes(ty, sl[k].len);
                    const uint32_t es_k = S->es[k];
                    if (((uint32_t)(uintptr_t)e & 15u) == 0 && (es_k & 15u) == 0) {
                        // the entry occupies whole 16 B chunks of the image: lane `sub` builds chunks sub, sub+gl, ... in
                        // registers (header fields; the data image straight from the slot / the staged payload) and
                        // writes each with ONE 16 B store; the two holes keep what the prefill put there
                        const uint64_t idx = S->idx0 + autoh + j, rq = sl[k].req_id;
                        const uint8_t *src = (S->flg[k] & 1u) ? ext + S->xoff[k] : sl[k].inl;
                        const uint32_t nch_e = es_k >> 4;
                        for (uint32_t c = (uint32_t)sub; c < nch_e; c += (uint32_t)gl) {
                            uint4 *dst = reinterpret_cast<uint4 *>(e) + c;
                            if (c == 0) *dst = make_uint4((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)cx->term, (uint32_t)(cx->term >> 32));
                            else if (c == 1) *dst = make_uint4((uint32_t)rq, (uint32_t)(rq >> 32),
                                                               ((uint32_t)sl[k].clt_id) | (ty << 16) | ((uint32_t)me << 24), 0u);
                            else if (c == 2) { const uint4 o = *dst; *dst = make_uint4(0u, 0u, o.z & 0xffffff00u, o.w); }
                            else {
                                const int nbv = (int)nb - 16 * (int)(c - 3);
                                if (nbv >= 16) *dst = *reinterpret_cast<const uint4 *>(src + 16u * (c - 3));
                                else if (nbv > 0) *dst = chunk_select(*reinterpret_cast<const uint4 *>(src + 16u * (c - 3)), *dst, nbv);
                            }
                        }
                    } else {
                        group_write_header(e, sub, gl, S->idx0 + autoh + j, cx->term, sl[k].req_id, sl[k].clt_id, ty, me, false);
                        if (nb) group_copy_smem(e + E_DATA, (S->flg[k] & 1u) ? ext + S->xoff[k] : sl[k].inl, nb, sub, gl);
                    }
                }
            }
            bar_sync(1, NT);
            PHASE(4);

            // ---- T5: push the byte range [a,b) to the local log and to every follower ----
            for (uint32_t c = tid; c < nchunks; c += NT)
                push_chunk(cx, S, a16 + 16ull * c, reinterpret_cast<const uint4 *>(img)[c], a, b);
            // entry-offset index: the c-th entry ever appended sits at index[c & idx_mask]
            if (!gap) {
                const uint64_t cum0 = S->cum_after - (m + autoh);
                for (uint32_t j = tid; j < m + autoh; j += NT) {
                    uint32_t w;
                    if (autoh && j == 0) w = (uint32_t)a | APUS_IDX_HEAD_FLAG;
                    else {
                        const uint32_t k = kbase + j - autoh;
                        w = (uint32_t)(a + S->rel[k]) | (S->ty[k] == T_HEAD ? APUS_IDX_HEAD_FLAG : 0u);
                    }
                    const uint32_t at = (uint32_t)(cum0 + 1 + j) & cx->idx_mask;
                    if (cx->mc_region) {
                        mst_u32(reinterpret_cast<uint32_t *>(cx->mc_region + APUS_INDEX_OFF) + at, w);
                    } else {
                        lindex[at] = w;
#pragma unroll 1
                        for (int f = 0; f < N; f++)
                            if (S->peer_index[f]) S->peer_index[f][at] = w;
                    }
                }
            }
            bar_sync(1, NT);
            PHASE(5);

            // ---- T6: publish the tail in claim order (data before tail, invariant I1) ----
            if (gap) {
                // nothing is published after a gap: the next sub-tile (at offset 0) carries it
                gap_bytes += b - a;
                bar_sync(1, NT);
                continue;
            }
            if (warp == 0) {
                const bool pubs = lane < N && lane != me && cx->peer[lane];
                // data before tail (invariant I1): all data stores of the tile -> bar.sync (above) -> one system
                // fence per publishing lane (cumulative over the barrier) -> the tail.  One fence costs 1.5 us;
                // fencing in every warp serializes 15 of them.
                if (pubs) __threadfence_system();
                // the publish turn: {slot number, record number} in one 16 B word.  Held for the N-1 tail stores
                // and the eight 16 B stores of the publish record -- no fence inside the turn
                if (lane == 0) {
                    if (!have_pub_turn) {
                        const uint64_t tw0 = prof ? globaltimer_ns() : 0;
                        S->abort = pub_turn_wait(seq, S->my_seq, S->pub_h);
                        if (prof) tn[2] += globaltimer_ns() - tw0;
                    }
                    if (!S->abort) S->abort = pub_room_wait(seq, S->pub_h, S->pub_tail_seen);
                }
                __syncwarp();
                const bool pub_ok = S->abort == 0;
                if (pubs && pub_ok) {
                    apus_ctrl_t *pc = reinterpret_cast<apus_ctrl_t *>(cx->peer[lane]);
                    st_relaxed_sys_2x64(&pc->pub_end, S->new_end, S->cum_after | ((cx->term & 0xffffull) << APUS_PUB_TERM_SHIFT));
                }
                if (pub_ok)
                    pub_record_write(pubring, S->pub_h, lane, S->cum_after, S->new_end, S->slot0 + kbase + m, S->t_dequeue,
                                     S->tail_after, S->hwm_after, S->idx0 + m + autoh, (b - a + gap_bytes) * (uint64_t)(N - 1));
                __syncwarp();
                if (lane == 0 && pub_ok) {
                    S->pub_h += 1;
                    if (S->last) pub_turn_pass(seq, S->my_seq + S->n_fetch, S->pub_h);
                    S->kbase = kbase + m;
                }
            }
            have_pub_turn = true;
            gap_bytes = 0;
            last_progress = globaltimer_ns();
            bar_sync(1, NT);
            if (S->abort) { aborted = true; break; }
            if (prof) {
                PHASE(6); ph[7]++;
                for (int i = 0; i < 8; i++) { ctrl->phase_ns[i] = ph[i]; ctrl->turn_ns[i] = tn[i]; }
            }
        }
        if (aborted) break;
    }
    if (prof) for (int i = 0; i < 8; i++) { ctrl->phase_ns[i] = ph[i]; ctrl->turn_ns[i] = tn[i]; }
    if (tid == 0) { __threadfence(); atomicAdd(reinterpret_cast<unsigned long long *>(&seq->workers_done), 1ull); }
}

// ---------------------------------------------------------------------------------
// FOLLOWER
// ---------------------------------------------------------------------------------
__device__ void follower_main(const apus_devctx_t *__restrict__ cx)
{
    FollowerShared *S = reinterpret_cast<FollowerShared *>(smem_raw);
    uint8_t *win = smem_raw + FS_BYTES;
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int me = cx->idx, ldr = cx->leader_idx;
    apus_ctrl_t *ctrl = reinterpret_cast<apus_ctrl_t *>(cx->region);
    apus_loghdr_t *hdr = reinterpret_cast<apus_loghdr_t *>(cx->region + APUS_HDR_OFF);
    uint8_t *entries = cx->region + cx->entries_off;
    apus_hostwords_t *hw = cx->hw;
    uint8_t *lregion = cx->peer[ldr];
    apus_ctrl_t *lctrl = reinterpret_cast<apus_ctrl_t *>(lregion);
    uint8_t *lentries = lregion + cx->entries_off;
    const uint64_t L = cx->log_len;
    const bool fenced = (cx->flags & APUS_FLAG_FENCED_ACK) != 0;
    const bool walk = (cx->flags & APUS_FLAG_WALK) != 0;
    const uint32_t *index = reinterpret_cast<const uint32_t *>(cx->region + APUS_INDEX_OFF);

    uint64_t old_end = hdr->old_end;     // walk position (dare_server.c:1795)
    uint64_t acked = ctrl->acked;        // entries walked (reply byte set) so far
    uint64_t applied = hdr->apply;       // apply offset (== commit as far as I hold the entries)
    uint64_t pend_val = ctrl->pend_head_val, pend_end = ctrl->pend_head_end;
    uint64_t last_progress = globaltimer_ns();
    uint32_t spins = 0;

    const uint64_t myterm16 = cx->term & 0xffffull;
    const bool host_apply = (cx->flags & APUS_FLAG_HOST_APPLY) != 0;
    uint64_t host_applied = hdr->apply;  // HOST_APPLY: the offset the application has replayed (what the leader may prune behind)
    uint64_t last_hb = ld_relaxed_sys(&ctrl->hb), last_hb_t = globaltimer_ns();
    bool suspected = false;
    const bool fstat = (cx->flags & APUS_FLAG_PROFILE) != 0;     // follower profiling: phase_ns[0] certificates verified,
    uint64_t cert_first_cum = 0, cert_first_t = 0, fbeat = globaltimer_ns() >> 8;               // [1] ns from first sight to verified, [2] verify retries

    for (;;) {
        if (tid < 32) {
            // warp 0 polls: lane 0 the tail publish {end, entries|term} (one 16 B acquire load), lane 1 its certificate half,
            // lane 2 the commit offset, lane 3 the heartbeat word
            const int lane = tid;
            uint64_t e = 0, cumt = 0, c = 0, cert_start = 0;
            uint32_t done = 0, is_cert = 0;
            for (;;) {
                uint64_t x0 = 0, x1 = 0;
                // lanes 4..15 read, SPECULATIVELY and in the same breath, the bytes where the next entry must land (a
                // self-certifying publish names exactly that offset): when its certificate shows up the bytes are already
                // in registers -- verification costs no second trip to memory
                const uint64_t spec_a = (old_end == L) ? 0 : old_end;
                const uint64_t spec_lo = (spec_a & ~15ull) + 16ull * (uint64_t)(lane - 4);
                uint4 spec = make_uint4(0, 0, 0, 0);
                if (lane == 0) ld_acquire_sys_2x64(&ctrl->pub_end, x0, x1);
                else if (lane == 1) ld_relaxed_sys_2x64(&ctrl->pub_csum, x0, x1);
                else if (lane == 2) x0 = ld_relaxed_sys(&hdr->commit);
                else if (lane == 3) x0 = ld_relaxed_sys(&ctrl->hb);
                else if (lane < 16 && spec_lo + 16 <= L) spec = ld_relaxed_sys_v4(entries + spec_lo);
                e = __shfl_sync(0xffffffffu, x0, 0); cumt = __shfl_sync(0xffffffffu, x1, 0);
                const uint64_t csum = __shfl_sync(0xffffffffu, x0, 1);
                cert_start = __shfl_sync(0xffffffffu, x1, 1);
                c = __shfl_sync(0xffffffffu, x0, 2);
                const uint64_t hbw = __shfl_sync(0xffffffffu, x0, 3);
                // term fence: a publish stamped with another term (a deposed leader still storing) is not looked at
                uint64_t cum = cumt & APUS_PUB_CUM_MASK;
                if ((cumt >> APUS_PUB_TERM_SHIFT) != myterm16) cum = 0;
                is_cert = (e & APUS_PUB_CERT) ? 1u : 0u;
                e &= ~APUS_PUB_CERT;
                bool new_entries = cum > acked;
                if (new_entries && is_cert && fstat && cum != cert_first_cum) { cert_first_cum = cum; cert_first_t = globaltimer_ns(); }
                if (new_entries && is_cert) {
                    // self-certifying publish of ONE entry at cert_start: the bytes may still be in flight -- read them back
                    // from my own HBM until they add up to the certificate
                    const uint64_t a = cert_start, b = (e == 0) ? L : e;
                    bool ok = cum == acked + 1 && a == ((old_end == L) ? 0 : old_end) && b > a && b - a <= 32u * 16u - 16u;
                    if (ok) {
                        const uint64_t a16 = a & ~15ull;
                        const uint32_t nch = (uint32_t)(((b + 15ull) & ~15ull) - a16) >> 4;
                        uint64_t cs = 0;
                        if (nch <= 12) {                  // the speculative read covers it (lane 4 + c holds chunk c)
                            if (lane >= 4 && lane < 4 + (int)nch) cs = cs_chunk(spec, spec_lo, a, b);
                        } else if (lane < (int)nch) cs = cs_chunk(ld_relaxed_sys_v4(entries + a16 + 16ull * lane), a16 + 16ull * lane, a, b);
#pragma unroll
                        for (int sft = 16; sft > 0; sft >>= 1) cs += __shfl_xor_sync(0xffffffffu, cs, sft);
                        ok = (cs + cs_key(cumt)) == csum;
                    }
                    if (fstat && lane == 0) { if (ok) { ctrl->phase_ns[0]++; ctrl->phase_ns[1] += globaltimer_ns() - cert_first_t; } else ctrl->phase_ns[2]++; }
                    if (!ok) { new_entries = false; cum = acked; }   // not there yet (or not verifiable: a fenced publish will follow);
                                                                     // nothing of it may be acked or walked
                }
                // commit moved, and I hold entries beyond what I applied
                const bool new_commit = (c != applied) && (old_end != L) && (applied != old_end);
                if (new_entries || new_commit) { cumt = cum; break; }
                // bounded launch: the leader says how many entries exist in total
                if (cx->target != ~0ull) {
                    uint64_t ft = 0;
                    if (lane == 0) ft = ld_acquire_sys(&ctrl->fin_target);
                    ft = __shfl_sync(0xffffffffu, ft, 0);
                    if (ft == cx->target) {
                        const uint64_t fe = ld_relaxed_sys(&ctrl->fin_entries);
                        if (acked >= fe && (old_end == L || (applied == old_end && c == old_end))) { done = 1; cumt = acked; break; }
                    }
                }
                if (hbw != last_hb) { last_hb = hbw; last_hb_t = globaltimer_ns(); if (lane == 0) st_relaxed_sys(&hw->hb_seen, hbw); }
                if ((++spins & 0xffu) == 0) {
                    uint32_t stopf = 0;
                    uint64_t ha = host_applied;
                    if (lane == 0) {
                        if (ld_relaxed_sys_u32(&hw->stop)) stopf = 1;
                        else if (cx->target != ~0ull && globaltimer_ns() - last_progress > WATCHDOG_NS) {
                            st_relaxed_sys(&hw->error, APUS_KERR_WATCHDOG_FOLLOWER);
                            stopf = 1;
                        }
                        // failure detector (hb_receive_cb, dare_server.c:866-993): the leader's beats stopped
                        if (cx->hb_timeout_ns && !suspected && globaltimer_ns() - last_hb_t > cx->hb_timeout_ns)
                            st_relaxed_sys(&hw->leader_suspect, 1 + cx->term);
                        if (host_apply) ha = ld_relaxed_sys(&hw->host_apply);
                    }
                    if (cx->hb_timeout_ns && globaltimer_ns() - last_hb_t > cx->hb_timeout_ns) suspected = true;
                    if (lane == 0) st_relaxed_sys(&lctrl->fbeat[me], ++fbeat);          // I am alive (leader's failure detector)
                    stopf = __shfl_sync(0xffffffffu, stopf, 0);
                    ha = __shfl_sync(0xffffffffu, ha, 0);
                    if (host_apply && ha != host_applied) {
                        // apply_committed_entries advances `apply` only after do_action (dare_server.c:1939-1962): what this
                        // replica reports to the leader's pruning rule is what the HOST has replayed
                        host_applied = ha;
                        if (lane == 0) { hdr->apply = ha; st_relaxed_sys(&lctrl->apply_off[me], ha); }
                    }
                    if (stopf) { done = 1; cumt = acked; break; }
                }
            }
            // early ack: the tail publish was observed with acquire semantics (or its certificate verified), so every
            // entry up to it is resident and visible here (invariant I2); the reply bytes follow behind the ack word
            // unless APUS_F_FENCED_ACK asks for them first
            if (lane == 0) {
                if (!done && !fenced && cumt > acked) st_relaxed_sys(&lctrl->ack[me], cumt);
                S->end_seen = e; S->cum_seen = cumt; S->commit_seen = c; S->done = done;
                S->cert = (cumt > acked) ? is_cert : 0u; S->cert_start = cert_start;
            }
        }
        __syncthreads();
        if (S->done) break;
        const uint64_t end_seen = S->end_seen, cum_seen = S->cum_seen, commit_seen = S->commit_seen;

        // ---- persist + ack every new entry in [old_end, end_seen) -----------------------
        if (cum_seen > acked && !walk) {
            // entry boundaries come from the offset index the leader wrote next to the bytes
            const uint64_t n = cum_seen - acked;
            if (tid == 0) S->head_j = 0;
            __syncthreads();
            for (uint64_t j = tid; j < n; j += nthr) {
                // (a self-certified publish names its one entry itself: its index word may still be in flight)
                const uint32_t w = S->cert ? (uint32_t)S->cert_start : ld_relaxed_sys_u32(&index[(uint32_t)(acked + 1 + j) & cx->idx_mask]);
                const uint64_t at = (uint64_t)(w & ~APUS_IDX_HEAD_FLAG) + E_REPLY + (uint64_t)me;
                st_relaxed_sys_u8(entries + at, 1);         // reply[me] = 1 in my copy and in the
                st_relaxed_sys_u8(lentries + at, 1);        // leader's (dare_ibv_rc.c:1833-1854)
                if (w & APUS_IDX_HEAD_FLAG) atomicMax(&S->head_j, (uint32_t)(j + 1));
            }
            __syncthreads();
            if (S->head_j) {
                // poll_config_entries (dare_server.c:2163-2170): remember the head this entry carries
                const uint32_t w = ld_relaxed_sys_u32(&index[(uint32_t)(acked + S->head_j) & cx->idx_mask]);
                const uint64_t off = (uint64_t)(w & ~APUS_IDX_HEAD_FLAG);
                pend_val = ld_relaxed_sys(entries + ((off + E_DATA) & ~7ull));
                if ((off + E_DATA) & 7ull) {
                    uint64_t hv = 0;
                    for (int q = 7; q >= 0; q--) hv = (hv << 8) | (uint64_t)(ld_relaxed_sys_u32(entries + ((off + E_DATA + q) & ~3ull)) >> (8 * ((off + E_DATA + q) & 3ull)) & 0xffu);
                    pend_val = hv;
                }
                pend_end = (off + APUS_HDR_BYTES == L) ? 0 : off + APUS_HDR_BYTES;
            }
            acked = cum_seen;
            old_end = end_seen;
            if (tid == 0) {
                if (fenced) {
                    __threadfence_system();                  // reply bytes before the ack word
                    st_relaxed_sys(&lctrl->ack[me], acked);
                }
                hdr->end = end_seen; hdr->old_end = old_end;
                ctrl->acked = acked;
                ctrl->pend_head_val = pend_val; ctrl->pend_head_end = pend_end;
            }
            last_progress = globaltimer_ns();
        } else if (cum_seen > acked) {
            uint64_t walked = 0;
            while (old_end != end_seen) {
                // window: contiguous bytes from old_end up to end_seen or the end of the ring
                if (tid == 0) {
                    uint64_t lo = (old_end == L) ? 0 : old_end;
                    if (L - lo < APUS_HDR_BYTES) lo = 0;                 // log_get_entry: header does not fit -> 0
                    uint64_t hi = (end_seen > lo) ? end_seen : L;       // wrapped: first run to the ring's end
                    if (lo == end_seen) hi = lo;
                    if (hi - (lo & ~15ull) > APUS_FOLLOWER_WIN_BYTES) hi = (lo & ~15ull) + APUS_FOLLOWER_WIN_BYTES;
                    S->win_lo = lo; S->win_hi = hi;
                }
                __syncthreads();
                const uint64_t lo = S->win_lo, hi = S->win_hi;
                if (lo == hi) { old_end = lo; break; }
                const uint64_t lo16 = lo & ~15ull;
                const uint32_t nch = (uint32_t)(((hi + 15ull) & ~15ull) - lo16) >> 4;
                {
                    uint32_t c = tid;
                    const uint8_t *src = entries + lo16;
                    for (; c + 3u * nthr < nch; c += 4u * nthr) {
                        const uint4 v0 = ld_relaxed_sys_v4(src + 16ull * c);
                        const uint4 v1 = ld_relaxed_sys_v4(src + 16ull * (c + nthr));
                        const uint4 v2 = ld_relaxed_sys_v4(src + 16ull * (c + 2u * nthr));
                        const uint4 v3 = ld_relaxed_sys_v4(src + 16ull * (c + 3u * nthr));
                        reinterpret_cast<uint4 *>(win)[c] = v0;
                        reinterpret_cast<uint4 *>(win)[c + nthr] = v1;
                        reinterpret_cast<uint4 *>(win)[c + 2u * nthr] = v2;
                        reinterpret_cast<uint4 *>(win)[c + 3u * nthr] = v3;
                    }
                    for (; c < nch; c += nthr) reinterpret_cast<uint4 *>(win)[c] = ld_relaxed_sys_v4(src + 16ull * c);
                }
                __syncthreads();
                // serial walk over headers in shared memory (log_get_entry / log_fit_entry / log_entry_len)
                if (tid == 0) {
                    uint64_t off = lo;
                    uint32_t n = 0;
                    uint64_t next = off;
                    bool wrapped = false;
                    uint64_t hv = 0, he = L;
                    while (off < hi) {
                        if (L - off < APUS_HDR_BYTES) { next = 0; wrapped = true; break; }   // jump to 0
                        if (hi - off < APUS_HDR_BYTES) { next = off; break; }                // header not in window yet
                        const uint8_t *e = win + (off - lo16);
                        const uint32_t ty = e[E_TYPE];
                        const uint32_t ln = (uint32_t)e[E_DATA] | ((uint32_t)e[E_DATA + 1] << 8);
                        const uint32_t es = entry_stride(ty, ln);
                        if (L - off < es) { next = 0; wrapped = true; break; }              // ghost: entry continues at 0
                        if (off + es > hi) { next = off; break; }                            // entry crosses the window
                        if (ty == T_HEAD) {                                                  // poll_config_entries (dare_server.c:2163-2170)
                            hv = 0;
                            for (int q = 7; q >= 0; q--) hv = (hv << 8) | e[E_DATA + q];
                            he = (off + es == L) ? 0 : off + es;
                        }
                        S->off[n++] = (uint32_t)(off - lo);
                        off += es;
                        next = off;
                    }
                    if (!wrapped && next == L) next = 0;      // rule E1 on walker offsets
                    S->n = n; S->next = next;
                    S->head_val = hv; S->head_end = he;
                }
                __syncthreads();
                const uint32_t n = S->n;
                // reply[me] = 1 in my copy and in the leader's copy (dare_ibv_rc.c:1833-1854)
                for (uint32_t k = tid; k < n; k += nthr) {
                    const uint64_t at = lo + S->off[k] + E_REPLY + (uint64_t)me;
                    st_relaxed_sys_u8(entries + at, 1);
                    st_relaxed_sys_u8(lentries + at, 1);
                }
                __syncthreads();
                const uint64_t next = S->next;
                if (n == 0 && next == old_end) {
                    // no progress possible inside this window: protocol error
                    if (tid == 0) st_relaxed_sys(&hw->error, APUS_KERR_BAD_ENTRY);
                    old_end = end_seen;
                    break;
                }
                if (S->head_end != L) { pend_val = S->head_val; pend_end = S->head_end; }
                walked += n;
                old_end = next;
            }
            if (acked + walked != cum_seen && tid == 0) st_relaxed_sys(&hw->error, APUS_KERR_COUNT_MISMATCH);
            acked = cum_seen;
            if (tid == 0) {
                if (fenced) {
                    __threadfence_system();                  // reply bytes before the ack word
                    st_relaxed_sys(&lctrl->ack[me], acked);  // the word the leader's quorum ranking polls
                }
                hdr->end = end_seen; hdr->old_end = old_end;
                ctrl->acked = acked;
                ctrl->pend_head_val = pend_val; ctrl->pend_head_end = pend_end;
            }
            last_progress = globaltimer_ns();
        }

        // ---- follow the commit offset (invariant I4: never beyond what I hold) ----------
        if (old_end != L && applied != old_end && commit_seen != applied) {
            const uint64_t from = applied;
            const uint64_t held = ring_dist(from, old_end, L);          // bytes I hold beyond `applied`
            uint64_t want = ring_dist(from, commit_seen, L);
            uint64_t to = commit_seen;
            if (want > held) { want = held; to = old_end; }             // the leader clamps the same way (dare_ibv_rc.c:1783-1787)
            if (want) {
                if (pend_end != L) {
                    const uint64_t dh = ring_dist(from, pend_end, L);
                    if (dh > 0 && dh <= want) {
                        // the HEAD entry is committed: adopt the head it carries (dare_server.c:2166-2169, 2182-2186)
                        if (tid == 0) { hdr->head = pend_val; ctrl->pend_head_end = L; }
                        pend_end = L;
                    }
                }
                applied = to;
                if (tid == 0) {
                    if (!host_apply) {
                        hdr->apply = applied;           // library use: nothing replays the log on the host
                        st_relaxed_sys(&lctrl->apply_off[me], applied);
                    }
                    // the host may replay [its apply, applied): everything before `applied` is committed and held here
                    st_relaxed_sys_2x64(&hw->commit_off, applied, acked);
                }
                last_progress = globaltimer_ns();
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
extern "C" __global__ void __launch_bounds__(APUS_KERNEL_THREADS, 1)
apus_replica_kernel(const apus_role_t *__restrict__ roles)
{
    const apus_role_t r = roles[blockIdx.x];
    if (r.kind == APUS_ROLE_LEADER) leader_main(r.ctx, r.worker);
    else if (r.kind == APUS_ROLE_FOLLOWER) follower_main(r.ctx);
}

extern "C" size_t apus_kernel_smem_bytes(void)
{
    size_t a = L_TOTAL, b = F_TOTAL;
    return a > b ? a : b;
}

extern "C" cudaError_t apus_launch_roles(const apus_role_t *d_roles, int n_roles, cudaStream_t stream)
{
    static bool attr_set[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    const size_t smem = apus_kernel_smem_bytes();
    if (dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(apus_replica_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    apus_replica_kernel<<<n_roles, APUS_KERNEL_THREADS, smem, stream>>>(d_roles);
    return cudaGetLastError();
}
