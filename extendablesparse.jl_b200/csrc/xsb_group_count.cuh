// xsb_group_count.cuh -- the counting half of the two-pass grouping (xsb_group.cu): per-chunk
// distinct columns and their record counts, as device functions of group_count_kernel.
#pragma once
#include "xsb_internal.h"

namespace xsb {

#ifndef XSB_GP_W
#define XSB_GP_W 512
#endif
constexpr int GP_W = XSB_GP_W;      // records per chunk (one warp)
constexpr int GP_NB = GP_W / 32;    // batches per chunk
constexpr int GP_HBITS = 9;
constexpr int GP_H = 1 << GP_HBITS; // hash slots per warp
constexpr int GP_DMAX = GP_H - 96;  // distinct columns a chunk may hold; more means "no locality" anyway
constexpr int GP_WARPS = 8;
constexpr u32 GP_EMPTY = 0xffffffffu;

__device__ __forceinline__ u32 gp_hash(u32 col) { return (col * 0x9E3779B1u) >> (32 - GP_HBITS); }

// where a chunk's (column, count) pairs go: fields of the grouping workspace (xsb_group.cu)
struct CountTarget
{
    u32 *pair_total;  // ticket: pairs appended so far
    u32 *flags;       // != 0: a chunk had too many distinct columns / the pair list is full
    Rec *pairs;       // (column, ticket position << 16 | count)
    u32 *chunkcols;   // column of pair p
    uint2 *chunkinfo; // per chunk: (first pair, pairs)
    u32 cap;          // room of the pair list
    int colshift;
    u32 colmask;
    unsigned short *chunkcnt; // records of pair p (1..chunk size)
};

struct CountSpace
{
    u32 key[GP_H];
    u32 cnt[GP_H];
    unsigned short cand[GP_H];
};

// ------------------------------------------------------------------------
// pass 1: distinct columns of every chunk and their record counts
// ------------------------------------------------------------------------
// One batch of 32 consecutive records.  FULL: every lane holds a record that takes part (whole
// chunk, no records of other ranks to skip).
template <bool FULL>
__device__ __forceinline__ void count_batch(CountSpace &ws, u64 key, bool valid, int colshift, u32 colmask, u32 lt,
                                            u32 &d)
{
    constexpr u32 full = 0xffffffffu;
    const u32 col = (u32)(key >> colshift) & colmask;
    u32 peers;
    if (FULL)
        peers = __match_any_sync(full, col);
    else
    {
        const u32 vm = __ballot_sync(full, valid);
        peers = 0;
        if (valid)
            peers = __match_any_sync(vm, col);
    }
    // the FIRST lane that holds a column speaks for it: the table sees one request per distinct column
    const bool leader = (FULL || valid) && (peers & lt) == 0u;
    u32 slot = gp_hash(col);
    bool fresh = false;
    if (leader)
    {
        for (;;)
        { // a plain look first: after a few batches nearly every column of the chunk is in the table
            u32 k = ws.key[slot];
            if (k == col)
                break;
            if (k == GP_EMPTY)
            {
                k = atomicCAS(&ws.key[slot], GP_EMPTY, col);
                if (k == GP_EMPTY)
                {
                    fresh = true;
                    break;
                }
                if (k == col)
                    break;
            }
            slot = (slot + 1) & (GP_H - 1);
        }
    }
    const u32 rb = __ballot_sync(full, fresh);
    if (fresh)
        ws.cand[d + __popc(rb & lt)] = (unsigned short)slot;
    d += __popc(rb);
    if (leader)
        ws.cnt[slot] += (u32)__popc(peers); // leaders hold distinct slots of a warp-private table
    __syncwarp();
}


__device__ __forceinline__ void count_space_init(CountSpace &ws, int lane)
{
    uint4 *kq = reinterpret_cast<uint4 *>(ws.key);
#pragma unroll
    for (int i = 0; i < GP_H / 128; ++i)
        kq[i * 32 + lane] = make_uint4(GP_EMPTY, GP_EMPTY, GP_EMPTY, GP_EMPTY);
    uint4 *cq = reinterpret_cast<uint4 *>(ws.cnt);
#pragma unroll
    for (int i = 0; i < GP_H / 128; ++i)
        cq[i * 32 + lane] = make_uint4(0, 0, 0, 0);
    __syncwarp();
}

// Appends the chunk's pairs.  Room is taken by atomic ticket: chunks land in completion order and
// the pair list is brought into chunk = stream order by pair_order_kernel before the sort.
__device__ __forceinline__ void count_publish(CountSpace &ws, const CountTarget &ct, u32 chunk, u32 d, bool crowded,
                                              int lane)
{
    constexpr u32 full = 0xffffffffu;
    __syncwarp();
    u32 base = 0;
    if (lane == 0)
        base = atomicAdd(ct.pair_total, d);
    base = __shfl_sync(full, base, 0);
    const bool room = !crowded && (u64)base + d <= (u64)ct.cap;
    if (lane == 0)
    {
        ct.chunkinfo[chunk] = make_uint2(base, room ? d : 0u);
        if (!room) // more pairs than the caller made room for: the stream has no column locality
            atomicOr(ct.flags, 1u);
    }
    if (!room)
        return;
    for (u32 j = lane; j < d; j += 32)
    {
        const u32 slot = ws.cand[j];
        const u32 col = ws.key[slot];
        const u32 cnt = ws.cnt[slot];
        ct.chunkcols[base + j] = col;
        ct.chunkcnt[base + j] = (unsigned short)cnt;
        Rec pr;
        pr.key = (u64)col;
        const u64 payload = ((u64)(base + j) << 16) | (u64)cnt;
        pr.val = __longlong_as_double((long long)payload);
        st_rec(ct.pairs + base + j, pr);
    }
}

} // namespace xsb
