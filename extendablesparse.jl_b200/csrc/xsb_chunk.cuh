// xsb_chunk.cuh -- "grouped chunks": the kernels that STAGE records (pack / emit kernels, xsb_insert.cu)
// bring every chunk of up to 32*NB consecutive insertions into column order before it is written, so
// that the records of one (chunk, column) pair -- a RUN -- sit next to each other in the staging buffer.
// The grouping is stable: inside a run the records keep their insertion order, and runs of the same
// column in different chunks are met in chunk = stream order, so every (column, row) still sees its
// insertions in stream order (what the deterministic left fold needs; reference: the per-column
// linked lists of SparseMatrixLNK ARE this grouping, src/matrix/sparsematrixlnk.jl:151-171,210-253).
//
// What a flush gains: it no longer moves the records at all.  The per-column fold (xsb_runs.cu) reads
// the runs where the producer left them, through the run index published here:
//     per chunk : (first pair, pairs) and the position of its first record
//     per pair  : the column (owner bits on top on slab handles) and (offset in the chunk, records)
//
// A warp owns a chunk.  Pass 1 finds the chunk's distinct columns with a warp-private open-addressing
// table in shared memory (one table request per distinct column of a 32-record batch: match.any
// first) and notes, per record, its column's table slot and its rank among the chunk's records of
// that column; a scan over the columns in order of first appearance gives every column its offset;
// pass 2 stores record k at offset[slot_k] + rank_k.
#pragma once
#include "xsb_internal.h"

namespace xsb {

constexpr u32 CH_EMPTY = 0xffffffffu;
constexpr int CH_RECORDS = 512; // records per chunk of the packing kernels and of the flush-time kernel
constexpr u32 CH_RUN_MAX = 2047; // records of one run: the count field of the flush's run descriptor (xsb_runs.cu)

template <int HB> struct ChunkSpaceT
{
    static constexpr int H = 1 << HB;
    static constexpr u32 DMAX = (u32)(H / 8 * 5); // distinct columns a chunk may hold
    u32 key[H];
    unsigned short cnt[H];   // records of the column
    unsigned short start[H]; // offset of its run inside the chunk
    unsigned short cand[H];  // slots in order of first appearance
};

__device__ __forceinline__ u32 ch_hash(u32 g, int hb) { return (g * 0x9E3779B1u) >> (32 - hb); }

template <int HB> __device__ __forceinline__ void chunk_space_init(ChunkSpaceT<HB> &ws, int lane)
{
    constexpr int H = ChunkSpaceT<HB>::H;
    uint4 *kq = reinterpret_cast<uint4 *>(ws.key);
#pragma unroll
    for (int i = 0; i < H / 128; ++i)
        kq[i * 32 + lane] = make_uint4(CH_EMPTY, CH_EMPTY, CH_EMPTY, CH_EMPTY);
    uint4 *cq = reinterpret_cast<uint4 *>(ws.cnt);
#pragma unroll
    for (int i = 0; i < H / 256; ++i)
        cq[i * 32 + lane] = make_uint4(0, 0, 0, 0);
    if (H < 256 && lane < H / 8)
        cq[lane] = make_uint4(0, 0, 0, 0);
    __syncwarp();
}

// One batch of 32 consecutive records: g = grouping key (column, owner bits on top) of this lane's
// record, valid = the lane holds a record (FULL: every lane does).  Returns (slot << 16 | rank of the record
// among the chunk's records of its column so far).  d = distinct columns of the chunk so far.
template <int HB, bool FULL = false>
__device__ __forceinline__ u32 chunk_count_batch(ChunkSpaceT<HB> &ws, u32 g, bool valid, u32 lt, u32 &d)
{
    constexpr u32 full = 0xffffffffu;
    constexpr int H = ChunkSpaceT<HB>::H;
    u32 peers;
    if (FULL)
        peers = __match_any_sync(full, g);
    else
    {
        const u32 vm = __ballot_sync(full, valid);
        peers = 0;
        if (valid)
            peers = __match_any_sync(vm, g);
    }
    // the FIRST lane that holds a column speaks for it: the table sees one request per distinct column
    const bool leader = (FULL || valid) && (peers & lt) == 0u;
    u32 slot = ch_hash(g, HB), old = 0;
    bool fresh = false;
    if (leader)
    {
        for (;;)
        { // a plain look first: after a few batches nearly every column of the chunk is in the table
            u32 k = ws.key[slot];
            if (k == g)
                break;
            if (k == CH_EMPTY)
            {
                k = atomicCAS(&ws.key[slot], CH_EMPTY, g);
                if (k == CH_EMPTY)
                {
                    fresh = true;
                    break;
                }
                if (k == g)
                    break;
            }
            slot = (slot + 1) & (H - 1);
        }
        old = ws.cnt[slot]; // leaders of a batch hold distinct slots of a warp-private table
        ws.cnt[slot] = (unsigned short)(old + (u32)__popc(peers));
    }
    const u32 rb = __ballot_sync(full, fresh);
    if (rb)
    { // warp-uniform: most batches bring no new column
        if (fresh)
            ws.cand[d + __popc(rb & lt)] = (unsigned short)slot;
        d += __popc(rb);
    }
    const int ldr = (FULL || peers) ? __ffs(peers) - 1 : 0;
    const u32 packed = __shfl_sync(full, (slot << 16) | old, ldr);
    __syncwarp();
    return packed + (u32)__popc(peers & lt);
}

// One KIND of visit of a producer that knows the structure of its stream (the stencil emitters): every valid lane
// holds a DIFFERENT grouping key and brings `weight` records for it -- no match.any, no leader election.  Returns
// (slot << 16 | records of the column before this visit); the column's count grows by `weight`.
template <int HB>
__device__ __forceinline__ u32 chunk_visit_batch(ChunkSpaceT<HB> &ws, u32 g, bool valid, u32 weight, u32 lt, u32 &d)
{
    constexpr u32 full = 0xffffffffu;
    constexpr int H = ChunkSpaceT<HB>::H;
    u32 slot = ch_hash(g, HB), old = 0;
    bool fresh = false;
    if (valid)
    {
        for (;;)
        {
            u32 k = ws.key[slot];
            if (k == g)
                break;
            if (k == CH_EMPTY)
            {
                k = atomicCAS(&ws.key[slot], CH_EMPTY, g);
                if (k == CH_EMPTY)
                {
                    fresh = true;
                    break;
                }
            }
            slot = (slot + 1) & (H - 1);
        }
        old = ws.cnt[slot]; // distinct keys: distinct slots
        ws.cnt[slot] = (unsigned short)(old + weight);
    }
    const u32 rb = __ballot_sync(full, fresh);
    if (rb)
    {
        if (fresh)
            ws.cand[d + __popc(rb & lt)] = (unsigned short)slot;
        d += __popc(rb);
    }
    __syncwarp();
    return (slot << 16) | old;
}

// offsets of the runs: exclusive sum of the columns' record counts in order of first appearance.
// mul: every counted request stands for mul records (a producer that knows that its records come in groups of
// mul per column counts the groups: emit_p1fem_grouped_kernel, 5; insert_elements_kernel, k at run time)
template <int HB> __device__ __forceinline__ void chunk_scan(ChunkSpaceT<HB> &ws, u32 d, int lane, u32 mul = 1)
{
    constexpr u32 full = 0xffffffffu;
    const u32 per = (d + 31u) >> 5;
    const u32 j0 = min((u32)lane * per, d), j1 = min(j0 + per, d);
    u32 sum = 0;
    for (u32 j = j0; j < j1; ++j)
        sum += mul * ws.cnt[ws.cand[j]];
    u32 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(full, incl, o);
        if (lane >= o)
            incl += t;
    }
    u32 run = incl - sum;
    for (u32 j = j0; j < j1; ++j)
    {
        const u32 s = ws.cand[j];
        ws.start[s] = (unsigned short)run;
        run += mul * ws.cnt[s];
    }
    __syncwarp();
}

__device__ __forceinline__ u32 chunk_dest(const unsigned short *start, u32 packed)
{
    return (u32)start[packed >> 16] + (packed & 0xffffu);
}

// Appends the chunk's pairs to the run index.  Room is taken by atomic ticket: chunks land in
// completion order, the flush orders the runs of a column by their position in the staging buffer.
// grouped == false: the chunk gave up (too many distinct columns: no column locality) and was stored
// in stream order; the flag sends the flush to the radix-sort path.
template <int HB>
__device__ __forceinline__ void chunk_publish(ChunkSpaceT<HB> &ws, const RunTarget &rt, u32 chunk, u32 abs_start, u32 d,
                                              bool grouped, int lane, u32 mul = 1)
{
    constexpr u32 full = 0xffffffffu;
    u32 base = 0;
    if (lane == 0)
        base = grouped ? atomicAdd(rt.counters, d) : 0u;
    base = __shfl_sync(full, base, 0);
    const bool room = grouped && (u64)base + d <= (u64)rt.cap;
    if (lane == 0)
    {
        rt.chunkinfo[chunk] = make_uint2(base, room ? d : 0u);
        rt.chunkstart[chunk] = abs_start;
        if (!room)
            atomicOr(rt.counters + 1, 1u);
    }
    if (!room)
        return;
    for (u32 j = lane; j < d; j += 32)
    {
        const u32 s = ws.cand[j];
        rt.pcol[base + j] = ws.key[s];
        rt.pinfo[base + j] = ((u32)ws.start[s] << 16) | (mul * (u32)ws.cnt[s]);
    }
}

// A chunk without column locality (more distinct columns than the table takes) stays in stream order and
// publishes every record as a run of its own: a small unordered batch on top of a large matrix still takes the
// grouped-chunk flush; a large one fills the pair list, and the flag sends the flush to the radix-sort path.
// g[b] / valid: grouping key of this lane's record of batch b.
template <int NB>
__device__ __forceinline__ void chunk_publish_singletons(const RunTarget &rt, u32 chunk, u32 abs_start, u32 len,
                                                         const u32 (&g)[NB], int lane)
{
    constexpr u32 full = 0xffffffffu;
    u32 base = 0;
    if (lane == 0)
        base = atomicAdd(rt.counters, len);
    base = __shfl_sync(full, base, 0);
    const bool room = (u64)base + len <= (u64)rt.cap;
    if (lane == 0)
    {
        rt.chunkinfo[chunk] = make_uint2(base, room ? len : 0u);
        rt.chunkstart[chunk] = abs_start;
        if (!room)
            atomicOr(rt.counters + 1, 1u);
    }
    if (!room)
        return;
#pragma unroll
    for (int b = 0; b < NB; ++b)
    {
        const u32 p = b * 32 + lane;
        if (p < len)
        {
            rt.pcol[base + p] = g[b];
            rt.pinfo[base + p] = (p << 16) | 1u;
        }
    }
}

// chunk_publish for a chunk in which a column holds more than CH_RUN_MAX records (more than a run descriptor
// counts; insert_elements_kernel with elements that repeat a dof): the column's records, neighbours in the grouped
// chunk, are published as several runs of at most CH_RUN_MAX records.  The flush orders a column's runs by position,
// so the pieces keep the records' order.
template <int HB>
__device__ __forceinline__ void chunk_publish_split(ChunkSpaceT<HB> &ws, const RunTarget &rt, u32 chunk, u32 abs_start, u32 d,
                                                    int lane, u32 mul)
{
    constexpr u32 full = 0xffffffffu;
    const u32 per = (d + 31u) >> 5;
    const u32 j0 = min((u32)lane * per, d), j1 = min(j0 + per, d);
    u32 sum = 0; // runs of this lane's columns
    for (u32 j = j0; j < j1; ++j)
        sum += (mul * ws.cnt[ws.cand[j]] + CH_RUN_MAX - 1u) / CH_RUN_MAX;
    u32 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(full, incl, o);
        if (lane >= o)
            incl += t;
    }
    const u32 total = __shfl_sync(full, incl, 31);
    u32 base = 0;
    if (lane == 0)
        base = atomicAdd(rt.counters, total);
    base = __shfl_sync(full, base, 0);
    const bool room = (u64)base + total <= (u64)rt.cap;
    if (lane == 0)
    {
        rt.chunkinfo[chunk] = make_uint2(base, room ? total : 0u);
        rt.chunkstart[chunk] = abs_start;
        if (!room)
            atomicOr(rt.counters + 1, 1u);
    }
    if (!room)
        return;
    u32 q = base + incl - sum;
    for (u32 j = j0; j < j1; ++j)
    {
        const u32 s = ws.cand[j];
        u32 off = ws.start[s], len = mul * (u32)ws.cnt[s];
        while (len > 0u)
        {
            const u32 piece = min(len, CH_RUN_MAX);
            rt.pcol[q] = ws.key[s];
            rt.pinfo[q] = (off << 16) | piece;
            ++q;
            off += piece;
            len -= piece;
        }
    }
}

} // namespace xsb
