// xsb_colfold.cu -- flush! after a stable COLUMN-ONLY radix sort, without ordering the rows of
// the records at all:
//
//   colscan kernels  : per-column record counts (taken by the sort's histogram kernel) -> compact
//                      list of the non-empty columns (nzcol) and where each one starts in the
//                      sorted records (nzstart); spans of CF_SPAN records -> first column (tilek).
//   colfold_kernel   : one warp per span, no block-wide staging.  The warp streams its columns'
//                      records straight from global memory, 32 at a time and in stream order.
//                      Every record finds the accumulator of its (column,row) in a small
//                      shared-memory hash table; the records of one batch that share an
//                      accumulator are folded by their first lane in lane (= stream) order, so every
//                      entry is the exact left fold of its insertions.  Only the DISTINCT entries
//                      are then sorted by row (in registers) and parked at the column's own offset.
//   colptr kernels   : entries per column -> colptr (+ nnz).
//   compact kernel   : parked entries -> rowval / nzval in the caller's index type and base.
//
// This is the reference's per-column structure (gather column, sort by row, accumulate equal rows:
// src/matrix/sparsematrixlnk.jl:328-377) with accumulate-on-insert (:210-253) done through the
// hash table instead of a list walk.  A group of columns whose distinct entries do not fit the
// table raises an overflow flag; the caller then finishes with the general (col,row) sort.
#include "xsb_fold.cuh"
#include "xsb_internal.h"

namespace xsb {

constexpr int CF_SPAN = 512;   // records per warp span
constexpr int CF_HBITS = 8;
constexpr int CF_H = 1 << CF_HBITS; // hash slots per warp
constexpr int CF_PIECE = 224;  // records folded per round: never more distinct entries than the table takes
constexpr u32 CF_EMPTY = 0xffffffffu;
constexpr int CF_MAXROWBITS = 26; // 5 bits of local column + row must stay below CF_EMPTY

// ------------------------------------------------------------------------
// per-column record counts -> compact list of non-empty columns
// ------------------------------------------------------------------------
constexpr int CS_THREADS = 256;
constexpr int CS_IPT = 8;
constexpr int CS_TILE = CS_THREADS * CS_IPT;

// block-wide sum of a u64 (all threads must call); result valid in thread 0
__device__ __forceinline__ u64 block_sum_u64(u64 s, u64 *s_w)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0)
        s_w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < CS_THREADS / 32; ++w)
            s += s_w[w];
    return s;
}

// tile sums of (records << 24 | non-empty columns): a tile has at most 2048 columns
__global__ void __launch_bounds__(CS_THREADS)
colscan_tilesum_kernel(const u32 *__restrict__ cnt, i64 n, u64 *__restrict__ trec, u32 *__restrict__ tnz)
{
    __shared__ u64 s_w[CS_THREADS / 32];
    const i64 b0 = (i64)blockIdx.x * CS_TILE;
    u64 rec = 0, nz = 0;
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        const i64 j = b0 + i * CS_THREADS + threadIdx.x;
        if (j < n)
        {
            const u32 c = cnt[j];
            rec += c;
            nz += c != 0u;
        }
    }
    const u64 r = block_sum_u64(rec, s_w);
    __syncthreads();
    const u64 z = block_sum_u64(nz, s_w);
    if (threadIdx.x == 0)
    {
        trec[blockIdx.x] = r;
        tnz[blockIdx.x] = (u32)z;
    }
}

// single block: exclusive scan of both tile sums in place; totals[0] = records, totals[1] = K
__global__ void __launch_bounds__(1024)
colscan_scan_kernel(u64 *__restrict__ trec, u32 *__restrict__ tnz, i64 nt, u64 *__restrict__ totals,
                    u32 *__restrict__ nzstart)
{
    __shared__ u64 s_wr[32], s_wz[32];
    __shared__ u64 s_cr, s_cz;
    if (threadIdx.x == 0)
    {
        s_cr = 0;
        s_cz = 0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (i64 b0 = 0; b0 < nt; b0 += 1024)
    {
        const i64 j = b0 + threadIdx.x;
        const u64 xr = j < nt ? trec[j] : 0ull, xz = j < nt ? (u64)tnz[j] : 0ull;
        u64 vr = xr, vz = xz;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 tr = __shfl_up_sync(0xffffffffu, vr, o);
            const u64 tz = __shfl_up_sync(0xffffffffu, vz, o);
            if (lane >= o)
            {
                vr += tr;
                vz += tz;
            }
        }
        if (lane == 31)
        {
            s_wr[warp] = vr;
            s_wz[warp] = vz;
        }
        __syncthreads();
        u64 pr = s_cr, pz = s_cz;
        for (int w = 0; w < warp; ++w)
        {
            pr += s_wr[w];
            pz += s_wz[w];
        }
        if (j < nt)
        {
            trec[j] = pr + vr - xr;
            tnz[j] = (u32)(pz + vz - xz);
        }
        __syncthreads();
        if (threadIdx.x == 1023)
        {
            s_cr = pr + vr;
            s_cz = pz + vz;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0)
    {
        totals[0] = s_cr;
        totals[1] = s_cz;
        nzstart[s_cz] = (u32)s_cr; // sentinel: one past the last record
    }
}

__global__ void __launch_bounds__(CS_THREADS)
colscan_emit_kernel(const u32 *__restrict__ cnt, const u64 *__restrict__ trec, const u32 *__restrict__ tnz,
                    i64 n, u32 *__restrict__ nzcol, u32 *__restrict__ nzstart)
{
    __shared__ u64 s_w[CS_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 b0 = (i64)blockIdx.x * CS_TILE + (i64)threadIdx.x * CS_IPT; // blocked: thread owns CS_IPT columns
    u32 c[CS_IPT];
    u64 sum = 0; // records << 24 | non-empty
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        const i64 j = b0 + i;
        c[i] = j < n ? cnt[j] : 0u;
        sum += ((u64)c[i] << 24) | (u64)(c[i] != 0u);
    }
    u64 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_w[warp] = incl;
    __syncthreads();
    u64 run = incl - sum;
    for (int w = 0; w < warp; ++w)
        run += s_w[w];
    u64 rec = trec[blockIdx.x] + (run >> 24);
    u32 k = tnz[blockIdx.x] + (u32)(run & 0xffffffu);
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        if (c[i])
        {
            nzcol[k] = (u32)(b0 + i);
            nzstart[k] = (u32)rec;
            ++k;
            rec += c[i];
        }
    }
}

// tilek[t] = first non-empty column (compact index) that starts at or after record t*CF_SPAN
__global__ void __launch_bounds__(256)
tilemap_kernel(const u32 *__restrict__ nzstart, const u64 *__restrict__ totals, u32 ntiles, u32 *__restrict__ tilek)
{
    const u64 K = totals[1];
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k > K)
        return;
    const u32 t0 = k ? nzstart[k - 1] / CF_SPAN + 1u : 0u;
    const u32 t1 = (k == K) ? ntiles : nzstart[k] / CF_SPAN;
    for (u32 t = t0; t <= t1; ++t)
        tilek[t] = (u32)k;
}

// ------------------------------------------------------------------------
// per-warp working space
// ------------------------------------------------------------------------
// A warp works on a GROUP: as many whole columns as fit in `chunk` records (at least one; a
// column longer than that is taken alone, in pieces of CF_PIECE records).  Per piece:
//   A. every record finds the slot of its (local column,row) in the hash table (insert on first
//      sight) and its rank among the piece's records of that slot, in stream order;
//   B. slot counts -> offsets (warp scan), the values are laid out slot by slot in stream order;
//   C. one lane per slot folds its list sequentially, seeded with the slot's state.
// After the last piece the distinct entries are sorted by (local column,row) and parked.
template <bool SIMPLE> struct WarpSpace;

enum : u32
{
    SF_EXISTS = 1,   // some record would have created the entry
    SF_OLDFIRST = 2, // the run starts with the resident CSC value
    SF_SEEDED = 4    // the accumulator already holds a partial fold
};

template <> struct WarpSpace<true>
{
    double acc[CF_H];
    double val[CF_PIECE];
    u32 key[CF_H];
    u32 ccnt[32];
    unsigned short cnt[CF_H];
    unsigned short cand[CF_H];
    unsigned char flag[CF_H];
    __device__ __forceinline__ void init_slot(u32 s)
    {
        acc[s] = 0.0;
        flag[s] = 0;
    }
    // leader of a batch group: first = the group's slot was created by this batch
    __device__ __forceinline__ void note(u32 s, bool first, u32 fl, bool creates)
    {
        u32 f = flag[s];
        if (creates)
            f |= SF_EXISTS;
        if (first && fl == FL_OLD)
            f |= SF_OLDFIRST;
        flag[s] = (unsigned char)f;
    }
    __device__ __forceinline__ void put(u32 pos, double v, u32) { val[pos] = v; }
    __device__ __forceinline__ void fold(u32 s, u32 o0, u32 o1, int)
    {
        double a = acc[s];
        u32 f = flag[s];
        if (o0 < o1)
        {
            if ((f & (SF_SEEDED | SF_OLDFIRST)) == SF_OLDFIRST)
                a = val[o0++]; // the old CSC value replaces the +0.0 seed: extendable.jl:165-166
            f |= SF_SEEDED;
            while (o0 + 4 <= o1)
            {
                const double v0 = val[o0], v1 = val[o0 + 1], v2 = val[o0 + 2], v3 = val[o0 + 3];
                a = (((a + v0) + v1) + v2) + v3;
                o0 += 4;
            }
            while (o0 < o1)
                a = a + val[o0++];
            acc[s] = a;
            flag[s] = (unsigned char)f;
        }
    }
    __device__ __forceinline__ bool settle(u32 s) { return (flag[s] & SF_EXISTS) != 0; }
    __device__ __forceinline__ double value(u32 s) const { return acc[s]; }
};

template <> struct WarpSpace<false>
{
    ColFold st[CF_H];
    double val[CF_PIECE];
    u32 meta[CF_PIECE];
    u32 key[CF_H];
    u32 ccnt[32];
    unsigned short cnt[CF_H];
    unsigned short cand[CF_H];
    __device__ __forceinline__ void init_slot(u32 s) { st[s] = ColFold(); }
    __device__ __forceinline__ void note(u32, bool, u32, bool) {}
    __device__ __forceinline__ void put(u32 pos, double v, u32 m)
    {
        val[pos] = v;
        meta[pos] = m;
    }
    __device__ __forceinline__ void fold(u32 s, u32 o0, u32 o1, int combine)
    {
        if (o0 < o1)
        {
            ColFold f = st[s];
            for (; o0 < o1; ++o0)
            {
                const u32 m = meta[o0];
                f.apply(m & 3u, m >> 2, val[o0], combine);
            }
            st[s] = f;
        }
    }
    __device__ __forceinline__ bool settle(u32 s)
    {
        ColFold f = st[s];
        f.finish();
        st[s].acc = f.acc;
        return f.exists;
    }
    __device__ __forceinline__ double value(u32 s) const { return st[s].acc; }
};

__device__ __forceinline__ u32 cf_hash(u32 hk) { return (hk * 0x9E3779B1u) >> (32 - CF_HBITS); }

// Sort the existing entries of a group by (local column, row) and park them at their column's
// offset; the per-column entry counts go to colcount.  dcount = slots in use (ws.cand).
template <int E, typename WS>
__device__ __forceinline__ void emit_group(WS &ws, u32 dcount, int rowbits, u32 a, u32 nc, u32 cstart, u32 ccol,
                                           Rec *__restrict__ tmp, u32 *__restrict__ colcount, int lane)
{
    constexpr u32 full = 0xffffffffu;
    const u32 rowmask = (1u << rowbits) - 1u;
    u32 k[E];
    u32 d = 0;
#pragma unroll
    for (int e = 0; e < E; ++e)
    {
        const u32 i = e * 32 + lane;
        k[e] = CF_EMPTY;
        if (i < dcount)
        {
            const u32 s = ws.cand[i];
            if (ws.settle(s))
                k[e] = ws.key[s];
        }
        d += __popc(__ballot_sync(full, k[e] != CF_EMPTY));
    }
    warp_bitonic<E>(k, lane);
    ws.ccnt[lane] = 0;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; ++e)
        if ((u32)(lane * E + e) < d)
            atomicAdd(&ws.ccnt[k[e] >> rowbits], 1u);
    __syncwarp();
    const u32 c = ws.ccnt[lane];
    u32 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(full, incl, o);
        if (lane >= o)
            incl += t;
    }
    const u32 excl = incl - c;
#pragma unroll
    for (int e = 0; e < E; ++e)
    {
        const u32 r = lane * E + e;
        const bool ok = r < d;
        const u32 lc = ok ? (k[e] >> rowbits) : 0u;
        const u32 first = __shfl_sync(full, excl, lc);
        const u32 cbeg = __shfl_sync(full, cstart, a + lc);
        if (ok)
        {
            u32 slot = cf_hash(k[e]);
            while (ws.key[slot] != k[e])
                slot = (slot + 1) & (CF_H - 1);
            Rec o;
            o.key = (u64)(k[e] & rowmask);
            o.val = ws.value(slot);
            st_rec(tmp + (cbeg + (r - first)), o);
        }
    }
    if ((u32)lane >= a && (u32)lane < a + nc)
        colcount[ccol] = ws.ccnt[lane - a];
    __syncwarp();
}

// LIST = false: warp `tile` takes the columns that start inside span `tile` (tilek).
// LIST = true : the warps walk `list` (compact column indices left over by colthread_kernel:
//               columns too long or too rich for a single thread), one column at a time.
template <bool SIMPLE, int WARPS, bool LIST>
__global__ void __launch_bounds__(WARPS * 32, SIMPLE ? 1024 / (WARPS * 32) : 384 / (WARPS * 32))
colfold_kernel(const Rec *__restrict__ sorted, KeyLayout L, int combine, u32 chunk, const u32 *__restrict__ nzcol,
               const u32 *__restrict__ nzstart, const u32 *__restrict__ tilek, u32 ntiles, Rec *__restrict__ tmp,
               u32 *__restrict__ colcount, u32 *__restrict__ d_overflow, const u32 *__restrict__ list,
               const u32 *__restrict__ list_count)
{
    typedef WarpSpace<SIMPLE> WS;
    constexpr u32 full = 0xffffffffu;
    constexpr int NB = CF_PIECE / 32; // batches of a piece
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    WS &ws = reinterpret_cast<WS *>(smem_raw)[warp];
    const u32 lt = lanemask_lt();
    const u32 le = lt | (1u << lane);
    const int rowbits = L.rowbits;
    const int low = L.low;
    const u32 rowmask = (1u << rowbits) - 1u;
    const u32 metamask = (1u << low) - 1u;
    const u32 tend = LIST ? *list_count : ntiles;
    const u32 tstep = LIST ? gridDim.x * WARPS : 0xffffffffu - ntiles; // one span per warp without a list
  for (u32 tile = blockIdx.x * WARPS + warp; tile < tend; tile += tstep)
  {
    const u32 k_begin = LIST ? list[tile] : tilek[tile];
    const u32 k_end = LIST ? k_begin + 1u : tilek[tile + 1];

    for (u32 kw = k_begin; kw < k_end; kw += 32)
    { // window of up to 32 non-empty columns: lane j holds column kw + j
        const u32 kj = kw + lane;
        const bool have = kj < k_end;
        const u32 cstart = have ? nzstart[kj] : 0u;
        const u32 cend = have ? nzstart[kj + 1] : 0u;
        const u32 ccol = have ? nzcol[kj] : 0u;
        const u32 nwin = min(32u, k_end - kw);
        u32 a = 0;
        while (a < nwin)
        {
            // ---- group: as many whole columns as fit in `chunk` records, at least one
            const u32 s0 = __shfl_sync(full, cstart, a);
            const bool fits = (u32)lane >= a && (u32)lane < nwin && (cend - s0) <= chunk;
            const u32 fm = __ballot_sync(full, fits) >> a;
            const u32 nc = (fm & 1u) ? ((~fm) ? (u32)(__ffs(~fm) - 1) : 32u) : 1u;
            const u32 e0 = __shfl_sync(full, cend, a + nc - 1);
            const bool inchunk = (u32)lane >= a && (u32)lane < a + nc;

            // ---- clear the table
            {
                uint4 *kq = reinterpret_cast<uint4 *>(ws.key);
#pragma unroll
                for (int i = 0; i < CF_H / 128; ++i)
                    kq[i * 32 + lane] = make_uint4(CF_EMPTY, CF_EMPTY, CF_EMPTY, CF_EMPTY);
            }
            u32 dcount = 0;
            bool ovf = false;
            for (u32 b = s0; b < e0 && !ovf; b += CF_PIECE)
            {
                // ---- A. slot and rank of every record of the piece
                {
                    uint4 *cq = reinterpret_cast<uint4 *>(ws.cnt); // CF_H u16 = CF_H/8 uint4
#pragma unroll
                    for (int i = 0; i < (CF_H / 8 + 31) / 32; ++i)
                        if (i * 32 + lane < CF_H / 8)
                            cq[i * 32 + lane] = make_uint4(0, 0, 0, 0);
                }
                __syncwarp();
                Rec r[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i)
                {
                    const u32 p = b + i * 32 + lane;
                    if (p < e0)
                        r[i] = ld_rec_stream(sorted + p);
                    else
                    {
                        r[i].key = 0;
                        r[i].val = 0.0;
                    }
                }
                u32 sr[NB]; // slot | rank << 16
#pragma unroll
                for (int i = 0; i < NB; ++i)
                {
                    const u32 bb = b + i * 32;
                    sr[i] = 0;
                    if (bb < e0 && !ovf) // warp-uniform
                    {
                        if (dcount + 32 > (u32)CF_H)
                        {
                            ovf = true; // not enough free slots left for this batch
                        }
                        else
                        {
                            const u32 p = bb + lane;
                            const bool valid = p < e0;
                            u32 lc = 0;
                            if (nc > 1)
                            { // local column of position p: how many of the group's columns end at or before p
                                const u32 bit = (inchunk && cend >= bb && cend < bb + 32u) ? (1u << (cend - bb)) : 0u;
                                const u32 B = __reduce_or_sync(full, bit);
                                const u32 cntlow = __popc(__ballot_sync(full, inchunk && cend < bb));
                                lc = cntlow + __popc(B & le);
                            }
                            const u64 key = r[i].key;
                            const u32 row = (u32)(key >> low) & rowmask;
                            const u32 fl = (u32)key & 3u;
                            const u32 hk = (lc << rowbits) | row;
                            u32 slot = cf_hash(hk);
                            bool fresh = false;
                            if (valid)
                            {
                                for (;;)
                                {
                                    const u32 prev = atomicCAS(&ws.key[slot], CF_EMPTY, hk);
                                    if (prev == CF_EMPTY)
                                    {
                                        fresh = true;
                                        break;
                                    }
                                    if (prev == hk)
                                        break;
                                    slot = (slot + 1) & (CF_H - 1);
                                }
                            }
                            const u32 fb = __ballot_sync(full, fresh);
                            if (fresh)
                            {
                                ws.cand[dcount + __popc(fb & lt)] = (unsigned short)slot;
                                ws.init_slot(slot);
                            }
                            dcount += __popc(fb);
                            const bool creates = valid && ((fl != FL_UPDATE) | (r[i].val != 0.0));
                            const u32 crb = __ballot_sync(full, creates);
                            const u32 vm = __ballot_sync(full, valid);
                            u32 peers = 1u << lane;
                            if (valid)
                                peers = __match_any_sync(vm, slot);
                            __syncwarp();
                            const int ldr = __ffs(peers) - 1;
                            u32 base = 0;
                            if (valid && lane == ldr)
                            {
                                base = ws.cnt[slot];
                                ws.cnt[slot] = (unsigned short)(base + __popc(peers));
                                if (SIMPLE)
                                    ws.note(slot, (fb & peers) != 0u, fl, (crb & peers) != 0u);
                            }
                            base = __shfl_sync(full, base, ldr);
                            sr[i] = slot | ((base + __popc(peers & lt)) << 16);
                            __syncwarp();
                        }
                    }
                }
                if (ovf)
                    break;
                // ---- B. counts -> exclusive offsets, values laid out slot by slot
                {
                    constexpr int PER = CF_H / 32; // slots per lane (8)
                    unsigned short *cp = ws.cnt + lane * PER;
                    u32 c[PER], sum = 0;
#pragma unroll
                    for (int q = 0; q < PER; ++q)
                    {
                        c[q] = cp[q];
                        sum += c[q];
                    }
                    u32 incl = sum;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1)
                    {
                        const u32 t = __shfl_up_sync(full, incl, o);
                        if (lane >= o)
                            incl += t;
                    }
                    u32 run = incl - sum;
#pragma unroll
                    for (int q = 0; q < PER; ++q)
                    {
                        cp[q] = (unsigned short)run;
                        run += c[q];
                    }
                }
                __syncwarp();
                const u32 piece_n = min((u32)CF_PIECE, e0 - b);
#pragma unroll
                for (int i = 0; i < NB; ++i)
                {
                    const u32 p = b + i * 32 + lane;
                    if (p < e0)
                    {
                        const u32 slot = sr[i] & 0xffffu;
                        ws.put(ws.cnt[slot] + (sr[i] >> 16), r[i].val, (u32)r[i].key & metamask);
                    }
                }
                __syncwarp();
                // ---- C. one lane per slot folds its list in stream order
                for (u32 q = lane; q < dcount; q += 32)
                {
                    const u32 slot = ws.cand[q];
                    const u32 o0 = ws.cnt[slot];
                    const u32 o1 = (slot + 1 < (u32)CF_H) ? ws.cnt[slot + 1] : piece_n;
                    ws.fold(slot, o0, o1, combine);
                }
                __syncwarp();
            }
            if (ovf)
            {
                if (lane == 0)
                    atomicExch(d_overflow, 1u);
                return;
            }

            // ---- the group's entries, sorted by (local column,row)
            if (dcount <= 32)
                emit_group<1>(ws, dcount, rowbits, a, nc, cstart, ccol, tmp, colcount, lane);
            else if (dcount <= 64)
                emit_group<2>(ws, dcount, rowbits, a, nc, cstart, ccol, tmp, colcount, lane);
            else if (dcount <= 128)
                emit_group<4>(ws, dcount, rowbits, a, nc, cstart, ccol, tmp, colcount, lane);
            else
                emit_group<8>(ws, dcount, rowbits, a, nc, cstart, ccol, tmp, colcount, lane);
            a += nc;
        }
    }
  }
}

// ------------------------------------------------------------------------
// one THREAD per column (plain += streams: one partition, no assign flavour, old values seed)
// ------------------------------------------------------------------------
// Thread k walks the records of non-empty column k in stream order.  Its accumulators live in
// shared memory, in a private open-addressing table laid out slot-major ([slot][lane]) so that a
// lane only ever touches its own bank: no conflicts whatever the slots are.  A table slot holds
// (row << HBITS | accumulator index); the accumulators are numbered in order of first appearance.
// Every record is one probe and one add: the exact left fold of the reference's
// accumulate-on-insert (src/matrix/sparsematrixlnk.jl:210-253) with the list walk replaced by the
// hash probe.  At the end the slots of the existing entries are insertion-sorted by row in place
// (src/matrix/sparsematrixlnk.jl:339) and the entries parked at the column's offset.
//
// Three table sizes (16/12, 32/24, 64/48 slots/accumulators) trade occupancy against capacity: a
// column with more distinct rows than the table takes is appended to `next` (the next size, or the
// warp-per-column kernel); columns longer than maxlen go straight to `longlist` (warp kernel).
constexpr int CT_WARPS = 4;
#ifndef XSB_CT_U
#define XSB_CT_U 2
#endif
constexpr int CT_U = XSB_CT_U; // 32-byte record pairs per step (the next step is prefetched)
constexpr u32 CT_EMPTY = 0xffffffffu;

// Table shapes, smallest first.  The template argument is the number of hash bits, except 15 = the
// 5-bit table with 16 instead of 24 accumulators: a P1 tetrahedral mesh has at most 15 rows per column,
// and the smaller accumulator array lets 5 instead of 4 blocks share an SM.
//   shape  4: 16 slots / 12 accumulators     shape 15: 32 / 16     shape 5: 32 / 24     shape 6: 64 / 32
template <int HBITS> struct CtShape
{
    static constexpr int HB = HBITS == 15 ? 5 : HBITS;
    static constexpr int H = 1 << HB;
    static constexpr int D = HBITS == 6 ? 32 : (HBITS == 5 ? 24 : (HBITS == 15 ? 16 : 12));
    static constexpr int kBlocks = HBITS == 4 ? 8 : (HBITS == 6 ? 2 : 5); // launch bound (registers)
    // table words + accumulators + row of every accumulator (first-appearance order)
    static constexpr size_t kBytesPerWarp = 32 * (sizeof(u32) * H + (sizeof(double) + sizeof(u32)) * D);
};

// Folds the records [cstart, cend) of one column.  Returns the number of existing entries j, their
// (row << HBITS | accumulator) words sorted in key[0 .. j), or -1 if the table is too small.
// d_out = distinct rows seen.
template <int HBITS>
__device__ __forceinline__ int ct_fold_column(const Rec *__restrict__ sorted, u32 cstart, u32 cend, int low,
                                              u32 rowmask, u32 *key, double *acc, u32 *rows, u32 &d_out)
{
    constexpr int H = CtShape<HBITS>::H;
    constexpr int HB = CtShape<HBITS>::HB;
    constexpr u32 D = CtShape<HBITS>::D;
#pragma unroll
    for (int s = 0; s < H; ++s)
        key[s * 32] = CT_EMPTY;

    u32 d = 0;       // accumulators in use
    u32 pending = 0; // of which not (yet) existing: only updateindex! of a zero touched them
    u64 exmask = 0;  // accumulator i holds an existing entry
    bool ovf = false;
    auto apply = [&](const Rec &r) {
        const u32 row = (u32)(r.key >> low) & rowmask;
        const double v = r.val;
        u32 s = (row * 0x9E3779B1u) >> (32 - HB);
        for (;;)
        {
            const u32 kk = key[s * 32];
            const u32 x = kk ^ (row << HB);
            if (x < D)
            { // same row (an empty slot reads as index H-1 >= D): x is the accumulator
                acc[x * 32] = acc[x * 32] + v;
                if (pending)
                {
                    const u32 fl = (u32)r.key & 3u;
                    if (!((exmask >> x) & 1ull) && ((fl != FL_UPDATE) | (v != 0.0)))
                    {
                        exmask |= 1ull << x;
                        --pending;
                    }
                }
                return;
            }
            if (kk == CT_EMPTY)
            {
                if (d >= D)
                {
                    ovf = true;
                    return;
                }
                const u32 fl = (u32)r.key & 3u;
                key[s * 32] = (row << HB) | d;
                rows[d * 32] = row;
                // a run starts from +0.0 (sparsematrixlnk.jl:225) unless the resident CSC value
                // seeds it (extendable.jl:165-166); updateindex! of a zero creates nothing (:212,223)
                acc[d * 32] = (fl == FL_OLD) ? v : 0.0 + v;
                if ((fl != FL_UPDATE) | (v != 0.0))
                    exmask |= 1ull << d;
                else
                    ++pending;
                ++d;
                return;
            }
            s = (s + 1) & (H - 1);
        }
    };

    // A lane streams its own column: every load instruction of the warp touches 32 different
    // lines, so the L1 sees one request per lane.  256-bit loads (two records per request, 32-byte
    // aligned: the records of an odd start and an odd end go alone) halve that.
    u32 p = cstart;
    if ((p & 1u) && p < cend)
        apply(sorted[p++]);
    const Rec *col = sorted + p;
    const u32 npair = (cend - p) >> 1;
    const u32 nfull = npair / CT_U;
    RecPair nxt[CT_U];
    if (nfull)
    {
#pragma unroll
        for (int i = 0; i < CT_U; ++i)
            nxt[i] = ld_pair_stream(col + 2 * i);
    }
    u32 g = 0;
    for (; g < nfull && !ovf; ++g)
    {
        RecPair cur[CT_U];
#pragma unroll
        for (int i = 0; i < CT_U; ++i)
            cur[i] = nxt[i];
        if (g + 1 < nfull)
        {
#pragma unroll
            for (int i = 0; i < CT_U; ++i)
                nxt[i] = ld_pair_stream(col + 2 * ((g + 1) * CT_U + i));
        }
#pragma unroll
        for (int i = 0; i < CT_U; ++i)
        {
            if (!ovf)
                apply(cur[i].a);
            if (!ovf)
                apply(cur[i].b);
        }
    }
    for (u32 q = p + 2 * nfull * CT_U; q < cend && !ovf; ++q)
        apply(sorted[q]);
    d_out = ovf ? D + 1 : d;
    if (ovf)
        return -1;
    // ---- existing entries as (row << HBITS | accumulator) words, insertion-sorted by row into the
    // (no longer needed) table.  They are taken in order of first appearance, which an assembly
    // stream visits nearly in row order: few shifts (src/matrix/sparsematrixlnk.jl:339 sorts here too).
    u32 j = 0;
    for (u32 i = 0; i < d; ++i)
    {
        if (!((exmask >> i) & 1ull))
            continue;
        const u32 kk = (rows[i * 32] << HB) | i;
        u32 q = j;
        while (q > 0)
        {
            const u32 prev = key[(q - 1) * 32];
            if (prev < kk)
                break;
            key[q * 32] = prev;
            --q;
        }
        key[q * 32] = kk;
        ++j;
    }
    return (int)j;
}

template <int HBITS, bool LIST>
__global__ void __launch_bounds__(CT_WARPS * 32, CtShape<HBITS>::kBlocks)
colthread_kernel(const Rec *__restrict__ sorted, int low, int rowbits, u32 maxlen, const u32 *__restrict__ nzcol,
                 const u32 *__restrict__ nzstart, const u64 *__restrict__ totals, Rec *__restrict__ tmp,
                 u32 *__restrict__ colcount, const u32 *__restrict__ src, const u32 *__restrict__ src_count,
                 u32 *__restrict__ next, u32 *__restrict__ next_count, u32 *__restrict__ longlist,
                 u32 *__restrict__ long_count, u32 *__restrict__ maxd)
{
    constexpr int H = CtShape<HBITS>::H;
    constexpr u32 D = CtShape<HBITS>::D;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *acc = reinterpret_cast<double *>(smem_raw) + warp * (D * 32) + lane; // accumulator i: acc[i * 32]
    u32 *key = reinterpret_cast<u32 *>(smem_raw + (size_t)CT_WARPS * D * 32 * sizeof(double)) + warp * (H * 32) + lane;
    u32 *rows = reinterpret_cast<u32 *>(smem_raw + (size_t)CT_WARPS * 32 * (D * sizeof(double) + H * sizeof(u32))) +
                warp * (D * 32) + lane;
    const u32 rowmask = (1u << rowbits) - 1u;
    const u64 K = LIST ? (u64)*src_count : totals[1];
    const u64 step = LIST ? (u64)gridDim.x * (CT_WARPS * 32) : ~0ull >> 1;
    for (u64 t = (u64)blockIdx.x * (CT_WARPS * 32) + threadIdx.x; t < K; t += step)
    {
        const u32 k = LIST ? src[t] : (u32)t;
        const u32 cstart = nzstart[k], cend = nzstart[k + 1];
        if (cend - cstart > maxlen)
        {
            longlist[atomicAdd(long_count, 1u)] = k;
            continue;
        }
        u32 d;
        const int j = ct_fold_column<HBITS>(sorted, cstart, cend, low, rowmask, key, acc, rows, d);
        if (j < 0)
        {
            next[atomicAdd(next_count, 1u)] = k;
            if (d > ld_relaxed_u32(maxd))
                atomicMax(maxd, d);
            continue;
        }
        Rec *dst = tmp + cstart;
        for (int e = 0; e < j; ++e)
        {
            const u32 pk = key[e * 32];
            Rec o;
            o.key = (u64)(pk >> CtShape<HBITS>::HB);
            o.val = acc[(pk & (H - 1)) * 32];
            st_rec(dst + e, o);
        }
        colcount[nzcol[k]] = (u32)j;
        if (d > ld_relaxed_u32(maxd))
            atomicMax(maxd, d);
    }
}

// The same fold writing the final CSC in ONE pass: the entries of column k go to
// rowval/nzval[sum of the entry counts of the columns before k ...], that sum coming from a block
// scan plus a decoupled look-back over the block totals (blocks are dispatched in index order).
// A column that needs another table size or the warp kernel raises *d_redo; the caller then runs
// the parking path (colthread_kernel + compact) instead.

template <int HBITS, typename Ti>
__global__ void __launch_bounds__(CT_WARPS * 32, CtShape<HBITS>::kBlocks)
colthread_direct_kernel(const Rec *__restrict__ sorted, int low, int rowbits, u32 maxlen,
                        const u32 *__restrict__ nzcol, const u32 *__restrict__ nzstart,
                        const u64 *__restrict__ totals, i64 ncols, Ti base, Ti *__restrict__ rowval,
                        double *__restrict__ nzval, Ti *__restrict__ colptr, u64 *__restrict__ status,
                        u32 *__restrict__ ticket, u64 *__restrict__ d_nnz, u32 *__restrict__ d_redo,
                        u32 *__restrict__ maxd)
{
    constexpr int H = CtShape<HBITS>::H;
    constexpr u32 D = CtShape<HBITS>::D;
    constexpr u32 full = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ u32 s_wsum[CT_WARPS];
    __shared__ u64 s_prefix;
    __shared__ u32 s_bid;
    // blocks take their columns in the order they START (ticket), so a block only ever waits for
    // blocks that are already running: the look-back cannot starve whatever the dispatch order
    if (threadIdx.x == 0)
        s_bid = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 bid = s_bid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *acc = reinterpret_cast<double *>(smem_raw) + warp * (D * 32) + lane;
    u32 *key = reinterpret_cast<u32 *>(smem_raw + (size_t)CT_WARPS * D * 32 * sizeof(double)) + warp * (H * 32) + lane;
    u32 *rows = reinterpret_cast<u32 *>(smem_raw + (size_t)CT_WARPS * 32 * (D * sizeof(double) + H * sizeof(u32))) +
                warp * (D * 32) + lane;
    const u32 rowmask = (1u << rowbits) - 1u;
    const u64 K = totals[1];
    const u64 k = (u64)bid * (CT_WARPS * 32) + threadIdx.x;
    int j = 0;
    u32 cstart = 0;
    if (k < K && ld_relaxed_u32(d_redo) == 0u)
    {
        cstart = nzstart[k];
        const u32 cend = nzstart[k + 1];
        if (cend - cstart > maxlen)
            atomicOr(d_redo, 2u);
        else
        {
            u32 d;
            j = ct_fold_column<HBITS>(sorted, cstart, cend, low, rowmask, key, acc, rows, d);
            if (j < 0)
            { // bit 2: not even the largest table takes this column
                atomicOr(d_redo, HBITS == 6 ? 5u : 1u);
                j = 0;
            }
            if (d > ld_relaxed_u32(maxd))
                atomicMax(maxd, d);
        }
    }
    // ---- entries before this column: warp scan, block scan, look-back over the blocks
    u32 incl = (u32)j;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(full, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_wsum[warp] = incl;
    __syncthreads();
    u32 wpre = 0, btotal = 0;
#pragma unroll
    for (int w = 0; w < CT_WARPS; ++w)
    {
        const u32 c = s_wsum[w];
        if (w < warp)
            wpre += c;
        btotal += c;
    }
    if (warp == 0)
    {
        const u64 prefix = warp_lookback(status, bid, (u64)btotal, lane);
        if (lane == 0)
            s_prefix = prefix;
    }
    __syncthreads();
    if (k >= K)
        return;
    const u64 o0 = s_prefix + wpre + (incl - (u32)j);
    // 256-bit stores where the destination is 32-byte aligned (rowval and nzval separately: their
    // bases differ): a lane writes its own run, so every store instruction costs one request per lane
    {
        Ti *rv = rowval + o0;
        auto row_at = [&](int e) { return (Ti)(key[e * 32] >> CtShape<HBITS>::HB) + base; };
        constexpr int V = 32 / (int)sizeof(Ti);
        int e = 0;
        for (; e < j && (reinterpret_cast<uintptr_t>(rv + e) & 31u); ++e)
            rv[e] = row_at(e);
        for (; e + V <= j; e += V)
        {
            if (sizeof(Ti) == 8)
                st_v4_u64(rv + e, (u64)row_at(e), (u64)row_at(e + 1), (u64)row_at(e + 2), (u64)row_at(e + 3));
            else
            {
                const u64 w0 = (u64)(u32)row_at(e) | ((u64)(u32)row_at(e + 1) << 32);
                const u64 w1 = (u64)(u32)row_at(e + 2) | ((u64)(u32)row_at(e + 3) << 32);
                const u64 w2 = (u64)(u32)row_at(e + 4) | ((u64)(u32)row_at(e + 5) << 32);
                const u64 w3 = (u64)(u32)row_at(e + 6) | ((u64)(u32)row_at(e + 7) << 32);
                st_v4_u64(rv + e, w0, w1, w2, w3);
            }
        }
        for (; e < j; ++e)
            rv[e] = row_at(e);
    }
    {
        double *nv = nzval + o0;
        auto val_at = [&](int e) { return (u64)__double_as_longlong(acc[(key[e * 32] & (H - 1)) * 32]); };
        int e = 0;
        for (; e < j && (reinterpret_cast<uintptr_t>(nv + e) & 31u); ++e)
            nv[e] = __longlong_as_double((long long)val_at(e));
        for (; e + 4 <= j; e += 4)
            st_v4_u64(nv + e, val_at(e), val_at(e + 1), val_at(e + 2), val_at(e + 3));
        for (; e < j; ++e)
            nv[e] = __longlong_as_double((long long)val_at(e));
    }
    // colptr of this column and of the empty columns right before it
    const i64 c1 = (i64)nzcol[k];
    const i64 c0 = k ? (i64)nzcol[k - 1] + 1 : 0;
    for (i64 c = c0; c <= c1; ++c)
        colptr[c] = (Ti)o0 + base;
    if (k == K - 1)
    {
        for (i64 c = c1 + 1; c <= ncols; ++c)
            colptr[c] = (Ti)(o0 + j) + base;
        *d_nnz = o0 + (u64)j;
    }
}

// ------------------------------------------------------------------------
// colptr = base + exclusive sum of the per-column entry counts
// ------------------------------------------------------------------------
__global__ void __launch_bounds__(CS_THREADS)
entrycount_tilesum_kernel(const u32 *__restrict__ colcount, i64 n, u64 *__restrict__ tsum)
{
    __shared__ u64 s_w[CS_THREADS / 32];
    const i64 b0 = (i64)blockIdx.x * CS_TILE;
    u64 s = 0;
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        const i64 j = b0 + i * CS_THREADS + threadIdx.x;
        if (j < n)
            s += colcount[j];
    }
    s = block_sum_u64(s, s_w);
    if (threadIdx.x == 0)
        tsum[blockIdx.x] = s;
}

__global__ void __launch_bounds__(1024)
entrycount_scan_kernel(u64 *__restrict__ tsum, i64 nt, u64 *__restrict__ d_nnz)
{
    __shared__ u64 s_w[32];
    __shared__ u64 s_carry;
    if (threadIdx.x == 0)
        s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (i64 b0 = 0; b0 < nt; b0 += 1024)
    {
        const i64 j = b0 + threadIdx.x;
        const u64 x = j < nt ? tsum[j] : 0;
        u64 v = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o)
                v += t;
        }
        if (lane == 31)
            s_w[warp] = v;
        __syncthreads();
        u64 pre = s_carry;
        for (int w = 0; w < warp; ++w)
            pre += s_w[w];
        if (j < nt)
            tsum[j] = pre + v - x;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = pre + v;
        __syncthreads();
    }
    if (threadIdx.x == 0)
        *d_nnz = s_carry;
}

template <typename Ti>
__global__ void __launch_bounds__(CS_THREADS)
colptr_emit_kernel(const u32 *__restrict__ colcount, const u64 *__restrict__ tsum, i64 n, Ti base,
                   Ti *__restrict__ colptr)
{
    __shared__ u64 s_w[CS_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 b0 = (i64)blockIdx.x * CS_TILE + (i64)threadIdx.x * CS_IPT;
    u64 c[CS_IPT], sum = 0;
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        const i64 j = b0 + i;
        c[i] = j < n ? (u64)colcount[j] : 0ull;
        sum += c[i];
    }
    u64 incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_w[warp] = incl;
    __syncthreads();
    u64 run = tsum[blockIdx.x];
    for (int w = 0; w < warp; ++w)
        run += s_w[w];
    run += incl - sum;
#pragma unroll
    for (int i = 0; i < CS_IPT; ++i)
    {
        const i64 j = b0 + i;
        if (j < n)
            colptr[j] = (Ti)run + base;
        run += c[i];
        if (j == n - 1)
            colptr[n] = (Ti)run + base;
    }
}

// parked entries -> rowval / nzval.  A half warp per non-empty column.
template <typename Ti>
__global__ void __launch_bounds__(256)
compact_entries_kernel(const Rec *__restrict__ tmp, const u32 *__restrict__ nzcol, const u32 *__restrict__ nzstart,
                       const u64 *__restrict__ totals, const Ti *__restrict__ colptr, Ti base, Ti *__restrict__ rowval,
                       double *__restrict__ nzval)
{
    const u64 K = totals[1];
    const int sub = threadIdx.x & 15;
    const u64 nhalf = ((u64)gridDim.x * blockDim.x) >> 4;
    for (u64 k = (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 4); k < K; k += nhalf)
    {
        const u32 col = nzcol[k];
        const u64 src = nzstart[k];
        const i64 dst = (i64)colptr[col] - (i64)base;
        const u32 cnt = (u32)(colptr[col + 1] - colptr[col]);
        for (u32 e = sub; e < cnt; e += 16)
        {
            const Rec r = tmp[src + e];
            rowval[dst + e] = (Ti)r.key + base;
            nzval[dst + e] = r.val;
        }
    }
}

// ------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------
namespace {
struct CtArgs
{
    const Rec *sorted;
    int low, rowbits;
    u32 maxlen;
    const u32 *nzcol, *nzstart;
    const u64 *totals;
    Rec *tmp;
    u32 *colcount;
    const u32 *src, *src_count;
    u32 *next, *next_count, *longlist, *long_count, *maxd;
};
template <int HBITS, bool LIST> void launch_colthread_t(cudaStream_t stream, unsigned blocks, const CtArgs &a)
{
    constexpr size_t smem = CT_WARPS * CtShape<HBITS>::kBytesPerWarp;
    static FuncAttrOnce once;
    once.set(colthread_kernel<HBITS, LIST>, (int)smem, true);
    colthread_kernel<HBITS, LIST><<<blocks, CT_WARPS * 32, smem, stream>>>(
        a.sorted, a.low, a.rowbits, a.maxlen, a.nzcol, a.nzstart, a.totals, a.tmp, a.colcount, a.src, a.src_count, a.next,
        a.next_count, a.longlist, a.long_count, a.maxd);
}
// level 0/1/2 = 16/32/64 table slots; list = false: every non-empty column, true: the columns of a.src
void launch_colthread(cudaStream_t stream, int level, bool list, unsigned blocks, const CtArgs &a)
{
    if (!list)
    {
        if (level == 0)
            launch_colthread_t<4, false>(stream, blocks, a);
        else if (level == 1)
            launch_colthread_t<5, false>(stream, blocks, a);
        else
            launch_colthread_t<6, false>(stream, blocks, a);
    }
    else
    {
        if (level == 1)
            launch_colthread_t<5, true>(stream, blocks, a);
        else
            launch_colthread_t<6, true>(stream, blocks, a);
    }
}
struct CfLayout
{
    size_t off_cnt, off_nzcol, off_nzstart, off_tilek, off_trec, off_tnz, off_tsum, off_tot, off_list, off_status, bytes;
};
CfLayout cf_layout(u64 nrec, i64 ncols)
{
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const u64 kmax = std::min<u64>((u64)ncols, nrec);
    const u64 ntiles = (nrec + CF_SPAN - 1) / CF_SPAN;
    const u64 ctiles = ((u64)ncols + CS_TILE - 1) / CS_TILE;
    CfLayout l{};
    size_t o = 0;
    l.off_cnt = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_nzcol = o;
    o = up(o + sizeof(u32) * (kmax + 1));
    l.off_nzstart = o;
    o = up(o + sizeof(u32) * (kmax + 2));
    l.off_tilek = o;
    o = up(o + sizeof(u32) * (ntiles + 2));
    l.off_trec = o;
    o = up(o + sizeof(u64) * (ctiles + 1));
    l.off_tnz = o;
    o = up(o + sizeof(u32) * (ctiles + 1));
    l.off_tsum = o;
    o = up(o + sizeof(u64) * (ctiles + 1));
    l.off_tot = o;
    o = up(o + sizeof(u64) * 4);
    l.off_list = o; // columns left over by the thread-per-column kernels: two hand-over lists + the long columns
    o = up(o + 3 * sizeof(u32) * (kmax + 1));
    l.off_status = o; // look-back words of the one-pass fold, one per block of CT_WARPS*32 columns
    o = up(o + sizeof(u64) * ((kmax + CT_WARPS * 32 - 1) / (CT_WARPS * 32) + 2));
    l.bytes = o;
    return l;
}
} // namespace

size_t colfold_workspace_bytes(u64 nrec, i64 ncols) { return cf_layout(nrec, ncols).bytes; }

void colscan_scan_launch(cudaStream_t stream, u64 *trec, u32 *tnz, i64 nt, u64 *totals, u32 *nzstart)
{
    colscan_scan_kernel<<<1, 1024, 0, stream>>>(trec, tnz, nt, totals, nzstart);
}

void colfold_lists(void *workspace, u64 nrec, i64 ncols, u32 **nzcol, u32 **nzstart, u64 **totals)
{
    const CfLayout l = cf_layout(nrec, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    *nzcol = reinterpret_cast<u32 *>(ws + l.off_nzcol);
    *nzstart = reinterpret_cast<u32 *>(ws + l.off_nzstart);
    *totals = reinterpret_cast<u64 *>(ws + l.off_tot);
}

bool colfold_supported(const KeyLayout &L, u64 nrec, i64 ncols)
{
    return L.rowbits <= CF_MAXROWBITS && L.low <= 32 && nrec < (1ull << 32) - (u64)CF_SPAN &&
           (u64)ncols < (1ull << 32) - 1ull;
}

u32 *colfold_counts(void *workspace, u64 nrec, i64 ncols)
{
    return reinterpret_cast<u32 *>(static_cast<unsigned char *>(workspace) + cf_layout(nrec, ncols).off_cnt);
}

void colfold_clear_counts(cudaStream_t stream, void *workspace, u64 nrec, i64 ncols)
{
    XSB_CUDA(cudaMemsetAsync(colfold_counts(workspace, nrec, ncols), 0, sizeof(u32) * ((size_t)ncols + 1), stream));
}

namespace {
template <int HBITS, typename Ti>
void launch_direct_t(cudaStream_t stream, unsigned blocks, const Rec *sorted, int low, int rowbits, u32 maxlen,
                     const u32 *nzcol, const u32 *nzstart, const u64 *totals, i64 ncols, i64 base, void *rowval,
                     double *nzval, void *colptr, u64 *status, u32 *ticket, u64 *d_nnz, u32 *d_redo, u32 *maxd)
{
    constexpr size_t smem = CT_WARPS * CtShape<HBITS>::kBytesPerWarp;
    static FuncAttrOnce once;
    once.set(colthread_direct_kernel<HBITS, Ti>, (int)smem, true);
    colthread_direct_kernel<HBITS, Ti><<<blocks, CT_WARPS * 32, smem, stream>>>(
        sorted, low, rowbits, maxlen, nzcol, nzstart, totals, ncols, (Ti)base, (Ti *)rowval, nzval, (Ti *)colptr, status,
        ticket, d_nnz, d_redo, maxd);
}
} // namespace

bool colfold_direct_supported(const KeyLayout &L, int combine, bool plain_adds)
{
    return plain_adds && L.tidbits == 0 && combine == 0;
}

// One-pass variant of the fold for plain += streams: records grouped by column -> final rowval / nzval /
// colptr (rowval_out / nzval_out need room for nrec entries).  *d_redo != 0 afterwards: a column did not
// fit the chosen table (bit 0) or is too long for one thread (bit 1); nothing valid was written and the
// caller runs colfold_reduce (lists_ready = true) + colfold_compact instead.
void colfold_direct(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, i64 ncols, int idx64, int base,
                    void *rowval_out, double *nzval_out, void *colptr_out, void *workspace, u64 *d_nnz, u32 *d_redo,
                    bool lists_ready, u32 *d_maxd, u32 hint_maxd, LaunchCounter &lc, StageTimer *timer)
{
    const CfLayout l = cf_layout(nrec, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *cnt = reinterpret_cast<u32 *>(ws + l.off_cnt);
    u32 *nzcol = reinterpret_cast<u32 *>(ws + l.off_nzcol);
    u32 *nzstart = reinterpret_cast<u32 *>(ws + l.off_nzstart);
    u64 *trec = reinterpret_cast<u64 *>(ws + l.off_trec);
    u32 *tnz = reinterpret_cast<u32 *>(ws + l.off_tnz);
    u64 *totals = reinterpret_cast<u64 *>(ws + l.off_tot);
    u64 *status = reinterpret_cast<u64 *>(ws + l.off_status);
    const u64 kmax = std::min<u64>((u64)ncols, nrec);
    const unsigned ctiles = (unsigned)(((u64)ncols + CS_TILE - 1) / CS_TILE);
    const unsigned blocks = (unsigned)((kmax + CT_WARPS * 32 - 1) / (CT_WARPS * 32));
    if (timer)
        timer->begin(stream);
    XSB_CUDA(cudaMemsetAsync(d_redo, 0, sizeof(u32), stream));
    XSB_CUDA(cudaMemsetAsync(d_maxd, 0, sizeof(u32), stream));
    XSB_CUDA(cudaMemsetAsync(status, 0, sizeof(u64) * ((size_t)blocks + 2), stream)); // look-back words + ticket
    u32 *ticket = reinterpret_cast<u32 *>(status + blocks + 1);
    if (!lists_ready)
    {
        colscan_tilesum_kernel<<<ctiles, CS_THREADS, 0, stream>>>(cnt, ncols, trec, tnz);
        colscan_scan_kernel<<<1, 1024, 0, stream>>>(trec, tnz, (i64)ctiles, totals, nzstart);
        colscan_emit_kernel<<<ctiles, CS_THREADS, 0, stream>>>(cnt, trec, tnz, ncols, nzcol, nzstart);
        lc.add(3);
    }
    if (timer)
        timer->end(stream, &StageTimes::colptr);
    if (timer)
        timer->begin(stream);
    const u64 avg = nrec / std::max<u64>(1, kmax);
    const int level = hint_maxd ? (hint_maxd <= 12 ? 0 : (hint_maxd <= 24 ? 1 : 2)) : (avg < 14 ? 0 : (avg < 40 ? 1 : 2));
    // 13..16 distinct rows in the previous flush (P1 FEM: 15): the 32-slot table with 16 accumulators
    const bool slim = level == 1 && hint_maxd != 0 && hint_maxd <= 16;
    const u32 maxlen = (u32)std::max<u64>(256, 6 * avg);
#define XSB_DIRECT(HB, TI)                                                                                              \
    launch_direct_t<HB, TI>(stream, blocks, sorted, L.low, L.rowbits, maxlen, nzcol, nzstart, totals, ncols, base,      \
                            rowval_out, nzval_out, colptr_out, status, ticket, d_nnz, d_redo, d_maxd)
    if (idx64)
    {
        if (level == 0)
            XSB_DIRECT(4, int64_t);
        else if (slim)
            XSB_DIRECT(15, int64_t);
        else if (level == 1)
            XSB_DIRECT(5, int64_t);
        else
            XSB_DIRECT(6, int64_t);
    }
    else
    {
        if (level == 0)
            XSB_DIRECT(4, int32_t);
        else if (slim)
            XSB_DIRECT(15, int32_t);
        else if (level == 1)
            XSB_DIRECT(5, int32_t);
        else
            XSB_DIRECT(6, int32_t);
    }
#undef XSB_DIRECT
    lc.add();
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::fold);
}

// Stage 1: records sorted by column (stable), per-column record counts already in the workspace
// -> entries parked in `tmp` (same capacity as `sorted`), colptr written, *d_nnz = entries,
// *d_overflow != 0 if a group of columns did not fit the in-warp table (outputs then undefined).
void colfold_reduce(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, int combine, bool plain_adds,
                    i64 ncols, int idx64, int base, Rec *tmp, void *colptr_out, void *workspace, u64 *d_nnz,
                    u32 *d_overflow, bool lists_ready, u32 *d_maxd, u32 hint_maxd, LaunchCounter &lc, StageTimer *timer)
{
    const CfLayout l = cf_layout(nrec, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *cnt = reinterpret_cast<u32 *>(ws + l.off_cnt);
    u32 *nzcol = reinterpret_cast<u32 *>(ws + l.off_nzcol);
    u32 *nzstart = reinterpret_cast<u32 *>(ws + l.off_nzstart);
    u32 *tilek = reinterpret_cast<u32 *>(ws + l.off_tilek);
    u64 *trec = reinterpret_cast<u64 *>(ws + l.off_trec);
    u32 *tnz = reinterpret_cast<u32 *>(ws + l.off_tnz);
    u64 *tsum = reinterpret_cast<u64 *>(ws + l.off_tsum);
    u64 *totals = reinterpret_cast<u64 *>(ws + l.off_tot);
    const u64 kmax = std::min<u64>((u64)ncols, nrec);
    const u32 ntiles = (u32)((nrec + CF_SPAN - 1) / CF_SPAN);
    const unsigned ctiles = (unsigned)(((u64)ncols + CS_TILE - 1) / CS_TILE);

    if (timer)
        timer->begin(stream);
    XSB_CUDA(cudaMemsetAsync(d_overflow, 0, sizeof(u32), stream));
    XSB_CUDA(cudaMemsetAsync(d_maxd, 0, sizeof(u32), stream));
    if (!lists_ready)
    { // column list from the per-column record counts (taken by the sort's histogram kernel)
        colscan_tilesum_kernel<<<ctiles, CS_THREADS, 0, stream>>>(cnt, ncols, trec, tnz);
        colscan_scan_kernel<<<1, 1024, 0, stream>>>(trec, tnz, (i64)ctiles, totals, nzstart);
        colscan_emit_kernel<<<ctiles, CS_THREADS, 0, stream>>>(cnt, trec, tnz, ncols, nzcol, nzstart);
        lc.add(3);
    }
    else // the grouping pass made the list; cnt only receives the entry counts of non-empty columns
        XSB_CUDA(cudaMemsetAsync(cnt, 0, sizeof(u32) * ((size_t)ncols + 1), stream));
    tilemap_kernel<<<(unsigned)((kmax + 1 + 255) / 256), 256, 0, stream>>>(nzstart, totals, ntiles, tilek);
    lc.add(1);
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::colptr);

    if (timer)
        timer->begin(stream);
    const bool simple = plain_adds && L.tidbits == 0 && combine == 0;
    // Groups of short columns hold many distinct entries per record (little duplication), and the
    // in-register sort of the distinct entries grows faster than linearly: keep such groups small.
    const u32 chunk = (nrec / std::max<u64>(1, std::min<u64>((u64)ncols, nrec)) >= 48) ? (u32)CF_PIECE : 128u;
    if (simple)
    { // one thread per column, smallest table first; what a size cannot take is handed to the next
      // one through a list, the rest (and the long columns) to the warp kernel
        u32 *listA = reinterpret_cast<u32 *>(ws + l.off_list);
        u32 *listB = listA + (kmax + 1);
        u32 *longlist = listB + (kmax + 1);
        u32 *counters = reinterpret_cast<u32 *>(totals + 2); // [0] listA, [1] listB, [2] long columns
        XSB_CUDA(cudaMemsetAsync(counters, 0, 4 * sizeof(u32), stream));
        const u64 avg = nrec / std::max<u64>(1, kmax);
        // table size to start with: what the previous flush of this handle needed, else the mean
        // column length (a column cannot hold more distinct rows than records)
        const int level = hint_maxd ? (hint_maxd <= 12 ? 0 : (hint_maxd <= 24 ? 1 : 2)) : (avg < 14 ? 0 : (avg < 40 ? 1 : 2));
        CtArgs a{sorted, L.low, L.rowbits, (u32)std::max<u64>(256, 6 * avg), nzcol, nzstart, totals, tmp, cnt,
                 nullptr, nullptr, nullptr, nullptr, longlist, counters + 2, d_maxd};
        // (nothing but skipped records: one block that finds no column)
        const unsigned blocks = (unsigned)std::max<u64>(1, (kmax + CT_WARPS * 32 - 1) / (CT_WARPS * 32));
        const unsigned lblocks = (unsigned)std::min<u64>(blocks, (u64)kNumSM * 8);
        u32 *lists[2] = {listA, listB};
        for (int lv = level, hop = 0; lv <= 2; ++lv, ++hop)
        {
            a.src = hop ? lists[(hop - 1) & 1] : nullptr;
            a.src_count = hop ? counters + ((hop - 1) & 1) : nullptr;
            a.next = lv == 2 ? longlist : lists[hop & 1];
            a.next_count = lv == 2 ? counters + 2 : counters + (hop & 1);
            launch_colthread(stream, lv, hop != 0, hop ? lblocks : blocks, a);
            lc.add();
        }
        constexpr int W = 8;
        const size_t smem = sizeof(WarpSpace<true>) * W;
        static FuncAttrOnce once;
        once.set(colfold_kernel<true, W, true>, (int)smem);
        colfold_kernel<true, W, true><<<kNumSM * 2, W * 32, smem, stream>>>(sorted, L, combine, chunk, nzcol, nzstart, tilek,
                                                                          ntiles, tmp, cnt, d_overflow, longlist, counters + 2);
    }
    else
    {
        constexpr int W = 4;
        const size_t smem = sizeof(WarpSpace<false>) * W;
        static FuncAttrOnce once;
        once.set(colfold_kernel<false, W, false>, (int)smem);
        colfold_kernel<false, W, false><<<std::max(1u, (ntiles + W - 1) / W), W * 32, smem, stream>>>(
            sorted, L, combine, chunk, nzcol, nzstart, tilek, ntiles, tmp, cnt, d_overflow, nullptr, nullptr);
    }
    lc.add();
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::fold);

    if (timer)
        timer->begin(stream);
    entrycount_tilesum_kernel<<<ctiles, CS_THREADS, 0, stream>>>(cnt, ncols, tsum);
    entrycount_scan_kernel<<<1, 1024, 0, stream>>>(tsum, (i64)ctiles, d_nnz);
    if (idx64)
        colptr_emit_kernel<int64_t><<<ctiles, CS_THREADS, 0, stream>>>(cnt, tsum, ncols, (int64_t)base, (int64_t *)colptr_out);
    else
        colptr_emit_kernel<int32_t><<<ctiles, CS_THREADS, 0, stream>>>(cnt, tsum, ncols, (int32_t)base, (int32_t *)colptr_out);
    lc.add(3);
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::colptr);
}

// Stage 2: parked entries -> rowval / nzval (caller's index type and base)
void colfold_compact(cudaStream_t stream, const Rec *tmp, u64 nrec, i64 ncols, int idx64, int base,
                     const void *colptr, void *rowval_out, double *nzval_out, void *workspace, LaunchCounter &lc,
                     StageTimer *timer)
{
    const CfLayout l = cf_layout(nrec, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    const u32 *nzcol = reinterpret_cast<const u32 *>(ws + l.off_nzcol);
    const u32 *nzstart = reinterpret_cast<const u32 *>(ws + l.off_nzstart);
    const u64 *totals = reinterpret_cast<const u64 *>(ws + l.off_tot);
    const u64 kmax = std::min<u64>((u64)ncols, nrec);
    if (timer)
        timer->begin(stream);
    const unsigned blocks = (unsigned)std::min<u64>(std::max<u64>((kmax * 16 + 255) / 256, 1), (u64)kNumSM * 32);
    if (idx64)
        compact_entries_kernel<int64_t><<<blocks, 256, 0, stream>>>(tmp, nzcol, nzstart, totals, (const int64_t *)colptr,
                                                                    (int64_t)base, (int64_t *)rowval_out, nzval_out);
    else
        compact_entries_kernel<int32_t><<<blocks, 256, 0, stream>>>(tmp, nzcol, nzstart, totals, (const int32_t *)colptr,
                                                                    (int32_t)base, (int32_t *)rowval_out, nzval_out);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::compact);
}

} // namespace xsb
