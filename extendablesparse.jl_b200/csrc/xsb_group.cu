// xsb_group.cu -- stable grouping of the staged records by column in TWO passes over the data,
// for insertion streams with column locality (FEM / FD / FV assembly: consecutive insertions
// touch few distinct columns).  A counting sort with 2^colbits bins whose per-chunk histograms
// are stored sparsely:
//
//   group_count_kernel   : a warp owns a chunk of GP_W consecutive records.  It finds the chunk's
//                          distinct columns with a shared-memory hash table and counts the records
//                          of each; the (column, chunk, count) pairs of all chunks are appended to
//                          one list (one atomic per chunk: no ordering between chunks is needed).
//   radix sort of the PAIRS by (column, chunk) (xsb_sort.cu): pairs of one column end up in chunk
//                          = stream order.  There are 4-12x fewer pairs than records.
//   pair_scan kernels    : exclusive sum of the counts in sorted order = where the records of
//                          (column, chunk) start in the output; column heads give the compact
//                          column list (nzcol, nzstart) the per-column kernels need.
//   group_scatter_kernel : the warp re-reads its chunk, ranks every record among the chunk's
//                          records of its column in stream order (warp match) and stores it.
//
// Against three onesweep passes (96 B of HBM traffic per record + the histogram read) this moves
// 48 B per record plus the pair traffic.  A stream without locality (about one pair per record)
// is detected after the counting pass; the caller then uses the plain radix sort.
//
// Reference counterpart: the per-column gather of Base.:+(lnk,csc), src/matrix/sparsematrixlnk.jl:330-338
// (the linked lists ARE the columns there); stdlib sparse! counting sort reached from
// src/matrix/sparsematrixdilnkc.jl:428-432.
#include "xsb_internal.h"
#include "xsb_group_count.cuh"

namespace xsb {

__global__ void __launch_bounds__(GP_WARPS * 32, 5)
group_count_kernel(const Rec *__restrict__ in, u64 nrec, int ownershift, u32 me, u32 nchunks, CountTarget ct)
{
    const int colshift = ct.colshift;
    const u32 colmask = ct.colmask;
    constexpr u32 full = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    CountSpace &ws = reinterpret_cast<CountSpace *>(smem_raw)[warp];
    const u32 chunk = blockIdx.x * GP_WARPS + warp;
    if (chunk >= nchunks)
        return;
    const u32 lt = lanemask_lt();
    const u64 r0 = (u64)chunk * GP_W;
    const u32 cnt_here = (u32)min((u64)GP_W, nrec - r0);

    count_space_init(ws, lane);

    u32 d = 0;
    bool crowded = false;
    const Rec *rec = in + r0 + lane;
    if (cnt_here == (u32)GP_W && ownershift < 0)
    { // whole chunk, every record takes part: no validity bookkeeping
        u64 key[4], nkey[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            nkey[i] = rec[i * 32].key;
#pragma unroll 1
        for (int g = 0; g < GP_NB && !crowded; g += 4)
        {
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                key[i] = nkey[i];
                if (g + 4 < GP_NB) // the next group's keys travel while this one is counted
                    nkey[i] = rec[(g + 4 + i) * 32].key;
            }
            if (d > (u32)GP_DMAX - 96u)
                crowded = true; // the table may not take another 4 x 32 columns
            else
            {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    count_batch<true>(ws, key[i], true, colshift, colmask, lt, d);
            }
        }
    }
    else
    {
        u64 key[4], nkey[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            const u32 p = i * 32 + lane;
            nkey[i] = p < cnt_here ? rec[i * 32].key : 0ull;
        }
#pragma unroll 1
        for (int g = 0; g < GP_NB && !crowded; g += 4)
        {
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                key[i] = nkey[i];
                const u32 p = (g + 4 + i) * 32 + lane;
                nkey[i] = p < cnt_here ? rec[(g + 4 + i) * 32].key : 0ull;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                const u32 bb = (g + i) * 32;
                if (bb < cnt_here && !crowded) // warp-uniform
                {
                    if (d > (u32)GP_DMAX)
                        crowded = true; // the table may not take another 32 columns
                    else
                    { // records owned by another rank (slab handles: already sent) do not take part
                        const bool valid =
                            bb + lane < cnt_here && (ownershift < 0 || (u32)(key[i] >> ownershift) == me);
                        count_batch<false>(ws, key[i], valid, colshift, colmask, lt, d);
                    }
                }
            }
        }
    }
    (void)full;
    __syncwarp();

    count_publish(ws, ct, chunk, d, crowded, lane);
}

// ------------------------------------------------------------------------
// pair list into chunk order: exclusive scan of the chunks' pair counts, then a copy
// ------------------------------------------------------------------------
constexpr int PO_THREADS = 256; // chunks per block

// Order in which the chunks' pairs are listed = order in which the fold meets the records of a
// column.  Physically a slab handle's buffer holds [old CSC | own | received from lower ranks |
// received from higher ranks] (each region a whole number of chunks); the fold must see
// [old | lower ranks | own | higher ranks]: the rank-ordered concatenation of the ranks' streams.
__device__ __forceinline__ u32 chunk_at(const ChunkOrder &o, u32 v)
{
    const u32 nl = o.c_low - o.c_own, no = o.c_own - o.c_old;
    if (v < o.c_old || v >= o.c_low)
        return v;
    if (v < o.c_old + nl)
        return o.c_own + (v - o.c_old);
    return o.c_old + (v - o.c_old - nl);
    (void)no;
}

__global__ void __launch_bounds__(PO_THREADS)
pair_order_tilesum_kernel(const uint2 *__restrict__ chunkinfo, u32 nchunks, ChunkOrder ord, u32 *__restrict__ tsum)
{
    __shared__ u32 s_w[PO_THREADS / 32];
    const u32 c = blockIdx.x * PO_THREADS + threadIdx.x;
    u32 v = c < nchunks ? chunkinfo[chunk_at(ord, c)].y : 0u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0)
        s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        u32 t = 0;
        for (int w = 0; w < PO_THREADS / 32; ++w)
            t += s_w[w];
        tsum[blockIdx.x] = t;
    }
}

// single block: exclusive scan of the tile sums in place
__global__ void __launch_bounds__(1024) pair_order_scan_kernel(u32 *__restrict__ tsum, u32 nt)
{
    __shared__ u32 s_w[32];
    __shared__ u32 s_carry;
    if (threadIdx.x == 0)
        s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (u32 b0 = 0; b0 < nt; b0 += 1024)
    {
        const u32 j = b0 + threadIdx.x;
        const u32 x = j < nt ? tsum[j] : 0u;
        u32 v = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o)
                v += t;
        }
        if (lane == 31)
            s_w[warp] = v;
        __syncthreads();
        u32 pre = s_carry;
        for (int w = 0; w < warp; ++w)
            pre += s_w[w];
        if (j < nt)
            tsum[j] = pre + v - x;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = pre + v;
        __syncthreads();
    }
}

// block = 256 chunks: in-block scan of the pair counts, then every warp copies the pairs of its 32
// chunks from their ticket position to their position in chunk order
__global__ void __launch_bounds__(PO_THREADS)
pair_order_kernel(const uint2 *__restrict__ chunkinfo, u32 nchunks, ChunkOrder ord, const u32 *__restrict__ tsum,
                  const Rec *__restrict__ pairs_in, Rec *__restrict__ pairs_out)
{
    __shared__ u32 s_w[PO_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 c = blockIdx.x * PO_THREADS + threadIdx.x;
    const uint2 info = c < nchunks ? chunkinfo[chunk_at(ord, c)] : make_uint2(0u, 0u);
    u32 incl = info.y;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_w[warp] = incl;
    __syncthreads();
    u32 dst = tsum[blockIdx.x] + incl - info.y;
    for (int w = 0; w < warp; ++w)
        dst += s_w[w];
    for (int q = 0; q < 32; ++q)
    { // chunk of lane q, all lanes copy
        const u32 src = __shfl_sync(0xffffffffu, info.x, q);
        const u32 cnt = __shfl_sync(0xffffffffu, info.y, q);
        const u32 to = __shfl_sync(0xffffffffu, dst, q);
        for (u32 j = lane; j < cnt; j += 32)
            pairs_out[to + j] = pairs_in[src + j];
    }
}

// ------------------------------------------------------------------------
// sorted pairs -> output offset of every (chunk, column) + compact column list
// ------------------------------------------------------------------------
constexpr int PS_THREADS = 256;
constexpr int PS_IPT = 8;
constexpr int PS_TILE = PS_THREADS * PS_IPT;

__device__ __forceinline__ u64 pair_payload(const Rec &r) { return (u64)__double_as_longlong(r.val); }

__global__ void __launch_bounds__(PS_THREADS)
pair_tilesum_kernel(const Rec *__restrict__ sp, u32 npairs, u64 *__restrict__ trec,
                    u32 *__restrict__ tnz)
{
    __shared__ u64 s_w[PS_THREADS / 32];
    const u32 b0 = blockIdx.x * PS_TILE;
    u64 rec = 0, heads = 0;
#pragma unroll
    for (int i = 0; i < PS_IPT; ++i)
    {
        const u32 j = b0 + i * PS_THREADS + threadIdx.x;
        if (j < npairs)
        {
            const Rec r = sp[j];
            rec += pair_payload(r) & 0xffffull;
            heads += (j == 0 || sp[j - 1].key != r.key) ? 1 : 0;
        }
    }
    // packed: records << 24 | heads (a tile holds at most 2048 heads)
    u64 s = (rec << 24) | heads;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0)
        s_w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        for (int w = 1; w < PS_THREADS / 32; ++w)
            s += s_w[w];
        trec[blockIdx.x] = s >> 24;
        tnz[blockIdx.x] = (u32)(s & 0xffffffull);
    }
}

__global__ void __launch_bounds__(PS_THREADS)
pair_emit_kernel(const Rec *__restrict__ sp, u32 npairs, const u64 *__restrict__ trec,
                 const u32 *__restrict__ tnz, u32 *__restrict__ offs, u32 *__restrict__ nzcol,
                 u32 *__restrict__ nzstart)
{
    __shared__ u64 s_w[PS_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 b0 = blockIdx.x * PS_TILE + threadIdx.x * PS_IPT; // blocked: thread owns PS_IPT consecutive pairs
    u32 cnt[PS_IPT], col[PS_IPT], tidx[PS_IPT];
    bool head[PS_IPT];
    u64 sum = 0;
    u32 prevcol = (b0 > 0 && b0 <= npairs) ? (u32)sp[b0 - 1].key : 0xffffffffu;
#pragma unroll
    for (int i = 0; i < PS_IPT; ++i)
    {
        const u32 j = b0 + i;
        cnt[i] = 0;
        col[i] = 0;
        tidx[i] = 0;
        head[i] = false;
        if (j < npairs)
        {
            const Rec r = sp[j];
            const u64 pl = pair_payload(r);
            cnt[i] = (u32)(pl & 0xffffull);
            tidx[i] = (u32)(pl >> 16);
            col[i] = (u32)r.key;
            head[i] = j == 0 || col[i] != prevcol;
            prevcol = col[i];
        }
        sum += ((u64)cnt[i] << 24) | (u64)(head[i] ? 1 : 0);
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
    for (int i = 0; i < PS_IPT; ++i)
    {
        if (b0 + i < npairs)
        {
            if (head[i])
            {
                nzcol[k] = col[i];
                nzstart[k] = (u32)rec;
                ++k;
            }
            offs[tidx[i]] = (u32)rec;
            rec += cnt[i];
        }
    }
}

// ------------------------------------------------------------------------
// Bucketed pair path: the pairs are NOT sorted.  The counting pass left, per column, its records and
// its pairs (colrec / colpairs, CountTarget).  A scan over the columns gives every column its bucket
// in a pair-sized array and its place in the output; the pairs are dropped into their column's
// bucket (atomic cursor), each bucket -- about a handful of pairs -- is put into chunk order by the
// thread that owns the column, and a running sum over it gives the output offset of every
// (chunk, column).  Against the radix sort of the pairs (3 passes of 32 B per pair + pair_order):
// two reads and one write of 8-byte bucket entries.
// ------------------------------------------------------------------------
constexpr int PB_TILE = 2048; // columns per tile of the per-column scan
constexpr int PB_THREADS = 256;
constexpr int PB_IPT = PB_TILE / PB_THREADS;

// per column: its records and its pairs (L2-resident arrays, one atomic each per pair)
__global__ void __launch_bounds__(256)
pair_totals_kernel(const u32 *__restrict__ pair_total, u32 cap, const u32 *__restrict__ chunkcols,
                   const unsigned short *__restrict__ chunkcnt, u32 *__restrict__ colrec, u32 *__restrict__ colpairs,
                   u32 *__restrict__ flags, u32 ncols)
{
    if (*flags & 1u) // a chunk gave up (no column locality): the pair list has holes and is not used
        return;
    const u32 np = min(*pair_total, cap);
    const u32 stride = gridDim.x * blockDim.x;
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < np; p += stride)
    {
        const u32 col = chunkcols[p];
        if (col >= ncols)
            continue;
        atomicAdd(colrec + col, (u32)chunkcnt[p]);
        if (atomicAdd(colpairs + col, 1u) >= kMaxColPairs)
            atomicOr(flags, 2u); // its pairs are ordered by the radix sort, not inside one thread
    }
}

// tile sums: a = records, b = pairs << 32 | non-empty columns
__global__ void __launch_bounds__(PB_THREADS)
colpair_tilesum_kernel(const u32 *__restrict__ colrec, const u32 *__restrict__ colpairs, i64 n, u64 *__restrict__ ta,
                       u64 *__restrict__ tb)
{
    __shared__ u64 s_a[PB_THREADS / 32], s_b[PB_THREADS / 32];
    const i64 b0 = (i64)blockIdx.x * PB_TILE;
    u64 a = 0, b = 0;
#pragma unroll
    for (int i = 0; i < PB_IPT; ++i)
    {
        const i64 j = b0 + i * PB_THREADS + threadIdx.x;
        if (j < n)
        {
            const u32 np = colpairs[j];
            a += colrec[j];
            b += ((u64)np << 32) | (u64)(np != 0u);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
    {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if ((threadIdx.x & 31) == 0)
    {
        s_a[threadIdx.x >> 5] = a;
        s_b[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        for (int w = 1; w < PB_THREADS / 32; ++w)
        {
            a += s_a[w];
            b += s_b[w];
        }
        ta[blockIdx.x] = a;
        tb[blockIdx.x] = b;
    }
}

// single block: exclusive scan of both tile sums in place; totals[0] = records, totals[1] = K (non-empty columns)
__global__ void __launch_bounds__(1024)
colpair_scan_kernel(u64 *__restrict__ ta, u64 *__restrict__ tb, i64 nt, u64 *__restrict__ totals, u32 *__restrict__ nzstart)
{
    __shared__ u64 s_wa[32], s_wb[32];
    __shared__ u64 s_ca, s_cb;
    if (threadIdx.x == 0)
    {
        s_ca = 0;
        s_cb = 0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (i64 b0 = 0; b0 < nt; b0 += 1024)
    {
        const i64 j = b0 + threadIdx.x;
        const u64 xa = j < nt ? ta[j] : 0ull, xb = j < nt ? tb[j] : 0ull;
        u64 va = xa, vb = xb;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 pa = __shfl_up_sync(0xffffffffu, va, o);
            const u64 pb = __shfl_up_sync(0xffffffffu, vb, o);
            if (lane >= o)
            {
                va += pa;
                vb += pb;
            }
        }
        if (lane == 31)
        {
            s_wa[warp] = va;
            s_wb[warp] = vb;
        }
        __syncthreads();
        u64 pa = s_ca, pb = s_cb;
        for (int w = 0; w < warp; ++w)
        {
            pa += s_wa[w];
            pb += s_wb[w];
        }
        if (j < nt)
        {
            ta[j] = pa + va - xa;
            tb[j] = pb + vb - xb;
        }
        __syncthreads();
        if (threadIdx.x == 1023)
        {
            s_ca = pa + va;
            s_cb = pb + vb;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0)
    {
        totals[0] = s_ca;
        totals[1] = s_cb & 0xffffffffull;
        nzstart[s_cb & 0xffffffffull] = (u32)s_ca; // sentinel: one past the last record
    }
}

// per column: pstart[col] = first slot of its bucket; per non-empty column k: nzcol[k], nzstart[k]
__global__ void __launch_bounds__(PB_THREADS)
colpair_emit_kernel(const u32 *__restrict__ colrec, const u32 *__restrict__ colpairs, const u64 *__restrict__ ta,
                    const u64 *__restrict__ tb, i64 n, u32 *__restrict__ pstart, u32 *__restrict__ nzcol,
                    u32 *__restrict__ nzstart)
{
    __shared__ u64 s_a[PB_THREADS / 32], s_b[PB_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 b0 = (i64)blockIdx.x * PB_TILE + (i64)threadIdx.x * PB_IPT; // blocked: a thread owns PB_IPT columns
    u32 rc[PB_IPT], np[PB_IPT];
    u64 sa = 0, sb = 0;
#pragma unroll
    for (int i = 0; i < PB_IPT; ++i)
    {
        const i64 j = b0 + i;
        rc[i] = j < n ? colrec[j] : 0u;
        np[i] = j < n ? colpairs[j] : 0u;
        sa += rc[i];
        sb += ((u64)np[i] << 32) | (u64)(np[i] != 0u);
    }
    u64 ia = sa, ib = sb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 pa = __shfl_up_sync(0xffffffffu, ia, o);
        const u64 pb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o)
        {
            ia += pa;
            ib += pb;
        }
    }
    if (lane == 31)
    {
        s_a[warp] = ia;
        s_b[warp] = ib;
    }
    __syncthreads();
    u64 ra = ia - sa, rb = ib - sb;
    for (int w = 0; w < warp; ++w)
    {
        ra += s_a[w];
        rb += s_b[w];
    }
    u64 rec = ta[blockIdx.x] + ra;
    const u64 bb = tb[blockIdx.x] + rb;
    u32 slot = (u32)(bb >> 32), k = (u32)(bb & 0xffffffffull);
#pragma unroll
    for (int i = 0; i < PB_IPT; ++i)
    {
        if (b0 + i < n)
            pstart[b0 + i] = slot;
        if (np[i])
        {
            nzcol[k] = (u32)(b0 + i);
            nzstart[k] = (u32)rec;
            ++k;
        }
        slot += np[i];
        rec += rc[i];
    }
}

// position of a chunk in the order the fold meets the chunks (inverse of chunk_at)
__device__ __forceinline__ u32 chunk_pos(const ChunkOrder &o, u32 c)
{
    if (c < o.c_old || c >= o.c_low)
        return c;
    if (c >= o.c_own)                     // region of the lower ranks: met right after the old entries
        return o.c_old + (c - o.c_own);
    return c + (o.c_low - o.c_own);       // own region: met after the lower ranks'
}

// bucket entry: [chunk position : 23][pair (ticket) index : 31][records - 1 : 9]
static_assert(GP_W <= 512, "a bucket entry keeps 9 bits for the records of a (chunk, column) pair");
__device__ __forceinline__ u64 pb_entry(u32 pos, u32 pair, u32 cnt) { return ((u64)pos << 40) | ((u64)pair << 9) | (u64)(cnt - 1u); }

// a warp per chunk: its pairs go into their columns' buckets
__global__ void __launch_bounds__(256)
pair_bucket_kernel(const uint2 *__restrict__ chunkinfo, u32 nchunks, ChunkOrder ord, const u32 *__restrict__ chunkcols,
                   const unsigned short *__restrict__ chunkcnt, const u32 *__restrict__ pstart,
                   u32 *__restrict__ pcursor, u64 *__restrict__ bucket)
{
    const int lane = threadIdx.x & 31;
    const u32 c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c >= nchunks)
        return;
    const uint2 info = chunkinfo[c];
    const u32 pos = chunk_pos(ord, c);
    for (u32 j = lane; j < info.y; j += 32)
    {
        const u32 p = info.x + j;
        const u32 col = chunkcols[p];
        const u32 slot = pstart[col] + atomicAdd(pcursor + col, 1u);
        bucket[slot] = pb_entry(pos, p, (u32)chunkcnt[p]);
    }
}

// a thread per non-empty column: bucket into chunk order (insertion sort in place: the entries arrive
// nearly in order), then offs[pair] = where the records of that (chunk, column) start in the output
__global__ void __launch_bounds__(256)
pair_offsets_kernel(const u32 *__restrict__ nzcol, const u32 *__restrict__ nzstart, const u64 *__restrict__ totals,
                    const u32 *__restrict__ pstart, const u32 *__restrict__ colpairs, u64 *__restrict__ bucket,
                    u32 *__restrict__ offs)
{
    const u64 K = totals[1];
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K)
        return;
    const u32 col = nzcol[k];
    u64 *b = bucket + pstart[col];
    const u32 np = colpairs[col];
    u32 run = nzstart[k];
    u64 prev = b[0];
    for (u32 i = 1; i < np; ++i)
    {
        const u64 e = b[i];
        if (e < prev)
        { // out of order: insert (prev stays the largest entry so far, now at b[i])
            u32 q = i;
            while (q > 0 && b[q - 1] > e)
            {
                b[q] = b[q - 1];
                --q;
            }
            b[q] = e;
        }
        else
            prev = e;
    }
    for (u32 i = 0; i < np; ++i)
    {
        const u64 e = b[i];
        offs[(u32)(e >> 9) & 0x7fffffffu] = run;
        run += (u32)(e & 0x1ffull) + 1u;
    }
}

// ------------------------------------------------------------------------
// pass 2: stable scatter
// ------------------------------------------------------------------------
struct ScatterSpace
{
    u32 key[GP_H];
    u32 cur[GP_H];
};

__global__ void __launch_bounds__(GP_WARPS * 32, 5)
group_scatter_kernel(const Rec *__restrict__ in, u64 nrec, int colshift, u32 colmask, int ownershift, u32 me,
                     u32 nchunks,
                     const u32 *__restrict__ chunkcols, const uint2 *__restrict__ chunkinfo,
                     const u32 *__restrict__ offs, Rec *__restrict__ out)
{
    constexpr u32 full = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ScatterSpace &ws = reinterpret_cast<ScatterSpace *>(smem_raw)[warp];
    const u32 chunk = blockIdx.x * GP_WARPS + warp;
    if (chunk >= nchunks)
        return;
    const u32 lt = lanemask_lt();
    const u64 r0 = (u64)chunk * GP_W;
    const u32 cnt_here = (u32)min((u64)GP_W, nrec - r0);
    const uint2 info = chunkinfo[chunk];
    const u32 base = info.x, d = info.y;
    {
        uint4 *kq = reinterpret_cast<uint4 *>(ws.key);
#pragma unroll
        for (int i = 0; i < GP_H / 128; ++i)
            kq[i * 32 + lane] = make_uint4(GP_EMPTY, GP_EMPTY, GP_EMPTY, GP_EMPTY);
    }
    __syncwarp();
    // the chunk's columns (all distinct) and where their records go
    for (u32 j = lane; j < d; j += 32)
    {
        const u32 col = chunkcols[base + j];
        const u32 o = offs[base + j];
        u32 slot = gp_hash(col);
        while (atomicCAS(&ws.key[slot], GP_EMPTY, col) != GP_EMPTY)
            slot = (slot + 1) & (GP_H - 1);
        ws.cur[slot] = o;
    }
    __syncwarp();
    Rec nxt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
    {
        const u32 p = i * 32 + lane;
        if (p < cnt_here)
            nxt[i] = ld_rec_stream(in + r0 + p);
        else
        {
            nxt[i].key = 0;
            nxt[i].val = 0.0;
        }
    }
#pragma unroll 1
    for (int g = 0; g < GP_NB; g += 4)
    {
        Rec r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            r[i] = nxt[i];
            const u32 p = (g + 4 + i) * 32 + lane; // the next group travels while this one is ranked
            if (p < cnt_here)
                nxt[i] = ld_rec_stream(in + r0 + p);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            const u32 bb = (g + i) * 32;
            if (bb < cnt_here) // warp-uniform
            {
                const bool valid = bb + lane < cnt_here && (ownershift < 0 || (u32)(r[i].key >> ownershift) == me);
                const u32 col = (u32)(r[i].key >> colshift) & colmask;
                const u32 vm = __ballot_sync(full, valid);
                u32 peers = 1u << lane;
                if (valid)
                    peers = __match_any_sync(vm, col);
                const int ldr = __ffs(peers) - 1;
                u32 b = 0;
                if (valid && lane == ldr)
                { // one lane per distinct column looks it up and advances its cursor
                    u32 slot = gp_hash(col);
                    while (ws.key[slot] != col)
                        slot = (slot + 1) & (GP_H - 1);
                    b = ws.cur[slot];
                    ws.cur[slot] = b + (u32)__popc(peers);
                }
                __syncwarp();
                b = __shfl_sync(full, b, ldr);
                if (valid)
                    st_rec(out + (b + __popc(peers & lt)), r[i]);
            }
        }
    }
}

// ------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------
namespace {
struct GpLayout
{
    size_t off_ticket, off_chunkinfo, off_chunkcols, off_offs, off_trec, off_tnz, off_status, bytes;
    size_t off_colrec, off_colpairs, off_pstart, off_pcursor, off_chunkcnt, off_ta, off_tb;
    u32 cap;
};
GpLayout gp_layout(u64 nrec, i64 ncols)
{
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const u64 nchunks = (nrec + GP_W - 1) / GP_W;
    GpLayout l{};
    l.cap = (u32)std::min<u64>(nrec / 8 * 3 + 4096, 0xfffffff0ull); // pairs we make room for (7-point FD streams: ~0.27 per record)
    const u64 ptiles = ((u64)l.cap + PS_TILE - 1) / PS_TILE;
    const u64 ctiles = ((u64)ncols + PB_TILE - 1) / PB_TILE;
    size_t o = 0;
    l.off_ticket = o;
    o = up(o + 256);
    // per-column totals right behind the ticket: one memset clears ticket, flags, colrec, colpairs and pcursor
    l.off_colrec = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_colpairs = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_pcursor = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_pstart = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_chunkinfo = o;
    o = up(o + sizeof(uint2) * (nchunks + 1));
    l.off_chunkcols = o;
    o = up(o + sizeof(u32) * ((size_t)l.cap + 1));
    l.off_chunkcnt = o;
    o = up(o + sizeof(unsigned short) * ((size_t)l.cap + 1));
    l.off_offs = o;
    o = up(o + sizeof(u32) * ((size_t)l.cap + 1));
    l.off_trec = o;
    o = up(o + sizeof(u64) * (ptiles + 1));
    l.off_tnz = o;
    o = up(o + sizeof(u32) * (ptiles + 1));
    l.off_ta = o;
    o = up(o + sizeof(u64) * (ctiles + 1));
    l.off_tb = o;
    o = up(o + sizeof(u64) * (ctiles + 1));
    l.off_status = o; // tile sums of the chunks' pair counts (pair_order kernels)
    o = up(o + sizeof(u32) * (nchunks / 256 + 2));
    l.bytes = o;
    return l;
}
} // namespace

size_t group_workspace_bytes(u64 nrec, i64 ncols) { return gp_layout(nrec, ncols).bytes; }
int group_chunk_records() { return GP_W; }

bool group_supported(const KeyLayout &L, u64 nrec, i64 ncols)
{
    return L.colbits <= 32 && L.colbits + 23 <= 8 * kMaxPasses && nrec >= 32768 && nrec < (1ull << 32) - (u64)GP_W && (u64)ncols < (1ull << 32) - 1ull;
}

// colscan_scan_kernel of xsb_colfold.cu (exclusive scan of the tile sums; totals; nzstart sentinel)
void colscan_scan_launch(cudaStream_t stream, u64 *trec, u32 *tnz, i64 nt, u64 *totals, u32 *nzstart);

// Groups `in` (nrec records) by column into `out`, stable.  `out` doubles as scratch for the pair
// sort before the scatter.  On success nzcol / nzstart / totals (workspace of xsb_colfold.cu) hold
// the compact column list.  Returns false -- with `in` untouched and `out` undefined -- when the
// stream has too many (chunk, column) pairs for this to pay off.

bool group_by_column(cudaStream_t stream, const Rec *in, Rec *out, u64 nrec, i64 ncols, const KeyLayout &L, void *workspace,
                     void *sort_workspace, u32 *nzcol, u32 *nzstart, u64 *totals, u64 *h_scal_pinned, LaunchCounter &lc,
                     StageTimer *timer, int *pair_passes, u64 *npairs_out, int ownershift, u32 me, const ChunkOrder *order)
{
    const GpLayout l = gp_layout(nrec, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *pair_total = reinterpret_cast<u32 *>(ws + l.off_ticket);
    u32 *flags = pair_total + 1;
    uint2 *chunkinfo = reinterpret_cast<uint2 *>(ws + l.off_chunkinfo);
    u32 *chunkcols = reinterpret_cast<u32 *>(ws + l.off_chunkcols);
    u32 *offs = reinterpret_cast<u32 *>(ws + l.off_offs);
    u64 *trec = reinterpret_cast<u64 *>(ws + l.off_trec);
    u32 *tnz = reinterpret_cast<u32 *>(ws + l.off_tnz);
    const u32 nchunks = (u32)((nrec + GP_W - 1) / GP_W);
    const int colshift = L.low + L.rowbits;
    const u32 colmask = L.colbits >= 32 ? 0xffffffffu : ((1u << L.colbits) - 1u);
    u32 *colrec = reinterpret_cast<u32 *>(ws + l.off_colrec);
    u32 *colpairs = reinterpret_cast<u32 *>(ws + l.off_colpairs);
    u32 *pcursor = reinterpret_cast<u32 *>(ws + l.off_pcursor);
    u32 *pstart = reinterpret_cast<u32 *>(ws + l.off_pstart);
    unsigned short *chunkcnt = reinterpret_cast<unsigned short *>(ws + l.off_chunkcnt);
    u64 *ta = reinterpret_cast<u64 *>(ws + l.off_ta);
    u64 *tb = reinterpret_cast<u64 *>(ws + l.off_tb);
    static FuncAttrOnce once[2];
    once[0].set(group_count_kernel, (int)(sizeof(CountSpace) * GP_WARPS));
    once[1].set(group_scatter_kernel, (int)(sizeof(ScatterSpace) * GP_WARPS));
    Rec *pairs_a = out;
    Rec *pairs_b = out + l.cap;

    // ---- pass 1
    if (timer)
        timer->begin(stream);
    XSB_CUDA(cudaMemsetAsync(ws + l.off_ticket, 0, 256, stream)); // pair ticket, flags
    // The bucketed pair path works on per-column arrays (12 bytes cleared + 12 bytes scanned per column and
    // flush); for a hypersparse flush (far more columns than records) the radix sort of the pairs is cheaper.
    const bool try_buckets = (u64)ncols <= 8ull * nrec;
    if (try_buckets) // per-column totals and bucket cursors
        XSB_CUDA(cudaMemsetAsync(ws + l.off_colrec, 0, l.off_pstart - l.off_colrec, stream));
    {
        CountTarget ct{pair_total, flags, pairs_b, chunkcols, chunkinfo, l.cap, colshift, colmask, chunkcnt};
        const unsigned cblocks = (nchunks + GP_WARPS - 1) / GP_WARPS;
        group_count_kernel<<<cblocks, GP_WARPS * 32, sizeof(CountSpace) * GP_WARPS, stream>>>(in, nrec, ownershift, me,
                                                                                              nchunks, ct);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    if (try_buckets)
    { // records and pairs per column (sizes of the buckets), "a column is met by very many chunks" flag
        pair_totals_kernel<<<kNumSM * 8, 256, 0, stream>>>(pair_total, l.cap, chunkcols, chunkcnt, colrec, colpairs, flags,
                                                           (u32)ncols);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    // pairs made, too-many flag
    XSB_CUDA(cudaMemcpyAsync(h_scal_pinned, pair_total, sizeof(u32), cudaMemcpyDeviceToHost, stream));
    XSB_CUDA(cudaMemcpyAsync(h_scal_pinned + 1, flags, sizeof(u32), cudaMemcpyDeviceToHost, stream));
    if (timer)
        timer->end(stream, &StageTimes::gcount);
    XSB_CUDA(cudaStreamSynchronize(stream));
    const u32 npairs = (u32)(h_scal_pinned[0] & 0xffffffffull);
    const u32 fl = (u32)(h_scal_pinned[1] & 0xffffffffull);
    const bool toomany = (fl & 1u) != 0u;
    const bool longcol = (fl & 2u) != 0u; // some column is met by more than kMaxColPairs chunks
    *npairs_out = npairs;
    if (toomany || npairs > l.cap || npairs == 0)
        return false;
    ChunkOrder ord = order ? *order : ChunkOrder{nchunks, nchunks, nchunks};

    if (!longcol && try_buckets)
    { // ---- bucketed pair path: no sort (see above)
        if (timer)
            timer->begin(stream);
        const unsigned ctiles = (unsigned)(((u64)ncols + PB_TILE - 1) / PB_TILE);
        u64 *bucket = reinterpret_cast<u64 *>(out);
        colpair_tilesum_kernel<<<ctiles, PB_THREADS, 0, stream>>>(colrec, colpairs, ncols, ta, tb);
        colpair_scan_kernel<<<1, 1024, 0, stream>>>(ta, tb, (i64)ctiles, totals, nzstart);
        colpair_emit_kernel<<<ctiles, PB_THREADS, 0, stream>>>(colrec, colpairs, ta, tb, ncols, pstart, nzcol, nzstart);
        pair_bucket_kernel<<<(nchunks + 7) / 8, 256, 0, stream>>>(chunkinfo, nchunks, ord, chunkcols, chunkcnt, pstart,
                                                                  pcursor, bucket);
        const u64 kmax = std::min<u64>((u64)ncols, (u64)npairs);
        pair_offsets_kernel<<<(unsigned)((kmax + 255) / 256), 256, 0, stream>>>(nzcol, nzstart, totals, pstart, colpairs,
                                                                                 bucket, offs);
        lc.add(5);
        XSB_CUDA(cudaGetLastError());
        *pair_passes = 0;
        if (timer)
            timer->end(stream, &StageTimes::sort);
        if (timer)
            timer->begin(stream);
    }
    else
    {
        // ---- pairs into chunk order, then sorted by column (stable: chunk order inside a column)
        if (timer)
            timer->begin(stream);
        {
            u32 *otsum = reinterpret_cast<u32 *>(ws + l.off_status);
            const unsigned oblocks = (nchunks + PO_THREADS - 1) / PO_THREADS;
            pair_order_tilesum_kernel<<<oblocks, PO_THREADS, 0, stream>>>(chunkinfo, nchunks, ord, otsum);
            pair_order_scan_kernel<<<1, 1024, 0, stream>>>(otsum, oblocks);
            pair_order_kernel<<<oblocks, PO_THREADS, 0, stream>>>(chunkinfo, nchunks, ord, otsum, pairs_b, pairs_a);
            lc.add(3);
            XSB_CUDA(cudaGetLastError());
        }
        if (timer)
            timer->end(stream, &StageTimes::sort);
        const SortPlan plan = make_sort_plan(0, L.colbits);
        *pair_passes = plan.npasses;
        Rec *sp = radix_sort_records(stream, pairs_a, pairs_b, npairs, plan, sort_workspace, lc, timer);

        // ---- offsets + column list
        if (timer)
            timer->begin(stream);
        const unsigned ptiles = (npairs + PS_TILE - 1) / PS_TILE;
        pair_tilesum_kernel<<<ptiles, PS_THREADS, 0, stream>>>(sp, npairs, trec, tnz);
        colscan_scan_launch(stream, trec, tnz, (i64)ptiles, totals, nzstart);
        pair_emit_kernel<<<ptiles, PS_THREADS, 0, stream>>>(sp, npairs, trec, tnz, offs, nzcol, nzstart);
        lc.add(3);
        XSB_CUDA(cudaGetLastError());
    }
    // ---- pass 2
    const unsigned sblocks = (nchunks + GP_WARPS - 1) / GP_WARPS;
    group_scatter_kernel<<<sblocks, GP_WARPS * 32, sizeof(ScatterSpace) * GP_WARPS, stream>>>(
        in, nrec, colshift, colmask, ownershift, me, nchunks, chunkcols, chunkinfo, offs, out);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::gscatter);
    return true;
}

} // namespace xsb
