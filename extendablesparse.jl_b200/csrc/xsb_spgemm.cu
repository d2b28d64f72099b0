// xsb_spgemm.cu -- C = A * B of two resident CSCs, SparseArrays' spmatmul bit for bit.
//
// spcolmul! builds column j of C by walking B[:, j]'s entries (k, b) in stored order and, for each, A[:, k]'s
// entries (i, a): the first product a * b of row i is assigned, every later one added (acc = acc + p).  So an
// entry of C is the left fold in ascending k of separately rounded products, and the pattern is the structural
// union (explicit zeros create entries).  The products are never written to memory:
//   classify  a warp per column of B: f(j) = products of column j (64 bits) and the row span they touch; the
//             column goes to the first warp-table bin whose table holds f(j) entries, else it is cut into row
//             tiles of kTile rows (pieces).  Columns without products get no work at all.
//   count     the same walks without values count the distinct rows u(j) of every column (and of every
//             piece); a scan of u gives colptr and nnz(C), which the caller reads before it allocates C.
//   write     a warp per column (or piece) walks the column's products flattened in (B position, A position)
//             order, 32 at a time.  Within such a batch a row occurs at most once per k and lane order is k
//             order: __match_any_sync groups the lanes of one row, the lowest lane of a group finds the row's
//             slot once and folds its peers' products in lane order, assigning when the row is new.  A table
//             column is then sorted by row (bitonic network in shared memory); a piece holds a dense tile and
//             reads its rows out in order.  Pieces of one column write disjoint row ranges at offsets from a
//             scan over the pieces' counts.
#include "xsb_internal.h"
#include "xsb_x86nan.cuh"

namespace xsb {
namespace {

constexpr u32 kEmpty = 0xffffffffu; // no row: rows are below m < 2^32 - 1
constexpr int kBins = 3;            // warp-table bins; bin kBins: row tiles; kBinNone: no products
constexpr u32 kBinNone = 4;
constexpr u32 kBinCap0 = 256, kBinCap1 = 1024, kBinCap2 = 4096; // table entries; f(j) <= cap
constexpr int kTile = 4096;                                      // rows of a piece's dense tile
constexpr int kTileWarps = 4;
constexpr u32 kTableMax = 4096;           // a column of u(j) <= kTableMax rows is written through a warp table
constexpr int kTableBlockSmem = 64 << 10; // shared memory of a table block: warps per block = this / warp's bytes
// counters at the head of the workspace
enum : int
{
    kCtBins = 0,     // [0, 4): columns of bins 0..2 and of the tiled bin
    kCtTiles = 4,    // pieces
    kCtNnz = 5,      // nnz(C)
    kCtCursor = 6,   // [6, 10): list fill cursors per bin
    kCtTileCur = 10, // piece fill cursor
    kCtUmax = 12,    // [12, 16): largest u(j) per bin (tiled bin: of the columns the tables write)
    kCtCount = 16
};

template <typename Ti> struct Mats
{
    const Ti *cpa, *rva;
    const double *nza;
    const Ti *cpb, *rvb;
    const double *nzb;
    Ti base;
};

template <typename Ti> Mats<Ti> mats(const Spgemm &g)
{
    return Mats<Ti>{static_cast<const Ti *>(g.a.colptr), static_cast<const Ti *>(g.a.rowval), g.a.nzval,
                    static_cast<const Ti *>(g.b.colptr), static_cast<const Ti *>(g.b.rowval), g.b.nzval,
                    (Ti)g.base};
}

// per-warp staging of one step of 32 B positions and of one batch of products
struct WarpStage
{
    i64 end[32];   // inclusive prefix of the lanes' product counts
    i64 start[32]; // first A position of each lane's k
    double bv[32]; // b of each lane's k
    double p[32];  // the batch's products
};

// Workspace over the columns of B (n = B.n): counters | bin | f (table bins) | span lo | span hi | column lists |
// u | scan sums
struct ColWs
{
    u64 *ct;
    u32 *bin, *f, *lo, *hi, *list;
    u64 *u, *bsum;
};

constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr i64 kScanTile = (i64)kScanThreads * kScanItems;
i64 scan_blocks(i64 n) { return (n + kScanTile - 1) / kScanTile; }
size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

ColWs col_ws(void *ws, i64 n)
{
    unsigned char *p = static_cast<unsigned char *>(ws);
    ColWs w;
    w.ct = reinterpret_cast<u64 *>(p);
    p += sizeof(u64) * kCtCount;
    w.bin = reinterpret_cast<u32 *>(p);
    p += align16(4 * (size_t)n);
    w.f = reinterpret_cast<u32 *>(p);
    p += align16(4 * (size_t)n);
    w.lo = reinterpret_cast<u32 *>(p);
    p += align16(4 * (size_t)n);
    w.hi = reinterpret_cast<u32 *>(p);
    p += align16(4 * (size_t)n);
    w.list = reinterpret_cast<u32 *>(p);
    p += align16(4 * (size_t)n);
    w.u = reinterpret_cast<u64 *>(p);
    p += align16(8 * (size_t)n);
    w.bsum = reinterpret_cast<u64 *>(p);
    return w;
}

// Workspace over the pieces: (column, first row, first piece of the column) | per-piece counts, then their
// exclusive scan (in place, one more entry) | scan sums
struct TileWs
{
    uint4 *piece;
    u64 *cnt, *bsum;
};

TileWs tile_ws(void *ws, u64 tiles)
{
    unsigned char *p = static_cast<unsigned char *>(ws);
    TileWs w;
    w.piece = reinterpret_cast<uint4 *>(p);
    p += sizeof(uint4) * (size_t)tiles;
    w.cnt = reinterpret_cast<u64 *>(p);
    p += align16(8 * (size_t)(tiles + 1));
    w.bsum = reinterpret_cast<u64 *>(p);
    return w;
}

// ---- classify: products f(j) and row span of every column, bin of the column
template <typename Ti>
__global__ void __launch_bounds__(256) spgemm_classify_kernel(Mats<Ti> M, i64 n, ColWs W)
{
    __shared__ u64 s_ct[kBins + 2];
    if (threadIdx.x < kBins + 2)
        s_ct[threadIdx.x] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const i64 wstride = ((i64)gridDim.x * blockDim.x) >> 5;
    for (i64 j = ((i64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += wstride)
    {
        const i64 b0 = (i64)M.cpb[j] - M.base, b1 = (i64)M.cpb[j + 1] - M.base;
        u64 f = 0;
        u32 lo = kEmpty, hi = 0;
        for (i64 q = b0 + lane; q < b1; q += 32)
        {
            const i64 k = (i64)M.rvb[q] - M.base;
            const i64 a0 = (i64)M.cpa[k] - M.base, a1 = (i64)M.cpa[k + 1] - M.base;
            if (a1 > a0)
            {
                f += (u64)(a1 - a0);
                lo = min(lo, (u32)((i64)M.rva[a0] - M.base));
                hi = max(hi, (u32)((i64)M.rva[a1 - 1] - M.base));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
        {
            f += __shfl_xor_sync(0xffffffffu, f, o);
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (lane == 0)
        {
            const u32 bin = f == 0 ? kBinNone : f <= kBinCap0 ? 0 : f <= kBinCap1 ? 1 : f <= kBinCap2 ? 2 : kBins;
            W.bin[j] = bin;
            W.f[j] = (u32)min(f, (u64)kEmpty);
            W.lo[j] = lo;
            W.hi[j] = hi;
            W.u[j] = 0;
            if (bin != kBinNone)
                atomicAdd(&s_ct[bin], 1ull);
            if (bin == kBins)
                atomicAdd(&s_ct[kBins + 1], (u64)((hi - lo) / kTile + 1));
        }
    }
    __syncthreads();
    if (threadIdx.x < kBins + 2 && s_ct[threadIdx.x])
        atomicAdd(&W.ct[kCtBins + threadIdx.x], s_ct[threadIdx.x]);
}

// ---- fill the per-bin column lists (bin b at offset binoff[b]) and the pieces
struct BinOffsets
{
    u64 off[kBins + 1];
};

__global__ void __launch_bounds__(256) spgemm_fill_kernel(i64 n, ColWs W, BinOffsets B, TileWs T)
{
    const int lane = threadIdx.x & 31;
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 j0 = (i64)blockIdx.x * blockDim.x; j0 < n; j0 += stride)
    {
        const i64 j = j0 + threadIdx.x;
        const u32 bin = j < n ? W.bin[j] : kBinNone;
#pragma unroll
        for (u32 b = 0; b <= (u32)kBins; ++b)
        { // warp-aggregated append
            const unsigned mask = __ballot_sync(0xffffffffu, bin == b);
            if (!mask)
                continue;
            const int leader = __ffs(mask) - 1;
            u64 base = 0;
            if (lane == leader)
                base = atomicAdd(&W.ct[kCtCursor + b], (u64)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (bin == b)
                W.list[B.off[b] + base + __popc(mask & ((1u << lane) - 1u))] = (u32)j;
        }
        if (bin == (u32)kBins)
        {
            const u32 lo = W.lo[j], np = (W.hi[j] - lo) / kTile + 1;
            const u64 p0 = atomicAdd(&W.ct[kCtTileCur], (u64)np);
            for (u32 t = 0; t < np; ++t)
                T.piece[p0 + t] = make_uint4((u32)j, lo + t * (u32)kTile, (u32)p0, 0);
        }
    }
}

// ---- largest u(j) per bin, over the columns a warp table writes (u(j) <= kTableMax)
__global__ void __launch_bounds__(256) spgemm_umax_kernel(i64 n, ColWs W)
{
    __shared__ unsigned long long s_max[kBins + 1];
    if (threadIdx.x <= kBins)
        s_max[threadIdx.x] = 0;
    __syncthreads();
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (i64)gridDim.x * blockDim.x)
    {
        const u32 b = W.bin[j];
        const u64 u = W.u[j];
        if (b <= (u32)kBins && u <= kTableMax)
            atomicMax(&s_max[b], u);
    }
    __syncthreads();
    if (threadIdx.x <= kBins && s_max[threadIdx.x])
        atomicMax(&W.ct[kCtUmax + threadIdx.x], s_max[threadIdx.x]);
}

// ---- the flattened walk over a column's products
// first position in [s, e) whose row is >= r (rows sorted)
template <typename Ti> __device__ __forceinline__ i64 lower_row(const Ti *rv, i64 s, i64 e, i64 r)
{
    while (s < e)
    {
        const i64 mid = s + ((e - s) >> 1);
        if ((i64)rv[mid] < r)
            s = mid + 1;
        else
            e = mid;
    }
    return s;
}

// Calls batch(active, row, product) on all lanes for every 32 products of column j in (B position, A position)
// order; RANGED: only the rows in [rlo, rhi).  !NUMERIC: product is 0.
template <typename Ti, bool NUMERIC, bool RANGED, class Batch>
__device__ __forceinline__ void walk_column(const Mats<Ti> &M, i64 j, i64 rlo, i64 rhi, WarpStage &st, Batch &&batch)
{
    const int lane = threadIdx.x & 31;
    const i64 b0 = (i64)M.cpb[j] - M.base, b1 = (i64)M.cpb[j + 1] - M.base;
    for (i64 c = b0; c < b1; c += 32)
    {
        i64 s = 0, e = 0;
        double bv = 0.0;
        if (c + lane < b1)
        {
            const i64 k = (i64)M.rvb[c + lane] - M.base;
            s = (i64)M.cpa[k] - M.base;
            e = (i64)M.cpa[k + 1] - M.base;
            if (NUMERIC)
                bv = M.nzb[c + lane];
            if (RANGED)
            {
                s = lower_row(M.rva, s, e, rlo + M.base);
                e = lower_row(M.rva, s, e, rhi + M.base);
            }
        }
        i64 incl = e - s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const i64 y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o)
                incl += y;
        }
        const i64 tot = __shfl_sync(0xffffffffu, incl, 31);
        st.end[lane] = incl;
        st.start[lane] = s;
        st.bv[lane] = bv;
        __syncwarp();
        for (i64 t0 = 0; t0 < tot; t0 += 32)
        {
            const i64 t = t0 + lane;
            const bool act = t < tot;
            u32 row = kEmpty;
            double p = 0.0;
            if (act)
            { // the lane (k) that product t belongs to: the first with end > t
                int lo = 0, hi = 31;
                while (lo < hi)
                {
                    const int mid = (lo + hi) >> 1;
                    if (st.end[mid] > t)
                        hi = mid;
                    else
                        lo = mid + 1;
                }
                const i64 q = st.start[lo] + t - (lo ? st.end[lo - 1] : 0);
                row = (u32)((i64)M.rva[q] - M.base);
                if (NUMERIC)
                    p = mul_x86(M.nza[q], st.bv[lo]);
            }
            batch(act, row, p);
        }
        __syncwarp();
    }
}

// where a row's value lives; fresh: the row was not in the table (or tile) before
struct Slot
{
    double *v;
    bool fresh;
};

// One batch of the numeric walk: the lanes of one row form a group; its lowest lane (first in k order) finds the
// row's value slot (locate(row)) and folds the group's products in lane order, assigning when fresh.
template <class Locate>
__device__ __forceinline__ void fold_batch(bool act, u32 row, double p, WarpStage &st, Locate &&locate)
{
    const int lane = threadIdx.x & 31;
    const unsigned grp = __match_any_sync(0xffffffffu, act ? row : kEmpty);
    st.p[lane] = p;
    __syncwarp();
    if (act && (grp & ((1u << lane) - 1u)) == 0u)
    {
        const Slot sl = locate(row);
        double acc = sl.fresh ? p : apply<kAlgAdd>(*sl.v, p);
        for (unsigned rest = grp & (grp - 1u); rest; rest &= rest - 1u)
            acc = apply<kAlgAdd>(acc, st.p[__ffs(rest) - 1]);
        *sl.v = acc;
    }
    __syncwarp();
}

__device__ __forceinline__ u32 warp_sum(u32 x)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// ---- warp tables: a warp per column, an open-addressing table in shared memory.  The count pass does not know
// u(j) yet: a column uses 2^lg >= max(f(j), 32) slots (keys only).  The write pass does: 2^lg >= max(2 u(j), 32)
// slots of keys and values, so its shared memory, and with it the warps an SM holds, follow the rows of the result
// rather than the products (block RD 32^3 x 8 squared: f(j) up to 3136, 190 rows per column on average).
__device__ __forceinline__ u32 table_slot(u32 *keys, int lg, u32 row, bool &fresh)
{
    u32 s = (row * 2654435769u) >> (32 - lg);
    for (;;)
    {
        const u32 old = atomicCAS(&keys[s], kEmpty, row);
        if (old == kEmpty || old == row)
        {
            fresh = old == kEmpty;
            return s;
        }
        s = (s + 1) & ((1u << lg) - 1u);
    }
}

__host__ __device__ constexpr size_t table_warp_bytes(bool numeric, int lgmax)
{
    return sizeof(WarpStage) + ((size_t)(numeric ? 12 : 4) << lgmax);
}

// 2^lgmax slots per warp; a column of the write pass with u(j) > 2^lgmax is left to the row tiles
template <typename Ti, bool NUMERIC>
__global__ void __launch_bounds__(256)
    spgemm_table_kernel(Mats<Ti> M, const u32 *__restrict__ cols, const u32 *__restrict__ fcol, u64 ncols, int lgmax,
                        u64 *__restrict__ ucount, const Ti *__restrict__ colptr, Ti *__restrict__ rowval,
                        double *__restrict__ nzval)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u64 ci = (u64)blockIdx.x * (blockDim.x >> 5) + w;
    if (ci >= ncols)
        return;
    unsigned char *my = smem + (size_t)w * table_warp_bytes(NUMERIC, lgmax);
    WarpStage &st = *reinterpret_cast<WarpStage *>(my);
    u32 *keys = reinterpret_cast<u32 *>(my + sizeof(WarpStage));
    double *vals = reinterpret_cast<double *>(my + sizeof(WarpStage) + ((size_t)4 << lgmax));
    const i64 j = cols[ci];
    i64 off = 0, u = 0;
    u32 need = fcol[j];
    if (NUMERIC)
    {
        off = (i64)colptr[j] - M.base;
        u = (i64)colptr[j + 1] - M.base - off;
        if (u > (i64)(1u << lgmax))
            return;
        need = 2 * (u32)u;
    }
    int lg = 5;
    while (lg < lgmax && (1u << lg) < need)
        ++lg;
    const u32 T = 1u << lg;
    for (u32 i = lane; i < T; i += 32)
        keys[i] = kEmpty;
    __syncwarp();
    if (!NUMERIC)
    {
        u32 fresh = 0;
        walk_column<Ti, false, false>(M, j, 0, 0, st, [&](bool act, u32 row, double) {
            bool f = false;
            if (act)
                table_slot(keys, lg, row, f);
            fresh += f;
        });
        fresh = warp_sum(fresh);
        if (lane == 0)
            ucount[j] = fresh;
        return;
    }
    walk_column<Ti, true, false>(M, j, 0, 0, st, [&](bool act, u32 row, double p) {
        fold_batch(act, row, p, st, [&](u32 r) {
            bool fresh;
            const u32 slot = table_slot(keys, lg, r, fresh);
            return Slot{&vals[slot], fresh};
        });
    });
    // the u occupied slots to the front in slot order (a chunk is read before any of its slots is written), padded
    // to S = 2^ceil(log2 u) with empty slots, then a bitonic sort of those S by row
    u32 cnt = 0;
    for (u32 c0 = 0; c0 < T; c0 += 32)
    {
        const u32 key = keys[c0 + lane];
        const double v = vals[c0 + lane];
        const unsigned occ = __ballot_sync(0xffffffffu, key != kEmpty);
        __syncwarp();
        if (key != kEmpty)
        {
            const u32 d = cnt + __popc(occ & ((1u << lane) - 1u));
            keys[d] = key;
            vals[d] = v;
        }
        cnt += __popc(occ);
        __syncwarp();
    }
    u32 S = 1;
    while (S < (u32)u)
        S <<= 1;
    for (u32 i = (u32)u + lane; i < S; i += 32)
        keys[i] = kEmpty;
    __syncwarp();
    for (u32 k = 2; k <= S; k <<= 1)
        for (u32 h = k >> 1; h > 0; h >>= 1)
        {
            for (u32 i = lane; i < S; i += 32)
            {
                const u32 x = i ^ h;
                if (x > i)
                {
                    const u32 a = keys[i], b = keys[x];
                    if ((a > b) == ((i & k) == 0))
                    {
                        keys[i] = b;
                        keys[x] = a;
                        const double t = vals[i];
                        vals[i] = vals[x];
                        vals[x] = t;
                    }
                }
            }
            __syncwarp();
        }
    for (i64 i = lane; i < u; i += 32)
    {
        rowval[off + i] = (Ti)((i64)keys[i] + M.base);
        nzval[off + i] = vals[i];
    }
}

// ---- tiled bin: a warp per piece (column, kTile rows), a dense tile of values and an occupancy bitmap
template <bool NUMERIC> __host__ __device__ constexpr size_t tile_warp_bytes()
{
    return sizeof(WarpStage) + 4 * (size_t)(kTile / 32) + (NUMERIC ? 8 * (size_t)kTile : 0);
}

template <typename Ti, bool NUMERIC>
__global__ void __launch_bounds__(32 * kTileWarps, 1)
    spgemm_tile_kernel(Mats<Ti> M, i64 m, TileWs T, u64 npieces, u64 *__restrict__ ucount,
                       const Ti *__restrict__ colptr, Ti *__restrict__ rowval, double *__restrict__ nzval)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u64 pi = (u64)blockIdx.x * kTileWarps + w;
    if (pi >= npieces)
        return;
    unsigned char *my = smem + (size_t)w * tile_warp_bytes<NUMERIC>();
    WarpStage &st = *reinterpret_cast<WarpStage *>(my);
    u32 *occ = reinterpret_cast<u32 *>(my + sizeof(WarpStage));
    double *vals = reinterpret_cast<double *>(my + sizeof(WarpStage) + 4 * (kTile / 32));
    const uint4 pc = T.piece[pi];
    const i64 j = pc.x, rlo = pc.y, rhi = min(rlo + (i64)kTile, m);
    if (NUMERIC && (i64)colptr[j + 1] - (i64)colptr[j] <= (i64)kTableMax)
        return; // written through a warp table
    for (int i = lane; i < kTile / 32; i += 32)
        occ[i] = 0;
    __syncwarp();
    if (!NUMERIC)
    {
        u32 fresh = 0;
        walk_column<Ti, false, true>(M, j, rlo, rhi, st, [&](bool act, u32 row, double) {
            if (act)
            {
                const u32 x = row - (u32)rlo, bit = 1u << (x & 31);
                fresh += (atomicOr(&occ[x >> 5], bit) & bit) == 0;
            }
        });
        fresh = warp_sum(fresh);
        if (lane == 0)
        {
            T.cnt[pi] = fresh;
            atomicAdd(&ucount[j], (u64)fresh);
        }
        return;
    }
    walk_column<Ti, true, true>(M, j, rlo, rhi, st, [&](bool act, u32 row, double p) {
        fold_batch(act, row, p, st, [&](u32 r) {
            const u32 x = r - (u32)rlo, bit = 1u << (x & 31);
            return Slot{&vals[x], (atomicOr(&occ[x >> 5], bit) & bit) == 0};
        });
    });
    // T.cnt holds the exclusive scan over the pieces: earlier pieces of this column come first
    i64 off = (i64)colptr[j] - M.base + (i64)(T.cnt[pi] - T.cnt[pc.z]);
    for (int w0 = 0; w0 < kTile / 32; w0 += 32)
    {
        u32 word = occ[w0 + lane];
        const u32 c = __popc(word);
        u32 incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o)
                incl += y;
        }
        i64 pos = off + incl - c;
        while (word)
        {
            const u32 x = (u32)(w0 + lane) * 32 + (u32)(__ffs(word) - 1);
            word &= word - 1u;
            rowval[pos] = (Ti)(rlo + (i64)x + M.base);
            nzval[pos] = vals[x];
            ++pos;
        }
        off += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// ---- exclusive scan of u64 counts: block sums, one block over the sums, then the scan itself
__device__ __forceinline__ u64 block_exclusive(u64 v, u64 *s_warp)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o)
            x += y;
    }
    if (lane == 31)
        s_warp[warp] = x;
    __syncthreads();
    u64 before = x - v;
    for (int w = 0; w < warp; ++w)
        before += s_warp[w];
    return before;
}

__global__ void __launch_bounds__(kScanThreads) scan_sum_kernel(const u64 *__restrict__ in, i64 n, u64 *__restrict__ bsum)
{
    __shared__ u64 s_warp[kScanThreads / 32];
    const i64 i0 = (i64)blockIdx.x * kScanTile + (i64)threadIdx.x * kScanItems;
    u64 s = 0;
#pragma unroll
    for (int q = 0; q < kScanItems; ++q)
        if (i0 + q < n)
            s += in[i0 + q];
    const u64 before = block_exclusive(s, s_warp);
    if (threadIdx.x == kScanThreads - 1)
        bsum[blockIdx.x] = before + s;
}

// exclusive scan of the block sums in place (one block); *total = their sum
__global__ void __launch_bounds__(1024) scan_blocks_kernel(u64 *__restrict__ bsum, i64 nblocks, u64 *__restrict__ total)
{
    __shared__ u64 s_warp[32];
    __shared__ u64 s_carry;
    if (threadIdx.x == 0)
        s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (i64 base = 0; base < nblocks; base += 1024)
    {
        const i64 k = base + threadIdx.x;
        const u64 v = k < nblocks ? bsum[k] : 0;
        u64 x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o)
                x += y;
        }
        if (lane == 31)
            s_warp[warp] = x;
        __syncthreads();
        if (warp == 0)
        {
            u64 w = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const u64 y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o)
                    w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const u64 incl = s_carry + x + (warp > 0 ? s_warp[warp - 1] : 0);
        if (k < nblocks)
            bsum[k] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0)
        *total = s_carry;
}

// out[i] = base + sum of in[0, i) for i <= n (out may be in: every thread reads its items before it writes them)
template <typename OutT>
__global__ void __launch_bounds__(kScanThreads)
    scan_write_kernel(const u64 *in, i64 n, const u64 *__restrict__ bsum, const u64 *__restrict__ total, OutT *out, i64 base)
{
    __shared__ u64 s_warp[kScanThreads / 32];
    const i64 i0 = (i64)blockIdx.x * kScanTile + (i64)threadIdx.x * kScanItems;
    u64 v[kScanItems];
    u64 s = 0;
#pragma unroll
    for (int q = 0; q < kScanItems; ++q)
    {
        v[q] = i0 + q < n ? in[i0 + q] : 0;
        s += v[q];
    }
    u64 run = block_exclusive(s, s_warp) + (n > 0 ? bsum[blockIdx.x] : 0);
#pragma unroll
    for (int q = 0; q < kScanItems; ++q)
        if (i0 + q < n)
        {
            out[i0 + q] = (OutT)((i64)run + base);
            run += v[q];
        }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0)
        out[n] = (OutT)((i64)*total + base);
}

template <typename OutT>
void exclusive_scan(cudaStream_t s, const u64 *in, i64 n, u64 *bsum, u64 *total, OutT *out, i64 base, LaunchCounter &lc)
{
    const i64 nb = scan_blocks(n);
    if (nb > 0)
    {
        scan_sum_kernel<<<(unsigned)nb, kScanThreads, 0, s>>>(in, n, bsum);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    scan_blocks_kernel<<<1, 1024, 0, s>>>(bsum, nb, total);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    scan_write_kernel<OutT><<<(unsigned)std::max<i64>(nb, 1), kScanThreads, 0, s>>>(in, n, bsum, total, out, base);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ---- launches
FuncAttrOnce g_attr_table[2][2], g_attr_tile[2][2];

template <typename Ti, bool NUMERIC>
void launch_table(cudaStream_t s, const Mats<Ti> &M, const u32 *cols, const u32 *fcol, u64 ncols, int lgmax,
                  u64 *ucount, const void *colptr, void *rowval, double *nzval, LaunchCounter &lc)
{
    if (ncols == 0)
        return;
    const size_t wb = table_warp_bytes(NUMERIC, lgmax);
    const int W = (int)std::max<size_t>(1, std::min<size_t>(8, kTableBlockSmem / wb));
    auto k = spgemm_table_kernel<Ti, NUMERIC>;
    g_attr_table[sizeof(Ti) == 8][NUMERIC].set(k, kTableBlockSmem);
    k<<<(unsigned)((ncols + W - 1) / W), 32 * W, W * wb, s>>>(M, cols, fcol, ncols, lgmax, ucount,
                                                              static_cast<const Ti *>(colptr),
                                                              static_cast<Ti *>(rowval), nzval);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

int ceil_log2(u64 x)
{
    int lg = 0;
    while ((1ull << lg) < x)
        ++lg;
    return lg;
}

// count: every table bin with the slots its f(j) bound needs; write: every bin, the tiled one included, with
// 2^ceil(log2 2 umax) slots (at least 32, at most kTableMax)
template <typename Ti, bool NUMERIC>
void launch_bins(cudaStream_t s, const Spgemm &g, const void *colptr, void *rowval, double *nzval, LaunchCounter &lc)
{
    const Mats<Ti> M = mats<Ti>(g);
    const ColWs W = col_ws(g.ws, g.n);
    const u32 caps[kBins] = {kBinCap0, kBinCap1, kBinCap2};
    u64 off = 0;
    for (int b = 0; b <= kBins; ++b)
    {
        if (NUMERIC ? g.umax[b] > 0 : b < kBins)
        {
            const int lgmax = NUMERIC ? std::min(std::max(ceil_log2(2 * g.umax[b]), 5), ceil_log2(kTableMax))
                                      : ceil_log2(caps[b]);
            launch_table<Ti, NUMERIC>(s, M, W.list + off, W.f, g.bins[b], lgmax, W.u, colptr, rowval, nzval, lc);
        }
        off += g.bins[b];
    }
    if (g.tiles == 0)
        return;
    const size_t smem = kTileWarps * tile_warp_bytes<NUMERIC>();
    auto k = spgemm_tile_kernel<Ti, NUMERIC>;
    g_attr_tile[sizeof(Ti) == 8][NUMERIC].set(k, (int)smem);
    k<<<(unsigned)((g.tiles + kTileWarps - 1) / kTileWarps), 32 * kTileWarps, smem, s>>>(
        M, g.m, tile_ws(g.tile_ws, g.tiles), g.tiles, W.u, static_cast<const Ti *>(colptr), static_cast<Ti *>(rowval),
        nzval);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

unsigned grid_for(i64 items, int per_block) { return (unsigned)std::max<i64>(1, std::min<i64>((items + per_block - 1) / per_block, 148 * 32)); }

template <typename Ti> void classify_t(cudaStream_t s, const Spgemm &g, LaunchCounter &lc)
{
    const ColWs W = col_ws(g.ws, g.n);
    XSB_CUDA(cudaMemsetAsync(W.ct, 0, sizeof(u64) * kCtCount, s));
    if (g.n == 0)
        return;
    spgemm_classify_kernel<Ti><<<grid_for(g.n, 8), 256, 0, s>>>(mats<Ti>(g), g.n, W);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

template <typename Ti> void count_t(cudaStream_t s, const Spgemm &g, void *colptr_out, LaunchCounter &lc)
{
    const ColWs W = col_ws(g.ws, g.n);
    const TileWs T = tile_ws(g.tile_ws, g.tiles);
    if (g.n > 0)
    {
        BinOffsets B;
        u64 o = 0;
        for (int b = 0; b <= kBins; ++b)
        {
            B.off[b] = o;
            o += g.bins[b];
        }
        spgemm_fill_kernel<<<grid_for(g.n, 256), 256, 0, s>>>(g.n, W, B, T);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    launch_bins<Ti, false>(s, g, nullptr, nullptr, nullptr, lc);
    if (g.n > 0)
    {
        spgemm_umax_kernel<<<grid_for(g.n, 256), 256, 0, s>>>(g.n, W);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    exclusive_scan<Ti>(s, W.u, g.n, W.bsum, W.ct + kCtNnz, static_cast<Ti *>(colptr_out), g.base, lc);
    if (g.tiles > 0) // piece offsets; the total lands in the unused counter slot after the cursors
        exclusive_scan<u64>(s, T.cnt, (i64)g.tiles, T.bsum, W.ct + kCtTileCur + 1, T.cnt, 0, lc);
}

} // namespace

size_t spgemm_workspace_bytes(i64 n)
{
    return sizeof(u64) * kCtCount + 5 * align16(4 * (size_t)n) + align16(8 * (size_t)n) +
           8 * (size_t)(scan_blocks(n) + 1);
}

size_t spgemm_tiles_bytes(u64 tiles)
{
    return sizeof(uint4) * (size_t)tiles + align16(8 * (size_t)(tiles + 1)) + 8 * (size_t)(scan_blocks((i64)tiles) + 1);
}

void spgemm_classify(cudaStream_t stream, const Spgemm &g, LaunchCounter &lc)
{
    if (g.idx64)
        classify_t<int64_t>(stream, g, lc);
    else
        classify_t<int32_t>(stream, g, lc);
}

void spgemm_count(cudaStream_t stream, const Spgemm &g, void *colptr_out, LaunchCounter &lc)
{
    if (g.idx64)
        count_t<int64_t>(stream, g, colptr_out, lc);
    else
        count_t<int32_t>(stream, g, colptr_out, lc);
}

void spgemm_write(cudaStream_t stream, const Spgemm &g, const void *colptr, void *rowval_out, double *nzval_out,
                  LaunchCounter &lc)
{
    if (g.idx64)
        launch_bins<int64_t, true>(stream, g, colptr, rowval_out, nzval_out, lc);
    else
        launch_bins<int32_t, true>(stream, g, colptr, rowval_out, nzval_out, lc);
}

} // namespace xsb
