// xsb_common.cuh -- shared device/host definitions of libxsparse_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdexcept>
#include <string>

namespace xsb {

typedef unsigned long long u64;
typedef long long i64;
typedef unsigned int u32;

// One staged insertion: packed key + Float64 value = one 16-byte vector load/store.
//
// key bits, low to high:  [flavour:2][tid:tidbits][row:rowbits][col:colbits]
// The radix sort covers only [low, low+rowbits+colbits): flavour and tid ride
// along unsorted, so a STABLE sort keeps the insertion order inside a run of
// equal (col,row) -- which is what the deterministic left fold needs.
struct __align__(16) Rec
{
    u64 key;
    double val;
};

enum : u32
{
    FL_UPDATE = 0,
    FL_RAW = 1,
    FL_ASSIGN = 2,
    FL_OLD = 3 // entry of the resident CSC, placed ahead of all staged entries
};

constexpr int kMaxRanks = 16;

struct KeyLayout
{
    int low;     // 2 + tidbits
    int tidbits; // bits of the partition id
    int rowbits;
    int colbits;
    // Slab (multi-GPU) handles only: the rank that owns the column rides in the bits above the
    // column ([owner:ownerbits] on top) and the column field is RELATIVE to the owner's slab, so a
    // record is already in its owner's flush layout wherever it is staged: records for other
    // ranks are picked out by their owner bits, the rest never moves.
    int ownerbits;
    int nranks;
    int self;        // this rank
    int cols_global; // pack() takes global columns (insertion side); 0: slab-local columns owned by self
    i64 self_lo;     // splits[self] and the width of the own slab: pack()'s fast path
    u64 self_width;
    i64 splits[kMaxRanks + 1]; // rank r owns columns [splits[r], splits[r+1]), 0-based
    __host__ __device__ __forceinline__ u64 pack(u64 col, u64 row, u32 tid, u32 fl) const
    {
        u64 o = 0;
        if (nranks > 0)
        {
            if (cols_global)
            {
                const u64 rel = col - (u64)self_lo; // a partitioned assembly mostly inserts into its own slab
                if (rel < self_width)
                {
                    col = rel;
                    o = (u64)self;
                }
                else
                {
                    int q = 0;
                    while (q + 1 < nranks && (i64)col >= splits[q + 1])
                        ++q;
                    col -= (u64)splits[q];
                    o = (u64)q;
                }
            }
            else
                o = (u64)self;
        }
        u64 k = (col << (rowbits + low)) | (row << low) | ((u64)tid << 2) | (u64)fl;
        if (ownerbits)
            k |= o << (low + rowbits + colbits);
        return k;
    }
    // pack(col,row,tid,fl) == colpart(col) | rowpart(row,tid,fl): producers that reuse a column or a
    // row for several records (element matrices) build the halves once
    __host__ __device__ __forceinline__ u64 colpart(u64 col) const { return pack(col, 0, 0u, 0u); }
    __host__ __device__ __forceinline__ u64 rowpart(u64 row, u32 tid, u32 fl) const
    {
        return (row << low) | ((u64)tid << 2) | (u64)fl;
    }
    __host__ __device__ __forceinline__ int ownershift() const { return low + rowbits + colbits; }
    __host__ __device__ __forceinline__ u32 owner(u64 key) const
    {
        return ownerbits ? (u32)(key >> (low + rowbits + colbits)) : 0u;
    }
    // global column of a staged record
    __host__ __device__ __forceinline__ u64 gcol(u64 key) const
    {
        return col(key) + (nranks > 0 ? (u64)splits[ownerbits ? owner(key) : (u32)self] : 0ull);
    }
    __host__ __device__ __forceinline__ u64 colrow(u64 key) const { return key >> low; }
    __host__ __device__ __forceinline__ u64 col(u64 key) const
    {
        return (key >> (rowbits + low)) & ((1ull << colbits) - 1ull);
    }
    __host__ __device__ __forceinline__ u64 row(u64 key) const
    {
        return (key >> low) & ((1ull << rowbits) - 1ull);
    }
    __host__ __device__ __forceinline__ u32 tid(u64 key) const
    {
        return (u32)((key >> 2) & ((1ull << tidbits) - 1ull));
    }
    __host__ __device__ __forceinline__ u32 flavour(u64 key) const { return (u32)(key & 3ull); }
    __host__ __device__ int sortbits() const { return rowbits + colbits; }
};

struct CudaError : std::runtime_error
{
    cudaError_t code;
    CudaError(cudaError_t c, const std::string &what) : std::runtime_error(what), code(c) {}
};

#define XSB_CUDA(expr)                                                                             \
    do                                                                                             \
    {                                                                                              \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            throw ::xsb::CudaError(_e, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    } while (0)

// number of SMs of a B200; grids are sized as multiples of it
constexpr int kNumSM = 148;

__device__ __forceinline__ u32 lanemask_lt()
{
    u32 m;
    asm volatile("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

__device__ __forceinline__ u32 ld_relaxed_u32(const u32 *p)
{
    u32 v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(u32 *p, u32 v)
{
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p)
{
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(u64 *p, u64 v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// streaming 16-byte record load / store (data touched once: keep it out of L1)
__device__ __forceinline__ Rec ld_rec_stream(const Rec *p)
{
    Rec r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];"
                 : "=l"(r.key), "=l"(*reinterpret_cast<u64 *>(&r.val))
                 : "l"(p));
    return r;
}
// two consecutive records in one 256-bit request (sm_100: LDG.256); p must be 32-byte aligned
struct RecPair
{
    Rec a, b;
};
__device__ __forceinline__ RecPair ld_pair_stream(const Rec *p)
{
    RecPair r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0, %1, %2, %3}, [%4];"
                 : "=l"(r.a.key), "=l"(*reinterpret_cast<u64 *>(&r.a.val)), "=l"(r.b.key),
                   "=l"(*reinterpret_cast<u64 *>(&r.b.val))
                 : "l"(p));
    return r;
}
// 256-bit store; p must be 32-byte aligned
__device__ __forceinline__ void st_v4_u64(void *p, u64 a, u64 b, u64 c, u64 d)
{
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
__device__ __forceinline__ void st_rec(Rec *p, const Rec &r)
{
    asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(r.key),
                 "l"(*reinterpret_cast<const u64 *>(&r.val))
                 : "memory");
}

// Slab handles: a producer that stages a record owned by another rank marks the tile of the
// staging buffer it lands in, so that routing only looks at marked tiles (xsb_route.cu).
constexpr int kRouteTileShift = 11; // tiles of 2048 records
struct StageFlags
{
    unsigned char *flags; // one byte per tile, relative to the first staged record; nullptr: not a slab handle
    i64 pos0;             // staged records ahead of out0
};
__device__ __forceinline__ void st_staged(Rec *p, const Rec &r, const KeyLayout &L, const StageFlags &sf,
                                          const Rec *out0)
{
    st_rec(p, r);
    if (sf.flags != nullptr && L.owner(r.key) != (u32)L.self)
        sf.flags[(sf.pos0 + (i64)(p - out0)) >> kRouteTileShift] = 1; // benign race: same value
}

// Decoupled look-back over per-tile totals (tiles are dispatched in index order): the calling WARP
// publishes `mine` for tile `index` and returns the sum of the totals of all tiles before it.
// status[] starts zeroed; values must stay below 2^62.
constexpr u64 LB_AGG = 1ull << 62, LB_INCL = 2ull << 62, LB_VALUE = (1ull << 62) - 1ull;
__device__ __forceinline__ u64 warp_lookback(u64 *__restrict__ status, u32 index, u64 mine, int lane)
{
    constexpr u32 full = 0xffffffffu;
    u64 prefix = 0;
    if (index == 0)
    {
        if (lane == 0)
            st_relaxed_u64(status, LB_INCL | mine);
        return 0;
    }
    if (lane == 0)
        st_relaxed_u64(status + index, LB_AGG | mine);
    long long b = (long long)index - 1;
    for (;;)
    { // lane l looks at tile b - l
        u64 v = LB_INCL;
        if (b - lane >= 0)
        {
            for (;;)
            {
                v = ld_relaxed_u64(status + (b - lane));
                if ((v >> 62) != 0ull)
                    break;
                __nanosleep(40); // the predecessor is still working: do not spend its issue slots on polling
            }
        }
        const u32 inc = __ballot_sync(full, (v >> 62) == 2ull);
        const int first = inc ? __ffs(inc) - 1 : 31; // nearest tile with an inclusive prefix, if in this window
        u64 c = (lane <= first) ? (v & LB_VALUE) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            c += __shfl_xor_sync(full, c, o);
        prefix += c;
        if (inc)
            break;
        b -= 32;
    }
    if (lane == 0)
        st_relaxed_u64(status + index, LB_INCL | (prefix + mine));
    return prefix;
}

} // namespace xsb
