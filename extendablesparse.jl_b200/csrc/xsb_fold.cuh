// xsb_fold.cuh -- how a column is folded and how the new CSC is written, for every flush path: the
// insertion-order fold of one run (RunFold), the thread-per-column fold with its table shapes
// (ThreadFold, FoldShape, fold_level_for), the thread-per-column write-out (column_offset,
// ThreadFold::store) and an in-register warp bitonic sort.
#pragma once
#include "xsb_common.cuh"

namespace xsb {

// Insertion-order fold of one run of equal (col,row): the semantics of the three insert
// flavours (src/matrix/sparsematrixlnk.jl:178-253) behind the CSC-hit router
// (src/matrix/extendable.jl:159-218), per partition buffer, then partitions summed in tid
// order with the first one copied (sparse! combine, src/matrix/sparsematrixdilnkc.jl:416-432).
struct RunFold
{
    bool seeded = false, has_old = false, exists = false, pexists = false;
    double old = 0.0, acc = 0.0, pacc = 0.0;
    u32 ptid = 0xffffffffu;

    __device__ __forceinline__ void commit()
    {
        if (pexists)
        {
            if (exists)
                acc = acc + pacc;
            else
            {
                acc = pacc;
                exists = true;
            }
            pexists = false;
        }
    }
    __device__ __forceinline__ void apply(u32 fl, u32 tid, double v, int combine)
    {
        if (fl == FL_OLD)
        {
            if (combine == 0)
            {
                seeded = true;
                exists = true;
                acc = v;
            }
            else
            {
                has_old = true;
                old = v;
            }
            return;
        }
        if (seeded)
        { // entry already in the CSC: in-place op, extendable.jl:164-166 / :210-212
            acc = (fl == FL_ASSIGN) ? v : acc + v;
            return;
        }
        if (tid != ptid)
        {
            commit();
            ptid = tid;
        }
        if (fl == FL_RAW)
        {
            pacc = pexists ? pacc + v : 0.0 + v;
            pexists = true;
        }
        else if (fl == FL_UPDATE)
        {
            if (pexists)
                pacc = pacc + v;
            else if (v != 0.0)
            {
                pexists = true;
                pacc = 0.0 + v;
            }
        }
        else
        { // FL_ASSIGN
            if (pexists)
                pacc = v;
            else if (v != 0.0)
            {
                pexists = true;
                pacc = v;
            }
        }
    }
    __device__ __forceinline__ void finish()
    {
        commit();
        if (has_old)
        { // csc.nzval + lnk.nzval, sparsematrixlnk.jl:363
            acc = exists ? old + acc : old;
            exists = true;
        }
    }
};

// ------------------------------------------------------------------------
// one THREAD per column
// ------------------------------------------------------------------------
// A thread folds its column in a private open-addressing table in shared memory, laid out [slot][lane] so that a
// lane only ever touches its own bank: one probe and one add per record, the exact left fold of the reference's
// accumulate-on-insert (src/matrix/sparsematrixlnk.jl:210-253) with the list walk replaced by the hash probe.

// Table shapes, smallest first.  The template argument is the number of hash bits, except 15 = the
// 5-bit table with 16 instead of 24 accumulators (a P1 tetrahedral mesh has at most 15 rows per column).
//   shape  4: 16 slots / 12 accumulators     shape 15: 32 / 16     shape 5: 32 / 24     shape 6: 64 / 32
template <int HBITS> struct FoldShape
{
    static constexpr int HB = HBITS == 15 ? 5 : HBITS;
    static constexpr int H = 1 << HB;
    static constexpr int D = HBITS == 6 ? 32 : (HBITS == 5 ? 24 : (HBITS == 15 ? 16 : 12));
    // shared memory of one warp's tables: accumulators, table slots, the slot of every accumulator
    static constexpr size_t kBytesPerWarp = 32 * (sizeof(u32) * H + (sizeof(double) + 1) * D);
};

// level 0..3 = table shapes 4, 15, 5, 6: the smallest that takes columns of at most `maxd` distinct rows
inline int fold_level_for(u32 maxd)
{
    return maxd <= (u32)FoldShape<4>::D ? 0 : (maxd <= (u32)FoldShape<15>::D ? 1 : (maxd <= (u32)FoldShape<5>::D ? 2 : 3));
}

constexpr u32 TF_EMPTY = 0xffffffffu;

// The fold state of one column.  A table slot holds (row << HB | accumulator index); accumulators are
// numbered in order of first appearance.  Flavour semantics (single partition): src/matrix/sparsematrixlnk.jl
// :178-253 behind the CSC-hit router src/matrix/extendable.jl:159-218.
template <int HBITS, bool ASSIGN> struct ThreadFold
{
    static constexpr int H = FoldShape<HBITS>::H;
    static constexpr int HB = FoldShape<HBITS>::HB;
    static constexpr u32 D = FoldShape<HBITS>::D;
    u32 *key;    // [slot * 32]
    double *acc; // [i * 32]
    unsigned char *ord; // [i * 32]: table slot of accumulator i (its row = key >> HB)
    u32 d = 0;       // accumulators in use
    u32 pending = 0; // of which not (yet) existing: only updateindex! / setindex! of a zero touched them
    u32 exmask = 0;  // accumulator i holds an existing entry (D <= 32)
    bool ovf = false;

    // the tables of thread `lane` of warp `warp` in a block of `warps` warps (FoldShape::kBytesPerWarp each)
    __device__ __forceinline__ ThreadFold(unsigned char *smem, int warps, int warp, int lane)
    {
        acc = reinterpret_cast<double *>(smem) + warp * (D * 32) + lane;
        key = reinterpret_cast<u32 *>(smem + (size_t)warps * D * 32 * sizeof(double)) + warp * (H * 32) + lane;
        ord = smem + (size_t)warps * 32 * (D * sizeof(double) + H * sizeof(u32)) + warp * (D * 32) + lane;
    }
    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int s = 0; s < H; ++s)
            key[s * 32] = TF_EMPTY;
    }
    // slot of `row`: x = its accumulator, or x >= D with s the empty slot where the probe ended (an empty slot reads
    // as index H-1 >= D).  One loop with one exit: the lanes of a warp leave it together before they touch an accumulator.
    __device__ __forceinline__ u32 find(u32 row, u32 &s) const
    {
        const u32 tag = row << HB;
        s = (row * 0x9E3779B1u) >> (32 - HB);
        for (;;)
        {
            const u32 kk = key[s * 32];
            const u32 x = kk ^ tag;
            if (x < D || kk == TF_EMPTY)
                return x;
            s = (s + 1) & (H - 1);
        }
    }
    // an entry of the resident CSC seeds its accumulator (extendable.jl:164-166); old rows are distinct
    __device__ __forceinline__ void seed(u32 row, double v)
    {
        u32 s;
        find(row, s);
        if (d >= D)
        {
            ovf = true;
            return;
        }
        key[s * 32] = (row << HB) | d;
        ord[d * 32] = (unsigned char)s;
        acc[d * 32] = v;
        exmask |= 1u << d;
        ++d;
    }
    // one staged insertion (update / rawupdate / assign flavour)
    __device__ __forceinline__ void apply(u32 row, double v, u32 fl)
    {
        u32 s;
        u32 x = find(row, s);
        if (x >= D)
        { // first insertion of this row: a new accumulator at +0.0 (sparsematrixlnk.jl:225), not an entry yet
            if (d >= D)
            {
                ovf = true;
                return;
            }
            x = d++;
            key[s * 32] = (row << HB) | x;
            ord[x * 32] = (unsigned char)s;
            acc[x * 32] = 0.0;
            ++pending;
        }
        if (ASSIGN && fl == FL_ASSIGN)
        { // A[i,j] = v: overwrites; creates only if v != 0 (sparsematrixlnk.jl:184-199)
            const bool ex = (exmask >> x) & 1u;
            if (ex | (v != 0.0))
            {
                acc[x * 32] = v;
                if (!ex)
                {
                    exmask |= 1u << x;
                    --pending;
                }
            }
            return;
        }
        acc[x * 32] = acc[x * 32] + v;
        if (pending)
        { // rawupdateindex! always creates the entry, updateindex! only with v != 0 (sparsematrixlnk.jl:212,223,239)
            if (!((exmask >> x) & 1u) && ((fl != FL_UPDATE) | (v != 0.0)))
            {
                exmask |= 1u << x;
                --pending;
            }
        }
    }
    // existing entries as (row << HB | accumulator) words, sorted by row into key[0 .. j).  All words are read into
    // registers first (the table is overwritten), ordered there by a bitonic network -- no branch, no
    // memory traffic, the same instruction stream for every lane whatever its column looks like -- and written back.
    // Entry e is then row key[e * 32] >> HB, value acc[(key[e * 32] & (H - 1)) * 32].
    __device__ __forceinline__ int finish()
    {
        constexpr int N = D <= 16 ? 16 : 32;
        u32 a[N];
#pragma unroll
        for (int i = 0; i < N; ++i)
        {
            a[i] = 0xffffffffu;
            if ((u32)i < D && (u32)i < d && ((exmask >> i) & 1u))
                a[i] = key[(u32)ord[i * 32] * 32]; // (row << HB) | i
        }
#pragma unroll
        for (int k = 2; k <= N; k <<= 1) // bitonic network: every index below is a compile-time constant
#pragma unroll
            for (int jj = k >> 1; jj > 0; jj >>= 1)
#pragma unroll
                for (int i = 0; i < N; ++i)
                {
                    const int l = i ^ jj;
                    if (l > i)
                    {
                        const u32 lo_ = min(a[i], a[l]), hi_ = max(a[i], a[l]);
                        a[i] = (i & k) == 0 ? lo_ : hi_;
                        a[l] = (i & k) == 0 ? hi_ : lo_;
                    }
                }
        const int j = __popc(exmask);
#pragma unroll
        for (int i = 0; i < N; ++i)
            if (i < H && i < j)
                key[i * 32] = a[i];
        return j;
    }
    // the j entries sorted by finish() -> rv[0 .. j) (row + base) and nv[0 .. j).  256-bit stores where the
    // destination is 32-byte aligned (rowval and nzval separately: their bases differ): a lane writes its own run,
    // so every store instruction costs one request per lane
    template <typename Ti> __device__ __forceinline__ void store(int j, Ti base, Ti *rv, double *nv) const
    {
        {
            auto row_at = [&](int e) { return (Ti)(key[e * 32] >> HB) + base; };
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
            auto val_at = [&](int e) { return (u64)__double_as_longlong(acc[(key[e * 32] & (H - 1)) * 32]); };
            int e = 0;
            for (; e < j && (reinterpret_cast<uintptr_t>(nv + e) & 31u); ++e)
                nv[e] = __longlong_as_double((long long)val_at(e));
            for (; e + 4 <= j; e += 4)
                st_v4_u64(nv + e, val_at(e), val_at(e + 1), val_at(e + 2), val_at(e + 3));
            for (; e < j; ++e)
                nv[e] = __longlong_as_double((long long)val_at(e));
        }
    }
};

// Where the j entries of this thread's column go in the new matrix: the entries of the columns before it, by a warp
// scan, a block scan over the WARPS warps (s_wsum[WARPS]) and a look-back over the blocks (block `bid`, its word in
// status).  Every thread of the block calls it.  Blocks must take their columns in the order they START (a ticket),
// so a block only ever waits for blocks that are already running: the look-back cannot starve whatever the
// dispatch order.
template <int WARPS>
__device__ __forceinline__ u64 column_offset(int j, u64 *__restrict__ status, u32 bid, u32 *s_wsum, u64 *s_prefix,
                                             int lane, int warp)
{
    u32 incl = (u32)j;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_wsum[warp] = incl;
    __syncthreads();
    u32 wpre = 0, btotal = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w)
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
            *s_prefix = prefix;
    }
    __syncthreads();
    return *s_prefix + wpre + (incl - (u32)j);
}

// bitonic sort of 32*E keys held E per lane (element index = lane*E + e), ascending
template <int E> __device__ __forceinline__ void warp_bitonic(u32 (&k)[E], int lane)
{
    constexpr int N = 32 * E;
#pragma unroll
    for (int size = 2; size <= N; size <<= 1)
    {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1)
        {
            if (stride >= E)
            { // partner in another lane, same register slot
                const int lstride = stride / E;
#pragma unroll
                for (int e = 0; e < E; ++e)
                {
                    const int g = lane * E + e;
                    const u32 other = __shfl_xor_sync(0xffffffffu, k[e], lstride);
                    const bool up = (g & size) == 0;      // ascending block
                    const bool lower = (g & stride) == 0; // this element is the lower index of the pair
                    const u32 mn = min(k[e], other), mx = max(k[e], other);
                    k[e] = (up == lower) ? mn : mx;
                }
            }
            else
            { // both elements in this lane
#pragma unroll
                for (int e = 0; e < E; ++e)
                {
                    if ((e & stride) == 0)
                    {
                        const int g = lane * E + e;
                        const bool up = (g & size) == 0;
                        const u32 a = k[e], b = k[e + stride];
                        const u32 mn = min(a, b), mx = max(a, b);
                        k[e] = up ? mn : mx;
                        k[e + stride] = up ? mx : mn;
                    }
                }
            }
        }
    }
}

} // namespace xsb
