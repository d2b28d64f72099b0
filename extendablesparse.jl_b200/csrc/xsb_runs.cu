// xsb_runs.cu -- flush! on GROUPED CHUNKS (xsb_chunk.cuh): the staged records are never moved.
//
//   chunk_sort_kernel : brings what the producers left in stream order (records received from other
//                       ranks, batches staged while grouping at insertion was off) into grouped chunks,
//                       in place, and appends their (chunk, column) pairs to the run index.
//   run_totals_kernel : pairs per column (one L2 atomic per pair).
//   runpair_scan_kernel: exclusive scan over the columns (single pass, decoupled look-back): every
//                       column's bucket in a pair-sized array.
//   run_bucket_kernel : a warp per chunk drops its pairs into their columns' buckets as 8-byte run
//                       descriptors [region rank | position in the staging buffer | records].
//   runfold_kernel    : ONE THREAD per column of the matrix.  It puts its handful of run descriptors
//                       into stream order, seeds a thread-private hash table (shared memory, laid out
//                       [slot][lane]) with the column of the RESIDENT CSC, walks its runs where they lie
//                       -- one probe and one add per record: the reference's accumulate-on-insert
//                       (src/matrix/sparsematrixlnk.jl:210-253, CSC hits: src/matrix/extendable.jl:164-166)
//                       as an exact left fold in insertion order -- sorts the entries by row
//                       (sparsematrixlnk.jl:339) and writes rowval / nzval / colptr of the new matrix in
//                       the same pass (block scan + look-back).  A column without new records is copied.
//                       This is the 3-way merge of Base.:+(lnk, csc) (sparsematrixlnk.jl:328-378): old
//                       entries are read once and written once, never turned back into records.
//
// HBM traffic of a flush: 16 B per staged record (read once) + the old CSC read once + the new CSC
// written once + 20 B per (chunk, column) pair -- SURVEY.md 8(d)'s algorithmic bytes plus the pairs.
#include "xsb_chunk.cuh"
#include "xsb_internal.h"

namespace xsb {

// ------------------------------------------------------------------------
// flush-time grouping of a region, in place
// ------------------------------------------------------------------------
constexpr int CS_WARPS = 8;
constexpr int CS_HB = 9;
constexpr int CS_NB = CH_RECORDS / 32;

__global__ void __launch_bounds__(CS_WARPS * 32)
chunk_sort_kernel(Rec *buf, u64 r0, u64 r1, u32 chunk0, u32 nchunks, RunTarget rt)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef ChunkSpaceT<CS_HB> Space;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 c = blockIdx.x * CS_WARPS + warp;
    if (c >= nchunks)
        return;
    Space &ws = reinterpret_cast<Space *>(smem_raw)[warp];
    chunk_space_init(ws, lane);
    const u32 lt = lanemask_lt();
    const u64 c0 = r0 + (u64)c * CH_RECORDS;
    const u32 len = (u32)min((u64)CH_RECORDS, r1 - c0);
    Rec *rec = buf + c0;
    Rec r[CS_NB];
#pragma unroll
    for (int b = 0; b < CS_NB; ++b)
    {
        const u32 p = b * 32 + lane;
        if (p < len)
            r[b] = ld_rec_stream(rec + p);
        else
        {
            r[b].key = 0;
            r[b].val = 0.0;
        }
    }
    u32 rs[CS_NB];
    u32 d = 0;
    bool grouped = true;
#pragma unroll
    for (int b = 0; b < CS_NB; ++b)
    {
        rs[b] = 0;
        if ((u32)(b * 32) < len && grouped) // warp-uniform
        {
            if (d > Space::DMAX - 32u)
                grouped = false; // the table may not take another 32 columns: no column locality here
            else
                rs[b] = chunk_count_batch(ws, (u32)(r[b].key >> rt.colshift) & rt.gmask, b * 32 + lane < len, lt, d);
        }
    }
    if (grouped)
    {
        chunk_scan(ws, d, lane);
#pragma unroll
        for (int b = 0; b < CS_NB; ++b)
            if ((u32)(b * 32 + lane) < len)
                st_rec(rec + chunk_dest(ws.start, rs[b]), r[b]);
        chunk_publish(ws, rt, chunk0 + c, (u32)c0, d, true, lane);
    }
    else
    { // no column locality in this chunk: it stays as it is, every record a run of its own
#pragma unroll
        for (int b = 0; b < CS_NB; ++b)
            rs[b] = (u32)(r[b].key >> rt.colshift) & rt.gmask;
        chunk_publish_singletons<CS_NB>(rt, chunk0 + c, (u32)c0, len, rs, lane);
    }
}

// ------------------------------------------------------------------------
// pairs per column; scan; buckets
// ------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
run_totals_kernel(const u32 *__restrict__ counters, u32 cap, const u32 *__restrict__ pcol, int colbits, u32 me,
                  u32 *__restrict__ colpairs)
{
    const u32 np = min(counters[0], cap);
    const u32 cmask = (1u << colbits) - 1u;
    const u32 stride = gridDim.x * blockDim.x;
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < np; p += stride)
    {
        const u32 g = pcol[p];
        if ((g >> colbits) == me) // records of other ranks (sent already) and padding are skipped
            atomicAdd(colpairs + (g & cmask), 1u);
    }
}

constexpr int SC_THREADS = 256;
constexpr int SC_IPT = 8;
constexpr int SC_TILE = SC_THREADS * SC_IPT;

// pstart[c] = pairs of the columns before c, c = 0..n (pstart[n] = all pairs of this rank)
__global__ void __launch_bounds__(SC_THREADS)
runpair_scan_kernel(const u32 *__restrict__ colpairs, i64 n, u32 *__restrict__ pstart, u64 *__restrict__ status,
                    u32 *__restrict__ ticket)
{
    __shared__ u32 s_w[SC_THREADS / 32];
    __shared__ u64 s_prefix;
    __shared__ u32 s_tile;
    if (threadIdx.x == 0)
        s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 b0 = (i64)tile * SC_TILE + (i64)threadIdx.x * SC_IPT; // a thread owns SC_IPT consecutive columns
    u32 v[SC_IPT];
    u32 sum = 0;
#pragma unroll
    for (int i = 0; i < SC_IPT; ++i)
    {
        v[i] = b0 + i < n ? colpairs[b0 + i] : 0u;
        sum += v[i];
    }
    u32 incl = sum;
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
    u32 wpre = 0, total = 0;
#pragma unroll
    for (int w = 0; w < SC_THREADS / 32; ++w)
    {
        const u32 c = s_w[w];
        if (w < warp)
            wpre += c;
        total += c;
    }
    if (warp == 0)
    {
        const u64 prefix = warp_lookback(status, tile, (u64)total, lane);
        if (lane == 0)
            s_prefix = prefix;
    }
    __syncthreads();
    u32 run = (u32)s_prefix + wpre + incl - sum;
#pragma unroll
    for (int i = 0; i < SC_IPT; ++i)
    {
        if (b0 + i <= n)
            pstart[b0 + i] = run;
        run += v[i];
    }
}

// run descriptor: [region rank : 2][position of the run's first record : 32][records : 11]
static_assert(CH_RUN_MAX < (1u << 11) && CH_RECORDS <= CH_RUN_MAX, "a run's records must fit the descriptor's count");
__device__ __forceinline__ u64 run_entry(u32 rank, u32 pos, u32 cnt) { return ((u64)rank << 43) | ((u64)pos << 11) | (u64)cnt; }

// A warp drops the pairs of RB_CHUNKS chunks into their columns' buckets; colpairs counts DOWN: afterwards it is zero
// again.  The way of a pair is a chain of four dependent memory operations (chunk info -> column -> bucket start and
// ticket -> store): the chunks of a warp travel it side by side (measured: one chunk per warp 0.103 ms for the FEM
// matrix's 10.7 M pairs, latency-bound at 86 % occupancy).
constexpr int RB_CHUNKS = 4;
__global__ void __launch_bounds__(256)
run_bucket_kernel(const uint2 *__restrict__ chunkinfo, const u32 *__restrict__ chunkstart, u32 nchunks,
                  const u32 *__restrict__ pcol, const u32 *__restrict__ pinfo, int colbits, u32 me, RunRegions reg,
                  const u32 *__restrict__ pstart, u32 *__restrict__ colpairs, u64 *__restrict__ bucket)
{
    const int lane = threadIdx.x & 31;
    const u32 c0 = (blockIdx.x * 8 + (threadIdx.x >> 5)) * RB_CHUNKS;
    if (c0 >= nchunks)
        return;
    const u32 cmask = (1u << colbits) - 1u;
    uint2 info[RB_CHUNKS];
    u32 start[RB_CHUNKS], most = 0;
#pragma unroll
    for (int u = 0; u < RB_CHUNKS; ++u)
    {
        info[u] = make_uint2(0u, 0u);
        start[u] = 0u;
        if (c0 + u < nchunks)
        {
            info[u] = chunkinfo[c0 + u];
            start[u] = chunkstart[c0 + u];
        }
        most = max(most, info[u].y);
    }
    for (u32 j = lane; j < most; j += 32)
    {
        u32 g[RB_CHUNKS], pi[RB_CHUNKS], slot[RB_CHUNKS];
        bool mine[RB_CHUNKS];
#pragma unroll
        for (int u = 0; u < RB_CHUNKS; ++u)
        {
            g[u] = j < info[u].y ? pcol[info[u].x + j] : ~0u;
            pi[u] = j < info[u].y ? pinfo[info[u].x + j] : 0u;
        }
#pragma unroll
        for (int u = 0; u < RB_CHUNKS; ++u)
        { // records of other ranks (sent already) and padding are skipped
            mine[u] = j < info[u].y && (g[u] >> colbits) == me;
            slot[u] = 0u;
            if (mine[u])
                slot[u] = pstart[g[u] & cmask] + atomicSub(colpairs + (g[u] & cmask), 1u) - 1u;
        }
#pragma unroll
        for (int u = 0; u < RB_CHUNKS; ++u)
            if (mine[u])
            {
                const u32 rank = start[u] < reg.own_end ? 1u : (start[u] < reg.low_end ? 0u : 2u);
                bucket[slot[u]] = run_entry(rank, start[u] + (pi[u] >> 16), pi[u] & 0xffffu);
            }
    }
}

// ------------------------------------------------------------------------
// one THREAD per column: merge the column of the resident CSC with the column's runs
// ------------------------------------------------------------------------
constexpr u32 RF_EMPTY = 0xffffffffu;

// Table shapes, smallest first.  The template argument is the number of hash bits, except 15 = the
// 5-bit table with 16 instead of 24 accumulators (a P1 tetrahedral mesh has at most 15 rows per column).
//   shape  4: 16 slots / 12 accumulators     shape 15: 32 / 16     shape 5: 32 / 24     shape 6: 64 / 32
template <int HBITS> struct RfShape
{
    static constexpr int HB = HBITS == 15 ? 5 : HBITS;
    static constexpr int H = 1 << HB;
    static constexpr int D = HBITS == 6 ? 32 : (HBITS == 5 ? 24 : (HBITS == 15 ? 16 : 12));
    // warps per block; blocks per SM that shared memory and the register file allow.  The largest shape takes
    // 544 B of shared memory per thread: one-warp blocks fit 12 warps per SM where four-warp blocks fit 8
    // (measured on the block reaction-diffusion system: 2.65 -> 2.34 ms; the small shapes lose with tiny blocks).
    // The 32/16 shape takes 272 B per thread: five blocks of five warps = 25 warps per SM (four-warp blocks: 24).
    static constexpr int kWarps = HBITS == 6 ? 1 : (HBITS == 15 ? 5 : 4);
    static constexpr int kBlocks = HBITS == 4 ? 8 : (HBITS == 6 ? 12 : 5);
    static constexpr size_t kBytesPerWarp = 32 * (sizeof(u32) * H + (sizeof(double) + 1) * D);
};

// The fold state of one column.  A table slot holds (row << HB | accumulator index); accumulators are
// numbered in order of first appearance.  Flavour semantics (single partition): src/matrix/sparsematrixlnk.jl
// :178-253 behind the CSC-hit router src/matrix/extendable.jl:159-218.
template <int HBITS, bool ASSIGN> struct ThreadFold
{
    static constexpr int H = RfShape<HBITS>::H;
    static constexpr int HB = RfShape<HBITS>::HB;
    static constexpr u32 D = RfShape<HBITS>::D;
    u32 *key;    // [slot * 32]
    double *acc; // [i * 32]
    unsigned char *ord; // [i * 32]: table slot of accumulator i (its row = key >> HB)
    u32 d = 0;       // accumulators in use
    u32 pending = 0; // of which not (yet) existing: only updateindex! / setindex! of a zero touched them
    u32 exmask = 0;  // accumulator i holds an existing entry (D <= 32)
    bool ovf = false;

    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int s = 0; s < H; ++s)
            key[s * 32] = RF_EMPTY;
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
            if (x < D || kk == RF_EMPTY)
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
};

template <int HBITS, typename Ti, bool ASSIGN>
__global__ void __launch_bounds__(RfShape<HBITS>::kWarps * 32, RfShape<HBITS>::kBlocks)
runfold_kernel(const Rec *__restrict__ buf, int low, int rowbits, u32 maxlen, const u32 *__restrict__ pstart,
               u64 *__restrict__ bucket, const Ti *__restrict__ old_colptr, const Ti *__restrict__ old_rowval,
               const double *__restrict__ old_nzval, i64 ncols, Ti base, Ti *__restrict__ rowval,
               double *__restrict__ nzval, Ti *__restrict__ colptr, u64 *__restrict__ status, u32 *__restrict__ ticket,
               u64 *__restrict__ d_nnz, u32 *__restrict__ d_redo, u32 *__restrict__ maxd)
{
    typedef RfShape<HBITS> Shape;
    constexpr int RF_WARPS = Shape::kWarps;
    constexpr int H = Shape::H;
    constexpr int HB = Shape::HB;
    constexpr u32 D = Shape::D;
    constexpr u32 full = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ u32 s_wsum[RF_WARPS];
    __shared__ u64 s_prefix;
    __shared__ u32 s_bid;
    // blocks take their columns in the order they START (ticket), so a block only ever waits for
    // blocks that are already running: the look-back cannot starve whatever the dispatch order
    if (threadIdx.x == 0)
        s_bid = atomicAdd(ticket, 1u);
    __syncthreads();
    const u32 bid = s_bid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ThreadFold<HBITS, ASSIGN> f;
    f.acc = reinterpret_cast<double *>(smem_raw) + warp * (D * 32) + lane;
    f.key = reinterpret_cast<u32 *>(smem_raw + (size_t)RF_WARPS * D * 32 * sizeof(double)) + warp * (H * 32) + lane;
    f.ord = smem_raw + (size_t)RF_WARPS * 32 * (D * sizeof(double) + H * sizeof(u32)) + warp * (D * 32) + lane;
    const u32 rowmask = (1u << rowbits) - 1u;
    const i64 k = (i64)bid * (RF_WARPS * 32) + threadIdx.x;
    int j = 0;           // entries of this column in the new matrix
    i64 os = 0, oe = 0;  // its entries in the resident matrix
    bool copy = false;   // no new records: the old column is copied
    if (k < ncols && ld_relaxed_u32(d_redo) == 0u)
    {
        if (old_colptr != nullptr)
        {
            os = (i64)old_colptr[k] - (i64)base;
            oe = (i64)old_colptr[k + 1] - (i64)base;
        }
        const u32 ps = pstart[k], np = pstart[k + 1] - ps;
        if (np == 0)
        {
            copy = true;
            j = (int)(oe - os);
        }
        else if (np > kMaxColPairs || (u64)(oe - os) > (u64)D)
            atomicOr(d_redo, np > kMaxColPairs ? 2u : (HBITS == 6 ? 5u : 1u));
        else
        {
            // ---- the column's run descriptors, in stream order.  Up to W of them (the usual case) are loaded at
            // once and ordered in registers by a sorting network; a column met by more chunks orders its bucket in
            // place first (insertion sort: the descriptors arrive nearly in order) and reads it W at a time.
            // W descriptors in registers (8; the small table shape serves short columns met by few chunks: 4)
            constexpr int W = HBITS == 4 ? 4 : 8;
            // Sectors in flight ahead of the one being folded.  With 24 warps per SM the warps hide each other's loads:
            // a deeper software pipeline only costs instructions and registers (FEM: depth 3 / 2 / 1 = 1.44 (at 20
            // warps) / 1.30 / 1.24 ms); the 12 warps of the largest shape want one more (1.78 / 1.69 / 1.85 at 1 / 2 / 4)
            constexpr int DEPTH = (HBITS == 4 || HBITS == 15) ? 1 : 2;
            u64 *b = bucket + ps;
            if (np > (u32)W)
            {
                u64 prev = b[0];
                for (u32 i = 1; i < np; ++i)
                {
                    const u64 e = b[i];
                    if (e < prev)
                    {
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
            }
            u64 e[W];
            u32 loaded = 0; // descriptors fetched so far
            auto fetch = [&]() {
#pragma unroll
                for (int i = 0; i < W; ++i)
                    e[i] = loaded + (u32)i < np ? b[loaded + (u32)i] : ~0ull;
                loaded += (u32)W;
            };
            fetch();
            u32 nrec = 0;
            if (np <= (u32)W)
            {
                auto cx = [&](int x, int y) {
                    const u64 lo_ = e[x] < e[y] ? e[x] : e[y], hi_ = e[x] < e[y] ? e[y] : e[x];
                    e[x] = lo_;
                    e[y] = hi_;
                };
                if (W == 8)
                { // 19-comparator network for 8 keys
                    cx(0, 1), cx(2, 3), cx(4, 5), cx(6, 7);
                    cx(0, 2), cx(1, 3), cx(4, 6), cx(5, 7);
                    cx(1, 2), cx(5, 6), cx(0, 4), cx(3, 7);
                    cx(1, 5), cx(2, 6);
                    cx(1, 4), cx(3, 6);
                    cx(2, 4), cx(3, 5);
                    cx(3, 4);
                }
                else
                {
                    cx(0, 1), cx(2, 3);
                    cx(0, 2), cx(1, 3);
                    cx(1, 2);
                }
#pragma unroll
                for (int i = 0; i < W; ++i)
                    nrec += e[i] != ~0ull ? (u32)(e[i] & 0x7ffull) : 0u;
            }
            else
            { // ordered in place above: read in order
                for (u32 i = 0; i < np; ++i)
                    nrec += (u32)(b[i] & 0x7ffull);
            }
            if (nrec > maxlen)
                atomicOr(d_redo, 2u); // a very long column would stall its warp: the caller takes another path
            else
            {
                f.init();
                // ---- the resident column seeds the table (CSC hits: extendable.jl:164-166)
                for (i64 eo = os; eo < oe; ++eo)
                    f.seed((u32)((i64)old_rowval[eo] - (i64)base), old_nzval[eo]);
                // ---- the runs, where the producers left them.  Every step a lane takes the aligned 32-byte
                // sector (two records, one LDG.256) its cursor stands in and folds the one or two records of it
                // that belong to its run: the same instruction stream for every lane whatever the run lengths;
                // DEPTH sectors travel ahead of the one being folded.
                // Positions are counted in records from the 32-byte boundary at or below buf: their parity is the
                // record's place inside its sector.
                const uintptr_t bufa = reinterpret_cast<uintptr_t>(buf);
                const u32 bias = (u32)(bufa >> 4) & 1u;
                const unsigned char *base32 = reinterpret_cast<const unsigned char *>(bufa & ~(uintptr_t)31);
                u32 used = 0, rem = 0, left = nrec, pos = 0; // used: descriptors of the register window consumed
                RecPair q[DEPTH];
                u32 m[DEPTH];
                auto gen = [&](RecPair &qq, u32 &mm) {
                    if (left == 0u)
                    {
                        mm = 0u;
                        return;
                    }
                    if (rem == 0u)
                    { // next run: the head of the register window
                        if (used == (u32)W)
                        {
                            fetch();
                            used = 0u;
                        }
                        pos = (u32)(e[0] >> 11) + bias;
                        rem = (u32)(e[0] & 0x7ffull);
#pragma unroll
                        for (int i = 0; i + 1 < W; ++i)
                            e[i] = e[i + 1];
                        ++used;
                    }
                    mm = (pos & 1u) ? 2u : (rem > 1u ? 3u : 1u); // which records of the sector belong to the run
                    const u32 take = (mm + 1u) >> 1;
                    const unsigned char *sec = base32 + (size_t)(pos >> 1) * 32u;
                    qq = ld_pair_stream(reinterpret_cast<const Rec *>(sec));
                    if (rem >= 8u) // long run: pull the sector some steps ahead from HBM into L2 meanwhile
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(sec + 96));
                    pos += take;
                    rem -= take;
                    left -= take;
                };
#pragma unroll
                for (int k = 0; k < DEPTH; ++k)
                    gen(q[k], m[k]);
                // one step: fold the records of sector k, then send its buffer for the sector DEPTH ahead
                for (bool done = false; !done;)
                {
#pragma unroll
                    for (int k = 0; k < DEPTH; ++k)
                    {
                        if (m[k] == 0u || f.ovf)
                        {
                            done = true;
                            break;
                        }
                        const RecPair c = q[k];
                        const u32 mm = m[k];
                        gen(q[k], m[k]);
                        if (mm & 1u)
                            f.apply((u32)(c.a.key >> low) & rowmask, c.a.val, (u32)c.a.key & 3u);
                        if ((mm & 2u) && !f.ovf)
                            f.apply((u32)(c.b.key >> low) & rowmask, c.b.val, (u32)c.b.key & 3u);
                    }
                }
                if (f.ovf)
                { // bit 2: not even the largest table takes this column
                    atomicOr(d_redo, HBITS == 6 ? 5u : 1u);
                    if (D + 1 > ld_relaxed_u32(maxd))
                        atomicMax(maxd, D + 1);
                }
                else
                {
                    j = f.finish();
                    if (f.d > ld_relaxed_u32(maxd))
                        atomicMax(maxd, f.d);
                }
            }
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
    for (int w = 0; w < RF_WARPS; ++w)
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
    if (k >= ncols)
        return;
    const u64 o0 = s_prefix + wpre + (incl - (u32)j);
    colptr[k] = (Ti)o0 + base;
    if (k == ncols - 1)
    {
        colptr[ncols] = (Ti)(o0 + (u64)j) + base;
        *d_nnz = o0 + (u64)j;
    }
    if (copy)
    { // untouched column: old entries move to their new place (read once, written once)
        const Ti *srv = old_rowval + os;
        const double *snv = old_nzval + os;
        Ti *rv = rowval + o0;
        double *nv = nzval + o0;
        for (int e = 0; e < j; ++e)
        {
            rv[e] = srv[e];
            nv[e] = snv[e];
        }
        return;
    }
    // 256-bit stores where the destination is 32-byte aligned (rowval and nzval separately: their
    // bases differ): a lane writes its own run, so every store instruction costs one request per lane
    {
        Ti *rv = rowval + o0;
        auto row_at = [&](int e) { return (Ti)(f.key[e * 32] >> HB) + base; };
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
        auto val_at = [&](int e) { return (u64)__double_as_longlong(f.acc[(f.key[e * 32] & (H - 1)) * 32]); };
        int e = 0;
        for (; e < j && (reinterpret_cast<uintptr_t>(nv + e) & 31u); ++e)
            nv[e] = __longlong_as_double((long long)val_at(e));
        for (; e + 4 <= j; e += 4)
            st_v4_u64(nv + e, val_at(e), val_at(e + 1), val_at(e + 2), val_at(e + 3));
        for (; e < j; ++e)
            nv[e] = __longlong_as_double((long long)val_at(e));
    }
}

// ------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------
namespace {
struct RwLayout
{
    size_t off_colpairs, off_status, off_fstatus, off_pstart, off_bucket, clear_bytes, bytes;
};
RwLayout rw_layout(u64 npairs, i64 ncols)
{
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const u64 stiles = ((u64)ncols + 1 + SC_TILE - 1) / SC_TILE;
    const u64 fblocks = ((u64)ncols + 31) / 32; // look-back words of the merge kernel: room for one-warp blocks
    RwLayout l{};
    size_t o = 0;
    // cleared by one memset: pairs per column, look-back words + tickets of the scan and of the fold
    l.off_colpairs = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 1));
    l.off_status = o;
    o = up(o + sizeof(u64) * (stiles + 2));
    l.off_fstatus = o;
    o = up(o + sizeof(u64) * (fblocks + 2));
    l.clear_bytes = o;
    l.off_pstart = o;
    o = up(o + sizeof(u32) * ((size_t)ncols + 2));
    l.off_bucket = o;
    o = up(o + sizeof(u64) * ((size_t)npairs + 1));
    l.bytes = o;
    return l;
}
} // namespace

RunIndexLayout run_index_layout(u64 cap_records)
{
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    RunIndexLayout l{};
    l.cap_pairs = (u32)std::min<u64>(cap_records / 8 * 3 + 4096, 0xfffffff0ull); // 7-point FD streams: ~0.27 per record
    l.cap_chunks = (u32)std::min<u64>(cap_records / 128 + 4096, 0xfffffff0ull);
    size_t o = 0;
    l.off_counters = o;
    o = up(o + 256);
    l.off_chunkinfo = o;
    o = up(o + sizeof(uint2) * ((size_t)l.cap_chunks + 1));
    l.off_chunkstart = o;
    o = up(o + sizeof(u32) * ((size_t)l.cap_chunks + 1));
    l.off_pcol = o;
    o = up(o + sizeof(u32) * ((size_t)l.cap_pairs + 1));
    l.off_pinfo = o;
    o = up(o + sizeof(u32) * ((size_t)l.cap_pairs + 1));
    l.bytes = o;
    return l;
}

RunTarget run_target(void *workspace, u64 cap_records, const KeyLayout &L)
{
    const RunIndexLayout l = run_index_layout(cap_records);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    RunTarget rt{};
    rt.counters = reinterpret_cast<u32 *>(ws + l.off_counters);
    rt.chunkinfo = reinterpret_cast<uint2 *>(ws + l.off_chunkinfo);
    rt.chunkstart = reinterpret_cast<u32 *>(ws + l.off_chunkstart);
    rt.pcol = reinterpret_cast<u32 *>(ws + l.off_pcol);
    rt.pinfo = reinterpret_cast<u32 *>(ws + l.off_pinfo);
    rt.cap = l.cap_pairs;
    rt.colshift = L.low + L.rowbits;
    rt.gmask = (1u << (L.colbits + L.ownerbits)) - 1u;
    return rt;
}

// records below 2^32 (positions are 32-bit), thread-table keys hold (row << 6 | index), the grouping key
// (column + owner bits) must stay below CH_EMPTY
bool runs_supported(const KeyLayout &L, u64 nrec, i64 ncols)
{
    return L.rowbits <= 26 && L.low <= 32 && L.tidbits == 0 && L.colbits + L.ownerbits <= 31 &&
           nrec < (1ull << 32) - 2048ull && (u64)ncols < (1ull << 31);
}

u32 chunk_sort_chunks(u64 count) { return (u32)((count + CH_RECORDS - 1) / CH_RECORDS); }

void chunk_sort(cudaStream_t stream, Rec *buf, u64 r0, u64 r1, const RunTarget &rt, u32 chunk0, LaunchCounter &lc)
{
    if (r1 <= r0)
        return;
    static FuncAttrOnce once;
    const int smem = (int)(sizeof(ChunkSpaceT<CS_HB>) * CS_WARPS);
    once.set(chunk_sort_kernel, smem);
    const u32 nchunks = chunk_sort_chunks(r1 - r0);
    chunk_sort_kernel<<<(nchunks + CS_WARPS - 1) / CS_WARPS, CS_WARPS * 32, smem, stream>>>(buf, r0, r1, chunk0, nchunks, rt);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

size_t runs_workspace_bytes(u64 npairs, i64 ncols) { return rw_layout(npairs, ncols).bytes; }

void runs_bucket(cudaStream_t stream, const RunTarget &rt, u32 nchunks, u32 npairs, i64 ncols, const KeyLayout &L,
                 RunRegions reg, void *workspace, LaunchCounter &lc)
{
    const RwLayout l = rw_layout(npairs, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *colpairs = reinterpret_cast<u32 *>(ws + l.off_colpairs);
    u64 *status = reinterpret_cast<u64 *>(ws + l.off_status);
    u32 *pstart = reinterpret_cast<u32 *>(ws + l.off_pstart);
    u64 *bucket = reinterpret_cast<u64 *>(ws + l.off_bucket);
    const u32 me = L.ownerbits ? (u32)L.self : 0u;
    XSB_CUDA(cudaMemsetAsync(ws, 0, l.clear_bytes, stream));
    run_totals_kernel<<<kNumSM * 8, 256, 0, stream>>>(rt.counters, rt.cap, rt.pcol, L.colbits, me, colpairs);
    const unsigned stiles = (unsigned)(((u64)ncols + 1 + SC_TILE - 1) / SC_TILE);
    runpair_scan_kernel<<<stiles, SC_THREADS, 0, stream>>>(colpairs, ncols, pstart, status,
                                                           reinterpret_cast<u32 *>(status + stiles + 1));
    run_bucket_kernel<<<(nchunks + 8 * RB_CHUNKS - 1) / (8 * RB_CHUNKS), 256, 0, stream>>>(rt.chunkinfo, rt.chunkstart, nchunks, rt.pcol, rt.pinfo,
                                                             L.colbits, me, reg, pstart, colpairs, bucket);
    lc.add(3);
    XSB_CUDA(cudaGetLastError());
}

namespace {
template <int HBITS, typename Ti, bool ASSIGN>
void launch_runfold_t(cudaStream_t stream, unsigned blocks, const Rec *buf, int low, int rowbits, u32 maxlen,
                      const u32 *pstart, u64 *bucket, const CscView &old, i64 ncols, i64 base, void *rowval, double *nzval,
                      void *colptr, u64 *status, u32 *ticket, u64 *d_nnz, u32 *d_redo, u32 *maxd)
{
    constexpr int RF_WARPS = RfShape<HBITS>::kWarps;
    constexpr size_t smem = RF_WARPS * RfShape<HBITS>::kBytesPerWarp;
    static FuncAttrOnce once;
    once.set(runfold_kernel<HBITS, Ti, ASSIGN>, (int)smem, true);
    const bool has_old = old.nnz > 0;
    runfold_kernel<HBITS, Ti, ASSIGN><<<blocks, RF_WARPS * 32, smem, stream>>>(
        buf, low, rowbits, maxlen, pstart, bucket, has_old ? (const Ti *)old.colptr : nullptr, (const Ti *)old.rowval,
        old.nzval, ncols, (Ti)base, (Ti *)rowval, nzval, (Ti *)colptr, status, ticket, d_nnz, d_redo, maxd);
}
} // namespace

// level 0..3 = table shapes 4, 15, 5, 6.  *d_redo afterwards: bit 0: a column did not fit the table (bit 2 as well:
// not even the largest one); bit 1: a column is too long / met by too many chunks for one thread.
void runs_fold(cudaStream_t stream, const Rec *buf, const KeyLayout &L, i64 ncols, int idx64, int base, const CscView &old,
               void *workspace, u32 npairs, int level, u32 maxlen, void *rowval_out, double *nzval_out, void *colptr_out,
               u64 *d_nnz, u32 *d_redo, u32 *d_maxd, bool first_try, bool has_assign, LaunchCounter &lc)
{
    const RwLayout l = rw_layout(npairs, ncols);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *pstart = reinterpret_cast<u32 *>(ws + l.off_pstart);
    u64 *bucket = reinterpret_cast<u64 *>(ws + l.off_bucket);
    u64 *status = reinterpret_cast<u64 *>(ws + l.off_fstatus);
    const unsigned tpb = 32u * (unsigned)(level == 3 ? RfShape<6>::kWarps
                                                      : (level == 2 ? RfShape<5>::kWarps
                                                                    : (level == 1 ? RfShape<15>::kWarps : RfShape<4>::kWarps)));
    const unsigned blocks = (unsigned)(((u64)ncols + tpb - 1) / tpb);
    u32 *ticket = reinterpret_cast<u32 *>(status + blocks + 1);
    if (!first_try) // look-back words + ticket were cleared with the bucket workspace the first time
        XSB_CUDA(cudaMemsetAsync(status, 0, sizeof(u64) * ((size_t)((u64)ncols + 31) / 32 + 2), stream));
    XSB_CUDA(cudaMemsetAsync(d_redo, 0, sizeof(u32), stream));
    XSB_CUDA(cudaMemsetAsync(d_maxd, 0, sizeof(u32), stream));
#define XSB_RUNFOLD(HB, TI)                                                                                             \
    do                                                                                                                  \
    {                                                                                                                   \
        if (has_assign)                                                                                                 \
            launch_runfold_t<HB, TI, true>(stream, blocks, buf, L.low, L.rowbits, maxlen, pstart, bucket, old, ncols,   \
                                           base, rowval_out, nzval_out, colptr_out, status, ticket, d_nnz, d_redo,     \
                                           d_maxd);                                                                     \
        else                                                                                                            \
            launch_runfold_t<HB, TI, false>(stream, blocks, buf, L.low, L.rowbits, maxlen, pstart, bucket, old, ncols,  \
                                            base, rowval_out, nzval_out, colptr_out, status, ticket, d_nnz, d_redo,    \
                                            d_maxd);                                                                    \
    } while (0)
    if (idx64)
    {
        if (level == 0)
            XSB_RUNFOLD(4, int64_t);
        else if (level == 1)
            XSB_RUNFOLD(15, int64_t);
        else if (level == 2)
            XSB_RUNFOLD(5, int64_t);
        else
            XSB_RUNFOLD(6, int64_t);
    }
    else
    {
        if (level == 0)
            XSB_RUNFOLD(4, int32_t);
        else if (level == 1)
            XSB_RUNFOLD(15, int32_t);
        else if (level == 2)
            XSB_RUNFOLD(5, int32_t);
        else
            XSB_RUNFOLD(6, int32_t);
    }
#undef XSB_RUNFOLD
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// table shape for columns with at most `maxd` distinct rows
int runs_level_for(u32 maxd) { return maxd <= 12 ? 0 : (maxd <= 16 ? 1 : (maxd <= 24 ? 2 : 3)); }

} // namespace xsb
