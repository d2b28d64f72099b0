// xsb_flush.cu -- the flush! kernels that follow the sort:
//   expand_csc_records : resident CSC -> FL_OLD records (so old entries seed the fold)
//   reduce_emit_kernel : stable segmented reduction of duplicate (col,row) runs and
//                        compaction into rowval/nzval, single pass with decoupled look-back
//   colptr kernels     : running maximum over per-column end markers -> colptr
//
// Reference counterpart: Base.:+(lnk,csc) src/matrix/sparsematrixlnk.jl:294-383 (gather,
// sort, 3-way merge per column) and the accumulate-on-insert of :210-253; multi-partition
// semantics of Base.sum(Vector{SparseMatrixDILNKC},csc) src/matrix/sparsematrixdilnkc.jl:397-435.
#include "xsb_fold.cuh"
#include "xsb_internal.h"

namespace xsb {

template <typename Ti>
__global__ void __launch_bounds__(256)
expand_csc_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, const double *__restrict__ nzval,
                  i64 n, Ti base, KeyLayout L, Rec *__restrict__ out)
{
    // one warp per column: lanes stride over the column's entries -> coalesced 16-byte stores
    const i64 warp = ((i64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const i64 nwarps = ((i64)gridDim.x * blockDim.x) >> 5;
    for (i64 j = warp; j < n; j += nwarps)
    {
        const i64 s = (i64)colptr[j] - base, e = (i64)colptr[j + 1] - base;
        for (i64 k = s + lane; k < e; k += 32)
        {
            Rec r;
            r.key = L.pack((u64)j, (u64)((i64)rowval[k] - base), 0u, FL_OLD);
            r.val = nzval[k];
            st_rec(out + k, r);
        }
    }
}

void expand_csc_records(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, KeyLayout L,
                        Rec *out, LaunchCounter &lc)
{
    if (csc.nnz == 0)
        return;
    const int threads = 256;
    const i64 want = (n * 32 + threads - 1) / threads;
    const int blocks = (int)std::min<i64>(std::max<i64>(want, 1), (i64)kNumSM * 16);
    if (idx64)
        expand_csc_kernel<int64_t><<<blocks, threads, 0, stream>>>(
            (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, csc.nzval, n, (int64_t)base, L, out);
    else
        expand_csc_kernel<int32_t><<<blocks, threads, 0, stream>>>(
            (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, csc.nzval, n, (int32_t)base, L, out);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------
// segmented duplicate reduction + compaction
// ------------------------------------------------------------------------
constexpr int RD_THREADS = 256;
constexpr int RD_WARPS = RD_THREADS / 32;
constexpr int RD_IPT = 8;
constexpr int RD_TILE = RD_THREADS * RD_IPT;
constexpr int RD_OVER = 64;

constexpr u64 RS_LOCAL = 1ull << 62;
constexpr u64 RS_INCL = 2ull << 62;
constexpr u64 RS_VALUE = (1ull << 62) - 1ull;

// Order-preserving compaction ranks for flags laid out as (step i, thread): returns the
// exclusive rank of every set flag and the total.  s_cnt/s_off hold RD_IPT*RD_WARPS words.
__device__ __forceinline__ u32 block_rank_flags(const bool (&flag)[RD_IPT], u32 (&rank)[RD_IPT], u32 *s_cnt,
                                                u32 *s_off, u32 *s_total, int lane, int warp, u32 lt)
{
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
    {
        const u32 bal = __ballot_sync(0xffffffffu, flag[i]);
        if (lane == 0)
            s_cnt[i * RD_WARPS + warp] = __popc(bal);
        rank[i] = __popc(bal & lt);
    }
    __syncthreads();
    if (warp == 0)
    {
        constexpr int PER = RD_IPT * RD_WARPS / 32;
        u32 c[PER], sum = 0;
#pragma unroll
        for (int k = 0; k < PER; ++k)
        {
            c[k] = s_cnt[lane * PER + k];
            sum += c[k];
        }
        u32 incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o)
                incl += t;
        }
        u32 run = incl - sum;
#pragma unroll
        for (int k = 0; k < PER; ++k)
        {
            s_off[lane * PER + k] = run;
            run += c[k];
        }
        if (lane == 31)
            *s_total = incl;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
        rank[i] += s_off[i * RD_WARPS + warp];
    return *s_total;
}

// One tile of RD_TILE sorted records: find the heads of the duplicate runs, compact them so that
// every lane folds one run (a run is folded sequentially in insertion order, which is what makes
// the result bit-exact), compact the created entries and write them at the tile's output offset
// (decoupled look-back over the tiles' entry counts).
// SIMPLE: single partition, no assign flavour, seed combine -- the fold is a plain running sum.
template <typename Ti, bool SIMPLE>
__global__ void __launch_bounds__(RD_THREADS)
reduce_emit_kernel(const Rec *__restrict__ sorted, u64 nrec, KeyLayout L, int combine, Ti base,
                   Ti *__restrict__ rowval, double *__restrict__ nzval, u64 *__restrict__ colend,
                   u64 *__restrict__ status, u32 *__restrict__ tile_counter, u64 *__restrict__ d_nnz, u32 ntiles)
{
    __shared__ Rec s_rec[RD_TILE + RD_OVER]; // tile + look-ahead for the run that crosses the tile's end
    __shared__ u32 s_col[RD_TILE]; // first the head positions, later the columns of the output entries
    __shared__ u32 s_cnt[RD_IPT * RD_WARPS];
    __shared__ u32 s_off[RD_IPT * RD_WARPS];
    __shared__ u64 s_prev, s_tileoff;
    __shared__ u32 s_tile, s_total;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0)
        s_tile = atomicAdd(tile_counter, 1u);
    __syncthreads();
    const u32 tile = s_tile;
    const u64 tbase = (u64)tile * RD_TILE;
    const u32 valid = (u32)min((u64)RD_TILE, nrec - tbase);

#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
    {
        const u32 e = i * RD_THREADS + tid;
        if (e < valid)
            s_rec[e] = ld_rec_stream(sorted + tbase + e);
    }
    const u32 avail = (u32)min((u64)(RD_TILE + RD_OVER), nrec - tbase);
    if (tid < RD_OVER && RD_TILE + tid < avail)
        s_rec[RD_TILE + tid] = ld_rec_stream(sorted + tbase + RD_TILE + tid);
    if (tid == 0)
        s_prev = tbase > 0 ? sorted[tbase - 1].key : 0ull;
    __syncthreads();

    const u32 lt = lanemask_lt();
    bool flag[RD_IPT];
    u32 rank[RD_IPT];

    // ---- heads of the runs of equal (col,row), compacted into s_col[0..nheads)
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
    {
        const u32 e = i * RD_THREADS + tid;
        bool head = false;
        if (e < valid)
        {
            const u64 cr = L.colrow(s_rec[e].key);
            if (e > 0)
                head = cr != L.colrow(s_rec[e - 1].key);
            else
                head = (tbase == 0) || cr != L.colrow(s_prev);
        }
        flag[i] = head;
    }
    const u32 nheads = block_rank_flags(flag, rank, s_cnt, s_off, &s_total, lane, warp, lt);
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
        if (flag[i])
            s_col[rank[i]] = i * RD_THREADS + tid;
    __syncthreads();

    // ---- one run per lane
    double myval[RD_IPT];
    u32 myrow[RD_IPT], mycol[RD_IPT];
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
    {
        const u32 hidx = i * RD_THREADS + tid;
        bool created = false;
        double out = 0.0;
        u32 row = 0, col = 0;
        if (i * RD_THREADS < nheads) // uniform: rounds beyond the last head are skipped by the whole block
        {
            if (hidx < nheads)
            {
                const u32 e0 = s_col[hidx];
                const bool last = hidx + 1 == nheads;
                const u32 e1 = last ? avail : s_col[hidx + 1]; // the last run ends where its key ends
                const u64 key = s_rec[e0].key;
                const u64 cr = L.colrow(key);
                row = (u32)L.row(key);
                col = (u32)L.col(key);
                if (SIMPLE)
                {
                    double acc = 0.0;
                    u32 q = e0;
                    for (; q < e1; ++q)
                    {
                        const Rec r = s_rec[q];
                        if (q >= valid && L.colrow(r.key) != cr)
                            break;
                        const u32 fl = L.flavour(r.key);
                        acc = (fl == FL_OLD) ? r.val : acc + r.val;
                        created |= (fl != FL_UPDATE) | (r.val != 0.0);
                    }
                    if (last && q == avail) // longer than the look-ahead: rare, walk global memory
                        for (u64 g = tbase + avail; g < nrec; ++g)
                        { // the tile's last run may continue into the following tiles
                            const Rec r = sorted[g];
                            if (L.colrow(r.key) != cr)
                                break;
                            acc = acc + r.val;
                            created |= (L.flavour(r.key) != FL_UPDATE) | (r.val != 0.0);
                        }
                    out = acc;
                }
                else
                {
                    RunFold f;
                    u32 q = e0;
                    for (; q < e1; ++q)
                    {
                        const Rec r = s_rec[q];
                        if (q >= valid && L.colrow(r.key) != cr)
                            break;
                        f.apply(L.flavour(r.key), L.tid(r.key), r.val, combine);
                    }
                    if (last && q == avail)
                        for (u64 g = tbase + avail; g < nrec; ++g)
                        {
                            const Rec r = sorted[g];
                            if (L.colrow(r.key) != cr)
                                break;
                            f.apply(L.flavour(r.key), L.tid(r.key), r.val, combine);
                        }
                    f.finish();
                    created = f.exists;
                    out = f.acc;
                }
            }
        }
        flag[i] = created;
        myval[i] = out;
        myrow[i] = row;
        mycol[i] = col;
    }
    __syncthreads(); // s_col (head positions) is dead from here on
    const u32 total = block_rank_flags(flag, rank, s_cnt, s_off, &s_total, lane, warp, lt);

    // ---- decoupled look-back over the tiles' entry counts, 32 predecessors per step
    if (warp == 0)
    {
        u64 prefix = 0;
        if (tile == 0)
        {
            if (lane == 0)
                st_relaxed_u64(status, RS_INCL | (u64)total);
        }
        else
        {
            if (lane == 0)
                st_relaxed_u64(status + tile, RS_LOCAL | (u64)total);
            i64 t = (i64)tile - 1;
            for (;;)
            {
                const i64 idx = t - lane;
                u64 v = RS_INCL; // tiles before the first contribute nothing
                if (idx >= 0)
                {
                    do
                    {
                        v = ld_relaxed_u64(status + idx);
                    } while ((v >> 62) == 0ull);
                }
                const u32 incl_mask = __ballot_sync(0xffffffffu, (v >> 62) == 2ull);
                u64 contrib = v & RS_VALUE;
                if (incl_mask)
                {
                    const int first = __ffs(incl_mask) - 1;
                    if (lane > first)
                        contrib = 0;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
                    contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
                prefix += contrib;
                if (incl_mask)
                    break;
                t -= 32;
            }
            if (lane == 0)
                st_relaxed_u64(status + tile, RS_INCL | (prefix + total));
        }
        if (lane == 0)
        {
            s_tileoff = prefix;
            if (tile == ntiles - 1)
                *d_nnz = prefix + total;
        }
    }
    __syncthreads();

    const u64 tileoff = s_tileoff;
#pragma unroll
    for (int i = 0; i < RD_IPT; ++i)
    {
        if (flag[i])
        {
            const u64 p = tileoff + rank[i];
            rowval[p] = (Ti)myrow[i] + base;
            nzval[p] = myval[i];
            s_col[rank[i]] = mycol[i];
        }
    }
    __syncthreads();
    // last output entry of a column inside this tile marks the column's end
    for (u32 q = tid; q < total; q += RD_THREADS)
    {
        const u32 c = s_col[q];
        if (q + 1 == total || s_col[q + 1] != c)
            atomicMax(colend + c, tileoff + q + 1);
    }
}

// ------------------------------------------------------------------------
// colptr = base + running maximum of colend
// ------------------------------------------------------------------------
constexpr int CP_THREADS = 256;
constexpr int CP_IPT = 8;
constexpr int CP_TILE = CP_THREADS * CP_IPT;

__global__ void __launch_bounds__(CP_THREADS)
colend_tilemax_kernel(const u64 *__restrict__ colend, i64 n, u64 *__restrict__ tmax)
{
    __shared__ u64 s_w[CP_THREADS / 32];
    const i64 b0 = (i64)blockIdx.x * CP_TILE;
    u64 m = 0;
#pragma unroll
    for (int i = 0; i < CP_IPT; ++i)
    {
        const i64 j = b0 + i * CP_THREADS + threadIdx.x;
        if (j < n)
            m = max(m, colend[j]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0)
        s_w[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        for (int w = 1; w < CP_THREADS / 32; ++w)
            m = max(m, s_w[w]);
        tmax[blockIdx.x] = m;
    }
}

// single block: in-place inclusive running maximum over the tile maxima
__global__ void __launch_bounds__(1024) tilemax_scan_kernel(u64 *__restrict__ tmax, i64 nt)
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
        u64 v = j < nt ? tmax[j] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u64 t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o)
                v = max(v, t);
        }
        if (lane == 31)
            s_w[warp] = v;
        __syncthreads();
        u64 pre = s_carry;
        for (int w = 0; w < warp; ++w)
            pre = max(pre, s_w[w]);
        v = max(v, pre);
        if (j < nt)
            tmax[j] = v;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = v;
        __syncthreads();
    }
}

template <typename Ti>
__global__ void __launch_bounds__(CP_THREADS)
colptr_emit_kernel(const u64 *__restrict__ colend, const u64 *__restrict__ tmax, i64 n, Ti base,
                   Ti *__restrict__ colptr)
{
    __shared__ u64 s_w[CP_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // blocked layout: thread t owns columns b0 + t*CP_IPT .. +CP_IPT-1
    const i64 b0 = (i64)blockIdx.x * CP_TILE + (i64)threadIdx.x * CP_IPT;
    u64 v[CP_IPT];
    u64 m = 0;
#pragma unroll
    for (int i = 0; i < CP_IPT; ++i)
    {
        const i64 j = b0 + i;
        const u64 c = j < n ? colend[j] : 0;
        m = max(m, c);
        v[i] = m;
    }
    u64 incl = m;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u64 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl = max(incl, t);
    }
    if (lane == 31)
        s_w[warp] = incl;
    __syncthreads();
    u64 pre = blockIdx.x > 0 ? tmax[blockIdx.x - 1] : 0;
    for (int w = 0; w < warp; ++w)
        pre = max(pre, s_w[w]);
    const u64 up = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane > 0)
        pre = max(pre, up);
#pragma unroll
    for (int i = 0; i < CP_IPT; ++i)
    {
        const i64 j = b0 + i;
        if (j < n)
            colptr[j + 1] = (Ti)max(v[i], pre) + base;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        colptr[0] = base;
}

size_t reduce_workspace_bytes(u64 nrec, i64 ncols)
{
    const u64 ntiles = (nrec + RD_TILE - 1) / RD_TILE;
    const u64 ctiles = ((u64)ncols + CP_TILE - 1) / CP_TILE;
    return sizeof(u64) * (size_t)ncols + sizeof(u64) * (ntiles + 1) + sizeof(u64) * (ctiles + 1) + 512;
}

void reduce_emit_csc(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, int combine, int mode,
                     bool plain_adds, i64 ncols, int idx64, int base, void *rowval_out, double *nzval_out,
                     void *colptr_out, void *workspace, u64 *d_nnz, LaunchCounter &lc, StageTimer *timer)
{
    (void)mode;
    const u64 ntiles = (nrec + RD_TILE - 1) / RD_TILE;
    const u64 ctiles = ((u64)ncols + CP_TILE - 1) / CP_TILE;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u32 *counter = reinterpret_cast<u32 *>(ws);
    u64 *colend = reinterpret_cast<u64 *>(ws + 256);
    u64 *status = colend + ncols;
    u64 *tmax = status + ntiles + 1;

    if (timer)
        timer->begin(stream);
    XSB_CUDA(cudaMemsetAsync(ws, 0, 256 + sizeof(u64) * ((size_t)ncols + ntiles + 1), stream));
    XSB_CUDA(cudaMemsetAsync(d_nnz, 0, sizeof(u64), stream));
    if (nrec > 0)
    {
        const bool simple = plain_adds && L.tidbits == 0 && combine == 0;
#define XSB_LAUNCH_REDUCE(TI, SIMPLE)                                                                            \
    reduce_emit_kernel<TI, SIMPLE><<<(unsigned)ntiles, RD_THREADS, 0, stream>>>(                                 \
        sorted, nrec, L, combine, (TI)base, (TI *)rowval_out, nzval_out, colend, status, counter, d_nnz, (u32)ntiles)
        if (idx64)
        {
            if (simple)
                XSB_LAUNCH_REDUCE(int64_t, true);
            else
                XSB_LAUNCH_REDUCE(int64_t, false);
        }
        else
        {
            if (simple)
                XSB_LAUNCH_REDUCE(int32_t, true);
            else
                XSB_LAUNCH_REDUCE(int32_t, false);
        }
#undef XSB_LAUNCH_REDUCE
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    if (timer)
        timer->end(stream, &StageTimes::reduce);

    if (timer)
        timer->begin(stream);
    colend_tilemax_kernel<<<(unsigned)ctiles, CP_THREADS, 0, stream>>>(colend, ncols, tmax);
    tilemax_scan_kernel<<<1, 1024, 0, stream>>>(tmax, (i64)ctiles);
    if (idx64)
        colptr_emit_kernel<int64_t><<<(unsigned)ctiles, CP_THREADS, 0, stream>>>(colend, tmax, ncols, (int64_t)base,
                                                                                 (int64_t *)colptr_out);
    else
        colptr_emit_kernel<int32_t><<<(unsigned)ctiles, CP_THREADS, 0, stream>>>(colend, tmax, ncols, (int32_t)base,
                                                                                 (int32_t *)colptr_out);
    lc.add(3);
    XSB_CUDA(cudaGetLastError());
    if (timer)
        timer->end(stream, &StageTimes::colptr);
}

} // namespace xsb
