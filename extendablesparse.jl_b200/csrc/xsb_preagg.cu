// xsb_preagg.cu -- XSB_FAST mode only: accumulate-on-insert inside small windows of the staged
// stream before anything is grouped or sorted.
//
// The reference never stores a duplicate: updateindex!/rawupdateindex! walk the column's list
// and add into the existing entry (src/matrix/sparsematrixlnk.jl:210-253).  Here a warp owns a
// chunk of PA_W consecutive staged records and folds them through a warp-private hash table in
// shared memory keyed by (column,row): an assembly stream revisits the same entries within a few
// elements (P1-FEM: 120 insertions per cube hit 46 entries), so 2.5-4x fewer records leave the
// kernel.  The partial sums are then grouped and folded per column like any other records; the
// value of an entry becomes a sum of partial sums instead of the left fold in insertion order
// (within gamma(N-1) * sum|x| of the exact sum, include/xsparse_b200.h XSB_FAST) and the pattern is unchanged:
//   rawupdateindex! always creates, updateindex! creates unless every value it saw was zero
//   (sparsematrixlnk.jl:212,223,239) -- a window whose records create nothing emits nothing.
// Not used when A[i,j] = v records are staged (assignment does not commute).
#include "xsb_internal.h"

namespace xsb {

constexpr int PA_W = 512;            // records per chunk (one warp)
constexpr int PA_NB = PA_W / 32;
constexpr int PA_HBITS = 9;
constexpr int PA_H = 1 << PA_HBITS;  // slots per warp: a chunk without duplicates fills it exactly
constexpr int PA_WARPS = 8;
constexpr u64 PA_EMPTY = ~0ull;

struct PreaggSpace
{
    u64 key[PA_H]; // (column,row) << 1 | creates
    double acc[PA_H];
};

__device__ __forceinline__ u32 pa_hash(u64 cr)
{
    const u32 x = (u32)cr ^ (u32)(cr >> 32) * 0x85EBCA6Bu;
    return (x * 0x9E3779B1u) >> (32 - PA_HBITS);
}

__global__ void __launch_bounds__(PA_WARPS * 32, 3)
preagg_kernel(const Rec *__restrict__ in, u64 nrec, int low, u32 nchunks, Rec *__restrict__ out,
              unsigned long long *__restrict__ out_count)
{
    constexpr u32 full = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    PreaggSpace &ws = reinterpret_cast<PreaggSpace *>(smem_raw)[warp];
    const u32 chunk = blockIdx.x * PA_WARPS + warp;
    if (chunk >= nchunks)
        return;
    const u32 lt = lanemask_lt();
    const u64 r0 = (u64)chunk * PA_W;
    const u32 cnt_here = (u32)min((u64)PA_W, nrec - r0);
#pragma unroll
    for (int i = 0; i < PA_H / 32; ++i)
        ws.key[i * 32 + lane] = PA_EMPTY;
    __syncwarp();

    Rec nxt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
    {
        const u32 p = i * 32 + lane;
        if (p < cnt_here)
            nxt[i] = ld_rec_stream(in + r0 + p);
    }
#pragma unroll 1
    for (int g = 0; g < PA_NB; g += 4)
    {
        Rec r[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            r[i] = nxt[i];
            const u32 p = (g + 4 + i) * 32 + lane;
            if (p < cnt_here)
                nxt[i] = ld_rec_stream(in + r0 + p);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            const u32 p = (g + i) * 32 + lane;
            if (p < cnt_here)
            {
                const u64 cr = r[i].key >> low;
                const u32 fl = (u32)r[i].key & 3u;
                const bool creates = (fl != FL_UPDATE) | (r[i].val != 0.0);
                const u64 want = cr << 1;
                u32 slot = pa_hash(cr);
                for (;;)
                {
                    u64 cur = ws.key[slot];
                    if (cur == PA_EMPTY)
                    {
                        cur = atomicCAS(reinterpret_cast<unsigned long long *>(&ws.key[slot]), PA_EMPTY, want);
                        if (cur == PA_EMPTY)
                        { // this lane made the slot: the sum starts from +0.0 (sparsematrixlnk.jl:225)
                            ws.acc[slot] = 0.0;
                            cur = want;
                        }
                    }
                    if ((cur >> 1) == cr)
                        break;
                    slot = (slot + 1) & (PA_H - 1);
                }
                if (creates && !(ws.key[slot] & 1ull))
                    atomicOr(reinterpret_cast<unsigned long long *>(&ws.key[slot]), 1ull);
            }
            __syncwarp(); // slots made in this batch hold their +0.0 before anybody adds
            if (p < cnt_here)
            {
                const u64 cr = r[i].key >> low;
                u32 slot = pa_hash(cr);
                while ((ws.key[slot] >> 1) != cr)
                    slot = (slot + 1) & (PA_H - 1);
                atomicAdd(&ws.acc[slot], r[i].val);
            }
            __syncwarp();
        }
    }
    // ---- the chunk's existing entries, packed: one ticket per chunk, coalesced stores
    u32 total = 0;
    u32 occ[PA_H / 32];
#pragma unroll
    for (int i = 0; i < PA_H / 32; ++i)
    {
        const u64 k = ws.key[i * 32 + lane];
        occ[i] = __ballot_sync(full, k != PA_EMPTY && (k & 1ull));
        total += __popc(occ[i]);
    }
    unsigned long long base = 0;
    if (lane == 0)
        base = atomicAdd(out_count, (unsigned long long)total);
    base = __shfl_sync(full, base, 0);
#pragma unroll
    for (int i = 0; i < PA_H / 32; ++i)
    {
        if ((occ[i] >> lane) & 1u)
        {
            const u64 k = ws.key[i * 32 + lane];
            Rec o;
            o.key = ((k >> 1) << low) | (u64)FL_RAW; // partition 0: the partial sums are not tied to a tid
            o.val = ws.acc[i * 32 + lane];
            st_rec(out + base + __popc(occ[i] & lt), o);
        }
        base += __popc(occ[i]);
    }
}

// in[0, nrec) -> out[0, *d_count): per-chunk partial sums.  d_count must be zeroed by the caller.
void preaggregate_records(cudaStream_t stream, const Rec *in, u64 nrec, const KeyLayout &L, Rec *out, u64 *d_count,
                          LaunchCounter &lc)
{
    if (nrec == 0)
        return;
    static FuncAttrOnce once;
    once.set(preagg_kernel, (int)(sizeof(PreaggSpace) * PA_WARPS));
    const u32 nchunks = (u32)((nrec + PA_W - 1) / PA_W);
    preagg_kernel<<<(nchunks + PA_WARPS - 1) / PA_WARPS, PA_WARPS * 32, sizeof(PreaggSpace) * PA_WARPS, stream>>>(
        in, nrec, L.low, nchunks, out, reinterpret_cast<unsigned long long *>(d_count));
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

} // namespace xsb
