// xsb_sort.cu -- stable LSD radix sort of 16-byte records on a bit range of the
// packed (col,row) key, "onesweep" style: one upfront digit histogram for all
// passes, then per pass a single kernel that ranks a tile with warp ballots,
// resolves its global offsets by decoupled look-back over per-tile digit counts
// and scatters through shared memory so that each digit's run leaves the SM as
// coalesced 16-byte stores.
//
// Reference counterpart (CPU): the per-column QuickSort of
// src/matrix/sparsematrixlnk.jl:339 and the counting sort inside stdlib
// sparse! reached from src/matrix/sparsematrixdilnkc.jl:428-432.
#include "xsb_internal.h"

namespace xsb {

// ------------------------------------------------------------------------
// digit histogram for all passes
// ------------------------------------------------------------------------
constexpr int HIST_THREADS = 512;

// With colcnt != nullptr the kernel also counts the records of every column (the field
// [colshift, colshift+colbits) of the key): one global atomic per distinct column of a warp's 32
// consecutive records.  The per-column kernels of xsb_colfold.cu take their column list from it.
__global__ void __launch_bounds__(HIST_THREADS)
histogram_kernel(const Rec *__restrict__ in, u64 n, SortPlan plan, u64 *__restrict__ ghist, u32 *__restrict__ colcnt,
                 int colshift, int colbits)
{
    __shared__ u32 s_hist[kMaxPasses][kRadix];
    for (int i = threadIdx.x; i < kMaxPasses * kRadix; i += HIST_THREADS)
        (&s_hist[0][0])[i] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * HIST_THREADS;
    const int lane = threadIdx.x & 31;
    const u32 lt = lanemask_lt();
    const u64 colmask = (1ull << colbits) - 1ull;
    // 32-bit shared counters: one block sees n/gridDim.x < 2^32 keys for every n that fits in HBM
    for (u64 k0 = (u64)blockIdx.x * HIST_THREADS + (threadIdx.x - lane); k0 < n; k0 += stride)
    { // k0 is warp-uniform
        const u64 k = k0 + lane;
        const bool valid = k < n;
        const u64 key = valid ? in[k].key : 0ull;
        if (valid)
        {
#pragma unroll
            for (int p = 0; p < kMaxPasses; ++p)
                if (p < plan.npasses)
                    atomicAdd(&s_hist[p][(key >> plan.shift[p]) & ((1u << plan.bits[p]) - 1u)], 1u);
        }
        if (colcnt != nullptr)
        {
            const u32 vm = __ballot_sync(0xffffffffu, valid);
            if (valid)
            {
                const u32 col = (u32)((key >> colshift) & colmask);
                const u32 peers = __match_any_sync(vm, col);
                if ((peers & lt) == 0u)
                    atomicAdd(&colcnt[col], (u32)__popc(peers));
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < plan.npasses * kRadix; i += HIST_THREADS)
    {
        u32 c = (&s_hist[0][0])[i];
        if (c)
            atomicAdd(&ghist[i], (u64)c);
    }
}

// exclusive scan of each pass's histogram -> first output index of every digit
__global__ void __launch_bounds__(kRadix) histogram_scan_kernel(u64 *__restrict__ ghist, int npasses)
{
    __shared__ u64 s_warp[kRadix / 32];
    const int p = blockIdx.x;
    if (p >= npasses)
        return;
    const int b = threadIdx.x, lane = b & 31, warp = b >> 5;
    const u64 c = ghist[p * kRadix + b];
    u64 incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        u64 t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o)
            incl += t;
    }
    if (lane == 31)
        s_warp[warp] = incl;
    __syncthreads();
    u64 pre = 0;
    for (int w = 0; w < warp; ++w)
        pre += s_warp[w];
    ghist[p * kRadix + b] = pre + incl - c;
}

// ------------------------------------------------------------------------
// one onesweep pass
// ------------------------------------------------------------------------
// look-back words carry 30-bit counts: longer inputs are sorted in portions
constexpr u32 ST_LOCAL = 1u << 30;
constexpr u32 ST_INCL = 2u << 30;
constexpr u32 ST_VALUE = (1u << 30) - 1u;

template <int THREADS, int IPT, int MINBLK>
__global__ void __launch_bounds__(THREADS, MINBLK)
onesweep_kernel(const Rec *__restrict__ in, Rec *__restrict__ out, u32 n, u32 ntiles, int shift,
                int bits, const u64 *__restrict__ gbase, u64 *__restrict__ gbase_next,
                u32 *__restrict__ status, u32 *__restrict__ tile_counter)
{
    constexpr int WARPS = THREADS / 32;
    constexpr int TILE = THREADS * IPT;
    static_assert(THREADS >= kRadix, "one thread per digit in the look-back");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Rec *s_rec = reinterpret_cast<Rec *>(smem_raw);
    __shared__ u32 s_whist[WARPS][kRadix];
    __shared__ u32 s_binstart[kRadix];
    __shared__ i64 s_gofs[kRadix];
    __shared__ u32 s_warpsum[kRadix / 32];
    __shared__ u32 s_tile;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0)
        s_tile = atomicAdd(tile_counter, 1u); // tiles are claimed in launch order: predecessors always run
    for (int i = tid; i < WARPS * kRadix; i += THREADS)
        (&s_whist[0][0])[i] = 0;
    __syncthreads();
    const u32 tile = s_tile;
    const u32 base = tile * TILE;
    const u32 valid = min((u32)TILE, n - base);
    const u32 mask = (1u << bits) - 1u;
    const u32 nbins = 1u << bits;

    // ---- load: warp-striped, one 16-byte vector per lane per step
    u64 key[IPT];
    double val[IPT];
    const u32 wbase = warp * (32 * IPT);
#pragma unroll
    for (int k = 0; k < IPT; ++k)
    {
        const u32 idx = wbase + k * 32 + lane;
        if (idx < valid)
        {
            Rec r = ld_rec_stream(in + base + idx);
            key[k] = r.key;
            val[k] = r.val;
        }
        else
        {
            key[k] = ~0ull; // padding sorts behind every real record of the tile
            val[k] = 0.0;
        }
    }

    // ---- rank inside the warp with ballots (stable: lower lane, lower step first)
    const u32 lt = lanemask_lt();
    u32 rank[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k)
    {
        const u32 d = (u32)(key[k] >> shift) & mask;
        u32 peers = 0xffffffffu;
#pragma unroll
        for (int b = 0; b < 8; ++b)
        {
            if (b < bits)
            {
                const bool bit = (d >> b) & 1u;
                const u32 bal = __ballot_sync(0xffffffffu, bit);
                peers &= bit ? bal : ~bal;
            }
        }
        const int leader = __ffs(peers) - 1;
        u32 pre = 0;
        if (lane == leader)
        {
            pre = s_whist[warp][d];
            s_whist[warp][d] = pre + __popc(peers);
        }
        pre = __shfl_sync(0xffffffffu, pre, leader);
        rank[k] = pre + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit: exclusive prefix over the warps, tile count, exclusive scan over digits
    u32 total = 0, incl = 0;
    if (tid < kRadix)
    {
#pragma unroll
        for (int w = 0; w < WARPS; ++w)
        {
            const u32 c = s_whist[w][tid];
            s_whist[w][tid] = total;
            total += c;
        }
        incl = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o)
                incl += t;
        }
        if (lane == 31)
            s_warpsum[warp] = incl;
    }
    __syncthreads();

    // ---- decoupled look-back: one thread per digit
    if (tid < kRadix)
    {
        u32 wpre = 0;
#pragma unroll
        for (int w = 0; w < kRadix / 32; ++w)
            if (w < warp)
                wpre += s_warpsum[w];
        const u32 excl = wpre + incl - total;
        s_binstart[tid] = excl;
        if ((u32)tid < nbins)
        {
            u32 *mine = status + (size_t)tile * nbins + tid;
            u32 prefix = 0;
            if (tile == 0)
            {
                st_relaxed_u32(mine, ST_INCL | total);
            }
            else
            {
                st_relaxed_u32(mine, ST_LOCAL | total);
                // LB predecessors are read per L2 round trip: the walk back to the nearest tile
                // with an inclusive prefix is latency bound, so the loads must overlap
                constexpr int LB = 8;
                bool done = false;
                for (i64 t = (i64)tile - 1; !done; t -= LB)
                {
                    u32 v[LB];
#pragma unroll
                    for (int j = 0; j < LB; ++j)
                        v[j] = (t - j >= 0) ? ld_relaxed_u32(status + (size_t)(t - j) * nbins + tid) : ST_INCL;
#pragma unroll
                    for (int j = 0; j < LB; ++j)
                    {
                        if (!done)
                        {
                            while ((v[j] >> 30) == 0u)
                                v[j] = ld_relaxed_u32(status + (size_t)(t - j) * nbins + tid);
                            prefix += v[j] & ST_VALUE;
                            done = (v[j] >> 30) == 2u;
                        }
                    }
                }
                st_relaxed_u32(mine, ST_INCL | (prefix + total));
            }
            const u64 g = gbase[tid];
            s_gofs[tid] = (i64)(g + prefix) - (i64)excl;
            if (gbase_next != nullptr && tile == ntiles - 1)
                gbase_next[tid] = g + prefix + total;
        }
    }
    __syncthreads();

    // ---- reorder through shared memory
#pragma unroll
    for (int k = 0; k < IPT; ++k)
    {
        const u32 d = (u32)(key[k] >> shift) & mask;
        const u32 pos = s_binstart[d] + s_whist[warp][d] + rank[k];
        Rec r;
        r.key = key[k];
        r.val = val[k];
        s_rec[pos] = r;
    }
    __syncthreads();

    // ---- scatter: consecutive threads hold consecutive ranks, so each digit's run is coalesced
#pragma unroll
    for (int i = 0; i < IPT; ++i)
    {
        const u32 idx = i * THREADS + tid;
        if (idx < valid)
        {
            const Rec r = s_rec[idx];
            const u32 d = (u32)(r.key >> shift) & mask;
            st_rec(out + (s_gofs[d] + (i64)idx), r);
        }
    }
}

// ------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------
// Onesweep tile: 512 threads x 8 records, 2 CTAs per SM -- the fastest of the tile shapes measured on B200.
constexpr int OS_THREADS = 512, OS_IPT = 8, OS_MINBLK = 2;
constexpr int OS_TILE = OS_THREADS * OS_IPT;
constexpr int kMinTile = 2048; // the workspace is sized for tiles this small (room to spare for OS_TILE)

static u64 sort_portion(int tile) { return ((1ull << 30) - 1ull) / (u64)tile * (u64)tile; }

SortPlan make_sort_plan(int begin_bit, int nbits)
{
    SortPlan p{};
    if (nbits <= 0)
    {
        p.npasses = 0;
        return p;
    }
    p.npasses = (nbits + 7) / 8;
    if (p.npasses > kMaxPasses)
        throw std::runtime_error("key too wide for the radix sort");
    int shift = begin_bit;
    for (int i = 0; i < p.npasses; ++i)
    {
        int b = nbits / p.npasses + (i < nbits % p.npasses ? 1 : 0);
        p.bits[i] = b;
        p.shift[i] = shift;
        shift += b;
    }
    return p;
}

size_t sort_workspace_bytes(u64 n)
{
    const u64 portion = std::min<u64>(n, sort_portion(kMinTile));
    const u64 ntiles = (portion + kMinTile - 1) / kMinTile;
    // ghist [kMaxPasses][256] u64, gbase_next [256] u64 x2, counter u32 (padded), status [ntiles][256] u32
    return sizeof(u64) * kMaxPasses * kRadix + 2 * sizeof(u64) * kRadix + 256 +
           sizeof(u32) * ntiles * kRadix;
}

// Sorts n records by key bits [begin_bit, begin_bit+nbits).  `a` holds the input;
// `b` is scratch of the same size.  Returns the buffer that holds the result.
Rec *radix_sort_records(cudaStream_t stream, Rec *a, Rec *b, u64 n, const SortPlan &plan, void *workspace,
                        LaunchCounter &lc, StageTimer *timer, u32 *colcnt, int colshift, int colbits)
{
    const bool nosort = n <= 1 || plan.npasses == 0;
    if (nosort && (colcnt == nullptr || n == 0))
        return a;
    static FuncAttrOnce once;
    once.set(onesweep_kernel<OS_THREADS, OS_IPT, OS_MINBLK>, (int)(OS_TILE * sizeof(Rec)));
    const u64 portion = sort_portion(OS_TILE);
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u64 *ghist = reinterpret_cast<u64 *>(ws);
    u64 *gnext0 = ghist + kMaxPasses * kRadix;
    u64 *gnext1 = gnext0 + kRadix;
    u32 *counter = reinterpret_cast<u32 *>(gnext1 + kRadix);
    u32 *status = counter + 64;

    if (timer)
        timer->begin(stream);
    XSB_CUDA(cudaMemsetAsync(ghist, 0, sizeof(u64) * kMaxPasses * kRadix, stream));
    {
        const u64 want = (n + HIST_THREADS * 8 - 1) / (HIST_THREADS * 8);
        const int blocks = (int)std::min<u64>(std::max<u64>(want, 1), (u64)kNumSM * 4);
        histogram_kernel<<<blocks, HIST_THREADS, 0, stream>>>(a, n, plan, ghist, colcnt, colshift, colbits);
        lc.add();
        if (plan.npasses > 0)
        {
            histogram_scan_kernel<<<plan.npasses, kRadix, 0, stream>>>(ghist, plan.npasses);
            lc.add();
        }
        XSB_CUDA(cudaGetLastError());
    }
    if (timer)
        timer->end(stream, &StageTimes::histogram);
    if (nosort)
        return a; // only the column counts were wanted

    if (timer)
        timer->begin(stream);
    Rec *src = a, *dst = b;
    for (int p = 0; p < plan.npasses; ++p)
    {
        const u32 nbins = 1u << plan.bits[p];
        const u64 *gbase = ghist + p * kRadix;
        u64 *gn[2] = {gnext0, gnext1};
        int flip = 0;
        for (u64 off = 0; off < n; off += portion)
        {
            const u32 cnt = (u32)std::min<u64>(portion, n - off);
            const u32 ntiles = (cnt + OS_TILE - 1) / OS_TILE;
            const bool more = off + portion < n;
            XSB_CUDA(cudaMemsetAsync(counter, 0, 256 + sizeof(u32) * (size_t)ntiles * nbins, stream));
            onesweep_kernel<OS_THREADS, OS_IPT, OS_MINBLK><<<ntiles, OS_THREADS, OS_TILE * sizeof(Rec), stream>>>(
                src + off, dst, cnt, ntiles, plan.shift[p], plan.bits[p], gbase, more ? gn[flip] : nullptr,
                status, counter);
            lc.add();
            if (more)
            {
                gbase = gn[flip];
                flip ^= 1;
            }
        }
        XSB_CUDA(cudaGetLastError());
        std::swap(src, dst);
    }
    if (timer)
        timer->end(stream, &StageTimes::sort);
    return src;
}

// Stable partition of n records by key bits [shift, shift+bits) into `out` (one onesweep pass);
// counts_host[d] receives the number of records of digit d.  Used to bucket staged records by
// owning rank before the all-to-all (the digit histogram doubles as the send counts).
void partition_records(cudaStream_t stream, const Rec *in, Rec *out, u64 n, int shift, int bits, void *workspace,
                       LaunchCounter &lc, u64 *counts_host)
{
    const int nb = 1 << bits;
    for (int d = 0; d < nb; ++d)
        counts_host[d] = 0;
    if (n == 0)
        return;
    SortPlan plan{};
    plan.npasses = 1;
    plan.shift[0] = shift;
    plan.bits[0] = bits;
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    u64 *ghist = reinterpret_cast<u64 *>(ws);
    XSB_CUDA(cudaMemsetAsync(ghist, 0, sizeof(u64) * kMaxPasses * kRadix, stream));
    const u64 want = (n + HIST_THREADS * 8 - 1) / (HIST_THREADS * 8);
    const int blocks = (int)std::min<u64>(std::max<u64>(want, 1), (u64)kNumSM * 4);
    histogram_kernel<<<blocks, HIST_THREADS, 0, stream>>>(in, n, plan, ghist, nullptr, 0, 0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    std::vector<u64> h((size_t)nb);
    XSB_CUDA(cudaMemcpyAsync(h.data(), ghist, sizeof(u64) * nb, cudaMemcpyDeviceToHost, stream));
    XSB_CUDA(cudaStreamSynchronize(stream));
    for (int d = 0; d < nb; ++d)
        counts_host[d] = h[d];
    histogram_scan_kernel<<<1, kRadix, 0, stream>>>(ghist, 1);
    lc.add();
    static FuncAttrOnce once;
    once.set(onesweep_kernel<OS_THREADS, OS_IPT, OS_MINBLK>, (int)(OS_TILE * sizeof(Rec)));
    const u64 portion = sort_portion(OS_TILE);
    u64 *gnext0 = ghist + kMaxPasses * kRadix;
    u64 *gnext1 = gnext0 + kRadix;
    u32 *counter = reinterpret_cast<u32 *>(gnext1 + kRadix);
    u32 *status = counter + 64;
    const u64 *gbase = ghist;
    u64 *gn[2] = {gnext0, gnext1};
    int flip = 0;
    for (u64 off = 0; off < n; off += portion)
    {
        const u32 cnt = (u32)std::min<u64>(portion, n - off);
        const u32 ntiles = (cnt + OS_TILE - 1) / OS_TILE;
        const bool more = off + portion < n;
        XSB_CUDA(cudaMemsetAsync(counter, 0, 256 + sizeof(u32) * (size_t)ntiles * nb, stream));
        onesweep_kernel<OS_THREADS, OS_IPT, OS_MINBLK><<<ntiles, OS_THREADS, OS_TILE * sizeof(Rec), stream>>>(
            in + off, out, cnt, ntiles, shift, bits, gbase, more ? gn[flip] : nullptr, status, counter);
        lc.add();
        if (more)
        {
            gbase = gn[flip];
            flip ^= 1;
        }
    }
    XSB_CUDA(cudaGetLastError());
}

} // namespace xsb
