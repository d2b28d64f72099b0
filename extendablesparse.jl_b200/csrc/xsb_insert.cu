// xsb_insert.cu -- producers of staged records:
//   pack_records   : caller (I,J,V) arrays -> 16-byte records, bounds-checked on device
//   emit_fdrand    : fdrand! call stream           (reference: src/matrix/sprand.jl:58-126)
//   emit_p1fem     : testassemble! call stream     (reference: test/femtools.jl:45-72)
//   emit_blockrd   : block reaction-diffusion stream (SURVEY.md 8d cfg 4, build-defined)
//   insert_elements: the caller's element loop, connectivity + dense element matrices (test/femtools.jl:45-72)
// The emitters batch whole elements/nodes per thread block, stage their records in
// shared memory and write them out as coalesced 16-byte vector stores, in exactly the
// order the reference's sequential loop would issue the insert calls.
//
// Compiled with -fmad=false: the element arithmetic must round like the CPU oracle's.
#include "xsb_internal.h"
#include "xsb_chunk.cuh"

namespace xsb {

// ------------------------------------------------------------------------
// pack / unpack
// ------------------------------------------------------------------------
template <typename Ti>
__global__ void __launch_bounds__(256)
pack_kernel(const Ti *__restrict__ I, const Ti *__restrict__ J, const double *__restrict__ V, i64 count, Ti base,
            i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *__restrict__ out, u64 *__restrict__ d_err,
            StageFlags sf)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        const i64 i = (i64)I[k] - base, j = (i64)J[k] - base;
        if (i < 0 || i >= m || j < 0 || j >= n)
        { // BoundsError: sparsematrixcsc.jl:8-10
            atomicMin(d_err, (u64)k);
            continue;
        }
        Rec r;
        r.key = L.pack((u64)j, (u64)i, tid, flavour);
        r.val = V[k];
        st_staged(out + k, r, L, sf, out);
    }
}

void pack_records(cudaStream_t stream, const void *I, const void *J, const double *V, i64 count, int idx64,
                  int base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *out, u64 *d_err,
                  LaunchCounter &lc, StageFlags sf)
{
    if (count <= 0)
        return;
    const int threads = 256;
    const int blocks = (int)std::min<i64>((count + threads - 1) / threads, (i64)kNumSM * 16);
    if (idx64)
        pack_kernel<int64_t><<<blocks, threads, 0, stream>>>((const int64_t *)I, (const int64_t *)J, V, count,
                                                             (int64_t)base, m, n, L, tid, flavour, out, d_err, sf);
    else
        pack_kernel<int32_t><<<blocks, threads, 0, stream>>>((const int32_t *)I, (const int32_t *)J, V, count,
                                                             (int32_t)base, m, n, L, tid, flavour, out, d_err, sf);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// 16-byte triplets {u32 row, u32 col, f64 val} -> staged records.  `in` may BE `out` (a host array
// is copied straight into the staging buffer and rewritten in place: every thread reads and writes
// its own 16 bytes), so neither pointer is __restrict__.
__global__ void __launch_bounds__(256)
pack_triplets_kernel(const uint4 *in, i64 count, u32 base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour,
                     Rec *out, u64 *__restrict__ d_err, StageFlags sf, i64 k0)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        const uint4 t = in[k];
        const i64 i = (i64)t.x - (i64)base, j = (i64)t.y - (i64)base;
        if (i < 0 || i >= m || j < 0 || j >= n)
        { // BoundsError: sparsematrixcsc.jl:8-10
            atomicMin(d_err, (u64)(k0 + k));
            continue;
        }
        Rec r;
        r.key = L.pack((u64)j, (u64)i, tid, flavour);
        r.val = __hiloint2double((int)t.w, (int)t.z);
        st_staged(out + k, r, L, sf, out);
    }
}

void pack_triplets(cudaStream_t stream, const void *T, i64 count, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                   u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf, i64 k0)
{
    if (count <= 0)
        return;
    const int threads = 256;
    const int blocks = (int)std::min<i64>((count + threads - 1) / threads, (i64)kNumSM * 16);
    pack_triplets_kernel<<<blocks, threads, 0, stream>>>(static_cast<const uint4 *>(T), count, (u32)base, m, n, L,
                                                         tid, flavour, out, d_err, sf, k0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------
// pack + group: the same conversion, a warp per chunk of CH_RECORDS insertions, and the chunk is brought
// into column order (xsb_chunk.cuh) while its records are in registers -- the flush then reads the
// records of a column where they were staged and never moves them.
// ------------------------------------------------------------------------
template <typename Ti> struct SrcIJV
{
    const Ti *I, *J;
    const double *V;
    i64 base;
    i64 k0 = 0; // position of entry 0 in the caller's batch (error reports)
    __device__ __forceinline__ void load(i64 k, i64 &i, i64 &j, double &v) const
    {
        i = (i64)I[k] - base;
        j = (i64)J[k] - base;
        v = V[k];
    }
    __device__ __forceinline__ void load_ij(i64 k, i64 &i, i64 &j) const
    {
        i = (i64)I[k] - base;
        j = (i64)J[k] - base;
    }
};
struct SrcTriplet
{
    const uint4 *T; // may alias the output: a warp reads its whole chunk before it writes any of it
    i64 base;
    i64 k0 = 0; // position of entry 0 in the caller's batch (a large host batch arrives in slices)
    __device__ __forceinline__ void load(i64 k, i64 &i, i64 &j, double &v) const
    {
        const uint4 t = T[k];
        i = (i64)t.x - base;
        j = (i64)t.y - base;
        v = __hiloint2double((int)t.w, (int)t.z);
    }
    __device__ __forceinline__ void load_ij(i64 k, i64 &i, i64 &j) const
    {
        const uint2 t = *reinterpret_cast<const uint2 *>(T + k);
        i = (i64)t.x - base;
        j = (i64)t.y - base;
    }
};

constexpr int PG_WARPS = 8;
constexpr int PG_HB = 9;
constexpr int PG_NB = CH_RECORDS / 32;

template <class Src>
__global__ void __launch_bounds__(PG_WARPS * 32)
pack_grouped_kernel(Src src, i64 count, u32 nchunks, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *out,
                    u64 *__restrict__ d_err, RunTarget rt, u32 chunk0, u32 pos0, StageFlags sf)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef ChunkSpaceT<PG_HB> Space;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 c = blockIdx.x * PG_WARPS + warp;
    if (c >= nchunks)
        return;
    Space &ws = reinterpret_cast<Space *>(smem_raw)[warp];
    chunk_space_init(ws, lane);
    const u32 lt = lanemask_lt();
    const i64 c0 = (i64)c * CH_RECORDS;
    const u32 len = (u32)min((i64)CH_RECORDS, count - c0);
    Rec r[PG_NB];
#pragma unroll
    for (int b = 0; b < PG_NB; ++b)
    {
        const u32 p = b * 32 + lane;
        r[b].key = 0;
        r[b].val = 0.0;
        if (p < len)
        {
            i64 i, j;
            double v;
            src.load(c0 + p, i, j, v);
            if (i < 0 || i >= m || j < 0 || j >= n)
            { // BoundsError (sparsematrixcsc.jl:8-10): the batch is rejected, whatever is written here is dropped
                atomicMin(d_err, (u64)(src.k0 + c0 + p));
                i = 0;
                j = 0;
            }
            r[b].key = L.pack((u64)j, (u64)i, tid, flavour);
            r[b].val = v;
        }
    }
    u32 rs[PG_NB];
    u32 d = 0;
    bool grouped = true;
#pragma unroll
    for (int b = 0; b < PG_NB; ++b)
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
        chunk_scan(ws, d, lane);
#pragma unroll
    for (int b = 0; b < PG_NB; ++b)
    {
        const u32 p = b * 32 + lane;
        if (p < len)
        {
            const u32 dst = grouped ? chunk_dest(ws.start, rs[b]) : p;
            st_rec(out + c0 + dst, r[b]);
            if (sf.flags != nullptr && L.owner(r[b].key) != (u32)L.self)
                sf.flags[(sf.pos0 + c0 + (i64)dst) >> kRouteTileShift] = 1; // benign race: same value
        }
    }
    if (grouped)
        chunk_publish(ws, rt, chunk0 + c, pos0 + (u32)c0, d, true, lane);
    else
    { // no column locality in this chunk: stored in call order, every record a run of its own
#pragma unroll
        for (int b = 0; b < PG_NB; ++b)
            rs[b] = (u32)(r[b].key >> rt.colshift) & rt.gmask;
        chunk_publish_singletons<PG_NB>(rt, chunk0 + c, pos0 + (u32)c0, len, rs, lane);
    }
}

// The same grouping for a source that does NOT alias the output (device arrays of the caller, the temporary copies
// of host (I,J,V) arrays).  pack_grouped_kernel holds a chunk's 512 records in registers (128 of them: 16 warps per
// SM) and stores each record on its own -- a half-filled 32-byte sector per store.  Here only the 4-byte grouping
// keys pass through shared memory: pass 1 reads the chunk (coalesced) and notes every record's key; the 16 batches
// run over the keys and leave (slot, rank) in their place; an inverse map (2 bytes per record) turns that into
// "which record goes to position t"; pass 3 walks the grouped chunk in DESTINATION order, reads the two records of a
// sector again (the chunk's 8 KB are in L2), and stores whole sectors, consecutive lanes to consecutive sectors.
// 8 KB of shared memory and ~50 registers per warp: 24 warps per SM.  Measured (FEM 128^3 as device triplets,
// 245.8 M): 3.9 -> see profiles/r2_summary.md.
constexpr int PG2_WARPS = 8;
struct Pg2WarpSpace
{
    u32 g[CH_RECORDS];              // grouping key of record p, then (slot << 16 | rank)
    unsigned short inv[CH_RECORDS]; // record that goes to position t of the grouped chunk
    ChunkSpaceT<PG_HB> tab;
};

template <class Src>
__global__ void __launch_bounds__(PG2_WARPS * 32, 3)
pack_grouped2_kernel(Src src, i64 count, u32 nchunks, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *__restrict__ out,
                     u64 *__restrict__ d_err, RunTarget rt, u32 chunk0, u32 pos0, StageFlags sf)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef ChunkSpaceT<PG_HB> Space;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 c = blockIdx.x * PG2_WARPS + warp;
    if (c >= nchunks)
        return;
    Pg2WarpSpace &sp = reinterpret_cast<Pg2WarpSpace *>(smem_raw)[warp];
    chunk_space_init(sp.tab, lane);
    const u32 lt = lanemask_lt();
    const i64 c0 = (i64)c * CH_RECORDS;
    const u32 len = (u32)min((i64)CH_RECORDS, count - c0);
    // an index outside the matrix is a BoundsError (sparsematrixcsc.jl:8-10): the batch is rejected, whatever is
    // written for it is dropped
    auto key_of = [&](i64 i, i64 j) {
        const bool bad = i < 0 || i >= m || j < 0 || j >= n;
        return L.pack(bad ? 0ull : (u64)j, bad ? 0ull : (u64)i, tid, flavour);
    };
    // pass 1: the chunk's indices, eight coalesced loads in flight per lane before the first one is used
#pragma unroll
    for (int b0 = 0; b0 < PG_NB; b0 += 8)
    {
        if ((u32)(b0 * 32) >= len) // warp-uniform
            break;
        i64 ii[8], jj[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
        {
            const u32 p = (b0 + u) * 32 + lane;
            ii[u] = jj[u] = 0;
            if (p < len)
                src.load_ij(c0 + p, ii[u], jj[u]);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
        {
            const u32 p = (b0 + u) * 32 + lane;
            if (p < len)
            {
                if (ii[u] < 0 || ii[u] >= m || jj[u] < 0 || jj[u] >= n)
                    atomicMin(d_err, (u64)(src.k0 + c0 + p));
                sp.g[p] = (u32)(key_of(ii[u], jj[u]) >> rt.colshift) & rt.gmask;
            }
        }
    }
    __syncwarp();
    u32 d = 0;
    bool grouped = true;
    for (int b = 0; b < PG_NB && grouped; ++b)
    {
        if ((u32)(b * 32) >= len) // warp-uniform
            break;
        if (d > Space::DMAX - 32u)
            grouped = false; // the table may not take another 32 columns: no column locality here
        else
        {
            const u32 p = b * 32 + lane;
            const u32 rs = chunk_count_batch(sp.tab, p < len ? sp.g[p] : 0u, p < len, lt, d);
            if (p < len)
                sp.g[p] = rs;
        }
    }
    if (grouped)
    {
        chunk_scan(sp.tab, d, lane);
        for (u32 p = lane; p < len; p += 32)
            sp.inv[chunk_dest(sp.tab.start, sp.g[p])] = (unsigned short)p;
    }
    else
        for (u32 p = lane; p < len; p += 32)
            sp.inv[p] = (unsigned short)p; // stored in call order
    __syncwarp();
    {
        Rec *dst = out + c0;
        const u32 a = (u32)(reinterpret_cast<uintptr_t>(dst) >> 4) & 1u; // dst[0] is the upper half of its sector
        auto mark = [&](const Rec &r, u32 t) {
            if (sf.flags != nullptr && L.owner(r.key) != (u32)L.self)
                sf.flags[(sf.pos0 + c0 + (i64)t) >> kRouteTileShift] = 1; // benign race: same value
        };
        auto make = [&](u32 p) {
            i64 i, j;
            Rec r;
            src.load(c0 + p, i, j, r.val);
            r.key = key_of(i, j);
            return r;
        };
        if (a && lane == 0 && len > 0)
        {
            const Rec r = make(sp.inv[0]);
            st_rec(dst, r);
            mark(r, 0);
        }
        const u32 pairs = (len - min(a, len)) >> 1;
        // pass 3: four sectors per lane and round: their eight records are requested before the first one is used
        for (u32 q0 = 0; q0 < pairs; q0 += 128)
        {
            i64 ii[8], jj[8];
            double vv[8];
#pragma unroll
            for (int u = 0; u < 4; ++u)
            {
                const u32 q = q0 + u * 32 + lane;
                ii[2 * u] = jj[2 * u] = ii[2 * u + 1] = jj[2 * u + 1] = 0;
                vv[2 * u] = vv[2 * u + 1] = 0.0;
                if (q < pairs)
                {
                    const u32 t = a + 2 * q;
                    const u32 pp = *reinterpret_cast<const u32 *>(reinterpret_cast<const unsigned char *>(sp.inv) + 2 * (t & ~1u));
                    // inv[t], inv[t + 1] (t odd: the pair straddles two words)
                    const u32 p0 = (t & 1u) ? (pp >> 16) : (pp & 0xffffu);
                    const u32 p1 = (t & 1u) ? (u32)sp.inv[t + 1] : (pp >> 16);
                    src.load(c0 + p0, ii[2 * u], jj[2 * u], vv[2 * u]);
                    src.load(c0 + p1, ii[2 * u + 1], jj[2 * u + 1], vv[2 * u + 1]);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
            {
                const u32 q = q0 + u * 32 + lane;
                if (q < pairs)
                {
                    const u32 t = a + 2 * q;
                    Rec r0, r1;
                    r0.key = key_of(ii[2 * u], jj[2 * u]);
                    r0.val = vv[2 * u];
                    r1.key = key_of(ii[2 * u + 1], jj[2 * u + 1]);
                    r1.val = vv[2 * u + 1];
                    st_v4_u64(dst + t, r0.key, (u64)__double_as_longlong(r0.val), r1.key, (u64)__double_as_longlong(r1.val));
                    mark(r0, t);
                    mark(r1, t + 1);
                }
            }
        }
        if (len > a && ((len - a) & 1u) && lane == 31)
        {
            const Rec r = make(sp.inv[len - 1]);
            st_rec(dst + len - 1, r);
            mark(r, len - 1);
        }
    }
    if (grouped)
        chunk_publish(sp.tab, rt, chunk0 + c, pos0 + (u32)c0, d, true, lane);
    else
    { // no column locality in this chunk: every record a run of its own
        u32 gk[PG_NB];
#pragma unroll
        for (int b = 0; b < PG_NB; ++b)
        {
            const u32 p = b * 32 + lane;
            gk[b] = 0u;
            if (p < len)
            {
                i64 i, j;
                src.load_ij(c0 + p, i, j);
                gk[b] = (u32)(key_of(i, j) >> rt.colshift) & rt.gmask;
            }
        }
        chunk_publish_singletons<PG_NB>(rt, chunk0 + c, pos0 + (u32)c0, len, gk, lane);
    }
}

template <class Src>
static u32 launch_pack_grouped(cudaStream_t stream, Src src, i64 count, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour,
                               Rec *out, u64 *d_err, const RunTarget &rt, u32 chunk0, u32 pos0, StageFlags sf,
                               LaunchCounter &lc, bool aliased)
{
    const u32 nchunks = (u32)((count + CH_RECORDS - 1) / CH_RECORDS);
    if (aliased)
    { // the source IS the staging buffer (triplets copied there from the host): every warp reads its whole chunk first
        static FuncAttrOnce once;
        const int smem = (int)(sizeof(ChunkSpaceT<PG_HB>) * PG_WARPS);
        once.set(pack_grouped_kernel<Src>, smem);
        const unsigned blocks = (nchunks + PG_WARPS - 1) / PG_WARPS;
        pack_grouped_kernel<Src><<<blocks, PG_WARPS * 32, smem, stream>>>(src, count, nchunks, m, n, L, tid, flavour, out,
                                                                          d_err, rt, chunk0, pos0, sf);
    }
    else
    {
        static FuncAttrOnce once;
        const int smem = (int)(sizeof(Pg2WarpSpace) * PG2_WARPS);
        once.set(pack_grouped2_kernel<Src>, smem, true);
        const unsigned blocks = (nchunks + PG2_WARPS - 1) / PG2_WARPS;
        pack_grouped2_kernel<Src><<<blocks, PG2_WARPS * 32, smem, stream>>>(src, count, nchunks, m, n, L, tid, flavour, out,
                                                                            d_err, rt, chunk0, pos0, sf);
    }
    lc.add();
    XSB_CUDA(cudaGetLastError());
    return nchunks;
}

u32 pack_chunks(i64 count) { return (u32)((count + CH_RECORDS - 1) / CH_RECORDS); }

// returns the chunks appended to the run index (pack_chunks(count))
u32 pack_records_grouped(cudaStream_t stream, const void *I, const void *J, const double *V, i64 count, int idx64,
                         int base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *out, u64 *d_err,
                         LaunchCounter &lc, const RunTarget &rt, u32 chunk0, u32 pos0, StageFlags sf)
{
    if (count <= 0)
        return 0;
    if (idx64)
        return launch_pack_grouped(stream, SrcIJV<int64_t>{(const int64_t *)I, (const int64_t *)J, V, (i64)base}, count, m,
                                   n, L, tid, flavour, out, d_err, rt, chunk0, pos0, sf, lc, false);
    return launch_pack_grouped(stream, SrcIJV<int32_t>{(const int32_t *)I, (const int32_t *)J, V, (i64)base}, count, m, n,
                               L, tid, flavour, out, d_err, rt, chunk0, pos0, sf, lc, false);
}

u32 pack_triplets_grouped(cudaStream_t stream, const void *T, i64 count, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                          u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, const RunTarget &rt, u32 chunk0, u32 pos0,
                          StageFlags sf, i64 k0)
{
    if (count <= 0)
        return 0;
    return launch_pack_grouped(stream, SrcTriplet{static_cast<const uint4 *>(T), (i64)base, k0}, count, m, n, L, tid, flavour,
                               out, d_err, rt, chunk0, pos0, sf, lc, static_cast<const void *>(T) == static_cast<const void *>(out));
}

template <typename Ti>
__global__ void __launch_bounds__(256)
unpack_kernel(const Rec *__restrict__ in, i64 count, Ti base, KeyLayout L, Ti *__restrict__ I, Ti *__restrict__ J,
              double *__restrict__ V, int *__restrict__ flavour)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        const Rec r = in[k];
        I[k] = (Ti)L.row(r.key) + base;
        J[k] = (Ti)L.gcol(r.key) + base;
        V[k] = r.val;
        if (flavour)
            flavour[k] = (int)L.flavour(r.key);
    }
}

void unpack_records(cudaStream_t stream, const Rec *in, i64 count, int idx64, int base, KeyLayout L, void *I,
                    void *J, double *V, int *flavour, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    const int threads = 256;
    const int blocks = (int)std::min<i64>((count + threads - 1) / threads, (i64)kNumSM * 16);
    if (idx64)
        unpack_kernel<int64_t><<<blocks, threads, 0, stream>>>(in, count, (int64_t)base, L, (int64_t *)I,
                                                               (int64_t *)J, V, flavour);
    else
        unpack_kernel<int32_t><<<blocks, threads, 0, stream>>>(in, count, (int32_t)base, L, (int32_t *)I,
                                                               (int32_t *)J, V, flavour);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------
// counter-based random numbers: Philox4x32-10, u = (w1:w0 >> 11) * 2^-53
// ------------------------------------------------------------------------
__host__ __device__ __forceinline__ double philox_uniform(u64 seed, u64 counter)
{
    u32 c0 = (u32)counter, c1 = (u32)(counter >> 32), c2 = 0u, c3 = 0u;
    u32 k0 = (u32)seed, k1 = (u32)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r)
    {
        const u64 p0 = (u64)0xD2511F53u * c0;
        const u64 p1 = (u64)0xCD9E8D57u * c2;
        const u32 n0 = (u32)(p1 >> 32) ^ c1 ^ k0;
        const u32 n1 = (u32)p1;
        const u32 n2 = (u32)(p0 >> 32) ^ c3 ^ k1;
        const u32 n3 = (u32)p0;
        c0 = n0;
        c1 = n1;
        c2 = n2;
        c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    const u64 bits = ((u64)c1 << 32) | (u64)c0;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);
}

// ------------------------------------------------------------------------
// fdrand! stream.  Per node (i,j,k), in this order (sprand.jl:100-124):
//   x-edge pair (4 records, if i<nx), x-boundary (1, if i==1||i==nx),
//   y-edge pair (if j<ny), y-boundary (if ny>2 && (j==1||j==ny)),
//   z-edge pair (if k<nz), z-boundary (if nz>2 && (k==1||k==nz)).
// Record and rand() counts before a node have a closed form, so every node
// can be emitted independently at its exact stream position.
// ------------------------------------------------------------------------
// node l0 (0-based, x fastest) -> 1-based (i,j,k); 32-bit arithmetic when the grid allows it (a 64-bit division by
// a run-time value costs about a hundred instructions)
__host__ __device__ __forceinline__ void node_ijk(i64 l0, i64 nx, i64 ny, i64 nz, i64 &i, i64 &j, i64 &k)
{
    if (nx * ny * nz < 0x7fffffffll)
    {
        const u32 l = (u32)l0, ux = (u32)nx, uy = (u32)ny;
        const u32 row = l / ux, lay = row / uy;
        i = (i64)(l - row * ux) + 1;
        j = (i64)(row - lay * uy) + 1;
        k = (i64)lay + 1;
    }
    else
    {
        i = l0 % nx + 1;
        j = (l0 / nx) % ny + 1;
        k = l0 / (nx * ny) + 1;
    }
}

struct FdGeom
{
    i64 nx, ny, nz;
    __host__ __device__ i64 bx(i64 i) const { return (i == 1 || i == nx) ? 1 : 0; }
    __host__ __device__ i64 by(i64 j) const { return (ny > 2 && (j == 1 || j == ny)) ? 1 : 0; }
    __host__ __device__ i64 bz(i64 k) const { return (nz > 2 && (k == 1 || k == nz)) ? 1 : 0; }
    // number of boundary hits / edges among indices 1..i-1
    __host__ __device__ i64 pbx(i64 i) const { return (i > 1 ? 1 : 0) + ((nx > 1 && i > nx) ? 1 : 0); }
    __host__ __device__ i64 pby(i64 j) const
    {
        return ny > 2 ? (j > 1 ? 1 : 0) + (j > ny ? 1 : 0) : 0;
    }
    __host__ __device__ i64 pbz(i64 k) const
    {
        return nz > 2 ? (k > 1 ? 1 : 0) + (k > nz ? 1 : 0) : 0;
    }
    __host__ __device__ static i64 pe(i64 i, i64 n) { return (i - 1) < (n - 1) ? (i - 1) : (n - 1); } // edges among 1..i-1

    // W = 4 for records, 1 for rand() calls (an edge pair is 4 records but one rand())
    template <int W> __host__ __device__ i64 cx(i64 i) const { return (i < nx ? W : 0) + bx(i); }
    template <int W> __host__ __device__ i64 cy(i64 j) const { return (j < ny ? W : 0) + by(j); }
    template <int W> __host__ __device__ i64 cz(i64 k) const { return (k < nz ? W : 0) + bz(k); }
    template <int W> __host__ __device__ i64 PX(i64 i) const { return W * pe(i, nx) + pbx(i); }
    template <int W> __host__ __device__ i64 PY(i64 j) const { return W * pe(j, ny) + pby(j); }
    template <int W> __host__ __device__ i64 PZ(i64 k) const { return W * pe(k, nz) + pbz(k); }
    // count over all nodes that precede (i,j,k) in the sweep (x fastest)
    template <int W> __host__ __device__ i64 before(i64 i, i64 j, i64 k) const
    {
        const i64 RX = PX<W>(nx + 1), RY = PY<W>(ny + 1);
        i64 s = (k - 1) * (ny * RX + nx * RY) + nx * ny * PZ<W>(k);
        s += (j - 1) * RX + nx * PY<W>(j) + (j - 1) * nx * cz<W>(k);
        s += PX<W>(i) + (i - 1) * (cy<W>(j) + cz<W>(k));
        return s;
    }
    template <int W> __host__ __device__ i64 before_node(i64 l0) const
    { // l0 = 0-based node index; l0 == nx*ny*nz gives the stream total
        if (l0 >= nx * ny * nz)
            return before<W>(1, 1, nz + 1);
        i64 i, j, k;
        node_ijk(l0, nx, ny, nz, i, j, k);
        return before<W>(i, j, k);
    }
};

i64 fdrand_prefix(i64 nx, i64 ny, i64 nz, i64 l)
{
    FdGeom g{nx, ny, nz};
    return g.before_node<4>(l);
}

constexpr int FD_THREADS = 128; // nodes per block
constexpr int FD_MAXREC = 15;   // records per node upper bound

// records of node l0 (0-based), in call order, to dst[0 ..); returns their number
// base: the tile's records start at stream position rec0; the node's go to base[before(node) - rec0 ...]
__device__ __forceinline__ int fd_node_records(const FdGeom &g, i64 l0, u64 seed, int ones, const KeyLayout &L, u32 tid,
                                               u32 flavour, Rec *base, i64 rec0)
{
    i64 i, j, k;
    node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
    Rec *dst = base + (g.before<4>(i, j, k) - rec0);
    int pos = 0;
    u64 call = (u64)g.before<1>(i, j, k);
    const double hx = 1.0 / (double)g.nx, hy = 1.0 / (double)g.ny, hz = 1.0 / (double)g.nz;
    const u64 l = (u64)l0; // 0-based unknown
    auto rnd = [&]() -> double {
        const double u = ones ? 1.0 : philox_uniform(seed, call);
        ++call;
        return u;
    };
    auto put = [&](double v, u64 row, u64 col) {
        Rec r;
        r.key = L.pack(col, row, tid, flavour);
        r.val = v;
        dst[pos++] = r;
    };
    auto pair = [&](double v, u64 a, u64 b) { // update_pair, sprand.jl:87-92
        put(-v, a, b);
        put(-v, b, a);
        put(v, a, a);
        put(v, b, b);
    };
    if (i < g.nx)
        pair(rnd() * hy * hz / hx, l, l + 1);
    if (i == 1 || i == g.nx)
        put(rnd() * hy * hz, l, l);
    if (j < g.ny)
        pair(rnd() * hx * hz / hy, l, l + (u64)g.nx);
    if (g.ny > 2 && (j == 1 || j == g.ny))
        put(rnd() * hx * hz, l, l);
    if (k < g.nz)
        pair(rnd() * hx * hy / hz, l, l + (u64)(g.nx * g.ny));
    if (g.nz > 2 && (k == 1 || k == g.nz))
        put(rnd() * hx * hy, l, l);
    return pos;
}

__global__ void __launch_bounds__(FD_THREADS)
emit_fdrand_kernel(FdGeom g, u64 seed, int ones, KeyLayout L, u32 tid, u32 flavour, i64 l_begin, i64 l_end,
                   i64 rec_begin, Rec *__restrict__ out, StageFlags sf)
{
    __shared__ Rec s_rec[FD_THREADS * FD_MAXREC];
    const i64 l_first = l_begin + (i64)blockIdx.x * FD_THREADS;
    const i64 l_last = min(l_first + FD_THREADS, l_end);
    const i64 blk_rec0 = g.before_node<4>(l_first);
    const i64 blk_rec1 = g.before_node<4>(l_last);
    const i64 l0 = l_first + threadIdx.x;
    if (l0 < l_last)
        fd_node_records(g, l0, seed, ones, L, tid, flavour, s_rec, blk_rec0);
    __syncthreads();
    const i64 nrec = blk_rec1 - blk_rec0;
    Rec *dst = out + (blk_rec0 - rec_begin);
    for (i64 q = threadIdx.x; q < nrec; q += FD_THREADS)
        st_staged(dst + q, s_rec[q], L, sf, out);
}

// Grouped chunks (xsb_chunk.cuh): the records of a warp's 32 nodes (at most 480) = one chunk -- grouped without
// looking at the records one by one.  Node l only touches four columns: its own (2 records per edge pair it emits
// plus its boundary terms), l+1, l+nx and l+nx*ny (2 records each, the far ends of its x / y / z pair).  The warp runs
// these (node, column) VISITS through its table, weighted by their record counts, kind after kind: z-ends of all
// nodes, y-ends, x-ends, own columns.  Inside one kind every lane holds a different column (no match.any, no
// leader election), and a column meets its visitors in node = call order: l - nx*ny (z-end), l - nx (y-end),
// l - 1 (x-end), l (own).  Then every lane computes its records and stores them straight to their place of the grouped
// chunk: a node's 6 .. 9 own-column records are neighbours there, and so are the two a far end receives, so they leave
// as 256-bit stores wherever two share a sector.  (Staging the chunk in shared memory first -- 7.7 KB per warp --
// left 30 % of the warp slots in use: 0.83 ms for 200^3; see profiles/r2_summary.md for this version.)
constexpr int FDG_HB = 8; // 256 slots for at most 128 distinct columns
struct FdWarpSpace
{
    ChunkSpaceT<FDG_HB> tab;
};

__global__ void __launch_bounds__(FD_THREADS)
emit_fdrand_grouped_kernel(FdGeom g, u64 seed, int ones, KeyLayout L, u32 tid, u32 flavour, i64 l_begin, i64 l_end,
                           i64 rec_begin, Rec *__restrict__ out, StageFlags sf, RunTarget rt, u32 chunk0, u32 pos_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr u32 full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FdWarpSpace &sp = reinterpret_cast<FdWarpSpace *>(smem_raw)[warp];
    const u32 wchunk = blockIdx.x * (FD_THREADS / 32) + warp;
    const i64 l_first = l_begin + (i64)wchunk * 32;
    if (l_first >= l_end)
        return;
    const i64 l_last = min(l_first + 32, l_end);
    chunk_space_init(sp.tab, lane);
    const i64 l0 = l_first + lane;
    const bool have = l0 < l_last;
    i64 i = 1, j = 1, k = 1;
    if (have)
        node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
    const bool ex = have && i < g.nx, ey = have && j < g.ny, ez = have && k < g.nz; // the node's edge pairs
    const bool bx = have && g.bx(i), by = have && g.by(j), bz = have && g.bz(k);    // its boundary terms
    const u64 l = (u64)l0;
    const u64 sx = 1, sy = (u64)g.nx, sz = (u64)(g.nx * g.ny);
    auto gkey = [&](u64 col) { return (u32)(L.pack(col, 0, tid, flavour) >> rt.colshift) & rt.gmask; };
    const u32 w_own = 2u * ((u32)ex + (u32)ey + (u32)ez) + (u32)bx + (u32)by + (u32)bz;
    const u32 lt = lanemask_lt();
    u32 d = 0;
    const u32 vz = chunk_visit_batch(sp.tab, ez ? gkey(l + sz) : 0u, ez, 2u, lt, d);
    const u32 vy = chunk_visit_batch(sp.tab, ey ? gkey(l + sy) : 0u, ey, 2u, lt, d);
    const u32 vx = chunk_visit_batch(sp.tab, ex ? gkey(l + sx) : 0u, ex, 2u, lt, d);
    const u32 vo = chunk_visit_batch(sp.tab, have ? gkey(l) : 0u, have, w_own, lt, d);
    chunk_scan(sp.tab, d, lane);
    // position of the chunk in the stream: the records of the nodes before the warp's first one (lane 0 holds it)
    i64 w_rec0 = lane == 0 ? g.before<4>(i, j, k) : 0;
    w_rec0 = __shfl_sync(full, w_rec0, 0);
    const i64 c0 = w_rec0 - rec_begin; // position of the chunk in this launch's output
    if (have)
    { // records straight from registers to their place: the own column's 6 .. 9 records are neighbours, and so are the two
      // a far end receives -- whole 32-byte sectors (STG.256) wherever two of them share one
        Rec *const dst = out + c0;
        Rec *own = dst + chunk_dest(sp.tab.start, vo);
        Rec pend;
        bool held = false; // pend waits for its sector's upper half
        u64 call = (u64)g.before<1>(i, j, k);
        const double hx = 1.0 / (double)g.nx, hy = 1.0 / (double)g.ny, hz = 1.0 / (double)g.nz;
        auto rnd = [&]() -> double {
            const double u = ones ? 1.0 : philox_uniform(seed, call);
            ++call;
            return u;
        };
        auto make = [&](double v, u64 row, u64 col) {
            Rec r;
            r.key = L.pack(col, row, tid, flavour);
            r.val = v;
            return r;
        };
        auto mark = [&](const Rec *p, const Rec &r) {
            if (sf.flags != nullptr && L.owner(r.key) != (u32)L.self)
                sf.flags[(sf.pos0 + c0 + (i64)(p - dst)) >> kRouteTileShift] = 1; // benign race: same value
        };
        auto pair256 = [&](Rec *p, const Rec &a, const Rec &b) {
            st_v4_u64(p, a.key, (u64)__double_as_longlong(a.val), b.key, (u64)__double_as_longlong(b.val));
        };
        auto put_own = [&](const Rec &r) {
            mark(own, r);
            if (held)
            {
                pair256(own - 1, pend, r);
                held = false;
            }
            else if (reinterpret_cast<uintptr_t>(own) & 16u)
                st_rec(own, r); // upper half of a sector whose lower half is somebody else's
            else
            {
                pend = r;
                held = true;
            }
            ++own;
        };
        // update_pair(v, a = l, b): (-v, a, b) (-v, b, a) (v, a, a) (v, b, b) in call order (sprand.jl:87-92):
        // the first and the last go to column b, the two in the middle to the node's own column
        auto pair = [&](double v, u64 b, u32 visit) {
            Rec *far = dst + chunk_dest(sp.tab.start, visit);
            const Rec f0 = make(-v, l, b), f1 = make(v, b, b);
            mark(far, f0);
            mark(far + 1, f1);
            if (reinterpret_cast<uintptr_t>(far) & 16u)
            {
                st_rec(far, f0);
                st_rec(far + 1, f1);
            }
            else
                pair256(far, f0, f1);
            put_own(make(-v, b, l));
            put_own(make(v, l, l));
        };
        if (ex)
            pair(rnd() * hy * hz / hx, l + sx, vx);
        if (bx)
            put_own(make(rnd() * hy * hz, l, l));
        if (ey)
            pair(rnd() * hx * hz / hy, l + sy, vy);
        if (by)
            put_own(make(rnd() * hx * hz, l, l));
        if (ez)
            pair(rnd() * hx * hy / hz, l + sz, vz);
        if (bz)
            put_own(make(rnd() * hx * hy, l, l));
        if (held)
            st_rec(own - 1, pend);
    }
    chunk_publish(sp.tab, rt, chunk0 + wchunk, pos_out + (u32)c0, d, true, lane);
}

void emit_fdrand(cudaStream_t stream, i64 nx, i64 ny, i64 nz, u64 seed, int ones, KeyLayout L, u32 tid,
                 u32 flavour, i64 l_begin, i64 l_end, Rec *out, LaunchCounter &lc, StageFlags sf)
{
    if (l_end <= l_begin)
        return;
    FdGeom g{nx, ny, nz};
    const i64 blocks = (l_end - l_begin + FD_THREADS - 1) / FD_THREADS;
    emit_fdrand_kernel<<<(unsigned)blocks, FD_THREADS, 0, stream>>>(g, seed, ones, L, tid, flavour, l_begin, l_end,
                                                                    g.before_node<4>(l_begin), out, sf);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

u32 emit_fdrand_chunks(i64 l_begin, i64 l_end) { return (u32)((l_end - l_begin + 31) / 32); }

u32 emit_fdrand_grouped(cudaStream_t stream, i64 nx, i64 ny, i64 nz, u64 seed, int ones, KeyLayout L, u32 tid, u32 flavour,
                        i64 l_begin, i64 l_end, Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0,
                        u32 pos0)
{
    if (l_end <= l_begin)
        return 0;
    FdGeom g{nx, ny, nz};
    static FuncAttrOnce once;
    const int smem = (int)(sizeof(FdWarpSpace) * (FD_THREADS / 32));
    once.set(emit_fdrand_grouped_kernel, smem, true);
    const i64 blocks = (l_end - l_begin + FD_THREADS - 1) / FD_THREADS;
    emit_fdrand_grouped_kernel<<<(unsigned)blocks, FD_THREADS, smem, stream>>>(
        g, seed, ones, L, tid, flavour, l_begin, l_end, g.before_node<4>(l_begin), out, sf, rt, chunk0, pos0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    return emit_fdrand_chunks(l_begin, l_end);
}

// ------------------------------------------------------------------------
// P1 FEM stream on the Kuhn tensor mesh: 20 rawupdateindex! calls per tetrahedron
// (test/femtools.jl:62-69).  One thread per tetrahedron, 128 tetrahedra per block.
// ------------------------------------------------------------------------
__constant__ int c_kuhn[6][3] = {{0, 1, 2}, {0, 2, 1}, {1, 0, 2}, {1, 2, 0}, {2, 0, 1}, {2, 1, 0}};

constexpr int FEM_THREADS = 128;
constexpr int FEM_REC = 20;
constexpr int FEM_PITCH = FEM_REC + 1;

// Element matrix of tetrahedron t: what its 20 rawupdateindex! calls (test/femtools.jl:62-69) insert.
struct FemTet
{
    u64 ckey[4], rkey[4]; // a node is the column of 5 and the row of 5 of the element's 20 records
    double vol;
    double S[4][4];
    int has_foreign; // slab handles: a column of this element belongs to another rank
    // record q = 5 il + w of the element: w == 0: mass term on (i,i); else stiffness (i, j = node[w-1])
    __device__ __forceinline__ u64 key(int il, int w) const { return (w == 0 ? ckey[il] : ckey[w - 1]) | rkey[il]; }
    __device__ __forceinline__ double val(int il, int w) const { return w == 0 ? 0.1 * vol / 4.0 : vol * S[il][w - 1]; }
};

// x / y for finite y != 0, bit for bit: a zero numerator (most cofactors of an axis-aligned tetrahedron, the
// coordinate of the first mesh plane) gives the signed zero directly instead of taking the division's slow path
__device__ __forceinline__ double div_finite(double x, double y)
{
    if (x == 0.0)
        return ((__double2hiint(x) ^ __double2hiint(y)) < 0) ? -0.0 : 0.0;
    return x / y;
}

__device__ __forceinline__ void fem_tet_compute(i64 t, i64 nxn, i64 nyn, i64 nzn, const KeyLayout &L, u32 tid, u32 flavour,
                                                bool slab, FemTet &e)
{
    e.has_foreign = 0;
    const i64 cxn = nxn - 1, cyn = nyn - 1;
    i64 idx[4][3];
    int perm;
    if (t < 0x7fffffffll)
    { // 32-bit index arithmetic (64-bit divisions by run-time values cost hundreds of instructions)
        const u32 t32 = (u32)t, cube = t32 / 6u, cx = (u32)cxn, cy = (u32)cyn;
        perm = (int)(t32 - cube * 6u);
        const u32 row = cube / cx;
        idx[0][0] = (i64)(cube - row * cx);
        const u32 lay = row / cy;
        idx[0][1] = (i64)(row - lay * cy);
        idx[0][2] = (i64)lay;
    }
    else
    {
        const i64 cube = t / 6;
        perm = (int)(t % 6);
        idx[0][0] = cube % cxn;
        idx[0][1] = (cube / cxn) % cyn;
        idx[0][2] = cube / (cxn * cyn);
    }
#pragma unroll
    for (int v = 1; v < 4; ++v)
    {
#pragma unroll
        for (int d = 0; d < 3; ++d)
            idx[v][d] = idx[v - 1][d] + (c_kuhn[perm][v - 1] == d ? 1 : 0);
    }
    const double dx = (double)(nxn - 1), dy = (double)(nyn - 1), dz = (double)(nzn - 1);
    // a vertex coordinate is index / cells; along an axis the four vertices only take the cube's lower
    // or upper index, so two divisions per axis (not four) give the same bits
    const double dd[3] = {dx, dy, dz};
    double lo[3], hi[3];
#pragma unroll
    for (int d = 0; d < 3; ++d)
    {
        lo[d] = div_finite((double)idx[0][d], dd[d]);
        hi[d] = (double)(idx[0][d] + 1) / dd[d];
    }
    double p[4][3];
    u64 node[4];
#pragma unroll
    for (int v = 0; v < 4; ++v)
    {
#pragma unroll
        for (int d = 0; d < 3; ++d)
            p[v][d] = idx[v][d] == idx[0][d] ? lo[d] : hi[d];
        node[v] = (u64)(idx[v][0] + nxn * idx[v][1] + nxn * nyn * idx[v][2]);
    }
    // P1 gradients from the inverse edge matrix; operation order mirrors the CPU oracle
    double a[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c)
            a[r][c] = p[c + 1][r] - p[0][r];
    const double c00 = a[1][1] * a[2][2] - a[1][2] * a[2][1];
    const double c01 = a[1][2] * a[2][0] - a[1][0] * a[2][2];
    const double c02 = a[1][0] * a[2][1] - a[1][1] * a[2][0];
    const double c10 = a[0][2] * a[2][1] - a[0][1] * a[2][2];
    const double c11 = a[0][0] * a[2][2] - a[0][2] * a[2][0];
    const double c12 = a[0][1] * a[2][0] - a[0][0] * a[2][1];
    const double c20 = a[0][1] * a[1][2] - a[0][2] * a[1][1];
    const double c21 = a[0][2] * a[1][0] - a[0][0] * a[1][2];
    const double c22 = a[0][0] * a[1][1] - a[0][1] * a[1][0];
    const double det = (a[0][0] * c00 + a[0][1] * c01) + a[0][2] * c02;
    double gr[4][3];
    gr[1][0] = div_finite(c00, det);
    gr[1][1] = div_finite(c10, det);
    gr[1][2] = div_finite(c20, det);
    gr[2][0] = div_finite(c01, det);
    gr[2][1] = div_finite(c11, det);
    gr[2][2] = div_finite(c21, det);
    gr[3][0] = div_finite(c02, det);
    gr[3][1] = div_finite(c12, det);
    gr[3][2] = div_finite(c22, det);
#pragma unroll
    for (int d = 0; d < 3; ++d)
        gr[0][d] = -((gr[1][d] + gr[2][d]) + gr[3][d]);
    e.vol = fabs(det) / 6.0;
#pragma unroll
    for (int il = 0; il < 4; ++il)
#pragma unroll
        for (int jl = il; jl < 4; ++jl)
        {
            double sum = 0.0;
#pragma unroll
            for (int d = 0; d < 3; ++d)
                sum += gr[jl][d] * gr[il][d];
            e.S[il][jl] = sum;
            e.S[jl][il] = sum;
        }
#pragma unroll
    for (int v = 0; v < 4; ++v)
    {
        e.ckey[v] = L.colpart(node[v]);
        e.rkey[v] = L.rowpart(node[v], tid, flavour);
        if (slab && L.owner(e.ckey[v]) != (u32)L.self)
            e.has_foreign = 1;
    }
}

// The 20 records of tetrahedron t, in call order, to dst[0..20).  Returns 1 if one of its columns belongs to
// another rank (slab handles).
__device__ __forceinline__ int fem_tet_records(i64 t, i64 nxn, i64 nyn, i64 nzn, const KeyLayout &L, u32 tid, u32 flavour,
                                               bool slab, Rec *dst)
{
    FemTet e;
    fem_tet_compute(t, nxn, nyn, nzn, L, tid, flavour, slab, e);
    int q = 0;
#pragma unroll
    for (int il = 0; il < 4; ++il)
#pragma unroll
        for (int w = 0; w < 5; ++w)
        {
            Rec r;
            r.key = e.key(il, w);
            r.val = e.val(il, w);
            dst[q++] = r;
        }
    return e.has_foreign;
}

// Stream order: a block's records through shared memory, coalesced 16-byte stores.
__global__ void __launch_bounds__(FEM_THREADS)
emit_p1fem_kernel(i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour, i64 tet_begin, i64 tet_end,
                  Rec *__restrict__ out, StageFlags sf)
{
    // a thread's 20 records sit FEM_PITCH records apart: with a pitch of 21 (84 words) the 16-byte
    // stores of a quarter warp fall into eight different bank groups instead of two
    __shared__ Rec s_rec[FEM_THREADS * FEM_PITCH];
    const i64 t_first = tet_begin + (i64)blockIdx.x * FEM_THREADS;
    const i64 t_last = min(t_first + FEM_THREADS, tet_end);
    const i64 t = t_first + threadIdx.x;
    int has_foreign = 0;
    if (t < t_last)
        has_foreign = fem_tet_records(t, nxn, nyn, nzn, L, tid, flavour, sf.flags != nullptr, s_rec + threadIdx.x * FEM_PITCH);
    // slab handles: only blocks at a slab face hold records of other ranks; every other block stores without
    // looking at owner bits (the emitter is issue-bound: the per-record checks cost 0.16 ms of 1.07 ms)
    if (!__syncthreads_or(has_foreign))
        sf.flags = nullptr;
    const i64 nrec = (t_last - t_first) * FEM_REC;
    const i64 pos0 = (t_first - tet_begin) * FEM_REC;
    Rec *dst = out + pos0;
#pragma unroll 2 // unrolled further, the loop needs more registers than the tetrahedron kernel above it
    for (i64 q = threadIdx.x; q < nrec; q += FEM_THREADS)
    {
        const int tt = (int)q / FEM_REC;
        const Rec r = s_rec[tt * FEM_PITCH + ((int)q - tt * FEM_REC)];
        st_staged(dst + q, r, L, sf, out);
    }
}

// Grouped chunks (xsb_chunk.cuh): a warp's 32 tetrahedra = one chunk of 640 records, brought into column
// order without a block-wide barrier -- and without looking at the records one by one: an element's 20 records
// fall on 4 columns (its nodes), 5 each, in a fixed order (record q = 5 il + w, FemTet), so the warp only runs
// the chunk's 128 (element, node) VISITS through its table, in call order (4 batches instead of 20), and every
// visit stands for 5 records: run offset = 5 x (visits of the column by earlier elements) + the record's fixed
// rank among its element's 5.  Keys, values and element matrices stay in the registers of the lane that
// computed them; only the 128 grouping keys pass through shared memory.
constexpr int FEMG_HB = 7; // 128 table slots: 32 neighbouring tetrahedra touch a few dozen nodes
struct FemWarpSpace
{
    u32 g[128]; // visit v = 4 element + node: grouping key, then (slot, visits before)
    ChunkSpaceT<FEMG_HB> tab;
};

__global__ void __launch_bounds__(FEM_THREADS, 7)
emit_p1fem_grouped_kernel(i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour, i64 tet_begin, i64 tet_end,
                          Rec *__restrict__ out, StageFlags sf, RunTarget rt, u32 chunk0, u32 pos_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr u32 full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FemWarpSpace &sp = reinterpret_cast<FemWarpSpace *>(smem_raw)[warp];
    const u32 wchunk = blockIdx.x * (FEM_THREADS / 32) + warp; // chunk of this warp
    const i64 t_first = tet_begin + (i64)wchunk * 32;
    if (t_first >= tet_end)
        return;
    const i64 t_last = min(t_first + 32, tet_end);
    const i64 t = t_first + lane;
    chunk_space_init(sp.tab, lane);
    FemTet e;
    e.has_foreign = 0;
    if (t < t_last)
    {
        fem_tet_compute(t, nxn, nyn, nzn, L, tid, flavour, sf.flags != nullptr, e);
        uint4 gq;
        gq.x = (u32)(e.ckey[0] >> rt.colshift) & rt.gmask;
        gq.y = (u32)(e.ckey[1] >> rt.colshift) & rt.gmask;
        gq.z = (u32)(e.ckey[2] >> rt.colshift) & rt.gmask;
        gq.w = (u32)(e.ckey[3] >> rt.colshift) & rt.gmask;
        reinterpret_cast<uint4 *>(sp.g)[lane] = gq;
    }
    if (!__any_sync(full, e.has_foreign))
        sf.flags = nullptr;
    __syncwarp();
    const u32 visits = (u32)(t_last - t_first) * 4u;
    const i64 c0 = (t_first - tet_begin) * FEM_REC; // position of the chunk in this launch's output
    const u32 lt = lanemask_lt();
    u32 d = 0;
#pragma unroll
    for (int b = 0; b < 4; ++b)
    { // at most 128 distinct columns: never more than the table takes
        if ((u32)(b * 32) < visits) // warp-uniform
        {
            const u32 v = b * 32 + lane;
            const u32 g = v < visits ? sp.g[v] : 0u;
            const u32 rs = (u32)(b * 32 + 32) <= visits ? chunk_count_batch<FEMG_HB, true>(sp.tab, g, true, lt, d)
                                                        : chunk_count_batch<FEMG_HB, false>(sp.tab, g, v < visits, lt, d);
            if (v < visits)
                sp.g[v] = rs; // (slot, visits of this column before this one)
        }
    }
    static_assert(ChunkSpaceT<FEMG_HB>::H >= 128, "a chunk's 128 visits must fit the table");
    chunk_scan(sp.tab, d, lane, 5u);
    __syncwarp();
    if (t < t_last)
    {
        Rec *dst = out + c0;
        const uint4 gq = reinterpret_cast<const uint4 *>(sp.g)[lane];
        const u32 rs[4] = {gq.x, gq.y, gq.z, gq.w};
        u32 base[4];
#pragma unroll
        for (int c = 0; c < 4; ++c)
            base[c] = (u32)sp.tab.start[rs[c] >> 16] + 5u * (rs[c] & 0xffffu);
#pragma unroll
        for (int c = 0; c < 4; ++c)
        { // the element's 5 records of column c sit next to each other, in call order: rows 0 .. c-1, the mass term
          // of row c, rows c .. 3 -- written as full 32-byte sectors (STG.256) where two of them share one
            Rec rr[5];
#pragma unroll
            for (int lr = 0; lr < 5; ++lr)
            {
                const int il = lr <= c ? lr : lr - 1;
                const int w = lr == c ? 0 : c + 1;
                rr[lr].key = e.key(il, w);
                rr[lr].val = e.val(il, w);
            }
            Rec *p = dst + base[c];
            auto pair = [&](Rec *q, const Rec &a, const Rec &b) {
                st_v4_u64(q, a.key, (u64)__double_as_longlong(a.val), b.key, (u64)__double_as_longlong(b.val));
            };
            if ((reinterpret_cast<uintptr_t>(p) & 16u) != 0)
            {
                st_rec(p, rr[0]);
                pair(p + 1, rr[1], rr[2]);
                pair(p + 3, rr[3], rr[4]);
            }
            else
            {
                pair(p, rr[0], rr[1]);
                pair(p + 2, rr[2], rr[3]);
                st_rec(p + 4, rr[4]);
            }
            if (sf.flags != nullptr && L.owner(e.ckey[c]) != (u32)L.self)
            { // (5 records: at most two tiles)
                sf.flags[(sf.pos0 + c0 + (i64)base[c]) >> kRouteTileShift] = 1; // benign race: same value
                sf.flags[(sf.pos0 + c0 + (i64)base[c] + 4) >> kRouteTileShift] = 1;
            }
        }
    }
    chunk_publish(sp.tab, rt, chunk0 + wchunk, pos_out + (u32)c0, d, true, lane, 5u);
}

void emit_p1fem(cudaStream_t stream, i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour,
                i64 cz_begin, i64 cz_end, Rec *out, LaunchCounter &lc, StageFlags sf)
{
    const i64 per_layer = 6 * (nxn - 1) * (nyn - 1);
    const i64 tet_begin = cz_begin * per_layer, tet_end = cz_end * per_layer;
    if (tet_end <= tet_begin)
        return;
    const i64 blocks = (tet_end - tet_begin + FEM_THREADS - 1) / FEM_THREADS;
    emit_p1fem_kernel<<<(unsigned)blocks, FEM_THREADS, 0, stream>>>(nxn, nyn, nzn, L, tid, flavour, tet_begin,
                                                                    tet_end, out, sf);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

u32 emit_p1fem_chunks(i64 nxn, i64 nyn, i64 cz_begin, i64 cz_end)
{
    const i64 tets = 6 * (nxn - 1) * (nyn - 1) * (cz_end - cz_begin);
    return (u32)((tets + 31) / 32);
}

// grouped variant: returns the chunks appended to the run index
u32 emit_p1fem_grouped(cudaStream_t stream, i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour, i64 cz_begin,
                       i64 cz_end, Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0, u32 pos0)
{
    const i64 per_layer = 6 * (nxn - 1) * (nyn - 1);
    const i64 tet_begin = cz_begin * per_layer, tet_end = cz_end * per_layer;
    if (tet_end <= tet_begin)
        return 0;
    static FuncAttrOnce once;
    const int smem = (int)(sizeof(FemWarpSpace) * (FEM_THREADS / 32));
    once.set(emit_p1fem_grouped_kernel, smem, true);
    const i64 blocks = (tet_end - tet_begin + FEM_THREADS - 1) / FEM_THREADS;
    emit_p1fem_grouped_kernel<<<(unsigned)blocks, FEM_THREADS, smem, stream>>>(nxn, nyn, nzn, L, tid, flavour, tet_begin,
                                                                               tet_end, out, sf, rt, chunk0, pos0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    return emit_p1fem_chunks(nxn, nyn, cz_begin, cz_end);
}

// ------------------------------------------------------------------------
// block reaction-diffusion stream: per node, per outgoing edge a dense ns x ns
// block applied as update_pair per block entry, then an ns x ns reaction block.
// One thread per (node, block entry): it writes 4 consecutive records per edge.
// ------------------------------------------------------------------------
struct RdGeom
{
    i64 nx, ny, nz, ns;
    __host__ __device__ i64 edges_before(i64 i, i64 j, i64 k) const
    { // edges leaving the nodes that precede (i,j,k)
        const i64 ex_row = nx - 1;
        auto ey = [&](i64 jj) { return jj < ny ? 1 : 0; };
        auto ez = [&](i64 kk) { return kk < nz ? 1 : 0; };
        const i64 pey = (j - 1) < (ny - 1) ? (j - 1) : (ny - 1);
        const i64 pez = (k - 1) < (nz - 1) ? (k - 1) : (nz - 1);
        const i64 pex = (i - 1) < (nx - 1) ? (i - 1) : (nx - 1);
        i64 s = (k - 1) * (ny * ex_row + nx * (ny - 1)) + nx * ny * pez;
        s += (j - 1) * ex_row + nx * pey + (j - 1) * nx * ez(k);
        s += pex + (i - 1) * (ey(j) + ez(k));
        return s;
    }
};

i64 blockrd_count(i64 nx, i64 ny, i64 nz, i64 ns)
{
    const i64 edges = (nx - 1) * ny * nz + nx * (ny - 1) * nz + nx * ny * (nz - 1);
    return edges * 4 * ns * ns + nx * ny * nz * ns * ns;
}

__global__ void __launch_bounds__(256)
emit_blockrd_kernel(RdGeom g, u64 seed, KeyLayout L, u32 tid, u32 flavour, Rec *__restrict__ out, StageFlags sf)
{
    const i64 ns2 = g.ns * g.ns;
    const i64 total = g.nx * g.ny * g.nz * ns2;
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 w = (i64)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += stride)
    {
        const i64 l0 = w / ns2;
        const i64 ab = w % ns2;
        const u64 a = (u64)(ab / g.ns), b = (u64)(ab % g.ns);
        i64 i, j, k;
        node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
        const i64 eb = g.edges_before(i, j, k);
        i64 rec = eb * 4 * ns2 + l0 * ns2;      // records before this node
        u64 call = (u64)(eb * ns2 + l0 * ns2);  // rand() calls before this node
        const i64 step[3] = {1, g.nx, g.nx * g.ny};
        const bool has[3] = {i < g.nx, j < g.ny, k < g.nz};
        const u64 ia = (u64)(g.ns * l0) + a, ib = (u64)(g.ns * l0) + b;
#pragma unroll
        for (int d = 0; d < 3; ++d)
        {
            if (!has[d])
                continue;
            const double v = philox_uniform(seed, call + (u64)ab);
            const u64 l2 = (u64)(l0 + step[d]);
            const u64 ja = (u64)g.ns * l2 + a, jb = (u64)g.ns * l2 + b;
            Rec *dst = out + rec + ab * 4;
            Rec r;
            r.val = -v;
            r.key = L.pack(jb, ia, tid, flavour); // (-v, i_a, j_b)
            st_staged(dst + 0, r, L, sf, out);
            r.key = L.pack(ib, ja, tid, flavour); // (-v, j_a, i_b)
            st_staged(dst + 1, r, L, sf, out);
            r.val = v;
            r.key = L.pack(ib, ia, tid, flavour); // ( v, i_a, i_b)
            st_staged(dst + 2, r, L, sf, out);
            r.key = L.pack(jb, ja, tid, flavour); // ( v, j_a, j_b)
            st_staged(dst + 3, r, L, sf, out);
            rec += 4 * ns2;
            call += (u64)ns2;
        }
        Rec r;
        r.val = philox_uniform(seed, call + (u64)ab);
        r.key = L.pack(ib, ia, tid, flavour);
        st_staged(out + rec + ab, r, L, sf, out);
    }
}

// Grouped chunks (xsb_chunk.cuh): a warp emits the records of `npw` consecutive nodes (at most 512 records:
// ns <= 6) into its own shared memory in call order, brings them into column order and stores them where the
// flush will read them.
constexpr int RDG_WARPS = 4;
constexpr int RDG_HB = 8;
struct RdWarpSpace
{
    u32 vis[4 * 32]; // visits [kind][lane]: (slot, records of the column before the visit)
    ChunkSpaceT<RDG_HB> tab;
};
__host__ __device__ inline i64 rd_node_rec(const RdGeom &g, i64 l0)
{ // records emitted by the nodes before l0 (l0 == number of nodes: all records)
    const i64 ns2 = g.ns * g.ns;
    const i64 N = g.nx * g.ny * g.nz;
    const i64 eb = l0 >= N ? g.edges_before(1, 1, g.nz + 1)
                           : [&]() {
                                 i64 i, j, k;
                                 node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
                                 return g.edges_before(i, j, k);
                             }();
    return eb * 4 * ns2 + (l0 >= N ? N : l0) * ns2;
}
static int rd_nodes_per_warp(i64 ns)
{
    const i64 ns2 = ns * ns;
    return (int)std::max<i64>(1, std::min<i64>(32 / ns2, CH_RECORDS / (13 * ns2)));
}

// Grouping by VISITS (see emit_fdrand_grouped_kernel): node l touches the ns columns of its own block row -- from every
// edge pair it emits 2 ns records per column, plus ns reaction records -- and the ns columns of each far end (2 ns
// records per column).  A warp holds npw nodes, so a kind of visit (z-ends, y-ends, x-ends, own) has npw * ns <= 32
// (node, species) visitors with different columns; a column meets its visitors in node = call order.  Every
// (node, a, b) item then computes its 13 records and stores them straight to their place of the grouped chunk (the two
// records a pair leaves in a column are neighbours: one 256-bit store where they share a sector):
//   far column (pair d, species b):  (-v, i_a, j_b) at 2 a, (v, j_a, j_b) at 2 a + 1
//   own column b: pair d (the dd-th existing one): (-v, j_a, i_b) at 2 ns dd + 2 a, (v, i_a, i_b) one behind it;
//                 reaction (i_a, i_b) at 2 ns nd + a
__global__ void __launch_bounds__(RDG_WARPS * 32)
emit_blockrd_grouped_kernel(RdGeom g, u64 seed, KeyLayout L, u32 tid, u32 flavour, int npw, Rec *__restrict__ out,
                            StageFlags sf, RunTarget rt, u32 chunk0, u32 pos_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr u32 full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    RdWarpSpace &sp = reinterpret_cast<RdWarpSpace *>(smem_raw)[warp];
    const i64 N = g.nx * g.ny * g.nz;
    const u32 wchunk = blockIdx.x * RDG_WARPS + warp;
    const i64 l_first = (i64)wchunk * npw;
    if (l_first >= N)
        return;
    const i64 l_last = min(l_first + npw, N);
    const u32 ns = (u32)g.ns, ns2 = ns * ns;
    const i64 w_rec0 = rd_node_rec(g, l_first);
    chunk_space_init(sp.tab, lane);
    const i64 step[3] = {1, g.nx, g.nx * g.ny};
    auto gkey = [&](u64 col) { return (u32)(L.pack(col, 0, tid, flavour) >> rt.colshift) & rt.gmask; };
    const u32 lt = lanemask_lt();
    u32 d = 0, len = 0;
    { // ---- the visits: lane v = (node v / ns, species v % ns)
        const u32 nvis = (u32)(l_last - l_first) * ns; // <= 32
        const bool have = (u32)lane < nvis;
        const u32 vn = (u32)lane / ns, vb = (u32)lane - vn * ns;
        const i64 l0 = l_first + (i64)vn;
        i64 i = 1, j = 1, k = 1;
        if (have)
            node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
        const bool has[3] = {have && i < g.nx, have && j < g.ny, have && k < g.nz};
        const u32 nd = (u32)has[0] + (u32)has[1] + (u32)has[2];
#pragma unroll
        for (int dd = 2; dd >= 0; --dd) // z-ends, y-ends, x-ends
            sp.vis[dd * 32 + lane] = chunk_visit_batch(sp.tab, has[dd] ? gkey((u64)ns * (u64)(l0 + step[dd]) + vb) : 0u,
                                                       has[dd], 2u * ns, lt, d);
        const u32 w_own = ns * (2u * nd + 1u);
        sp.vis[3 * 32 + lane] = chunk_visit_batch(sp.tab, have ? gkey((u64)ns * (u64)l0 + vb) : 0u, have, w_own, lt, d);
        len = have ? w_own + 2u * ns * nd : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            len += __shfl_xor_sync(full, len, o);
    }
    chunk_scan(sp.tab, d, lane);
    const u32 nitems = (u32)(l_last - l_first) * ns2;
    for (u32 it = lane; it < nitems; it += 32)
    {
        const u32 nl = it / ns2;
        const i64 l0 = l_first + (i64)nl;
        const u32 ab = it - nl * ns2;
        const u32 a = ab / ns, b = ab - a * ns;
        i64 i, j, k;
        node_ijk(l0, g.nx, g.ny, g.nz, i, j, k);
        const i64 eb = g.edges_before(i, j, k);
        u64 call = (u64)(eb * (i64)ns2 + l0 * (i64)ns2); // rand() calls before this node
        const bool has[3] = {i < g.nx, j < g.ny, k < g.nz};
        const u64 ia = (u64)((i64)ns * l0) + a, ib = (u64)((i64)ns * l0) + b;
        const u32 v = nl * ns + b; // the visitor that speaks for this item's columns
        Rec *const dst = out + w_rec0;
        Rec *own = dst + chunk_dest(sp.tab.start, sp.vis[3 * 32 + v]) + 2u * a;
        auto mark = [&](const Rec *p, const Rec &r) {
            if (sf.flags != nullptr && L.owner(r.key) != (u32)L.self)
                sf.flags[(sf.pos0 + w_rec0 + (i64)(p - dst)) >> kRouteTileShift] = 1; // benign race: same value
        };
        // two neighbouring records: one 256-bit store when they share a sector
        auto put2 = [&](Rec *p, const Rec &r0, const Rec &r1) {
            mark(p, r0);
            mark(p + 1, r1);
            if (reinterpret_cast<uintptr_t>(p) & 16u)
            {
                st_rec(p, r0);
                st_rec(p + 1, r1);
            }
            else
                st_v4_u64(p, r0.key, (u64)__double_as_longlong(r0.val), r1.key, (u64)__double_as_longlong(r1.val));
        };
#pragma unroll
        for (int dd = 0; dd < 3; ++dd)
        {
            if (!has[dd])
                continue;
            const double val = philox_uniform(seed, call + (u64)ab);
            const u64 l2 = (u64)(l0 + step[dd]);
            const u64 ja = (u64)ns * l2 + a, jb = (u64)ns * l2 + b;
            Rec *far = dst + chunk_dest(sp.tab.start, sp.vis[dd * 32 + v]) + 2u * a;
            Rec f0, f1, o0, o1;
            f0.val = -val;
            f0.key = L.pack(jb, ia, tid, flavour); // (-v, i_a, j_b)
            o0.val = -val;
            o0.key = L.pack(ib, ja, tid, flavour); // (-v, j_a, i_b)
            o1.val = val;
            o1.key = L.pack(ib, ia, tid, flavour); // ( v, i_a, i_b)
            f1.val = val;
            f1.key = L.pack(jb, ja, tid, flavour); // ( v, j_a, j_b)
            put2(far, f0, f1);
            put2(own, o0, o1);
            own += 2u * ns;
            call += (u64)ns2;
        }
        Rec r;
        r.val = philox_uniform(seed, call + (u64)ab);
        r.key = L.pack(ib, ia, tid, flavour);
        Rec *rp = own - (int)a; // the reaction block follows the pairs: position 2 ns nd + a (own stands at ... + 2 a)
        mark(rp, r);
        st_rec(rp, r);
    }
    chunk_publish(sp.tab, rt, chunk0 + wchunk, pos_out + (u32)w_rec0, d, true, lane);
}

// 0: this species count is emitted in stream order only (a node's records exceed a chunk)
u32 emit_blockrd_chunks(i64 nx, i64 ny, i64 nz, int ns)
{
    if (13 * (i64)ns * ns > CH_RECORDS)
        return 0;
    const i64 npw = rd_nodes_per_warp(ns);
    return (u32)((nx * ny * nz + npw - 1) / npw);
}

u32 emit_blockrd_grouped(cudaStream_t stream, i64 nx, i64 ny, i64 nz, int ns, u64 seed, KeyLayout L, u32 tid, u32 flavour,
                         Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0, u32 pos0)
{
    RdGeom g{nx, ny, nz, (i64)ns};
    const u32 chunks = emit_blockrd_chunks(nx, ny, nz, ns);
    static FuncAttrOnce once;
    const int smem = (int)(sizeof(RdWarpSpace) * RDG_WARPS);
    once.set(emit_blockrd_grouped_kernel, smem, true);
    emit_blockrd_grouped_kernel<<<(chunks + RDG_WARPS - 1) / RDG_WARPS, RDG_WARPS * 32, smem, stream>>>(
        g, seed, L, tid, flavour, rd_nodes_per_warp(ns), out, sf, rt, chunk0, pos0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
    return chunks;
}

void emit_blockrd(cudaStream_t stream, i64 nx, i64 ny, i64 nz, int ns, u64 seed, KeyLayout L, u32 tid,
                  u32 flavour, Rec *out, LaunchCounter &lc, StageFlags sf)
{
    RdGeom g{nx, ny, nz, (i64)ns};
    const i64 total = nx * ny * nz * ns * ns;
    const int threads = 256;
    const int blocks = (int)std::min<i64>((total + threads - 1) / threads, (i64)kNumSM * 32);
    emit_blockrd_kernel<<<blocks, threads, 0, stream>>>(g, seed, L, tid, flavour, out, sf);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------
// Element-by-element insertion (test/femtools.jl:45-72 with the caller's mesh): row connectivity rdofs[kr x ncells],
// column connectivity cdofs[kc x ncells] and dense element matrices Aloc[kr x kc x ncells], all column-major (the
// square loop: kr == kc, rdofs == cdofs).  Call p = kr kc c + kr jl + il is
// (row = rdofs[il, c], col = cdofs[jl, c], v = Aloc[il, jl, c]): the records of one (element, column) VISIT are kr
// neighbours in call order.
//
// A warp owns a chunk of whole elements (at most EL_VISITS visits and EL_VISITS row dofs).  Grouped (xsb_chunk.cuh):
// the chunk's visits run through the warp's table with match.any (neighbouring elements share columns) and every
// visit stands for kr records, so a record goes to start[slot] + kr x (visits of its column before its own) + il --
// stable, also when an element repeats a dof.  A column holds at most 128 min(kr, kc) records of a chunk; repeated
// column dofs can pile up more than one run may hold (CH_RUN_MAX): such a column is published as several runs
// (chunk_publish_split).  Call order (ungrouped): record p goes to p.  Either way the lanes walk the
// chunk's values in memory order (coalesced 8-byte loads) and store one 16-byte record each; consecutive lanes store
// consecutive records wherever they belong to one visit, so the stores merge into whole sectors there.
// ------------------------------------------------------------------------
constexpr int EL_WARPS = 4;
constexpr int EL_VISITS = 128; // visits per chunk: records (<= 128 min(kr, kc) <= 8192) fit the 16-bit run offsets
constexpr int EL_HB = 8;       // 256 table slots for at most 128 distinct columns
struct ElWarpSpace
{
    u64 ckey[EL_VISITS]; // visit v = element * kc + jl of the chunk: column half of its keys
    u64 rkey[EL_VISITS]; // row dof l = element * kr + il of the chunk: row half of its keys
    u32 vis[EL_VISITS];  // visit v: (slot << 16 | visits of its column before it)
    ChunkSpaceT<EL_HB> tab;
};
static_assert(ChunkSpaceT<EL_HB>::DMAX >= EL_VISITS, "a chunk's visits must fit the table");

__host__ __device__ __forceinline__ int el_cells_per_chunk(int kr, int kc) { return EL_VISITS / (kr > kc ? kr : kc); }

u32 insert_elements_chunks(int kr, int kc, i64 ncells)
{
    const i64 e = el_cells_per_chunk(kr, kc);
    return (u32)((ncells + e - 1) / e);
}

// x / k for x < 128 k: (x * ceil(2^22 / k)) >> 22 is exact there (k <= 64) and stays in 32 bits
struct DivK
{
    u32 inv;
    __device__ __forceinline__ explicit DivK(u32 k) : inv(((1u << 22) + k - 1u) / k) {}
    __device__ __forceinline__ u32 operator()(u32 x) const { return (x * inv) >> 22; }
};

template <typename Ti, bool GROUPED>
__global__ void __launch_bounds__(EL_WARPS * 32)
insert_elements_kernel(const Ti *__restrict__ rdofs, const Ti *__restrict__ cdofs, const double *__restrict__ Aloc, int kr,
                       int kc, i64 ncells, i64 base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour,
                       Rec *__restrict__ out, u64 *__restrict__ d_err, StageFlags sf, RunTarget rt, u32 chunk0, u32 pos0)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    ElWarpSpace &sp = reinterpret_cast<ElWarpSpace *>(smem_raw)[warp];
    const u32 chunk = blockIdx.x * EL_WARPS + warp;
    const i64 per = el_cells_per_chunk(kr, kc);
    const i64 e0 = (i64)chunk * per;
    if (e0 >= ncells)
        return;
    const u32 ukr = (u32)kr, ukc = (u32)kc;
    const u32 ne = (u32)min(per, ncells - e0);
    const u32 nvis = ne * ukc; // visits = column dofs of the chunk
    const u32 nrow = ne * ukr; // row dofs of the chunk
    const u32 nrec = nvis * ukr;
    const i64 c0 = e0 * kr * kc; // position of the chunk's first record (call order)
    // every quotient below has a dividend under 128 x its divisor: p < nrec <= 128 min(kr, kc), v < nvis <= 128
    const DivK divr(ukr), divc(ukc);
    // *d_err: 2 x element + (1 for a column dof), so the first offending element wins
    bool foreign = false;
    for (u32 l = lane; l < nvis; l += 32)
    {
        i64 d = (i64)cdofs[e0 * kc + l] - base;
        if (d < 0 || d >= n)
        { // BoundsError (sparsematrixcsc.jl:8-10): the batch is rejected, whatever is written for it is dropped
            atomicMin(d_err, ((u64)(e0 + divc(l)) << 1) | 1u);
            d = 0;
        }
        const u64 ck = L.colpart((u64)d);
        sp.ckey[l] = ck;
        foreign |= sf.flags != nullptr && L.owner(ck) != (u32)L.self;
    }
    for (u32 l = lane; l < nrow; l += 32)
    {
        i64 d = (i64)rdofs[e0 * kr + l] - base;
        if (d < 0 || d >= m)
        {
            atomicMin(d_err, (u64)(e0 + divr(l)) << 1);
            d = 0;
        }
        sp.rkey[l] = L.rowpart((u64)d, tid, flavour);
    }
    // slab handles: only chunks that hold a column of another rank mark route tiles
    if (!__any_sync(0xffffffffu, foreign))
        sf.flags = nullptr;
    __syncwarp();
    u32 d = 0;
    bool split = false; // a column of the chunk holds more records than one run may
    if (GROUPED)
    {
        chunk_space_init(sp.tab, lane);
        const u32 lt = lanemask_lt();
#pragma unroll
        for (int b = 0; b < EL_VISITS / 32; ++b)
        {
            if ((u32)(b * 32) < nvis) // warp-uniform
            {
                const u32 v = b * 32 + lane;
                const u32 g = v < nvis ? (u32)(sp.ckey[v] >> rt.colshift) & rt.gmask : 0u;
                const u32 rs = (u32)(b * 32 + 32) <= nvis ? chunk_count_batch<EL_HB, true>(sp.tab, g, true, lt, d)
                                                          : chunk_count_batch<EL_HB, false>(sp.tab, g, v < nvis, lt, d);
                if (v < nvis)
                    sp.vis[v] = rs;
            }
        }
        __syncwarp();
        if (nrec > CH_RUN_MAX) // warp-uniform
        {                      // a column holds kr x (its visits) records of the chunk
            bool over = false;
            for (u32 v = lane; v < nvis; v += 32)
                over |= ((sp.vis[v] & 0xffffu) + 1u) * ukr > CH_RUN_MAX;
            split = __any_sync(0xffffffffu, over);
        }
        chunk_scan(sp.tab, d, lane, ukr);
    }
    const double *src = Aloc + c0;
    Rec *dst = out + c0;
    auto put = [&](u32 p, double val) {
        const u32 v = divr(p), il = p - v * ukr; // visit (element, column dof) and row rank inside it
        const u32 e = divc(v);                   // the chunk's element
        Rec r;
        r.key = sp.ckey[v] | sp.rkey[e * ukr + il];
        r.val = val;
        u32 t = p;
        if (GROUPED)
        {
            const u32 vs = sp.vis[v];
            t = (u32)sp.tab.start[vs >> 16] + ukr * (vs & 0xffffu) + il;
        }
        st_rec(dst + t, r);
        if (sf.flags != nullptr && L.owner(r.key) != (u32)L.self)
            sf.flags[(sf.pos0 + c0 + (i64)t) >> kRouteTileShift] = 1; // benign race: same value
    };
    // four loads in flight per lane before the first record is built
    u32 p0 = 0;
    for (; p0 + 128 <= nrec; p0 += 128)
    {
        double vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
            vv[u] = __ldcs(src + p0 + u * 32 + lane);
#pragma unroll
        for (int u = 0; u < 4; ++u)
            put(p0 + u * 32 + lane, vv[u]);
    }
    for (u32 p = p0 + lane; p < nrec; p += 32)
        put(p, __ldcs(src + p));
    if (GROUPED && !split)
        chunk_publish(sp.tab, rt, chunk0 + chunk, pos0 + (u32)c0, d, true, lane, ukr);
    else if (GROUPED)
        chunk_publish_split(sp.tab, rt, chunk0 + chunk, pos0 + (u32)c0, d, lane, ukr);
}

template <typename Ti, bool GROUPED>
static void launch_insert_elements(cudaStream_t stream, const ElementBatch &eb, int base, i64 m, i64 n, const KeyLayout &L,
                                   u32 tid, u32 flavour, Rec *out, u64 *d_err, StageFlags sf, const RunTarget &rt,
                                   u32 chunk0, u32 pos0, LaunchCounter &lc)
{
    static FuncAttrOnce once;
    const int smem = (int)(sizeof(ElWarpSpace) * EL_WARPS);
    once.set(insert_elements_kernel<Ti, GROUPED>, smem, true);
    const u32 chunks = insert_elements_chunks(eb.kr, eb.kc, eb.ncells);
    insert_elements_kernel<Ti, GROUPED><<<(chunks + EL_WARPS - 1) / EL_WARPS, EL_WARPS * 32, smem, stream>>>(
        (const Ti *)eb.rdofs, (const Ti *)eb.cdofs, eb.Aloc, eb.kr, eb.kc, eb.ncells, (i64)base, m, n, L, tid, flavour, out,
        d_err, sf, rt, chunk0, pos0);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void insert_elements(cudaStream_t stream, const ElementBatch &eb, int idx64, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                     u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf)
{
    if (eb.ncells <= 0)
        return;
    const RunTarget none{};
    if (idx64)
        launch_insert_elements<int64_t, false>(stream, eb, base, m, n, L, tid, flavour, out, d_err, sf, none, 0, 0, lc);
    else
        launch_insert_elements<int32_t, false>(stream, eb, base, m, n, L, tid, flavour, out, d_err, sf, none, 0, 0, lc);
}

u32 insert_elements_grouped(cudaStream_t stream, const ElementBatch &eb, int idx64, int base, i64 m, i64 n, KeyLayout L,
                            u32 tid, u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf,
                            const RunTarget &rt, u32 chunk0, u32 pos0)
{
    if (eb.ncells <= 0)
        return 0;
    if (idx64)
        launch_insert_elements<int64_t, true>(stream, eb, base, m, n, L, tid, flavour, out, d_err, sf, rt, chunk0, pos0, lc);
    else
        launch_insert_elements<int32_t, true>(stream, eb, base, m, n, L, tid, flavour, out, d_err, sf, rt, chunk0, pos0, lc);
    return insert_elements_chunks(eb.kr, eb.kc, eb.ncells);
}

} // namespace xsb
