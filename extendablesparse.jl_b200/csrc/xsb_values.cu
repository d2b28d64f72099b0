// xsb_values.cu -- values-only work on the resident CSC:
//   lookup_slots / gather_values : findindex + getindex    (src/matrix/sparsematrixcsc.jl:7-23,
//                                                           src/matrix/extendable.jl:226-238)
//   frozen-pattern re-assembly   : the CSC-hit branch of updateindex! (extendable.jl:164-166)
//                                  resolved once into an entry->nzval map
//   Dirichlet passes             : mark_dirichlet / eliminate_dirichlet! (sparsematrixcsc.jl:97-148)
//   pattern fingerprint          : stands in for phash (sparsematrixcsc.jl:74)
#include "xsb_internal.h"

namespace xsb {

__global__ void __launch_bounds__(256) zero_kernel(double *__restrict__ x, i64 n)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
        x[k] = 0.0;
}

static inline int grid_for(i64 n, int threads, int waves = 16)
{
    return (int)std::min<i64>(std::max<i64>((n + threads - 1) / threads, 1), (i64)kNumSM * waves);
}

template <typename Ti> __global__ void __launch_bounds__(256) fill_index_kernel(Ti *__restrict__ x, i64 n, Ti v)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
        x[k] = v;
}

void fill_index(cudaStream_t stream, void *x, i64 count, int idx64, i64 value, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    if (idx64)
        fill_index_kernel<int64_t><<<grid_for(count, 256), 256, 0, stream>>>((int64_t *)x, count, (int64_t)value);
    else
        fill_index_kernel<int32_t><<<grid_for(count, 256), 256, 0, stream>>>((int32_t *)x, count, (int32_t)value);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void zero_values(cudaStream_t stream, double *nzval, i64 nnz, LaunchCounter &lc)
{
    if (nnz <= 0)
        return;
    zero_kernel<<<grid_for(nnz, 256), 256, 0, stream>>>(nzval, nnz);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// searchsortedfirst over one CSC column, sparsematrixcsc.jl:11-22
template <typename Ti>
__device__ __forceinline__ i64 find_slot(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, Ti base,
                                         i64 i, i64 j)
{
    i64 lo = (i64)colptr[j] - base, hi = (i64)colptr[j + 1] - base;
    const i64 end = hi;
    const Ti want = (Ti)i + base;
    while (lo < hi)
    {
        const i64 mid = lo + ((hi - lo) >> 1);
        if (rowval[mid] < want)
            lo = mid + 1;
        else
            hi = mid;
    }
    return (lo < end && rowval[lo] == want) ? lo : -1;
}

// where the positions of a lookup come from: (I[p], J[p]) arrays, or call p of an element loop
template <typename Ti> struct PosIJ
{
    const Ti *I, *J;
    __device__ __forceinline__ void at(i64 p, i64 &i, i64 &j) const
    {
        i = (i64)I[p];
        j = (i64)J[p];
    }
};
template <typename Ti> struct PosElements
{
    const Ti *dofs; // k x ncells, column-major
    i64 k;
    // call p = k^2 c + k jl + il is (dofs[il, c], dofs[jl, c])
    __device__ __forceinline__ void at(i64 p, i64 &i, i64 &j) const
    {
        const i64 kk = k * k, c = p / kk, r = p - c * kk, jl = r / k;
        i = (i64)dofs[c * k + (r - jl * k)];
        j = (i64)dofs[c * k + jl];
    }
};
template <typename Ti> struct PosElementsRect
{
    const Ti *rdofs, *cdofs; // kr x ncells and kc x ncells, column-major
    i64 kr, kc;
    // call p = kr kc c + kr jl + il is (rdofs[il, c], cdofs[jl, c])
    __device__ __forceinline__ void at(i64 p, i64 &i, i64 &j) const
    {
        const i64 kk = kr * kc, c = p / kk, r = p - c * kk, jl = r / kr;
        i = (i64)rdofs[c * kr + (r - jl * kr)];
        j = (i64)cdofs[c * kc + jl];
    }
};

// the square loop (one connectivity for rows and columns) reads it through PosElements, anything else through
// PosElementsRect
template <typename Ti, class F> static void with_element_pos(const ElementBatch &eb, F &&f)
{
    if (eb.rdofs == eb.cdofs && eb.kr == eb.kc)
        f(PosElements<Ti>{(const Ti *)eb.rdofs, (i64)eb.kr});
    else
        f(PosElementsRect<Ti>{(const Ti *)eb.rdofs, (const Ti *)eb.cdofs, (i64)eb.kr, (i64)eb.kc});
}

template <typename Ti, class Pos>
__global__ void __launch_bounds__(256)
lookup_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, Ti base, i64 m, i64 n, Pos pos, i64 count,
              i64 *__restrict__ slot, u64 *__restrict__ d_missing, u64 *__restrict__ d_oob)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        i64 i, j;
        pos.at(k, i, j);
        i -= base;
        j -= base;
        i64 s = -1;
        if (i < 0 || i >= m || j < 0 || j >= n)
            atomicMin(d_oob, (u64)k);
        else
        {
            s = find_slot<Ti>(colptr, rowval, base, i, j);
            if (s < 0)
                atomicAdd(d_missing, 1ull);
        }
        slot[k] = s;
    }
}

template <typename Ti, class Pos>
static void launch_lookup(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int base, Pos pos, i64 count, i64 *slot,
                          u64 *d_missing, u64 *d_oob, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    lookup_kernel<Ti, Pos><<<grid_for(count, 256), 256, 0, stream>>>((const Ti *)csc.colptr, (const Ti *)csc.rowval, (Ti)base,
                                                                      m, n, pos, count, slot, d_missing, d_oob);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void lookup_slots(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base, const void *I,
                  const void *J, i64 count, i64 *slot, u64 *d_missing, u64 *d_oob, LaunchCounter &lc)
{
    if (idx64)
        launch_lookup<int64_t>(stream, csc, m, n, base, PosIJ<int64_t>{(const int64_t *)I, (const int64_t *)J}, count, slot,
                               d_missing, d_oob, lc);
    else
        launch_lookup<int32_t>(stream, csc, m, n, base, PosIJ<int32_t>{(const int32_t *)I, (const int32_t *)J}, count, slot,
                               d_missing, d_oob, lc);
}

void lookup_slots_elements(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base,
                           const ElementBatch &eb, i64 count, i64 *slot, u64 *d_missing, u64 *d_oob, LaunchCounter &lc)
{
    if (idx64)
        with_element_pos<int64_t>(eb, [&](auto pos) {
            launch_lookup<int64_t>(stream, csc, m, n, base, pos, count, slot, d_missing, d_oob, lc);
        });
    else
        with_element_pos<int32_t>(eb, [&](auto pos) {
            launch_lookup<int32_t>(stream, csc, m, n, base, pos, count, slot, d_missing, d_oob, lc);
        });
}

__global__ void __launch_bounds__(256)
gather_kernel(const double *__restrict__ nzval, const i64 *__restrict__ slot, i64 count, double *__restrict__ out)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        const i64 s = slot[k];
        out[k] = s >= 0 ? nzval[s] : 0.0;
    }
}

void gather_values(cudaStream_t stream, const double *nzval, const i64 *slot, i64 count, double *out,
                   LaunchCounter &lc)
{
    if (count <= 0)
        return;
    gather_kernel<<<grid_for(count, 256), 256, 0, stream>>>(nzval, slot, count, out);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ---- frozen pattern: sort (slot, stream index) pairs by slot (stable) ----
__global__ void __launch_bounds__(256)
slots_to_records_kernel(const i64 *__restrict__ slot, i64 count, Rec *__restrict__ out)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        Rec r;
        r.key = (u64)slot[k];
        *reinterpret_cast<u64 *>(&r.val) = (u64)k;
        st_rec(out + k, r);
    }
}

void slots_to_records(cudaStream_t stream, const i64 *slot, i64 count, Rec *out, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    slots_to_records_kernel<<<grid_for(count, 256), 256, 0, stream>>>(slot, count, out);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// staged records whose (row, column) is not an entry of the CSC (MT wrapper: setindex! of a new entry is an error)
template <typename Ti>
__global__ void __launch_bounds__(256)
count_missing_kernel(const Rec *__restrict__ recs, i64 count, KeyLayout L, const Ti *__restrict__ colptr,
                     const Ti *__restrict__ rowval, Ti base, u64 *__restrict__ d_missing)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        const u64 key = recs[k].key;
        const i64 j = (i64)L.col(key), i = (i64)L.row(key);
        i64 lo = (i64)colptr[j] - base, hi = (i64)colptr[j + 1] - base;
        while (lo < hi)
        {
            const i64 mid = (lo + hi) >> 1;
            if ((i64)rowval[mid] - base < i)
                lo = mid + 1;
            else
                hi = mid;
        }
        const i64 end = (i64)colptr[j + 1] - base;
        if (!(lo < end && (i64)rowval[lo] - base == i))
            atomicAdd(reinterpret_cast<unsigned long long *>(d_missing), 1ull);
    }
}

void count_missing_records(cudaStream_t stream, const Rec *recs, i64 count, const KeyLayout &L, const CscView &csc,
                           int idx64, int base, u64 *d_missing, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    if (idx64)
        count_missing_kernel<int64_t><<<grid_for(count, 256), 256, 0, stream>>>(
            recs, count, L, (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, (int64_t)base, d_missing);
    else
        count_missing_kernel<int32_t><<<grid_for(count, 256), 256, 0, stream>>>(
            recs, count, L, (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, (int32_t)base, d_missing);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// sorted (slot,index) records -> perm[] and segstart[0..nnz]
__global__ void __launch_bounds__(256)
frozen_map_kernel(const Rec *__restrict__ sorted, i64 count, i64 nnz, u32 *__restrict__ perm,
                  u32 *__restrict__ segstart, u32 *__restrict__ slot32)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 s = (i64)blockIdx.x * blockDim.x + threadIdx.x; s < count; s += stride)
    {
        const Rec r = sorted[s];
        const u32 k = (u32) * reinterpret_cast<const u64 *>(&r.val); // position in the stream
        perm[s] = k;
        const i64 z = (i64)r.key;
        slot32[k] = (u32)z; // the 4-byte entry -> nzval map of the stream (fast mode)
        const i64 zprev = s > 0 ? (i64)sorted[s - 1].key : -1;
        // slots zprev+1 .. z start at s (slots without entries get an empty range)
        for (i64 q = zprev + 1; q <= z; ++q)
            segstart[q] = (u32)s;
        if (s == count - 1)
            for (i64 q = z + 1; q <= nnz; ++q)
                segstart[q] = (u32)count;
    }
}

void build_frozen_map(cudaStream_t stream, const Rec *sorted, i64 count, i64 nnz, u32 *perm, u32 *segstart, u32 *slot32,
                      LaunchCounter &lc)
{
    if (count <= 0)
    {
        XSB_CUDA(cudaMemsetAsync(segstart, 0, sizeof(u32) * (size_t)(nnz + 1), stream));
        return;
    }
    frozen_map_kernel<<<grid_for(count, 256), 256, 0, stream>>>(sorted, count, nnz, perm, segstart, slot32);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// Where value k of a re-assembly lives.  Plain handles: V[k].  SLAB (a stream frozen across column slabs): k runs
// over the combined index space [received from lower ranks | own stream | received from higher ranks], whose parts
// sit in two arrays -- the received values and the caller's V, which is read in place.
template <bool SLAB>
__device__ __forceinline__ const double *value_at(const double *V, const SlabValues &sv, u32 k)
{
    if constexpr (!SLAB)
        return V + k;
    else
        return k < sv.low ? sv.recv + k : (k - sv.low < sv.own ? V + (k - sv.low) : sv.recv + (k - sv.own));
}

// nzval[z] = ((nzval[z] + V[p0]) + V[p1]) + ...  in stream order: bit-exact with the reference's in-place CSC-hit
// updates (extendable.jl:164-166).  One thread per entry walks its piece of the permutation built at freeze time.
// The gathers of V go through L1: the threads of a block hold consecutive entries (a few dozen neighbouring columns),
// whose values come from a few short windows of the stream, so the 32-byte sectors of V are shared inside the block
// and HBM sees every value about once.  ZERO: the entries start from +0.0 instead of the resident value
// (nonzeros(A) .= 0 fused in: nzval is written, never read).  `sv` comes last so that the plain instantiations keep
// the parameter layout (and the code) they had before slab streams existed.
template <bool ZERO, bool SLAB>
__global__ void __launch_bounds__(256)
reassemble_det_kernel(const double *__restrict__ V, const u32 *__restrict__ perm, const u32 *__restrict__ segstart,
                      i64 nnz, double *__restrict__ nzval, SlabValues sv)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 z = (i64)blockIdx.x * blockDim.x + threadIdx.x; z < nnz; z += stride)
    {
        const u32 s0 = segstart[z], s1 = segstart[z + 1];
        if (s1 == s0)
        {
            if (ZERO)
                nzval[z] = 0.0;
            continue;
        }
        double acc = ZERO ? 0.0 : nzval[z];
        u32 s = s0;
        for (; s + 2 <= s1; s += 2)
        { // two gathers in flight, folded in order
            const double v0 = __ldg(value_at<SLAB>(V, sv, perm[s])), v1 = __ldg(value_at<SLAB>(V, sv, perm[s + 1]));
            acc = acc + v0;
            acc = acc + v1;
        }
        if (s < s1)
            acc = acc + __ldg(value_at<SLAB>(V, sv, perm[s]));
        nzval[z] = acc;
    }
}

void reassemble_deterministic(cudaStream_t stream, const double *V, const u32 *perm, const u32 *segstart, i64 nnz,
                              double *nzval, bool zero_first, LaunchCounter &lc, const SlabValues *sv)
{
    if (nnz <= 0)
        return;
    const int blocks = (int)std::min<i64>((nnz + 255) / 256, (i64)kNumSM * 64);
    const SlabValues none{};
    if (sv && zero_first)
        reassemble_det_kernel<true, true><<<blocks, 256, 0, stream>>>(V, perm, segstart, nnz, nzval, *sv);
    else if (sv)
        reassemble_det_kernel<false, true><<<blocks, 256, 0, stream>>>(V, perm, segstart, nnz, nzval, *sv);
    else if (zero_first)
        reassemble_det_kernel<true, false><<<blocks, 256, 0, stream>>>(V, perm, segstart, nnz, nzval, none);
    else
        reassemble_det_kernel<false, false><<<blocks, 256, 0, stream>>>(V, perm, segstart, nnz, nzval, none);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// fast mode: one atomic add per insertion through the 4-byte entry -> nzval map, in whatever order the hardware takes.
// SLAB: k runs over the combined index space; the own stream's positions in other ranks' columns carry kNoSlot.
template <bool SLAB>
__global__ void __launch_bounds__(256)
reassemble_fast_kernel(const double *__restrict__ V, const u32 *__restrict__ slot, i64 count,
                       double *__restrict__ nzval, SlabValues sv)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        if constexpr (!SLAB)
            atomicAdd(nzval + slot[k], V[k]);
        else
        {
            const u32 z = slot[k];
            if (z != kNoSlot)
                atomicAdd(nzval + z, __ldg(value_at<true>(V, sv, (u32)k)));
        }
    }
}

void reassemble_fast(cudaStream_t stream, const double *V, const u32 *slot, i64 count, double *nzval,
                     LaunchCounter &lc, const SlabValues *sv)
{
    if (count <= 0)
        return;
    if (sv)
        reassemble_fast_kernel<true><<<grid_for(count, 256, 32), 256, 0, stream>>>(V, slot, count, nzval, *sv);
    else
        reassemble_fast_kernel<false><<<grid_for(count, 256, 32), 256, 0, stream>>>(V, slot, count, nzval, SlabValues{});
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ---- frozen streams of slab handles (xsb_freeze_slab*): positions in GLOBAL columns, some owned by other ranks ----
// One pass over the stream: bounds, owner (KeyLayout::pack, the search the producers use), own positions -> nzval
// slot, foreign ones -> a routing tag {owner << 32 | stream index, (row, owner-relative column)} that the stable
// copy-out of xsb_route.cu gathers destination after destination.  Own positions (and bad ones) get tag owner self.
template <typename Ti, class Pos>
__global__ void __launch_bounds__(256)
slab_classify_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, Ti base, i64 m, i64 n_global,
                     KeyLayout Ls, Pos pos, i64 count, i64 *__restrict__ slot, Rec *__restrict__ tags,
                     u64 *__restrict__ d_missing, u64 *__restrict__ d_oob)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += stride)
    {
        i64 i, j;
        pos.at(k, i, j);
        i -= base;
        j -= base;
        i64 s = -1;
        u64 owner = (u64)Ls.self, where = 0;
        if (i < 0 || i >= m || j < 0 || j >= n_global)
            atomicMin(d_oob, (u64)k);
        else
        {
            const u64 key = Ls.colpart((u64)j);
            const u64 lc = Ls.col(key);
            owner = Ls.owner(key);
            if (owner == (u64)Ls.self)
            {
                s = find_slot<Ti>(colptr, rowval, base, i, (i64)lc);
                if (s < 0)
                    atomicAdd(d_missing, 1ull);
            }
            else
                where = (u64)i | (lc << 32);
        }
        slot[k] = s;
        Rec r;
        r.key = (owner << 32) | (u64)k;
        *reinterpret_cast<u64 *>(&r.val) = where;
        st_rec(tags + k, r);
    }
}

template <typename Ti, class Pos>
static void launch_classify(cudaStream_t stream, const CscView &csc, i64 m, i64 n_global, const KeyLayout &Ls, int base,
                            Pos pos, i64 count, i64 *slot, Rec *tags, u64 *d_missing, u64 *d_oob, LaunchCounter &lc)
{
    if (count <= 0)
        return;
    slab_classify_kernel<Ti, Pos><<<grid_for(count, 256), 256, 0, stream>>>(
        (const Ti *)csc.colptr, (const Ti *)csc.rowval, (Ti)base, m, n_global, Ls, pos, count, slot, tags, d_missing, d_oob);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void slab_classify(cudaStream_t stream, const CscView &csc, i64 m, i64 n_global, const KeyLayout &Ls, int idx64, int base,
                   const void *I, const void *J, i64 count, i64 *slot, Rec *tags, u64 *d_missing, u64 *d_oob,
                   LaunchCounter &lc)
{
    if (idx64)
        launch_classify<int64_t>(stream, csc, m, n_global, Ls, base, PosIJ<int64_t>{(const int64_t *)I, (const int64_t *)J},
                                 count, slot, tags, d_missing, d_oob, lc);
    else
        launch_classify<int32_t>(stream, csc, m, n_global, Ls, base, PosIJ<int32_t>{(const int32_t *)I, (const int32_t *)J},
                                 count, slot, tags, d_missing, d_oob, lc);
}

void slab_classify_elements(cudaStream_t stream, const CscView &csc, i64 m, i64 n_global, const KeyLayout &Ls, int idx64,
                            int base, const ElementBatch &eb, i64 count, i64 *slot, Rec *tags, u64 *d_missing,
                            u64 *d_oob, LaunchCounter &lc)
{
    if (idx64)
        with_element_pos<int64_t>(eb, [&](auto pos) {
            launch_classify<int64_t>(stream, csc, m, n_global, Ls, base, pos, count, slot, tags, d_missing, d_oob, lc);
        });
    else
        with_element_pos<int32_t>(eb, [&](auto pos) {
            launch_classify<int32_t>(stream, csc, m, n_global, Ls, base, pos, count, slot, tags, d_missing, d_oob, lc);
        });
}

// the gathered tags -> stream indices (kept for every step) and 8-byte positions {row, owner-relative column}
__global__ void __launch_bounds__(256)
slab_split_kernel(const Rec *__restrict__ tags, i64 n, u32 *__restrict__ idx, u64 *__restrict__ where)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride)
    {
        const Rec r = tags[q];
        idx[q] = (u32)r.key;
        where[q] = *reinterpret_cast<const u64 *>(&r.val);
    }
}

void slab_split(cudaStream_t stream, const Rec *tags, i64 n, u32 *idx, u64 *where, LaunchCounter &lc)
{
    if (n <= 0)
        return;
    slab_split_kernel<<<grid_for(n, 256), 256, 0, stream>>>(tags, n, idx, where);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// (slot, combined index) records over [received from lower ranks | own stream | received from higher ranks]: received
// positions are looked up in the slab, own ones bring the slot found at freeze time; foreign own positions and bad
// received ones get slot `nnz`, which sorts behind every real slot and stays out of the map
template <typename Ti>
__global__ void __launch_bounds__(256)
slab_records_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, Ti base, i64 m, i64 n,
                    const i64 *__restrict__ own_slot, i64 own, const uint2 *__restrict__ recv, i64 low, i64 total,
                    i64 nnz, Rec *__restrict__ out, u64 *__restrict__ d_missing, u64 *__restrict__ d_oob)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += stride)
    {
        i64 s;
        if (k >= low && k - low < own)
        {
            s = own_slot[k - low];
            if (s < 0)
                s = nnz;
        }
        else
        {
            const i64 q = k < low ? k : k - own;
            const uint2 p = recv[q];
            s = nnz;
            if ((i64)p.x >= m || (i64)p.y >= n)
                atomicMin(d_oob, (u64)q);
            else
            {
                const i64 f = find_slot<Ti>(colptr, rowval, base, (i64)p.x, (i64)p.y);
                if (f < 0)
                    atomicAdd(d_missing, 1ull);
                else
                    s = f;
            }
        }
        Rec r;
        r.key = (u64)s;
        *reinterpret_cast<u64 *>(&r.val) = (u64)k;
        st_rec(out + k, r);
    }
}

void slab_records(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base, const i64 *own_slot, i64 own,
                  const void *recv, i64 low, i64 total, Rec *out, u64 *d_missing, u64 *d_oob, LaunchCounter &lc)
{
    if (total <= 0)
        return;
    if (idx64)
        slab_records_kernel<int64_t><<<grid_for(total, 256), 256, 0, stream>>>(
            (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, (int64_t)base, m, n, own_slot, own,
            (const uint2 *)recv, low, total, csc.nnz, out, d_missing, d_oob);
    else
        slab_records_kernel<int32_t><<<grid_for(total, 256), 256, 0, stream>>>(
            (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, (int32_t)base, m, n, own_slot, own,
            (const uint2 *)recv, low, total, csc.nnz, out, d_missing, d_oob);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// per step: the values of the foreign positions, bucket after bucket, in the order of xsb_freeze_slab_prepare
__global__ void __launch_bounds__(256)
slab_pack_kernel(const double *__restrict__ V, const u32 *__restrict__ idx, i64 n, double *__restrict__ send)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride)
        send[q] = __ldg(V + idx[q]);
}

void slab_pack_values(cudaStream_t stream, const double *V, const u32 *idx, i64 n, double *send, LaunchCounter &lc)
{
    if (n <= 0)
        return;
    slab_pack_kernel<<<grid_for(n, 256), 256, 0, stream>>>(V, idx, n, send);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ---- Dirichlet passes (square matrices; sparsematrixcsc.jl:97-148) ----
template <typename Ti>
__global__ void __launch_bounds__(256)
mark_dirichlet_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval,
                      const double *__restrict__ nzval, i64 n, Ti base, double penalty,
                      unsigned char *__restrict__ marker)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    {
        unsigned char mk = 0;
        const i64 s = (i64)colptr[i] - base, e = (i64)colptr[i + 1] - base;
        for (i64 k = s; k < e; ++k)
            if ((i64)rowval[k] - base == i && nzval[k] >= penalty)
                mk = 1;
        marker[i] = mk;
    }
}

void mark_dirichlet(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, double penalty,
                    unsigned char *marker, LaunchCounter &lc)
{
    const int blocks = grid_for(n, 256);
    if (idx64)
        mark_dirichlet_kernel<int64_t><<<blocks, 256, 0, stream>>>(
            (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, csc.nzval, n, (int64_t)base, penalty, marker);
    else
        mark_dirichlet_kernel<int32_t><<<blocks, 256, 0, stream>>>(
            (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, csc.nzval, n, (int32_t)base, penalty, marker);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// The reference sweeps columns sequentially, but each nzval[k] is decided by
// (marker[col], marker[row], row==col) alone, so one thread per column is exact:
//   marked column: diagonal -> 1, rest -> 0;  then any off-diagonal in a marked row -> 0.
template <typename Ti>
__global__ void __launch_bounds__(256)
eliminate_dirichlet_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval,
                           double *__restrict__ nzval, i64 n, Ti base, const unsigned char *__restrict__ marker)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    {
        const bool mi = marker[i] != 0;
        const i64 s = (i64)colptr[i] - base, e = (i64)colptr[i + 1] - base;
        for (i64 k = s; k < e; ++k)
        {
            const i64 r = (i64)rowval[k] - base;
            if (mi)
                nzval[k] = (r == i) ? 1.0 : 0.0;
            if (r != i && marker[r] != 0)
                nzval[k] = 0.0;
        }
    }
}

void eliminate_dirichlet(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base,
                         const unsigned char *marker, LaunchCounter &lc)
{
    const int blocks = grid_for(n, 256);
    if (idx64)
        eliminate_dirichlet_kernel<int64_t><<<blocks, 256, 0, stream>>>(
            (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, csc.nzval, n, (int64_t)base, marker);
    else
        eliminate_dirichlet_kernel<int32_t><<<blocks, 256, 0, stream>>>(
            (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, csc.nzval, n, (int32_t)base, marker);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ---- pattern fingerprint: order-sensitive polynomial hash, combined with atomics ----
__device__ __forceinline__ u64 mix64(u64 x)
{ // splitmix64 finaliser
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

template <typename Ti>
__global__ void __launch_bounds__(256)
pattern_hash_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, i64 n, i64 nnz,
                    u64 *__restrict__ d_hash)
{
    // sum over positions of mix(position, value) is order sensitive and associative
    const i64 stride = (i64)gridDim.x * blockDim.x;
    u64 acc = 0;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < n + 1 + nnz; k += stride)
    {
        const u64 v = k <= n ? (u64)colptr[k] : (u64)rowval[k - n - 1];
        acc += mix64(mix64((u64)k + 0x9e3779b97f4a7c15ull) ^ v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc)
        atomicAdd(d_hash, acc);
}

// pattern_equal(a, b): a.colptr == b.colptr && a.rowval == b.rowval (sparsematrixcsc.jl:83-85); counts the differing
// positions (index bases may differ: both patterns are compared 0-based)
template <typename Ta, typename Tb>
__global__ void __launch_bounds__(256)
pattern_diff_kernel(const Ta *__restrict__ cpa, const Ta *__restrict__ rva, Ta basea, const Tb *__restrict__ cpb,
                    const Tb *__restrict__ rvb, Tb baseb, i64 n, i64 nnz, u64 *__restrict__ d_diff)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    u32 bad = 0;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < n + 1 + nnz; k += stride)
    {
        const i64 a = k <= n ? (i64)cpa[k] - (i64)basea : (i64)rva[k - n - 1] - (i64)basea;
        const i64 b = k <= n ? (i64)cpb[k] - (i64)baseb : (i64)rvb[k - n - 1] - (i64)baseb;
        bad += a != b;
    }
    if (bad)
        atomicAdd(reinterpret_cast<unsigned long long *>(d_diff), (unsigned long long)bad);
}

void pattern_diff(cudaStream_t stream, const CscView &a, int idx64a, int basea, const CscView &b, int idx64b, int baseb,
                  i64 n, u64 *d_diff, LaunchCounter &lc)
{
    const int blocks = grid_for(n + 1 + a.nnz, 256);
#define XSB_PD(TA, TB)                                                                                               \
    pattern_diff_kernel<TA, TB><<<blocks, 256, 0, stream>>>((const TA *)a.colptr, (const TA *)a.rowval, (TA)basea,      \
                                                            (const TB *)b.colptr, (const TB *)b.rowval, (TB)baseb, n,   \
                                                            a.nnz, d_diff)
    if (idx64a && idx64b)
        XSB_PD(int64_t, int64_t);
    else if (idx64a)
        XSB_PD(int64_t, int32_t);
    else if (idx64b)
        XSB_PD(int32_t, int64_t);
    else
        XSB_PD(int32_t, int32_t);
#undef XSB_PD
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void pattern_hash(cudaStream_t stream, const CscView &csc, i64 n, int idx64, u64 *d_hash, LaunchCounter &lc)
{
    XSB_CUDA(cudaMemsetAsync(d_hash, 0, sizeof(u64), stream));
    const int blocks = grid_for(n + 1 + csc.nnz, 256);
    if (idx64)
        pattern_hash_kernel<int64_t><<<blocks, 256, 0, stream>>>((const int64_t *)csc.colptr,
                                                                 (const int64_t *)csc.rowval, n, csc.nnz, d_hash);
    else
        pattern_hash_kernel<int32_t><<<blocks, 256, 0, stream>>>((const int32_t *)csc.colptr,
                                                                 (const int32_t *)csc.rowval, n, csc.nnz, d_hash);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------
// pointblock(A, blocksize): src/matrix/extendable.jl:292-318.
// The reference walks A in CSC order (column i, entries k) and, for the entry in row j, calls
// rawupdateindex!(Ab, +, block, iblock, jblock) with iblock = (i-1)/bs+1 taken from the COLUMN,
// jblock from the ROW and block[ii,jj] = nzval[k] (ii from the column, jj from the row).
//   pointblock_emit_kernel : entry k -> staged record (row iblock, column jblock, +0.0) of the block
//                            pattern matrix, at stream position k (the reference's call order)
//   pointblock_fill_kernel : entry k -> its value into block (iblock, jblock) of the flushed pattern,
//                            column-major position ii + jj*bs.  Every (block, position) receives
//                            exactly one entry, so the sum of single-entry blocks is 0.0 + v.
// ------------------------------------------------------------------------
template <typename Ti>
__device__ __forceinline__ i64 column_of_entry(const Ti *__restrict__ colptr, Ti base, i64 n, i64 k)
{ // the column c with colptr[c] <= k < colptr[c+1]: the largest c whose start is <= k
    i64 lo = 0, hi = n - 1;
    while (lo < hi)
    {
        const i64 mid = (lo + hi + 1) >> 1;
        if ((i64)colptr[mid] - base <= k)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

template <typename Ti>
__global__ void __launch_bounds__(256)
pointblock_emit_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, Ti base, i64 n, i64 nnz, i64 bs,
                       i64 nb, KeyLayout Lb, Rec *__restrict__ out, u64 *__restrict__ d_err)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += stride)
    {
        const i64 col = column_of_entry<Ti>(colptr, base, n, k);
        const i64 row = (i64)rowval[k] - base;
        const i64 ib = col / bs, jb = row / bs;
        Rec r;
        r.val = 0.0;
        if (ib >= nb || jb >= nb)
        { // BoundsError of rawupdateindex!(Ab, ...): sparsematrixcsc.jl:8-10
            atomicMin(d_err, (u64)k);
            r.key = Lb.pack(0, 0, 0u, FL_RAW);
        }
        else
            r.key = Lb.pack((u64)jb, (u64)ib, 0u, FL_RAW);
        st_rec(out + k, r);
    }
}

template <typename Ti>
__global__ void __launch_bounds__(256)
pointblock_fill_kernel(const Ti *__restrict__ colptr, const Ti *__restrict__ rowval, const double *__restrict__ nzval,
                       Ti base, i64 n, i64 nnz, i64 bs, const Ti *__restrict__ bcolptr,
                       const Ti *__restrict__ browval, double *__restrict__ blocks, u64 *__restrict__ d_err)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += stride)
    {
        const i64 col = column_of_entry<Ti>(colptr, base, n, k);
        const i64 row = (i64)rowval[k] - base;
        const i64 ib = col / bs, jb = row / bs, ii = col % bs, jj = row % bs;
        const i64 pos = find_slot<Ti>(bcolptr, browval, base, ib, jb);
        if (pos < 0)
        {
            atomicMin(d_err, (u64)k);
            continue;
        }
        blocks[pos * bs * bs + ii + jj * bs] = 0.0 + nzval[k];
    }
}

void pointblock_emit(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, i64 bs, i64 nb,
                     KeyLayout Lb, Rec *out, u64 *d_err, LaunchCounter &lc)
{
    if (csc.nnz <= 0)
        return;
    const int blocks = grid_for(csc.nnz, 256);
    if (idx64)
        pointblock_emit_kernel<int64_t><<<blocks, 256, 0, stream>>>((const int64_t *)csc.colptr,
                                                                    (const int64_t *)csc.rowval, (int64_t)base, n,
                                                                    csc.nnz, bs, nb, Lb, out, d_err);
    else
        pointblock_emit_kernel<int32_t><<<blocks, 256, 0, stream>>>((const int32_t *)csc.colptr,
                                                                    (const int32_t *)csc.rowval, (int32_t)base, n,
                                                                    csc.nnz, bs, nb, Lb, out, d_err);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

void pointblock_fill(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, i64 bs,
                     const CscView &pattern, double *blocks, u64 *d_err, LaunchCounter &lc)
{
    if (csc.nnz <= 0)
        return;
    const int grid = grid_for(csc.nnz, 256);
    if (idx64)
        pointblock_fill_kernel<int64_t><<<grid, 256, 0, stream>>>(
            (const int64_t *)csc.colptr, (const int64_t *)csc.rowval, csc.nzval, (int64_t)base, n, csc.nnz, bs,
            (const int64_t *)pattern.colptr, (const int64_t *)pattern.rowval, blocks, d_err);
    else
        pointblock_fill_kernel<int32_t><<<grid, 256, 0, stream>>>(
            (const int32_t *)csc.colptr, (const int32_t *)csc.rowval, csc.nzval, (int32_t)base, n, csc.nnz, bs,
            (const int32_t *)pattern.colptr, (const int32_t *)pattern.rowval, blocks, d_err);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

} // namespace xsb
