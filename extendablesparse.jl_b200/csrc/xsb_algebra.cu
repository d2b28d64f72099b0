// xsb_algebra.cu -- A + B, A - B and dropzeros! on resident CSCs: one merge-and-filter over the entry
// sequences of two CSCs (SparseArrays' map(+/-, A, B), i.e. _map_zeropres!, and fkeep!(!iszero)).
//
// Both CSCs are sorted by (column, row) as a whole, so the merged sequence has nA + nB positions and position
// d of column c lies in [S(c), S(c+1)) with S(c) = colptrA[c] + colptrB[c] - 2 base.  Every thread owns kItems
// consecutive merged positions (merge path): it finds its column by a binary search over S and its place inside
// the column by a merge-path search over the two row lists, so a column of 2^20 entries is shared by 2^17
// threads and runs of empty columns cost nothing.  Ties go to A: an entry of both lands as the A position, which
// sees its partner as the next B row and emits f(a, b); the B position sees its partner as the previous A row
// and emits nothing.  Three passes: count (kept entries per block), scan (block offsets), write (rowval, nzval
// and the colptr of every non-empty column); a last pass fills the colptr of the empty columns.
#include "xsb_internal.h"

namespace xsb {
namespace {

constexpr int kAlgThreads = 256;
constexpr int kAlgItems = 8;
constexpr i64 kAlgTile = (i64)kAlgThreads * kAlgItems;

// One IEEE add or subtract, NaN results with the bits x86-64 gives them (the first NaN operand, quieted;
// Inf - Inf is the negative default NaN): nzval is compared bit for bit with the reference's host arithmetic.
__device__ __forceinline__ double quiet(double x)
{
    return __longlong_as_double(__double_as_longlong(x) | 0x0008000000000000ll);
}
template <int OP> __device__ __forceinline__ double apply(double a, double b)
{
    const double r = OP == kAlgSub ? __dsub_rn(a, b) : __dadd_rn(a, b);
    if (r == r)
        return r;
    if (a != a)
        return quiet(a);
    if (b != b)
        return quiet(b);
    return __longlong_as_double((long long)0xfff8000000000000ull);
}

template <typename Ti, int OP> struct Operands
{
    const Ti *cpa, *rva;
    const double *nza;
    const Ti *cpb, *rvb; // OP == kAlgKeep: no B
    const double *nzb;
    i64 n, total;
    Ti base;
    __device__ __forceinline__ i64 sa(i64 c) const { return (i64)cpa[c] - base; }
    __device__ __forceinline__ i64 sb(i64 c) const { return OP == kAlgKeep ? 0 : (i64)cpb[c] - base; }
    __device__ __forceinline__ i64 s(i64 c) const { return sa(c) + sb(c); }
    // the column holding merged position d: the largest c in [lo, hi) with S(c) <= d (S(lo) <= d < S(hi))
    __device__ __forceinline__ i64 locate(i64 d, i64 lo, i64 hi) const
    {
        if (lo + 1 < hi && s(lo + 1) > d)
            return lo;
        while (hi - lo > 1)
        {
            const i64 mid = lo + ((hi - lo) >> 1);
            if (s(mid) <= d)
                lo = mid;
            else
                hi = mid;
        }
        return lo;
    }
};

// Walks merged positions [d0, d0 + kItems) (those below total); calls visit(first position of column c or -1,
// column, row, value, kept) for each.  [clo, chi): columns that can hold these positions.
template <typename Ti, int OP, class Visit>
__device__ __forceinline__ void merge_walk(const Operands<Ti, OP> &P, i64 d0, i64 clo, i64 chi, Visit &&visit)
{
    if (d0 >= P.total)
        return;
    i64 c = P.locate(d0, clo, chi);
    i64 a0 = P.sa(c), a1 = P.sa(c + 1), b0 = P.sb(c), b1 = P.sb(c + 1);
    i64 ia = a0, jb = b0;
    const i64 k = d0 - a0 - b0;
    if (OP == kAlgKeep)
        ia = a0 + k;
    else if (k > 0)
    { // merge path inside the column: the A rows among its first k merged positions (ties to A)
        i64 lo = k > b1 - b0 ? k - (b1 - b0) : 0, hi = k < a1 - a0 ? k : a1 - a0;
        while (lo < hi)
        {
            const i64 mid = (lo + hi) >> 1;
            if (P.rva[a0 + mid] <= P.rvb[b0 + k - 1 - mid])
                lo = mid + 1;
            else
                hi = mid;
        }
        ia = a0 + lo;
        jb = b0 + k - lo;
    }
    bool colstart = k == 0;
#pragma unroll 1
    for (int t = 0; t < kAlgItems; ++t)
    {
        const i64 d = d0 + t;
        if (d >= P.total)
            break;
        if (ia == a1 && jb == b1)
        { // next non-empty column starts at d
            c = P.locate(d, c + 1, chi);
            a0 = ia;
            a1 = P.sa(c + 1);
            b0 = jb;
            b1 = P.sb(c + 1);
            colstart = true;
        }
        const bool takeA = ia < a1 && (OP == kAlgKeep || jb >= b1 || P.rva[ia] <= P.rvb[jb]);
        Ti row;
        double x;
        bool keep;
        if (OP == kAlgKeep)
        {
            row = P.rva[ia];
            x = P.nza[ia];
            keep = !(x == 0.0);
            ++ia;
        }
        else if (takeA)
        {
            row = P.rva[ia];
            const bool both = jb < b1 && P.rvb[jb] == row;
            x = apply<OP>(P.nza[ia], both ? P.nzb[jb] : 0.0);
            keep = !(x == 0.0);
            ++ia;
        }
        else
        {
            row = P.rvb[jb];
            const bool both = ia > a0 && P.rva[ia - 1] == row; // emitted by the A position
            x = both ? 0.0 : apply<OP>(0.0, P.nzb[jb]);
            keep = !both && !(x == 0.0);
            ++jb;
        }
        visit(colstart ? c : (i64)-1, row, x, keep);
        colstart = false;
    }
}

// columns that can hold the positions of this block
template <typename Ti, int OP> __device__ __forceinline__ void block_columns(const Operands<Ti, OP> &P, i64 *s_cols)
{
    const i64 first = (i64)blockIdx.x * kAlgTile;
    if (threadIdx.x < 2)
    {
        const i64 d = threadIdx.x == 0 ? first : (first + kAlgTile < P.total ? first + kAlgTile : P.total) - 1;
        s_cols[threadIdx.x] = P.locate(d, 0, P.n) + threadIdx.x;
    }
    __syncthreads();
}

template <typename Ti, int OP>
__global__ void __launch_bounds__(kAlgThreads) merge_count_kernel(Operands<Ti, OP> P, u64 *__restrict__ blockcnt)
{
    __shared__ i64 s_cols[2];
    __shared__ u32 s_warp[kAlgThreads / 32];
    block_columns(P, s_cols);
    u32 cnt = 0;
    merge_walk(P, (i64)blockIdx.x * kAlgTile + (i64)threadIdx.x * kAlgItems, s_cols[0], s_cols[1],
               [&](i64, Ti, double, bool keep) { cnt += keep; });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0)
        s_warp[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        u32 sum = 0;
        for (int w = 0; w < kAlgThreads / 32; ++w)
            sum += s_warp[w];
        blockcnt[blockIdx.x] = sum;
    }
}

// exclusive scan of the block counts in place (one block); *total = their sum
__global__ void __launch_bounds__(1024) merge_scan_kernel(u64 *__restrict__ blockcnt, i64 nblocks, u64 *__restrict__ total)
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
        const u64 v = k < nblocks ? blockcnt[k] : 0;
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
        const u64 carry = s_carry;
        const u64 incl = carry + x + (warp > 0 ? s_warp[warp - 1] : 0);
        if (k < nblocks)
            blockcnt[k] = incl - v;
        __syncthreads();
        if (threadIdx.x == 1023)
            s_carry = incl;
        __syncthreads();
    }
    if (threadIdx.x == 0)
        *total = s_carry;
}

template <typename Ti, int OP>
__global__ void __launch_bounds__(kAlgThreads)
    merge_write_kernel(Operands<Ti, OP> P, const u64 *__restrict__ blockoff, Ti *__restrict__ colptr,
                       Ti *__restrict__ rowval, double *__restrict__ nzval)
{
    __shared__ i64 s_cols[2];
    __shared__ u32 s_warp[kAlgThreads / 32];
    block_columns(P, s_cols);
    const i64 d0 = (i64)blockIdx.x * kAlgTile + (i64)threadIdx.x * kAlgItems;
    u32 cnt = 0;
    merge_walk(P, d0, s_cols[0], s_cols[1], [&](i64, Ti, double, bool keep) { cnt += keep; });
    // exclusive scan of the threads' counts
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 x = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const u32 y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o)
            x += y;
    }
    if (lane == 31)
        s_warp[warp] = x;
    __syncthreads();
    u32 before = x - cnt;
    for (int w = 0; w < warp; ++w)
        before += s_warp[w];
    i64 pos = (i64)blockoff[blockIdx.x] + before;
    merge_walk(P, d0, s_cols[0], s_cols[1], [&](i64 cstart, Ti row, double v, bool keep) {
        if (cstart >= 0)
            colptr[cstart] = (Ti)(pos + P.base);
        if (keep)
        {
            rowval[pos] = row;
            nzval[pos] = v;
            ++pos;
        }
    });
}

// colptr of the columns without merged positions (and colptr[n]): that of the next non-empty column
template <typename Ti, int OP>
__global__ void __launch_bounds__(256) merge_fill_kernel(Operands<Ti, OP> P, const u64 *__restrict__ total_out,
                                                         Ti *__restrict__ colptr)
{
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c <= P.n; c += stride)
    {
        const i64 d = P.s(c);
        if (c < P.n && P.s(c + 1) > d)
            continue; // written by the write pass
        if (d == P.total)
            colptr[c] = (Ti)((i64)*total_out + P.base);
        else
            colptr[c] = colptr[P.locate(d, c + 1, P.n)];
    }
}

template <typename Ti, int OP>
Operands<Ti, OP> operands(const CscView &a, const CscView *b, i64 n, int base)
{
    Operands<Ti, OP> P;
    P.cpa = static_cast<const Ti *>(a.colptr);
    P.rva = static_cast<const Ti *>(a.rowval);
    P.nza = a.nzval;
    P.cpb = b ? static_cast<const Ti *>(b->colptr) : nullptr;
    P.rvb = b ? static_cast<const Ti *>(b->rowval) : nullptr;
    P.nzb = b ? b->nzval : nullptr;
    P.n = n;
    P.total = a.nnz + (b ? b->nnz : 0);
    P.base = (Ti)base;
    return P;
}

i64 merge_blocks(const CscView &a, const CscView *b) { return (a.nnz + (b ? b->nnz : 0) + kAlgTile - 1) / kAlgTile; }

template <typename Ti, int OP>
void count_t(cudaStream_t s, const CscView &a, const CscView *b, i64 n, int base, u64 *ws, LaunchCounter &lc)
{
    const auto P = operands<Ti, OP>(a, b, n, base);
    const i64 nb = merge_blocks(a, b);
    if (nb > 0)
    {
        merge_count_kernel<Ti, OP><<<(unsigned)nb, kAlgThreads, 0, s>>>(P, ws + 1);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    merge_scan_kernel<<<1, 1024, 0, s>>>(ws + 1, nb, ws);
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

template <typename Ti, int OP>
void write_t(cudaStream_t s, const CscView &a, const CscView *b, i64 n, int base, const u64 *ws, void *colptr,
             void *rowval, double *nzval, LaunchCounter &lc)
{
    const auto P = operands<Ti, OP>(a, b, n, base);
    const i64 nb = merge_blocks(a, b);
    if (nb > 0)
    {
        merge_write_kernel<Ti, OP><<<(unsigned)nb, kAlgThreads, 0, s>>>(P, ws + 1, static_cast<Ti *>(colptr),
                                                                       static_cast<Ti *>(rowval), nzval);
        lc.add();
        XSB_CUDA(cudaGetLastError());
    }
    const i64 cols = n + 1;
    const i64 fb = std::min<i64>((cols + 255) / 256, 148 * 16);
    merge_fill_kernel<Ti, OP><<<(unsigned)fb, 256, 0, s>>>(P, ws, static_cast<Ti *>(colptr));
    lc.add();
    XSB_CUDA(cudaGetLastError());
}

template <int OP> struct Dispatch
{
    static void count(cudaStream_t s, const CscView &a, const CscView *b, i64 n, int idx64, int base, u64 *ws,
                      LaunchCounter &lc)
    {
        if (idx64)
            count_t<int64_t, OP>(s, a, b, n, base, ws, lc);
        else
            count_t<int32_t, OP>(s, a, b, n, base, ws, lc);
    }
    static void write(cudaStream_t s, const CscView &a, const CscView *b, i64 n, int idx64, int base, const u64 *ws,
                      void *colptr, void *rowval, double *nzval, LaunchCounter &lc)
    {
        if (idx64)
            write_t<int64_t, OP>(s, a, b, n, base, ws, colptr, rowval, nzval, lc);
        else
            write_t<int32_t, OP>(s, a, b, n, base, ws, colptr, rowval, nzval, lc);
    }
};

} // namespace

size_t merge_workspace_bytes(i64 nnz_a, i64 nnz_b) { return sizeof(u64) * (size_t)(1 + (nnz_a + nnz_b + kAlgTile - 1) / kAlgTile); }

void merge_count(cudaStream_t stream, int op, const CscView &a, const CscView *b, i64 n, int idx64, int base, void *ws,
                 LaunchCounter &lc)
{
    u64 *w = static_cast<u64 *>(ws);
    if (op == kAlgAdd)
        Dispatch<kAlgAdd>::count(stream, a, b, n, idx64, base, w, lc);
    else if (op == kAlgSub)
        Dispatch<kAlgSub>::count(stream, a, b, n, idx64, base, w, lc);
    else
        Dispatch<kAlgKeep>::count(stream, a, nullptr, n, idx64, base, w, lc);
}

void merge_write(cudaStream_t stream, int op, const CscView &a, const CscView *b, i64 n, int idx64, int base,
                 const void *ws, void *colptr_out, void *rowval_out, double *nzval_out, LaunchCounter &lc)
{
    const u64 *w = static_cast<const u64 *>(ws);
    if (op == kAlgAdd)
        Dispatch<kAlgAdd>::write(stream, a, b, n, idx64, base, w, colptr_out, rowval_out, nzval_out, lc);
    else if (op == kAlgSub)
        Dispatch<kAlgSub>::write(stream, a, b, n, idx64, base, w, colptr_out, rowval_out, nzval_out, lc);
    else
        Dispatch<kAlgKeep>::write(stream, a, nullptr, n, idx64, base, w, colptr_out, rowval_out, nzval_out, lc);
}

} // namespace xsb
