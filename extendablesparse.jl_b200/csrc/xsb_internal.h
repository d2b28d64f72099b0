// xsb_internal.h -- host-side declarations shared by the translation units of libxsparse_b200.
#pragma once
#include "xsb_common.cuh"
#include <algorithm>
#include <atomic>
#include <cstddef>
#include <vector>

namespace xsb {

constexpr int kRadix = 256;
constexpr int kMaxPasses = 8;

struct SortPlan
{
    int npasses;
    int shift[kMaxPasses];
    int bits[kMaxPasses];
};

struct LaunchCounter
{
    long long total = 0;
    int in_flush = 0;
    void add(int k = 1)
    {
        total += k;
        in_flush += k;
    }
};

struct StageTimes
{
    float expand = 0, histogram = 0, sort = 0, reduce = 0, colptr = 0, other = 0, total = 0;
    float gcount = 0, gscatter = 0, fold = 0, compact = 0, preagg = 0; // two-pass grouping and per-column fold, in detail
};

// Optional CUDA-event bracket around pipeline stages (profiling mode only).
struct StageTimer
{
    struct Span
    {
        cudaEvent_t a, b;
        float StageTimes::*slot;
    };
    std::vector<Span> spans;
    cudaEvent_t cur = nullptr;
    void begin(cudaStream_t s)
    {
        XSB_CUDA(cudaEventCreate(&cur));
        XSB_CUDA(cudaEventRecord(cur, s));
    }
    void end(cudaStream_t s, float StageTimes::*slot)
    {
        cudaEvent_t b;
        XSB_CUDA(cudaEventCreate(&b));
        XSB_CUDA(cudaEventRecord(b, s));
        spans.push_back({cur, b, slot});
        cur = nullptr;
    }
    // call after the stream has been synchronised
    void collect(StageTimes &t)
    {
        for (auto &sp : spans)
        {
            float ms = 0;
            cudaEventElapsedTime(&ms, sp.a, sp.b);
            t.*(sp.slot) += ms;
            cudaEventDestroy(sp.a);
            cudaEventDestroy(sp.b);
        }
        spans.clear();
    }
};

// cudaFuncSetAttribute applies to the device that is current when it is called, and a process may hold
// handles on several GPUs: remember per device what was set (devices >= 32: set on every launch).
struct FuncAttrOnce
{
    std::atomic<unsigned> done{0};
    template <class K> void set(K kernel, int smem_bytes, bool max_carveout = false)
    {
        int dev = 0;
        XSB_CUDA(cudaGetDevice(&dev));
        if (dev < 32 && ((done.load(std::memory_order_acquire) >> dev) & 1u))
            return;
        XSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        if (max_carveout)
            XSB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                          (int)cudaSharedmemCarveoutMaxShared));
        if (dev < 32)
            done.fetch_or(1u << dev, std::memory_order_release);
    }
};

// ---- xsb_sort.cu
SortPlan make_sort_plan(int begin_bit, int nbits);
size_t sort_workspace_bytes(u64 n);
// colcnt != nullptr: the histogram kernel also counts the records per column (key field
// [colshift, colshift+colbits)) into colcnt[], which the caller has zeroed
Rec *radix_sort_records(cudaStream_t stream, Rec *a, Rec *b, u64 n, const SortPlan &plan, void *workspace,
                        LaunchCounter &lc, StageTimer *timer, u32 *colcnt = nullptr, int colshift = 0,
                        int colbits = 0);

void partition_records(cudaStream_t stream, const Rec *in, Rec *out, u64 n, int shift, int bits, void *workspace,
                       LaunchCounter &lc, u64 *counts_host);

// ---- xsb_flush.cu
struct CscView
{
    void *colptr; // Ti[n+1]
    void *rowval; // Ti[nnz]
    double *nzval;
    i64 nnz;
};
// old CSC -> FL_OLD records at out[0..nnz)
void expand_csc_records(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, KeyLayout L,
                        Rec *out, LaunchCounter &lc);
size_t reduce_workspace_bytes(u64 nrec, i64 ncols);
// sorted records -> rowval/nzval (compacted, user index type/base) + colptr; returns nnz via *d_nnz (device)
void reduce_emit_csc(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, int combine, int mode,
                     bool plain_adds, i64 ncols, int idx64, int base, void *rowval_out, double *nzval_out,
                     void *colptr_out, void *workspace, u64 *d_nnz, LaunchCounter &lc, StageTimer *timer);

// ---- xsb_colfold.cu
size_t colfold_workspace_bytes(u64 nrec, i64 ncols);
bool colfold_supported(const KeyLayout &L, u64 nrec, i64 ncols);
u32 *colfold_counts(void *workspace, u64 nrec, i64 ncols);
void colfold_clear_counts(cudaStream_t stream, void *workspace, u64 nrec, i64 ncols);
// records sorted by column only (stable) + per-column record counts -> entries parked in tmp, colptr, nnz
void colfold_reduce(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, int combine, bool plain_adds,
                    i64 ncols, int idx64, int base, Rec *tmp, void *colptr_out, void *workspace, u64 *d_nnz,
                    u32 *d_overflow, bool lists_ready, u32 *d_maxd, u32 hint_maxd, LaunchCounter &lc, StageTimer *timer);
// d_maxd receives the largest number of distinct rows a thread-folded column held (0: path not taken);
// hint_maxd is that number from the handle's previous flush (0: unknown) and picks the first table size
bool colfold_direct_supported(const KeyLayout &L, int combine, bool plain_adds);
// one-pass fold of plain += streams straight into rowval / nzval / colptr; *d_redo != 0: run colfold_reduce instead
void colfold_direct(cudaStream_t stream, const Rec *sorted, u64 nrec, KeyLayout L, i64 ncols, int idx64, int base,
                    void *rowval_out, double *nzval_out, void *colptr_out, void *workspace, u64 *d_nnz, u32 *d_redo,
                    bool lists_ready, u32 *d_maxd, u32 hint_maxd, LaunchCounter &lc, StageTimer *timer);
void colfold_lists(void *workspace, u64 nrec, i64 ncols, u32 **nzcol, u32 **nzstart, u64 **totals);

// ---- xsb_group.cu
// chunk index boundaries of the regions of a slab handle's buffer: old CSC [0, c_old), own records
// [c_old, c_own), received from lower ranks [c_own, c_low), from higher ranks [c_low, nchunks)
struct ChunkOrder
{
    u32 c_old, c_own, c_low;
};
constexpr u32 kMaxColPairs = 128; // a column met by more chunks than this sends the flush to the pair SORT

int group_chunk_records();
size_t group_workspace_bytes(u64 nrec, i64 ncols);
bool group_supported(const KeyLayout &L, u64 nrec, i64 ncols);
// stable grouping by column in two passes (sparse per-chunk histograms); false: no column locality
bool group_by_column(cudaStream_t stream, const Rec *in, Rec *out, u64 nrec, i64 ncols, const KeyLayout &L, void *workspace,
                     void *sort_workspace, u32 *nzcol, u32 *nzstart, u64 *totals, u64 *h_scal_pinned, LaunchCounter &lc,
                     StageTimer *timer, int *pair_passes, u64 *npairs_out, int ownershift = -1, u32 me = 0,
                     const ChunkOrder *order = nullptr);
// ownershift >= 0: records whose key >> ownershift != me belong to other ranks and are skipped
// parked entries -> rowval / nzval
void colfold_compact(cudaStream_t stream, const Rec *tmp, u64 nrec, i64 ncols, int idx64, int base,
                     const void *colptr, void *rowval_out, double *nzval_out, void *workspace, LaunchCounter &lc,
                     StageTimer *timer);

// ---- xsb_runs.cu / xsb_chunk.cuh: flush on grouped chunks (the product path)
// Where the kernels that stage records publish the runs of their chunks (the run index of a handle).
struct RunTarget
{
    u32 *counters;    // [0] pairs appended so far (ticket), [1] != 0: a chunk gave up / the pair list is full
    uint2 *chunkinfo; // per chunk: (first pair, pairs)
    u32 *chunkstart;  // per chunk: position of its first record in the staging buffer
    u32 *pcol;        // per pair: grouping key = column (owner bits on top on slab handles)
    u32 *pinfo;       // per pair: (offset of the run inside its chunk << 16) | records
    u32 cap;          // room of the pair list
    int colshift;
    u32 gmask;        // mask of the grouping key
};
struct RunIndexLayout
{
    size_t off_counters, off_chunkinfo, off_chunkstart, off_pcol, off_pinfo, bytes;
    u32 cap_pairs, cap_chunks;
};
// regions of a slab handle's staged records by position: own [0, own_end), received from lower ranks
// [own_end, low_end), from higher ranks [low_end, ...).  The fold meets a column's runs as
// [lower ranks | own | higher ranks], each in stream order.  Plain handles: own_end = low_end = 2^32-1.
struct RunRegions
{
    u32 own_end, low_end;
};
RunIndexLayout run_index_layout(u64 cap_records);
RunTarget run_target(void *workspace, u64 cap_records, const KeyLayout &L);
bool runs_supported(const KeyLayout &L, u64 nrec, i64 ncols);
u32 chunk_sort_chunks(u64 count);
// groups buf[r0, r1) in place, chunk by chunk; chunk ids from chunk0
void chunk_sort(cudaStream_t stream, Rec *buf, u64 r0, u64 r1, const RunTarget &rt, u32 chunk0, LaunchCounter &lc);
size_t runs_workspace_bytes(u64 npairs, i64 ncols);
void runs_bucket(cudaStream_t stream, const RunTarget &rt, u32 nchunks, u32 npairs, i64 ncols, const KeyLayout &L,
                 RunRegions reg, void *workspace, LaunchCounter &lc);
void runs_fold(cudaStream_t stream, const Rec *buf, const KeyLayout &L, i64 ncols, int idx64, int base, const CscView &old,
               void *workspace, u32 npairs, int level, u32 maxlen, void *rowval_out, double *nzval_out, void *colptr_out,
               u64 *d_nnz, u32 *d_redo, u32 *d_maxd, bool first_try, bool has_assign, LaunchCounter &lc);

// ---- xsb_route.cu
size_t route_workspace_bytes(u64 n, int nranks);
// tileflags != nullptr: only tiles whose byte is set can hold records of other ranks (StageFlags)
void route_count(cudaStream_t stream, const Rec *in, u64 n, const KeyLayout &L, void *workspace, u64 *counts_host,
                 LaunchCounter &lc, const unsigned char *tileflags = nullptr);
void route_extract(cudaStream_t stream, const Rec *in, u64 n, const KeyLayout &L, void *workspace,
                   const u64 *counts_host, Rec *send, LaunchCounter &lc);
void route_fill_skipped(cudaStream_t stream, Rec *out, i64 count, const KeyLayout &L, LaunchCounter &lc);
// fixed-capacity exchange (no count visits the host): see xsb_route.cu
// flags in device memory (own or a peer's) with the values to wait for / to store; addr 0 = unused entry
struct PeerFlags
{
    u64 addr[kMaxRanks];
    u64 value[kMaxRanks];
};
void route_pack(cudaStream_t stream, const Rec *in, u64 n, const KeyLayout &L, void *workspace, const i64 *caps,
                u64 *pinned_addr, u64 *pinned_caps, const PeerFlags &sig, u64 *d_flags, LaunchCounter &lc,
                const unsigned char *tileflags);
void route_tailcheck(cudaStream_t stream, const Rec *in, u64 from, u64 n, const KeyLayout &L, const unsigned char *tileflags,
                     u64 *d_flags, LaunchCounter &lc);
void peer_wait(cudaStream_t stream, const PeerFlags &w, u64 timeout_ns, u64 *d_flags, LaunchCounter &lc);
void peer_signal(cudaStream_t stream, const PeerFlags &sgn, LaunchCounter &lc);
void route_unpack(cudaStream_t stream, const Rec *block, i64 cap, Rec *out, const KeyLayout &L, i64 ncols, u64 *d_flags,
                  u64 *d_counts, int which, LaunchCounter &lc);
void route_check(cudaStream_t stream, const Rec *in, i64 count, const KeyLayout &L, i64 ncols, u64 *d_err,
                 u64 *d_has_assign, LaunchCounter &lc);

// ---- xsb_preagg.cu
// XSB_FAST: in[0, nrec) -> out[0, *d_count): partial sums of windows of the stream; d_count zeroed by the caller
void preaggregate_records(cudaStream_t stream, const Rec *in, u64 nrec, const KeyLayout &L, Rec *out, u64 *d_count,
                          LaunchCounter &lc);

// ---- xsb_insert.cu
// (I,J,V) -> records; *d_err receives the smallest offending index (or ~0)
void pack_records(cudaStream_t stream, const void *I, const void *J, const double *V, i64 count, int idx64,
                  int base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *out, u64 *d_err,
                  LaunchCounter &lc, StageFlags sf = StageFlags{nullptr, 0});
// pack + group (xsb_insert.cu, xsb_chunk.cuh): a warp per chunk brings its records into column order while it
// packs them and publishes the chunk's runs; pos0 = position of out[0] among the staged records.  Return the
// chunks appended to the run index.
u32 pack_chunks(i64 count);
u32 pack_records_grouped(cudaStream_t stream, const void *I, const void *J, const double *V, i64 count, int idx64,
                         int base, i64 m, i64 n, KeyLayout L, u32 tid, u32 flavour, Rec *out, u64 *d_err,
                         LaunchCounter &lc, const RunTarget &rt, u32 chunk0, u32 pos0, StageFlags sf);
u32 pack_triplets_grouped(cudaStream_t stream, const void *T, i64 count, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                          u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, const RunTarget &rt, u32 chunk0, u32 pos0,
                          StageFlags sf, i64 k0 = 0);
u32 emit_fdrand_chunks(i64 l_begin, i64 l_end);
u32 emit_fdrand_grouped(cudaStream_t stream, i64 nx, i64 ny, i64 nz, u64 seed, int ones, KeyLayout L, u32 tid, u32 flavour,
                        i64 l_begin, i64 l_end, Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0,
                        u32 pos0);
u32 emit_blockrd_chunks(i64 nx, i64 ny, i64 nz, int ns); // 0: not available for this species count
u32 emit_blockrd_grouped(cudaStream_t stream, i64 nx, i64 ny, i64 nz, int ns, u64 seed, KeyLayout L, u32 tid, u32 flavour,
                         Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0, u32 pos0);
u32 emit_p1fem_chunks(i64 nxn, i64 nyn, i64 cz_begin, i64 cz_end);
u32 emit_p1fem_grouped(cudaStream_t stream, i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour, i64 cz_begin,
                       i64 cz_end, Rec *out, LaunchCounter &lc, StageFlags sf, const RunTarget &rt, u32 chunk0, u32 pos0);
// element-by-element insertion: an element loop given as connectivity and dense element matrices, Julia's
// column-major arrays (rdofs kr x ncells and cdofs kc x ncells in the handle's index type, Aloc kr x kc x ncells;
// the square loop passes rdofs == cdofs): call p = kr kc c + kr jl + il is (rdofs[il, c], cdofs[jl, c], Aloc[il, jl, c])
struct ElementBatch
{
    const void *rdofs, *cdofs;
    const double *Aloc;
    int kr, kc;
    i64 ncells;
};
// -> the kr kc ncells records of the loop; a row dof must lie below m, a column dof below n.  *d_err receives
// 2 x (first offending element) + (1 if a column dof is at fault).  insert_elements stores call order,
// insert_elements_grouped groups chunks of whole elements and returns the chunks appended to the run index
// (insert_elements_chunks(kr, kc, ncells)).
u32 insert_elements_chunks(int kr, int kc, i64 ncells);
void insert_elements(cudaStream_t stream, const ElementBatch &eb, int idx64, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                     u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf);
u32 insert_elements_grouped(cudaStream_t stream, const ElementBatch &eb, int idx64, int base, i64 m, i64 n, KeyLayout L,
                            u32 tid, u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf,
                            const RunTarget &rt, u32 chunk0, u32 pos0);
// pointblock (xsb_values.cu): CSC entries -> records of the block pattern; values into the blocks
void pointblock_emit(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, i64 bs, i64 nb,
                     KeyLayout Lb, Rec *out, u64 *d_err, LaunchCounter &lc);
void pointblock_fill(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, i64 bs,
                     const CscView &pattern, double *blocks, u64 *d_err, LaunchCounter &lc);
void pack_triplets(cudaStream_t stream, const void *T, i64 count, int base, i64 m, i64 n, KeyLayout L, u32 tid,
                   u32 flavour, Rec *out, u64 *d_err, LaunchCounter &lc, StageFlags sf, i64 k0 = 0);
void unpack_records(cudaStream_t stream, const Rec *in, i64 count, int idx64, int base, KeyLayout L, void *I,
                    void *J, double *V, int *flavour, LaunchCounter &lc);
i64 fdrand_prefix(i64 nx, i64 ny, i64 nz, i64 l); // records emitted by nodes [0,l)
void emit_fdrand(cudaStream_t stream, i64 nx, i64 ny, i64 nz, u64 seed, int ones, KeyLayout L, u32 tid,
                 u32 flavour, i64 l_begin, i64 l_end, Rec *out, LaunchCounter &lc,
                 StageFlags sf = StageFlags{nullptr, 0});
void emit_p1fem(cudaStream_t stream, i64 nxn, i64 nyn, i64 nzn, KeyLayout L, u32 tid, u32 flavour,
                i64 cz_begin, i64 cz_end, Rec *out, LaunchCounter &lc, StageFlags sf = StageFlags{nullptr, 0});
i64 blockrd_count(i64 nx, i64 ny, i64 nz, i64 ns);
void emit_blockrd(cudaStream_t stream, i64 nx, i64 ny, i64 nz, int ns, u64 seed, KeyLayout L, u32 tid,
                  u32 flavour, Rec *out, LaunchCounter &lc, StageFlags sf = StageFlags{nullptr, 0});

// ---- xsb_values.cu
void zero_values(cudaStream_t stream, double *nzval, i64 nnz, LaunchCounter &lc);
void fill_index(cudaStream_t stream, void *x, i64 count, int idx64, i64 value, LaunchCounter &lc);
// slot[k] = nz index of (I[k],J[k]) or -1; *d_missing counts the absent ones
void lookup_slots(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base, const void *I,
                  const void *J, i64 count, i64 *slot, u64 *d_missing, u64 *d_oob, LaunchCounter &lc);
// the same for the calls of an element loop (eb.Aloc unused; count = kr kc ncells)
void lookup_slots_elements(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base,
                           const ElementBatch &eb, i64 count, i64 *slot, u64 *d_missing, u64 *d_oob, LaunchCounter &lc);
void gather_values(cudaStream_t stream, const double *nzval, const i64 *slot, i64 count, double *out,
                   LaunchCounter &lc);
void count_missing_records(cudaStream_t stream, const Rec *recs, i64 count, const KeyLayout &L, const CscView &csc,
                           int idx64, int base, u64 *d_missing, LaunchCounter &lc);
void slots_to_records(cudaStream_t stream, const i64 *slot, i64 count, Rec *out, LaunchCounter &lc);
void build_frozen_map(cudaStream_t stream, const Rec *sorted, i64 count, i64 nnz, u32 *perm, u32 *segstart, u32 *slot32,
                      LaunchCounter &lc);
// A stream frozen across column slabs (xsb_freeze_slab*): the map indexes the combined space [received from lower
// ranks | own stream | received from higher ranks].  Index k < low: recv[k]; low <= k < low + own: V[k - low] (the
// caller's values, read in place); else recv[k - own].  In the fast map the own positions that other ranks own
// carry kNoSlot.
struct SlabValues
{
    const double *recv;
    u32 low, own;
};
constexpr u32 kNoSlot = 0xffffffffu;
// sv == nullptr: plain frozen stream, V indexed by stream position
void reassemble_deterministic(cudaStream_t stream, const double *V, const u32 *perm, const u32 *segstart, i64 nnz,
                              double *nzval, bool zero_first, LaunchCounter &lc, const SlabValues *sv = nullptr);
void reassemble_fast(cudaStream_t stream, const double *V, const u32 *slot, i64 count, double *nzval,
                     LaunchCounter &lc, const SlabValues *sv = nullptr);
// slab freeze, one pass over the stream: global bounds (*d_oob: first bad position), owner, own positions -> slot[k]
// (nzval slot, -1 when absent: *d_missing), every position -> tags[k] {owner << 32 | k, row | column in the owner's
// slab << 32} for the stable copy-out of route_count / route_extract (layout with ownershift 32)
void slab_classify(cudaStream_t stream, const CscView &csc, i64 m, i64 n_global, const KeyLayout &Ls, int idx64, int base,
                   const void *I, const void *J, i64 count, i64 *slot, Rec *tags, u64 *d_missing, u64 *d_oob,
                   LaunchCounter &lc);
void slab_classify_elements(cudaStream_t stream, const CscView &csc, i64 m, i64 n_global, const KeyLayout &Ls, int idx64,
                            int base, const ElementBatch &eb, i64 count, i64 *slot, Rec *tags, u64 *d_missing,
                            u64 *d_oob, LaunchCounter &lc);
// gathered tags -> stream indices and {row, column} positions
void slab_split(cudaStream_t stream, const Rec *tags, i64 n, u32 *idx, u64 *where, LaunchCounter &lc);
// (slot, combined index) records of the combined space; received positions recv[q] = {row, slab column}
// (*d_oob: first bad q, *d_missing: absent ones); slot nnz = no entry of the map
void slab_records(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base, const i64 *own_slot, i64 own,
                  const void *recv, i64 low, i64 total, Rec *out, u64 *d_missing, u64 *d_oob, LaunchCounter &lc);
// send[q] = V[idx[q]]
void slab_pack_values(cudaStream_t stream, const double *V, const u32 *idx, i64 n, double *send, LaunchCounter &lc);
void mark_dirichlet(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base, double penalty,
                    unsigned char *marker, LaunchCounter &lc);
void eliminate_dirichlet(cudaStream_t stream, const CscView &csc, i64 n, int idx64, int base,
                         const unsigned char *marker, LaunchCounter &lc);
void pattern_hash(cudaStream_t stream, const CscView &csc, i64 n, int idx64, u64 *d_hash, LaunchCounter &lc);
void pattern_diff(cudaStream_t stream, const CscView &a, int idx64a, int basea, const CscView &b, int idx64b, int baseb,
                  i64 n, u64 *d_diff, LaunchCounter &lc);

// ---- xsb_algebra.cu
// C = A + B, A - B (SparseArrays' map(op, A, B): an entry of C is stored unless it == 0) and dropzeros! (kAlgKeep:
// A's entries that are not +-0.0, bits unchanged; b unused).  Both CSCs sorted by (column, row), same n, index type
// and base.  merge_count leaves C's nnz at ((u64 *)ws)[0]; merge_write then fills colptr_out (n + 1) and
// rowval_out / nzval_out (that many entries) in the same index type and base.
enum : int
{
    kAlgAdd = 0,
    kAlgSub = 1,
    kAlgKeep = 2
};
size_t merge_workspace_bytes(i64 nnz_a, i64 nnz_b);
void merge_count(cudaStream_t stream, int op, const CscView &a, const CscView *b, i64 n, int idx64, int base, void *ws,
                 LaunchCounter &lc);
void merge_write(cudaStream_t stream, int op, const CscView &a, const CscView *b, i64 n, int idx64, int base,
                 const void *ws, void *colptr_out, void *rowval_out, double *nzval_out, LaunchCounter &lc);

// ---- xsb_spgemm.cu
// C = A * B (SparseArrays' spmatmul): the structural pattern, and per entry the left fold in ascending k of the
// separately rounded products a * b, the first one assigned.  A is m x k, B k x n, both sorted by (column, row),
// same index type and base; m < 2^32 - 1, n < 2^32.  spgemm_classify leaves at ((u64 *)ws)[0..5) the columns of
// the three warp-table bins and of the tiled bin, then the number of row tiles; the caller copies them into
// bins / tiles and allocates tile_ws.  spgemm_count fills colptr_out (n + 1) and leaves nnz(C) at
// ((u64 *)ws)[5] and at ((u64 *)ws)[12..16) the largest u(j) per bin that spgemm_write sizes its tables by (the
// caller copies them into umax); spgemm_write then fills rowval_out / nzval_out (that many entries).
struct Spgemm
{
    CscView a, b;
    i64 m, n;
    int idx64, base;
    void *ws;      // spgemm_workspace_bytes(n)
    void *tile_ws; // spgemm_tiles_bytes(tiles)
    u64 bins[4], tiles;
    u64 umax[4];
};
size_t spgemm_workspace_bytes(i64 n);
size_t spgemm_tiles_bytes(u64 tiles);
void spgemm_classify(cudaStream_t stream, const Spgemm &g, LaunchCounter &lc);
void spgemm_count(cudaStream_t stream, const Spgemm &g, void *colptr_out, LaunchCounter &lc);
void spgemm_write(cudaStream_t stream, const Spgemm &g, const void *colptr, void *rowval_out, double *nzval_out,
                  LaunchCounter &lc);

// ---- xsb_mul.cu
size_t csr_map_bytes(i64 m, i64 nnz);
void build_csr_map(cudaStream_t stream, const CscView &csc, i64 m, i64 n, int idx64, int base, Rec *tags_a, Rec *tags_b,
                   void *sort_ws, u32 *map, LaunchCounter &lc);
void csr_mul(cudaStream_t stream, const u32 *map, i64 m, i64 nnz, const double *nzval, const double *x, double *y,
             LaunchCounter &lc);

} // namespace xsb
