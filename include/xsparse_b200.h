/*
 * xsparse_b200.h -- C ABI of libxsparse_b200.so
 *
 * A B200 (sm_100a) implementation of the assembly hot path of
 * ExtendableSparse.jl: batched insertion/accumulation of possibly duplicate
 * (i,j,v) entries and the flush! that merges them with the resident CSC matrix
 * into a new sorted CSC matrix; a values-only path for frozen patterns; and the
 * synthetic stencil/FEM emitters the benchmarks are defined on.
 *
 * The entry points are what a Julia `ccall` (or any FFI) binding of the
 * reference's extension plug-in interface needs
 * (reference: src/matrix/abstractsparsematrixextension.jl:1-19).  Each entry
 * point cites the reference interface it stands in for; paths are relative to
 * the ExtendableSparse.jl v1.5.1 source tree.
 *
 * Conventions
 *  - Plain C: opaque handle, plain pointers and sizes, no C++/torch types.
 *  - Every function returns an int32 status (XSB_OK == 0).  No exception ever
 *    crosses the boundary.  xsb_last_error(h) returns the message of the last
 *    failing call on that handle (h == NULL: last failure of a call that had no
 *    handle, per thread).
 *  - Array arguments may be HOST or DEVICE pointers (resolved through unified
 *    virtual addressing).  The library never frees, keeps or reallocates a
 *    caller pointer: outputs are written into caller-allocated buffers, hence
 *    the two-phase flush (xsb_flush returns nnz; the caller allocates; then
 *    xsb_fetch_csc).
 *  - Index arrays have the element type `idx_type` and the base `index_base`
 *    chosen at creation (Julia: XSB_I64, base 1).  Values are Float64.
 *  - Threading: every call locks its handle, so calls on one handle from several
 *    threads are safe and run one after the other.  What the reference's contract
 *    needs (test/femtools.jl:88-105) -- xsb_insert_batch / xsb_insert_triplets /
 *    xsb_emit_* issued concurrently with DISTINCT `tid` -- therefore works; the
 *    order in which such calls reach a partition's buffer is the order in which its
 *    own thread issued them.  flush!/reset! are expected from one thread while no
 *    insertion is in flight (test/femtools.jl:109), as in the reference.
 *  - Streams: all work of a handle runs on the handle's own non-blocking CUDA stream
 *    (xsb_get_stream).  DEVICE-pointer arguments (I/J/V, triplets, x, received records,
 *    markers) are read on that stream: the caller must have finished writing them
 *    (synchronise the producing stream, or make it wait on an event) before the call.
 *    HOST-pointer arguments are copied before the call returns.
 *  - There is no CPU fallback: without a CUDA device xsb_create fails with
 *    XSB_ECUDA.
 */
#ifndef XSPARSE_B200_H
#define XSPARSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XSB_VERSION 100 /* 0.1.0 */

/* status codes */
#define XSB_OK 0
#define XSB_EBOUNDS 1  /* Julia BoundsError: sparsematrixcsc.jl:8-10, sparsematrixlnk.jl:121-123 */
#define XSB_ESIZE 2    /* size-mismatch @assert: sparsematrixlnk.jl:296-297 */
#define XSB_EILLEGAL 3 /* error(...) of the MT wrapper: genericmtextendablesparsematrixcsc.jl:67,80 */
#define XSB_EINVAL 4   /* bad argument */
#define XSB_ECUDA 5    /* CUDA runtime failure, or no device */
#define XSB_ENOMEM 6   /* device allocation failed */
#define XSB_ESTATE 7   /* call not valid in the current state (e.g. pending inserts) */

/* value / index element types */
#define XSB_F64 0
#define XSB_I32 0
#define XSB_I64 1

/* insertion flavours */
#define XSB_UPDATE 0 /* updateindex!(A,+,v,i,j): no new entry if v==0   extendable.jl:159-174, sparsematrixlnk.jl:210-228 */
#define XSB_RAW 1    /* rawupdateindex!(A,+,v,i,j): always creates      extendable.jl:181-197, sparsematrixlnk.jl:237-253 */
#define XSB_ASSIGN 2 /* A[i,j]=v: overwrite; creates only if v!=0       extendable.jl:205-218, sparsematrixlnk.jl:178-201 */

/* summation modes */
#define XSB_DETERMINISTIC 0 /* left fold in insertion order: bit-exact with the reference   */
#define XSB_FAST 1          /* summation order free, pattern bit-exact.  Each entry is within gamma(N-1) * sum|x| of
                               the exact sum of its N contributions x (resident value included), gamma(k) = k u /
                               (1 - k u), u = 2^-53; exact (and so equal to XSB_DETERMINISTIC up to the sign of a zero
                               result) whenever every partial sum is representable, e.g. integers or one common power
                               of two.  No relative bound holds once contributions cancel.  xsb_flush: duplicates
                               may be accumulated per chunk of the stream before the per-column merge (off unless
                               xsb_set_preaggregation; otherwise the exact merge runs); xsb_reassemble_values: one
                               atomic add per insertion instead of the ordered per-entry fold */

/* how resident CSC values combine with new duplicates */
#define XSB_COMBINE_SEED 0 /* ((old + v1) + v2)...  the wrapper's CSC-hit branch, extendable.jl:164-166 */
#define XSB_COMBINE_ADD 1  /* old + ((0 + v1) + v2)  stand-alone `lnk + csc`, sparsematrixlnk.jl:359-366 */

typedef struct xsb_matrix xsb_matrix;

/* Timings and traffic of the most recent xsb_flush, for roofline reporting. */
typedef struct xsb_flush_stats
{
    int64_t n_inserted;       /* staged insertions consumed            */
    int64_t nnz_old;          /* entries of the CSC before the flush   */
    int64_t nnz_new;          /* entries of the CSC after the flush    */
    int32_t sort_passes;      /* onesweep passes executed              */
    int32_t sort_bits;        /* key bits sorted                       */
    int32_t kernel_launches;  /* kernels launched by the flush         */
    int32_t column_path;      /* 0: (col,row) sort + flat reduction; 2: column sort + hash fold; 3: two-pass grouping by column + hash fold;
                                 4: grouped chunks (records grouped by column while they were staged) +
                                    thread-per-column merge with the resident CSC -- the product path */
    float ms_total;           /* device time of the whole flush (CUDA events; 0 unless profiling on) */
    float ms_expand;          /* old CSC -> records                    */
    float ms_histogram;       /* digit histogram + scan                */
    float ms_sort;            /* all onesweep passes                   */
    float ms_reduce;          /* segmented duplicate reduction + CSC emit */
    float ms_colptr;          /* colptr scan                           */
    float ms_other;           /* buffer management, shrink copy        */
    float ms_host_alloc;      /* host wall time spent in device allocations during the flush */
    int64_t group_pairs;      /* (chunk, column) pairs of the two-pass grouping; 0 when it was not tried */
    /* detail of the column paths (already included in ms_histogram / ms_sort / ms_reduce above) */
    float ms_group_count;     /* grouping pass 1: per-chunk column histograms             */
    float ms_pair_sort;       /* radix sort of the (column, chunk) pairs                  */
    float ms_group_scatter;   /* pair offsets + grouping pass 2: stable scatter by column */
    float ms_fold;            /* per-column fold of duplicates (entries parked)           */
    float ms_compact;         /* parked entries -> rowval / nzval                         */
    int32_t direct_fold;      /* 1: the fold wrote rowval / nzval / colptr in one pass (no park + compact) */
    int64_t preagg_records;   /* XSB_FAST: staged records left after accumulate-on-insert in windows; 0: not used */
    float ms_preagg;          /* ... and its device time (also inside ms_total)                */
    float precounted;         /* share of the staged records whose chunks were grouped by column by the kernels that
                                 staged them; ms_group_count covers the rest (grouped in place by the flush) */
} xsb_flush_stats;

/* ------------------------------------------------------------------ */
/* life cycle                                                          */
/* ------------------------------------------------------------------ */
int32_t xsb_version(void);
int32_t xsb_device_count(int32_t *count);

/* T_ext(m,n) constructor of the plug-in contract (abstractsparsematrixextension.jl:10)
 * together with the wrapper's empty CSC (extendable.jl:39-41, genericmt...:16-22).
 * n_tid = number of partition buffers (length(xmatrices)); device = CUDA ordinal. */
int32_t xsb_create(int64_t m, int64_t n, int32_t val_type, int32_t idx_type, int32_t index_base,
                   int32_t n_tid, int32_t device, xsb_matrix **out);
int32_t xsb_destroy(xsb_matrix *h);
const char *xsb_last_error(const xsb_matrix *h);

/* reset!(A): extendable.jl:269-272, genericmt...:31-42 */
int32_t xsb_reset(xsb_matrix *h);

/* ExtendableSparseMatrixCSC(csc) constructor: extendable.jl:61-67.  Replaces the
 * resident CSC (colptr[n+1], rowval[nnz], nzval[nnz]); pending inserts are dropped. */
int32_t xsb_set_csc(xsb_matrix *h, const void *colptr, const void *rowval, const void *nzval);

/* After a flush the CSC lives in a buffer sized for the staged insertions (no copy on the
 * hot path); this moves it into exactly nnz entries and releases idle staging buffers
 * (the resize! of sparsematrixlnk.jl:380-381). */
int32_t xsb_shrink_to_fit(xsb_matrix *h);

/* Base.size(ext), SparseArrays.nnz(csc part) */
int32_t xsb_size(const xsb_matrix *h, int64_t *m, int64_t *n);
int32_t xsb_nnz(const xsb_matrix *h, int64_t *nnz);

/* ------------------------------------------------------------------ */
/* insertion                                                           */
/* ------------------------------------------------------------------ */
/* Pre-size the staging buffer of partition `tid` (0-based) for `count` more entries. */
int32_t xsb_reserve(xsb_matrix *h, int32_t tid, int64_t count);

/* `count` calls of updateindex!/rawupdateindex!/setindex!(A,[+,]V[k],I[k],J[k][,tid])
 * in the order k = 0..count-1 (genericmt...:87-114, extendable.jl:159-218).
 * Out-of-range indices reject the whole batch with XSB_EBOUNDS. */
int32_t xsb_insert_batch(xsb_matrix *h, int32_t tid, const void *I, const void *J, const void *V,
                         int64_t count, int32_t flavour);

/* The same `count` calls as xsb_insert_batch, handed over as ONE array of 16-byte triplets: the
 * layout the Julia glue appends to in updateindex!/rawupdateindex!(A,+,v,i,j[,tid]) (one 16-byte
 * store per call instead of three 8-byte ones) and the cheapest one to ship: a host array goes
 * over PCIe straight into the staging buffer (16 B per call instead of 24 B with Int64 indices) and
 * is turned into staged records in place.  row/col carry the handle's index_base; the matrix must
 * have fewer than 2^32 rows and columns (XSB_EINVAL otherwise).  Out-of-range indices reject the
 * whole batch with XSB_EBOUNDS (findindex, sparsematrixcsc.jl:8-10). */
typedef struct xsb_triplet
{
    uint32_t row;
    uint32_t col;
    double val;
} xsb_triplet;
int32_t xsb_insert_triplets(xsb_matrix *h, int32_t tid, const xsb_triplet *T, int64_t count, int32_t flavour);

/* k*k*ncells calls of updateindex!/rawupdateindex!/setindex!(A,[+,]v,i,j[,tid]) of an element loop
 * (test/femtools.jl:45-72), given as connectivity and dense element matrices, Julia's column-major arrays:
 *   dofs  k x ncells, the handle's idx_type and index_base: dofs[l + k*c] = cellnodes[l+1, c+1];
 *   Aloc  k x k x ncells Float64:                         Aloc[il + k*jl + k*k*c] = Aloc[il+1, jl+1, c+1].
 * Value p of Aloc in memory order is call p: (row = dofs[il,c], col = dofs[jl,c], v = Aloc[il,jl,c]) -- elements
 * in order, inside an element column by column, inside a column row by row.  The result equals xsb_insert_batch of
 * that expanded stream bit for bit (any flavour, tid, slab handle -- global dofs --, host or device pointers), and
 * xsb_reassemble_values[_zeroed](h, Aloc, k*k*ncells, mode) after xsb_freeze_elements takes Aloc unchanged.
 * 1 <= k <= 64, else XSB_EINVAL.  A dof outside the matrix rejects the whole batch with XSB_EBOUNDS; the message
 * names the first offending element by its position in the batch.  The staging follows the handle's precount and
 * grouping settings like the emitters: whole elements are grouped by column while they are staged. */
int32_t xsb_insert_elements(xsb_matrix *h, int32_t tid, int32_t k, int64_t ncells, const void *dofs, const double *Aloc,
                            int32_t flavour);
/* The element loop whose rows and columns come from different connectivities: coupling blocks of multi-field
 * problems (test space != trial space, e.g. the pressure-velocity block of Stokes), rectangular operators (P0 x P1
 * divergence, interpolation between meshes).  Julia's column-major arrays again:
 *   rdofs kr x ncells, cdofs kc x ncells (idx_type, index_base), Aloc kr x kc x ncells Float64.
 * Call p = kr*kc*c + kr*jl + il is (row = rdofs[il,c], col = cdofs[jl,c], v = Aloc[il,jl,c]) -- the order of
 * xsb_insert_elements, whose calls are these with kr = kc = k and rdofs = cdofs = dofs.  The result equals
 * xsb_insert_batch of the expanded stream bit for bit, as for the square loop.  1 <= kr, kc <= 64, else XSB_EINVAL.
 * A row dof must lie in the m rows, a column dof in the n_global columns; one outside rejects the whole batch with
 * XSB_EBOUNDS, and the message names the first offending element and whether a row or a column dof is at fault. */
int32_t xsb_insert_elements_rect(xsb_matrix *h, int32_t tid, int32_t kr, int32_t kc, int64_t ncells,
                                 const void *rdofs, const void *cdofs, const double *Aloc, int32_t flavour);

/* Number of staged insertions (an upper bound of nnznew(A), genericextendable...:21). */
int32_t xsb_pending(const xsb_matrix *h, int64_t *count);

/* ------------------------------------------------------------------ */
/* flush! / sparse(A)                                                  */
/* ------------------------------------------------------------------ */
/* flush!(A): extendable.jl:248-255 = Base.:+(lnk,csc) sparsematrixlnk.jl:294-383;
 * multi-partition: Base.sum(xmatrices,csc) sparsematrixdilnkc.jl:397-435.
 * pattern_changed != 0 iff colptr/rowval changed (the phash contract, extendable.jl:252). */
int32_t xsb_flush(xsb_matrix *h, int32_t mode, int64_t *nnz_out, int32_t *pattern_changed);
int32_t xsb_flush_ex(xsb_matrix *h, int32_t mode, int32_t combine, int64_t *nnz_out,
                     int32_t *pattern_changed);

/* sparse(A) after flush!: copy the resident CSC out.  Any pointer may be NULL. */
int32_t xsb_fetch_csc(xsb_matrix *h, void *colptr_out, void *rowval_out, void *nzval_out);

/* getindex(A,i,j) for `count` positions on the flushed CSC (extendable.jl:226-238,
 * findindex sparsematrixcsc.jl:7-23); absent entries read 0. XSB_ESTATE if inserts are pending. */
int32_t xsb_get_values(xsb_matrix *h, const void *I, const void *J, void *V_out, int64_t count);

/* nonzeros(A) .= 0 (sprand.jl:80-85, test_parallel.jl:55) */
int32_t xsb_zero_values(xsb_matrix *h);

/* ------------------------------------------------------------------ */
/* multi-GPU: column-slab ownership, one process (and handle) per GPU  */
/* ------------------------------------------------------------------ */
/* Rank `rank` of `n_ranks` owns columns [col_splits[rank], col_splits[rank+1]) (0-based) of an
 * m x n_global matrix.  Insertions and emitters take GLOBAL indices on any rank; the resident
 * CSC, xsb_flush and xsb_fetch_csc work on the owned slab (colptr has slab_width+1 entries,
 * row indices stay global).  The reference has no counterpart (single process); its
 * per-partition analogue is genericmtextendablesparsematrixcsc.jl:45-51 /
 * sparsematrixdilnkc.jl:416-426, whose partition order becomes the source-rank order here. */
int32_t xsb_create_slab(int64_t m, int64_t n_global, int32_t n_ranks, int32_t rank,
                        const int64_t *col_splits, int32_t val_type, int32_t idx_type,
                        int32_t index_base, int32_t device, xsb_matrix **out);
int32_t xsb_slab_info(const xsb_matrix *h, int64_t *col_begin, int64_t *col_end, int64_t *n_global);
/* A staged record carries its owner and its column relative to the owner's slab, so it is already
 * in its owner's flush layout: routing only COPIES OUT what other ranks own; the rest never moves
 * (the flush skips the copied-out records by their owner bits).
 * Step 0 (optional): xsb_route_count -> send_counts[n_ranks] (host): staged records per owning rank
 *   (own rank: the ones that stay); lets the caller size the send buffer.  One read of the keys.
 * Step 1: xsb_route_prepare copies the records of the OTHER ranks into `send_records` (device,
 *   16 B each), destination after destination, each bucket in stream order; capacity >= their number.
 * Step 2 (caller): all-to-all-v of the buckets (NCCL).
 * Step 3: xsb_route_finish once per source rank != own, in ascending rank order; then xsb_flush.
 * The fold meets the records of an entry as [resident CSC | lower ranks | own | higher ranks], each
 * in stream order: the distributed result equals the serial reference applied to the rank-ordered
 * concatenation of the ranks' streams, bit for bit in XSB_DETERMINISTIC mode. */
int32_t xsb_route_count(xsb_matrix *h, int64_t *send_counts);
/* The same exchange with FIXED capacities, for assembly loops that repeat a step (Newton, time stepping): no
 * count ever visits the host, so the whole step -- insertion, routing, all-to-all, flush -- is stream-ordered
 * apart from the flush's own two synchronisations.  Sender and receiver agree on caps[][] beforehand (e.g. twice
 * what the previous step sent).
 *   xsb_route_pack(h, send, caps, capacity): one BLOCK per destination d != own rank, block after block in `send`
 *     (device): a 16-byte header {records of the bucket, magic} + caps[d] record slots; capacity >= sum(caps[d] + 1).
 *   all-to-all of the blocks (split sizes caps[d] + 1 records, known on the host).
 *   xsb_route_unpack(h, recv, caps): `recv` = the blocks of the sources src != own rank in ascending order, block
 *     src = header + caps[src] slots; every block becomes caps[src] staged records (the bucket, then skipped ones).
 *   xsb_flush.  A bucket that did not fit its block, a record of another owner or a missing header make the FLUSH
 *     fail (XSB_ESTATE / XSB_EBOUNDS / XSB_EINVAL) with the resident matrix untouched: xsb_reset and repeat the step
 *     through xsb_route_count / xsb_route_prepare / xsb_route_finish, or with larger capacities. */
int32_t xsb_route_pack(xsb_matrix *h, void *send_records, const int64_t *caps, int64_t send_capacity);
int32_t xsb_route_unpack(xsb_matrix *h, const void *recv_records, const int64_t *caps);
int32_t xsb_route_prepare(xsb_matrix *h, void *send_records, int64_t capacity, int64_t *send_counts);
int32_t xsb_route_finish(xsb_matrix *h, int32_t src_rank, const void *recv_records, int64_t count);
/* PEER EXCHANGE: the fixed-capacity exchange over NVLink peer memory, for ranks that are processes (or handles of one
 * process) on ONE node whose GPUs have peer access.  No communication library on the records' path: the kernel that
 * copies a bucket out of the staging buffer stores it straight into the MAILBOX of the receiving rank (that GPU's
 * memory, mapped through CUDA IPC) -- the copy-out is the transfer -- and raises a flag there; the receiver's
 * stream waits for the flags of the step, takes the blocks and tells the senders that the blocks are free again.  Two
 * blocks per (sender, receiver) pair let a sender run one step ahead.  Everything is stream-ordered on the handles'
 * streams; nothing visits the host.  (The reference has no counterpart: its partitions share one address space,
 * src/matrix/genericmtextendablesparsematrixcsc.jl:87-114; this is that shared address space across GPUs.)
 *   setup    xsb_peer_exchange_create(h, caps, ipc_handle)  caps[dst * n_ranks + src] = slots of the block src -> dst
 *              (0: the pair exchanges nothing), the SAME matrix on every rank; writes the 64-byte CUDA IPC handle
 *              of this rank's mailbox to ipc_handle (may be NULL for xsb_peer_exchange_connect_local)
 *            all-gather the handles by any means (plain bytes)
 *            xsb_peer_exchange_connect(h, ipc_handles)       n_ranks * 64 bytes, handle of rank r at 64 r
 *            (ranks inside one process: xsb_peer_exchange_connect_local(h, handles_of_all_ranks))
 *   step     insertions -> xsb_route_pack_peer(h) -> xsb_route_unpack_peer(h) -> xsb_flush(h, ...); EVERY rank makes
 *              both calls in every step (ranks that send or receive nothing launch nothing).  xsb_route_pack_peer
 *              may come BEFORE the step's last insertion -- an assembly loop that visits its interface elements
 *              first hides the transfer behind the interior --: records staged after it must be owned by this
 *              rank (one of another rank makes the flush fail, XSB_ESTATE).  Errors surface at the
 *              flush as for xsb_route_pack / _unpack; additionally XSB_ESTATE when a peer did not deliver or take a
 *              block within XSB_PEER_TIMEOUT_MS (environment, default 30000): the ranks are out of step.
 *   teardown xsb_peer_exchange_disconnect on every rank, a barrier, xsb_peer_exchange_destroy (frees the mailbox;
 *              xsb_destroy does both for a handle that still has one). */
int32_t xsb_peer_exchange_create(xsb_matrix *h, const int64_t *caps, void *ipc_handle_out);
int32_t xsb_peer_exchange_connect(xsb_matrix *h, const void *ipc_handles);
int32_t xsb_peer_exchange_connect_local(xsb_matrix *h, xsb_matrix *const *peers);
int32_t xsb_peer_exchange_disconnect(xsb_matrix *h);
int32_t xsb_peer_exchange_destroy(xsb_matrix *h);
int32_t xsb_route_pack_peer(xsb_matrix *h);
int32_t xsb_route_unpack_peer(xsb_matrix *h);

/* ------------------------------------------------------------------ */
/* values-only re-assembly into a frozen pattern (Newton / transient loops) */
/* ------------------------------------------------------------------ */
/* Records, for an insertion stream (I[k],J[k]), the nzval slot of every entry
 * (the CSC-hit branch extendable.jl:164-166 resolved once instead of per insert).
 * Every (i,j) must already be in the pattern, else XSB_EILLEGAL. */
int32_t xsb_freeze_pattern(xsb_matrix *h, const void *I, const void *J, int64_t count);
/* xsb_freeze_pattern for the stream xsb_insert_elements(h, ., k, ncells, dofs, ., .) would stage: the element
 * loop's positions from its connectivity alone; errors as xsb_freeze_pattern (XSB_EBOUNDS names the call). */
int32_t xsb_freeze_elements(xsb_matrix *h, int32_t k, int64_t ncells, const void *dofs);
/* xsb_freeze_elements for the stream xsb_insert_elements_rect(h, ., kr, kc, ncells, rdofs, cdofs, ., .) would stage;
 * xsb_reassemble_values[_zeroed](h, Aloc, kr*kc*ncells, mode) then takes Aloc unchanged. */
int32_t xsb_freeze_elements_rect(xsb_matrix *h, int32_t kr, int32_t kc, int64_t ncells, const void *rdofs,
                                 const void *cdofs);
/* nzval[slot(k)] += V[k] for the frozen stream; deterministic mode folds every entry's values in stream order,
 * starting from the resident value (bit-exact with the in-place CSC-hit updates); fast mode is one atomic add
 * per insertion through the 4-byte entry -> nzval map. */
int32_t xsb_reassemble_values(xsb_matrix *h, const void *V, int64_t count, int32_t mode);
/* nonzeros(A) .= 0 (sprand.jl:80-85, test_parallel.jl:55) followed by xsb_reassemble_values, as ONE pass: the
 * entries start from +0.0 and nzval is written, never read (a Newton / time step re-assembles from zero). */
int32_t xsb_reassemble_values_zeroed(xsb_matrix *h, const void *V, int64_t count, int32_t mode);
int32_t xsb_unfreeze(xsb_matrix *h);
/* On slab handles xsb_freeze_pattern / xsb_freeze_elements[_rect] / xsb_get_values take slab-relative columns and the
 * rank's own entries only.  A distributed element loop is sharded by elements instead: the interface elements of
 * every rank write into columns a neighbour owns.  The calls below freeze such a stream -- GLOBAL positions, any
 * owner -- across the ranks (slab handles only; on a plain handle, or with insertions pending: XSB_ESTATE).
 * A counted exchange runs once, at freeze time; every step then moves the values of the foreign positions with sizes
 * fixed since the freeze.
 *   freeze  xsb_freeze_slab(h, I, J, count, send_counts) or xsb_freeze_slab_elements(h, k, ncells, dofs, send_counts):
 *             resolves the own positions and counts the foreign ones per owner: send_counts[n_ranks] (host; own rank:
 *             the positions kept).  count < 2^32 (else XSB_EINVAL); a position outside the matrix: XSB_EBOUNDS naming
 *             the stream position; an own position absent from the pattern: XSB_EILLEGAL.  The handle is now HALF
 *             frozen: the re-assembly calls return XSB_ESTATE, and insertions, xsb_flush, xsb_set_csc, xsb_reset and
 *             xsb_unfreeze drop the half-made freeze.
 *           xsb_freeze_slab_prepare(h, send_positions, capacity): the foreign positions, destination after destination,
 *             each bucket in stream order, 8 bytes each {u32 row (0-based), u32 column relative to the owner's slab},
 *             into device memory; capacity >= their number.
 *           (caller) exchange the counts, then the positions, all-to-all-v (own rank: nothing).
 *           xsb_freeze_slab_finish(h, recv_positions, recv_counts): the received buckets, sources ascending, own rank
 *             left out (recv_counts[own] is ignored); device memory.  Resolves them against the slab's CSC (absent:
 *             XSB_EILLEGAL, outside the slab: XSB_EBOUNDS) and builds the map.  Received positions plus count must
 *             stay below 2^32 (XSB_EINVAL).  On any error of the three calls the handle is left unfrozen.
 *           xsb_frozen_slab_counts(h, send_counts, recv_counts): the sizes of the per-step exchange.
 *   step    xsb_reassemble_slab_pack(h, V, count, send_values): V holds one value per position of the rank's frozen
 *             stream (count must match: XSB_ESIZE); the values of the foreign positions go to send_values (device),
 *             laid out as the positions at prepare.
 *           (caller) exchange the values with the counts of the freeze (point-to-point, no count on the host).
 *           xsb_reassemble_slab_values(h, V, count, recv_values, mode, zero_first): folds own and received values into
 *             the slab's nzval; recv_values laid out as the positions at finish.
 *   The map indexes the combined space [received from lower ranks | own stream | received from higher ranks]; every
 *   entry folds its resident value (+0.0 with zero_first), then the values of rank 0, 1, ..., each rank's in its
 *   stream order.  So rank r's slab equals, bit for bit in XSB_DETERMINISTIC mode, its columns of one plain handle
 *   that froze the concatenated streams S_0 ++ S_1 ++ ... and re-assembled V_0 ++ V_1 ++ ...  XSB_FAST: one atomic add
 *   per value.  xsb_reassemble_values[_zeroed] on a handle frozen this way returns XSB_ESTATE; a flush that changes the
 *   slab's pattern drops the map. */
int32_t xsb_freeze_slab(xsb_matrix *h, const void *I, const void *J, int64_t count, int64_t *send_counts);
int32_t xsb_freeze_slab_elements(xsb_matrix *h, int32_t k, int64_t ncells, const void *dofs, int64_t *send_counts);
/* the first step of the slab freeze for the stream of xsb_insert_elements_rect; then _prepare and _finish as above */
int32_t xsb_freeze_slab_elements_rect(xsb_matrix *h, int32_t kr, int32_t kc, int64_t ncells, const void *rdofs,
                                      const void *cdofs, int64_t *send_counts);
int32_t xsb_freeze_slab_prepare(xsb_matrix *h, void *send_positions, int64_t capacity);
int32_t xsb_freeze_slab_finish(xsb_matrix *h, const void *recv_positions, const int64_t *recv_counts);
int32_t xsb_frozen_slab_counts(const xsb_matrix *h, int64_t *send_counts, int64_t *recv_counts);
int32_t xsb_reassemble_slab_pack(xsb_matrix *h, const double *V, int64_t count, double *send_values);
int32_t xsb_reassemble_slab_values(xsb_matrix *h, const double *V, int64_t count, const double *recv_values,
                                   int32_t mode, int32_t zero_first);

/* y = A*x on the resident CSC (x: n values, y: m values; host or device pointers).  mul!(r,A,x):
 * src/matrix/abstractextendablesparsematrixcsc.jl:170-181 (flush, then the stdlib kernel: columns
 * ascending, y[rowval[k]] += nzval[k]*x[j]).  Every y[i] is that left fold in column order with
 * separately rounded products: bit-identical to the reference.  The row-major view of the pattern
 * it needs is built on first use and dropped when a flush changes the pattern.  On a slab handle
 * x holds the slab's columns and y is the slab's contribution (sum over the ranks = A*x). */
int32_t xsb_mul(xsb_matrix *h, const void *x, void *y);

/* ------------------------------------------------------------------ */
/* values-only passes over the resident CSC                            */
/* ------------------------------------------------------------------ */
/* mark_dirichlet / eliminate_dirichlet!: sparsematrixcsc.jl:97-148 (square matrices) */
int32_t xsb_mark_dirichlet(xsb_matrix *h, double penalty, uint8_t *marker_out);
int32_t xsb_eliminate_dirichlet(xsb_matrix *h, const uint8_t *marker);
/* 64-bit fingerprint of (colptr,rowval): stands in for phash (sparsematrixcsc.jl:74);
 * equal patterns give equal values, it is NOT Julia's hash(). */
int32_t xsb_pattern_hash(xsb_matrix *h, uint64_t *hash_out);

/* pattern_equal(a, b): src/matrix/sparsematrixcsc.jl:77-85 -- a.colptr == b.colptr && a.rowval == b.rowval, compared
 * element by element on the device (exact, unlike comparing two xsb_pattern_hash values); matrices of different size
 * or nnz are unequal.  Both matrices flushed (XSB_ESTATE otherwise).  Handles on different devices fall back to
 * comparing fingerprints. */
int32_t xsb_pattern_equal(xsb_matrix *a, xsb_matrix *b, int32_t *equal_out);

/* ------------------------------------------------------------------ */
/* pattern-changing operations on flushed matrices                     */
/* ------------------------------------------------------------------ */
/* A + B and A - B: src/matrix/abstractextendablesparsematrixcsc.jl (flush both, then SparseArrays'
 * map(+/-, A, B)).  Column by column over the sorted rows of both: a row in both gives f(a, b), a row
 * in A only f(a, 0.0), a row in B only f(0.0, b), and the result is stored unless it == 0 (so +-0.0 are
 * dropped, NaN is kept, explicit zeros of the inputs disappear).  Every value is one IEEE add or
 * subtract; NaN results carry x86-64's bits (the first NaN operand, quieted; Inf - Inf is the negative
 * default NaN), as the reference computes them on its hosts.
 * Returns a NEW plain handle *out = C with one partition and A's device, index type and base: a full
 * assembly target (insert, flush, freeze, mul).  Its CSC is built on the device.  The caller destroys it.
 * a == b is allowed (A - A is empty).  Pending inserts on either, a slab handle or a pointblock result:
 * XSB_ESTATE; different sizes: XSB_ESIZE (DimensionMismatch); different index type, base or device, an
 * unknown op, or a result nnz the index type cannot hold: XSB_EINVAL.  On any error *out is NULL and A
 * and B are unchanged. */
#define XSB_OP_ADD 0
#define XSB_OP_SUB 1
int32_t xsb_add(xsb_matrix *a, xsb_matrix *b, int32_t op, xsb_matrix **out);

/* dropzeros!(A): src/matrix/abstractextendablesparsematrixcsc.jl:110 (fkeep! with !iszero): removes
 * the stored +-0.0 in place, order and the other values' bits unchanged.  *pattern_changed = 1 exactly
 * when an entry was dropped; only then are the frozen map (plain or slab), the row-major view of xsb_mul
 * and a half-made slab freeze dropped, so a dropzeros that drops nothing leaves a frozen handle frozen.
 * Plain and slab handles (each rank filters its own slab, no communication).  Pending inserts or a
 * pointblock result: XSB_ESTATE. */
int32_t xsb_dropzeros(xsb_matrix *h, int64_t *nnz_out, int32_t *pattern_changed);

/* pointblock(A, blocksize): src/matrix/extendable.jl:292-318 (feeds PointBlockILUZeroPreconditioner,
 * src/factorizations/iluzero.jl:61-71).  Returns a NEW handle *out holding the nblock x nblock block
 * matrix Ab, nblock = n / blocksize: its CSC pattern is read with xsb_nnz / xsb_fetch_csc, its values
 * -- one dense blocksize x blocksize block per pattern entry, column-major (SMatrix layout), in CSC
 * order -- with xsb_fetch_blocks.  As in the reference the block index taken from A's COLUMN becomes
 * the block ROW: Ab[(i-1)/bs+1, (j-1)/bs+1][(i-1)%bs+1, (j-1)%bs+1] = A[j,i] for every stored A[j,i]
 * (the reference's loop variable i runs over columns).  An entry that falls outside nblock blocks is
 * the reference's BoundsError (XSB_EBOUNDS).  Pending inserts: XSB_ESTATE (flush first).  The caller
 * destroys *out with xsb_destroy; it is a result, not an assembly target. */
int32_t xsb_pointblock(xsb_matrix *h, int32_t blocksize, xsb_matrix **out);
int32_t xsb_block_size(const xsb_matrix *hb, int32_t *blocksize);
int32_t xsb_fetch_blocks(xsb_matrix *hb, void *blocks_out);

/* ------------------------------------------------------------------ */
/* on-device emitters of the benchmark insertion streams               */
/* ------------------------------------------------------------------ */
/* fdrand!(A,nx,ny,nz) call stream: sprand.jl:58-126.  ones != 0: rand = ()->1. */
int32_t xsb_emit_fdrand(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz,
                        uint64_t seed, int32_t ones, int32_t flavour);
/* Same stream restricted to nodes l in [l_begin, l_end) (0-based), for sharded generation. */
int32_t xsb_emit_fdrand_range(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz,
                              uint64_t seed, int32_t ones, int32_t flavour, int64_t l_begin,
                              int64_t l_end);
/* testassemble!(A,grid) call stream on the Kuhn tensor mesh: test/femtools.jl:45-72 */
int32_t xsb_emit_p1fem(xsb_matrix *h, int32_t tid, int64_t nxn, int64_t nyn, int64_t nzn,
                       int32_t flavour);
/* Same, cubes cz in [cz_begin, cz_end) only; node numbering stays global. */
int32_t xsb_emit_p1fem_range(xsb_matrix *h, int32_t tid, int64_t nxn, int64_t nyn, int64_t nzn,
                             int32_t flavour, int64_t cz_begin, int64_t cz_end);
/* block reaction-diffusion stream (SURVEY.md 8d cfg 4) */
int32_t xsb_emit_blockrd(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz,
                         int32_t ns, uint64_t seed, int32_t flavour);

/* Lengths of those streams (host arithmetic, no device needed). */
int32_t xsb_stream_count_fdrand(int64_t nx, int64_t ny, int64_t nz, int64_t *count);
int32_t xsb_stream_count_p1fem(int64_t nxn, int64_t nyn, int64_t nzn, int64_t *count);
int32_t xsb_stream_count_blockrd(int64_t nx, int64_t ny, int64_t nz, int32_t ns, int64_t *count);

/* Copy staged records of partition `tid` back as (I,J,V,flavour) in stream order (testing aid). */
int32_t xsb_debug_fetch_staged(xsb_matrix *h, int32_t tid, void *I, void *J, void *V,
                               int32_t *flavour, int64_t capacity, int64_t *count);

/* ------------------------------------------------------------------ */
/* streams, timing                                                     */
/* ------------------------------------------------------------------ */
int32_t xsb_synchronize(xsb_matrix *h);
/* The CUDA stream (cudaStream_t) all kernels of this handle are launched on. */
int32_t xsb_get_stream(xsb_matrix *h, void **stream_out);
/* CUDA-event timer on that stream. */
int32_t xsb_timer_start(xsb_matrix *h);
int32_t xsb_timer_stop(xsb_matrix *h, float *ms_out);
/* Per-stage CUDA-event timing inside xsb_flush (off by default). */
int32_t xsb_set_profiling(xsb_matrix *h, int32_t enable);
/* Flush algorithm.  AUTO: records brought together by column (grouped chunks, two-pass grouping or
 * a stable radix sort on the column bits); per column, duplicates are folded through a hash table in
 * stream order and only the distinct entries are sorted by row (falls back to the FULLSORT path by
 * itself when a column does not fit).  FULLSORT: (col,row) radix sort + flat segmented reduction.
 * Both give the same bits; any other value returns XSB_EINVAL. */
#define XSB_STRATEGY_AUTO 0
#define XSB_STRATEGY_FULLSORT 1
int32_t xsb_set_strategy(xsb_matrix *h, int32_t strategy);
/* How STRATEGY_AUTO brings the records of a column together.  AUTO: try the two-pass grouping
 * (sparse per-chunk column histograms; pays off when consecutive insertions touch few distinct
 * columns, as element-by-element assembly does) and use the radix sort when the stream has no
 * such locality; after two such misses in a row the handle stops trying.  OFF: always the radix
 * sort.  ON: always try. */
#define XSB_GROUPING_AUTO 0
#define XSB_GROUPING_OFF 1
#define XSB_GROUPING_ON 2
int32_t xsb_set_grouping(xsb_matrix *h, int32_t grouping);
/* XSB_FAST flushes only (ignored otherwise, and when A[i,j]=v records are staged): fold the staged
 * stream inside windows of 512 insertions first -- the reference's accumulate-on-insert
 * (src/matrix/sparsematrixlnk.jl:210-253) -- so that fewer records are grouped.  Pattern unchanged,
 * each value within gamma(N-1) * sum|x| of the exact sum of its N contributions (XSB_FAST), summation
 * order not reproducible from run to run.  Streams of fewer than 4096 staged records are not folded;
 * a handle stops trying after two flushes in a row whose windows kept more than 3/4 of the records,
 * until xsb_set_preaggregation is called again.  Off by default:
 * on B200 it only pays when the windows shrink the stream more than about 3x (DESIGN.md section 5). */
int32_t xsb_set_preaggregation(xsb_matrix *h, int32_t enable);
/* Grouping at insertion (default on): the kernels behind xsb_insert_batch / xsb_insert_triplets / xsb_emit_* bring
 * every chunk of ~512 consecutive insertions into column order while its records are in registers or shared memory
 * and publish where each column's records lie; xsb_flush then reads them in place and never moves a record.  Off:
 * records are staged in call order and the flush groups the chunks itself (one more read + write of the records).
 * Applies to partition 0 of single-partition handles (slab handles included); results are identical either way.
 * xsb_debug_fetch_staged returns grouped chunks in their grouped order. */
int32_t xsb_set_precount(xsb_matrix *h, int32_t enable);
int32_t xsb_get_flush_stats(const xsb_matrix *h, xsb_flush_stats *out);
/* Total kernels launched by this handle since creation. */
int32_t xsb_kernel_launches(const xsb_matrix *h, int64_t *count);

#ifdef __cplusplus
}
#endif
#endif /* XSPARSE_B200_H */
