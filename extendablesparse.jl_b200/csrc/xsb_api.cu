// xsb_api.cu -- the C ABI of libxsparse_b200 (include/xsparse_b200.h): handle, device
// memory, staging buffers and the flush pipeline that strings the kernels together.
#include "../../include/xsparse_b200.h"
#include "xsb_internal.h"

#include <chrono>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

using namespace xsb;

namespace {

struct ApiError : std::runtime_error
{
    int32_t code;
    ApiError(int32_t c, const std::string &w) : std::runtime_error(w), code(c) {}
};

thread_local std::string g_err;

int ceil_log2(i64 x)
{
    int b = 0;
    while (((i64)1 << b) < x)
        ++b;
    return b < 1 ? 1 : b;
}

bool is_device_ptr(const void *p)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

struct Stage
{
    Rec *buf = nullptr;
    i64 cap = 0;   // records the allocation holds (front included)
    i64 front = 0; // slots reserved ahead of the staged records for the old CSC (single-partition handles)
    i64 count = 0; // staged records
};

} // namespace

struct xsb_matrix
{
    i64 m = 0, n = 0;
    int idx64 = 1, base = 1, n_tid = 1, device = 0;
    KeyLayout L{};  // layout the flush sorts and reduces on (columns relative to the slab)
    KeyLayout Ls{}; // layout of staged records before routing (global columns + owner bits); == L without ranks
    i64 n_global = 0, col_begin = 0; // slab handles own columns [col_begin, col_begin + n) of an m x n_global matrix
    int nranks = 0, rank = 0;        // nranks == 0: plain single-GPU handle
    bool routed = false;             // staged records already went through xsb_route_prepare / xsb_route_finish
    i64 foreign = 0;                 // staged records owned by other ranks (sent; the flush skips them)
    void *route_ws = nullptr;        // tile counts between xsb_route_count and xsb_route_prepare
    unsigned char *tileflags = nullptr; // slab handles: tiles of the staged records that hold records of other ranks
    i64 tileflags_cap = 0;
    u64 route_counts[kMaxRanks] = {0};
    i64 route_counted = -1;          // staged count route_counts was taken at
    // regions of the staged records of a slab handle after routing (offsets from stage.front, chunk aligned):
    // own [0, own_end), received from lower ranks [own_end, low_end), from higher ranks [low_end, count)
    i64 own_end = 0, low_end = -1, n_low = 0, n_high = 0, n_pad = 0;
    int last_src = -1;
    cudaStream_t stream = nullptr;
    std::string err;
    // Calls on one handle are serialised here: insertions with distinct `tid` may be ISSUED concurrently
    // (the reference's threading contract, test/femtools.jl:88-105), their host side runs one at a time.
    std::recursive_mutex mu;

    // resident CSC, in the caller's index type and base
    void *colptr = nullptr;
    void *csc_store = nullptr; // holds rowval then nzval
    size_t csc_store_bytes = 0;
    void *rowval = nullptr;
    double *nzval = nullptr;
    i64 nnz = 0;

    std::vector<Stage> stage;
    bool has_assign = false;

    // frozen pattern
    bool frozen = false;
    i64 f_count = 0;
    u32 *f_slot = nullptr;     // 4-byte entry -> nzval map of the frozen stream (fast mode)
    u32 *f_perm = nullptr;     // stream positions in nzval order (deterministic mode)
    u32 *f_segstart = nullptr; // first of them per nzval entry
    // stream frozen across column slabs (xsb_freeze_slab*): global positions, those in other ranks' columns travel
    // to their owner.  The map above then indexes [received from lower ranks | own stream | from higher ranks].
    int fs_state = 0;                  // 0: none, 1: half frozen (until xsb_freeze_slab_finish), 2: frozen
    i64 fs_send[kMaxRanks] = {0};      // positions per owner (own rank: the ones kept)
    i64 fs_recv[kMaxRanks] = {0};      // positions received per source (own rank: 0)
    i64 fs_foreign = 0, fs_low = 0, fs_total = 0; // sent; received from lower ranks; size of the combined space
    u32 *fs_send_idx = nullptr;        // stream indices of the sent positions, destination after destination
    u64 *fs_send_pos = nullptr;        // their {row, owner-relative column} (until the freeze is complete)
    i64 *fs_slot = nullptr;            // nzval slot per own stream position, -1: foreign (until complete)

    double *blocks = nullptr; // result handle of xsb_pointblock: nnz dense bs x bs blocks, column-major, CSC order
    int block_size = 0;
    u32 *csr_map = nullptr; // row-major view of the resident pattern for xsb_mul (rebuilt when the pattern changes)
    u64 *d_scal = nullptr; // 8 device scalars
    u64 *h_scal = nullptr; // pinned mirror
    // fixed-capacity exchange (xsb_route_pack / xsb_route_unpack): nothing of it visits the host until the flush
    u64 *d_route = nullptr;    // [0] error flags of the received blocks, [1] records taken from lower ranks, [2] from higher
    u64 *h_route = nullptr;    // pinned: block bases / capacities handed to the kernels (2 * kMaxRanks), results (4)
    bool fixed_exchange = false; // the staged regions of other ranks are capacity-sized blocks (n_low / n_high: upper bounds)

    // Peer exchange (xsb_peer_exchange_*): the blocks of the fixed-capacity exchange are written straight into the
    // MAILBOX of the receiving rank (its GPU's memory, mapped here through CUDA IPC or, inside one process, used
    // directly) by the copy-out kernel; flags in the mailboxes order the steps.  Mailbox of rank r:
    //   u64 ready[kMaxRanks]  ready[s] = last step whose block from s is complete   (written by s)
    //   u64 done[kMaxRanks]   done[d]  = last step whose block TO d was taken by d  (written by d)
    //   at 512 B: for every source s with caps[r][s] > 0, ascending: two blocks (step parity) of
    //             round16(1 + caps[r][s]) records each
    struct PeerExchange
    {
        bool created = false, connected = false, packed = false;
        unsigned char *box = nullptr;
        size_t box_bytes = 0;
        unsigned char *peer[kMaxRanks] = {};
        bool peer_ipc[kMaxRanks] = {};
        i64 caps[kMaxRanks * kMaxRanks] = {}; // [dst * nranks + src]
        u64 seq = 0;                          // steps packed so far
        i64 packed_upto = 0;                  // staged records when xsb_route_pack_peer ran
        u64 timeout_ns = 30000000000ull;
    } px;

    LaunchCounter lc;
    bool profiling = false;
    xsb_flush_stats stats{};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // host triplets arrive in slices on a second stream while the slices before them are packed (xsb_insert_triplets)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_slice[3] = {nullptr, nullptr, nullptr};

    float alloc_ms = 0.f; // host time spent inside cudaMallocAsync (reset per flush)
    static constexpr size_t kBigBytes = (size_t)32 << 20;
    std::unordered_map<void *, size_t> big_live;         // large allocations currently handed out
    std::vector<std::pair<void *, size_t>> big_cache;    // large allocations waiting for reuse
    size_t isz() const { return idx64 ? 8 : 4; }
    void *dalloc(size_t bytes)
    {
        void *p = nullptr;
        if (bytes == 0)
            bytes = 16;
        if (bytes >= kBigBytes)
        { // size classes of four significant bits (at most 1/8 more than asked for): a CSC store that grows by a
          // per cent per flush keeps fitting the block the flush before last gave back
            const int sh = 60 - __builtin_clzll((unsigned long long)bytes);
            const size_t m = ((size_t)1 << sh) - 1;
            bytes = (bytes + m) & ~m;
        }
        if (bytes >= kBigBytes)
        { // large buffers (staging, sort scratch, CSC store) rotate through a per-handle cache:
          // in a steady assembly loop a flush allocates nothing (measured: the CUDA pool re-maps
          // gigabytes per flush once small allocations have split its free blocks)
            int best = -1;
            for (int k = 0; k < (int)big_cache.size(); ++k)
                if (big_cache[k].second >= bytes && big_cache[k].second <= 4 * bytes &&
                    (best < 0 || big_cache[k].second < big_cache[best].second))
                    best = k;
            if (best >= 0)
            {
                p = big_cache[best].first;
                big_live[p] = big_cache[best].second;
                big_cache.erase(big_cache.begin() + best);
                return p;
            }
        }
        const auto t0 = std::chrono::steady_clock::now();
        cudaError_t e = cudaMallocAsync(&p, bytes, stream);
        if (e == cudaErrorMemoryAllocation && !big_cache.empty())
        { // give the cache back and retry once
            cudaGetLastError();
            release_cache();
            e = cudaMallocAsync(&p, bytes, stream);
        }
        alloc_ms += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (e != cudaSuccess)
        {
            cudaGetLastError();
            throw ApiError(e == cudaErrorMemoryAllocation ? XSB_ENOMEM : XSB_ECUDA,
                           std::string("device allocation of ") + std::to_string(bytes) +
                               " bytes failed: " + cudaGetErrorString(e));
        }
        if (bytes >= kBigBytes)
            big_live[p] = bytes;
        return p;
    }
    void dfree(void *p)
    {
        if (!p)
            return;
        auto it = big_live.find(p);
        if (it == big_live.end())
        {
            cudaFreeAsync(p, stream);
            return;
        }
        big_cache.emplace_back(p, it->second);
        big_live.erase(it);
        if (big_cache.size() > 6)
        { // keep the cache bounded: drop the smallest buffer
            int k = 0;
            for (int q = 1; q < (int)big_cache.size(); ++q)
                if (big_cache[q].second < big_cache[k].second)
                    k = q;
            cudaFreeAsync(big_cache[k].first, stream);
            big_cache.erase(big_cache.begin() + k);
        }
    }
    void release_cache()
    {
        for (auto &b : big_cache)
            cudaFreeAsync(b.first, stream);
        big_cache.clear();
    }
    void sync() { XSB_CUDA(cudaStreamSynchronize(stream)); }
    i64 pending() const
    {
        i64 s = 0;
        for (auto &st : stage)
            s += st.count;
        return s;
    }
    CscView view() const { return CscView{colptr, rowval, nzval, nnz}; }
    void drop_blocks()
    {
        dfree(blocks);
        blocks = nullptr;
        block_size = 0;
    }
    static i64 chunk_up(i64 x)
    {
        const i64 w = group_chunk_records();
        return (x + w - 1) / w * w;
    }
    void drop_frozen()
    {
        dfree(csr_map);
        csr_map = nullptr;
        dfree(f_slot);
        dfree(f_perm);
        dfree(f_segstart);
        f_slot = nullptr;
        f_perm = nullptr;
        f_segstart = nullptr;
        frozen = false;
        f_count = 0;
        dfree(fs_send_idx);
        dfree(fs_send_pos);
        dfree(fs_slot);
        fs_send_idx = nullptr;
        fs_send_pos = nullptr;
        fs_slot = nullptr;
        fs_state = 0;
        fs_foreign = fs_low = fs_total = 0;
        for (int r = 0; r < kMaxRanks; ++r)
            fs_send[r] = fs_recv[r] = 0;
    }
    // insertions and flushes abandon a slab freeze that is still waiting for xsb_freeze_slab_finish
    void drop_half_freeze()
    {
        if (fs_state == 1)
            drop_frozen();
    }
    void clear_staging(bool release)
    {
        for (auto &st : stage)
        {
            st.count = 0;
            st.front = 0;
            routed = false;
            foreign = 0;
            route_counted = -1;
            own_end = 0;
            low_end = -1;
            n_low = n_high = n_pad = 0;
            last_src = -1;
            if (fixed_exchange && d_route)
                cudaMemsetAsync(d_route, 0, sizeof(u64) * 4, stream);
            fixed_exchange = false;
            if (release)
            {
                dfree(st.buf);
                st.buf = nullptr;
                st.cap = 0;
            }
        }
        has_assign = false;
        if (runs.ws && (runs.nchunks > 0 || runs.dead))
            cudaMemsetAsync(runs.ws, 0, 256, stream); // pair ticket and flags of the run index
        runs.nchunks = 0;
        runs.sorted_end = 0;
        runs.dead = false;
        if (tileflags)
            cudaMemsetAsync(tileflags, 0, (size_t)tileflags_cap, stream);
    }
    void set_empty_csc()
    {
        dfree(colptr);
        dfree(csc_store);
        colptr = dalloc(isz() * (size_t)(n + 1));
        fill_index(stream, colptr, n + 1, idx64, base, lc); // spzeros: colptr[:] = base
        csc_store = nullptr;
        csc_store_bytes = 0;
        rowval = nullptr;
        nzval = nullptr;
        nnz = 0;
    }
    size_t shrink_surplus_bytes = (size_t)16 << 30;
    int strategy = XSB_STRATEGY_AUTO;
    int grouping = XSB_GROUPING_AUTO; // two-pass grouping by column before the hash fold
    int grouping_misses = 0;          // consecutive flushes whose stream had no column locality
    int runs_misses = 0;              // consecutive flushes whose columns were too long / rich for the thread-per-column merge
    i64 stats_pairs = 0;
    bool no_direct_fold = false; // the one-pass fold met columns it cannot take: park + compact instead
    int stats_direct = 0;
    i64 stats_preagg = 0;
    i64 stats_precounted = 0;
    bool preagg = false;   // xsb_set_preaggregation
    int preagg_misses = 0; // consecutive XSB_FAST flushes whose windows held few duplicates
    u32 fold_hint = 0; // most distinct rows a column held in the previous thread-per-column fold
    // Grouping at insertion (xsb_chunk.cuh): the kernels that stage records (pack / emit) bring every chunk
    // into column order while its records are in registers / shared memory and publish its runs in the run
    // index; the flush (xsb_runs.cu) reads the runs in place.  Partition 0 of single-partition handles.
    struct RunIndexState
    {
        void *ws = nullptr;  // run index laid out for cap_records staged records
        i64 cap_records = 0;
        u32 cap_chunks = 0;
        u32 nchunks = 0;     // chunks published so far
        i64 sorted_end = 0;  // staged records [0, sorted_end) are grouped chunks whose runs are published
        bool dead = false;   // a rejected batch left runs behind: the index is rebuilt at flush time
    } runs;
    bool precount = true; // xsb_set_precount: producers group their chunks (else the flush does)
    void runs_release()
    {
        dfree(runs.ws);
        runs = RunIndexState{};
    }
    // room in the run index for `records` staged records (contents are kept)
    void runs_reserve(i64 records)
    {
        if (runs.ws && runs.cap_records >= records)
            return;
        const i64 want = std::max<i64>(records + records / 4, 65536);
        const RunIndexLayout nl = run_index_layout((u64)want);
        void *nw = dalloc(nl.bytes);
        XSB_CUDA(cudaMemsetAsync(nw, 0, 256, stream));
        if (runs.ws && runs.nchunks > 0 && !runs.dead)
        { // an assembly in progress outgrew the index: move what was published
            const RunIndexLayout ol = run_index_layout((u64)runs.cap_records);
            unsigned char *o = static_cast<unsigned char *>(runs.ws), *n2 = static_cast<unsigned char *>(nw);
            XSB_CUDA(cudaMemcpyAsync(n2 + nl.off_counters, o + ol.off_counters, 256, cudaMemcpyDeviceToDevice, stream));
            XSB_CUDA(cudaMemcpyAsync(n2 + nl.off_chunkinfo, o + ol.off_chunkinfo, sizeof(uint2) * (size_t)runs.nchunks,
                                     cudaMemcpyDeviceToDevice, stream));
            XSB_CUDA(cudaMemcpyAsync(n2 + nl.off_chunkstart, o + ol.off_chunkstart, sizeof(u32) * (size_t)runs.nchunks,
                                     cudaMemcpyDeviceToDevice, stream));
            XSB_CUDA(cudaMemcpyAsync(n2 + nl.off_pcol, o + ol.off_pcol, sizeof(u32) * (size_t)ol.cap_pairs,
                                     cudaMemcpyDeviceToDevice, stream));
            XSB_CUDA(cudaMemcpyAsync(n2 + nl.off_pinfo, o + ol.off_pinfo, sizeof(u32) * (size_t)ol.cap_pairs,
                                     cudaMemcpyDeviceToDevice, stream));
        }
        dfree(runs.ws);
        runs.ws = nw;
        runs.cap_records = want;
        runs.cap_chunks = nl.cap_chunks;
    }
    // move rowval/nzval into an allocation of exactly nnz entries
    void shrink_store()
    {
        const size_t rv_bytes = (isz() * (size_t)nnz + 15) & ~(size_t)15;
        if (!csc_store || csc_store_bytes <= rv_bytes + 8 * (size_t)nnz)
            return;
        unsigned char *st = static_cast<unsigned char *>(dalloc(rv_bytes + 8 * (size_t)nnz));
        if (nnz)
        {
            XSB_CUDA(cudaMemcpyAsync(st, rowval, isz() * (size_t)nnz, cudaMemcpyDeviceToDevice, stream));
            XSB_CUDA(cudaMemcpyAsync(st + rv_bytes, nzval, 8 * (size_t)nnz, cudaMemcpyDeviceToDevice, stream));
        }
        dfree(csc_store);
        csc_store = st;
        csc_store_bytes = rv_bytes + 8 * (size_t)nnz;
        rowval = st;
        nzval = reinterpret_cast<double *>(st + rv_bytes);
    }
    // make room for `extra` more records in partition t
    void ensure_stage(int t, i64 extra)
    {
        Stage &st = stage[t];
        if (st.count == 0)
        {
            st.front = (n_tid == 1) ? nnz : 0;
            if (L.ownerbits > 0) // slab handles: every region of the buffer is a whole number of chunks
                st.front = chunk_up(st.front);
        }
        const i64 need = st.front + st.count + extra;
        if (need <= st.cap)
        {
            ensure_tileflags(st.cap);
            return;
        }
        i64 cap = std::max<i64>(need, st.cap + st.cap / 2);
        cap = (std::max<i64>(cap, 1024) + 1) & ~(i64)1; // even: the merge reads whole 32-byte sectors (two records)
        Rec *nb = static_cast<Rec *>(dalloc(sizeof(Rec) * (size_t)cap));
        if (st.buf && st.count > 0)
            XSB_CUDA(cudaMemcpyAsync(nb + st.front, st.buf + st.front, sizeof(Rec) * (size_t)st.count,
                                     cudaMemcpyDeviceToDevice, stream));
        dfree(st.buf);
        st.buf = nb;
        st.cap = cap;
        ensure_tileflags(cap);
    }
    // one byte per 2048 staged records, set by the producers (StageFlags) where another rank's record lands
    void ensure_tileflags(i64 cap_records)
    {
        if (L.ownerbits == 0)
            return;
        const i64 need = (cap_records >> kRouteTileShift) + 2;
        if (need <= tileflags_cap)
            return;
        unsigned char *nf = static_cast<unsigned char *>(dalloc((size_t)need));
        XSB_CUDA(cudaMemsetAsync(nf, 0, (size_t)need, stream));
        if (tileflags)
            XSB_CUDA(cudaMemcpyAsync(nf, tileflags, (size_t)tileflags_cap, cudaMemcpyDeviceToDevice, stream));
        dfree(tileflags);
        tileflags = nf;
        tileflags_cap = need;
    }
    StageFlags stage_flags(int t) const { return StageFlags{n_tid == 1 ? tileflags : nullptr, stage[t].count}; }
};

namespace {

void set_err(xsb_matrix *h, const std::string &s)
{
    if (h)
        h->err = s;
    else
        g_err = s;
}

template <class F> int32_t guard(xsb_matrix *h, F &&f)
{
    std::unique_lock<std::recursive_mutex> lock;
    if (h)
        lock = std::unique_lock<std::recursive_mutex>(h->mu);
    try
    {
        if (h)
            XSB_CUDA(cudaSetDevice(h->device));
        return f();
    }
    catch (const ApiError &e)
    {
        set_err(h, e.what());
        return e.code;
    }
    catch (const CudaError &e)
    {
        set_err(h, e.what());
        cudaGetLastError();
        return e.code == cudaErrorMemoryAllocation ? XSB_ENOMEM : XSB_ECUDA;
    }
    catch (const std::bad_alloc &)
    {
        set_err(h, "host allocation failed");
        return XSB_ENOMEM;
    }
    catch (const std::exception &e)
    {
        set_err(h, e.what());
        return XSB_EINVAL;
    }
    catch (...)
    {
        set_err(h, "unknown failure");
        return XSB_EINVAL;
    }
}

#define REQUIRE(cond, code, msg)                                                                   \
    do                                                                                             \
    {                                                                                              \
        if (!(cond))                                                                               \
            throw ApiError((code), (msg));                                                         \
    } while (0)

// A caller array made visible to the device: device pointers pass through,
// host pointers are staged through a stream-ordered temporary.
struct DevIn
{
    xsb_matrix *h;
    const void *ptr = nullptr;
    void *tmp = nullptr;
    DevIn(xsb_matrix *h_, const void *p, size_t bytes) : h(h_)
    {
        if (bytes == 0 || p == nullptr)
        {
            ptr = p;
            return;
        }
        if (is_device_ptr(p))
            ptr = p;
        else
        {
            tmp = h->dalloc(bytes);
            XSB_CUDA(cudaMemcpyAsync(tmp, p, bytes, cudaMemcpyHostToDevice, h->stream));
            ptr = tmp;
        }
    }
    ~DevIn() { h->dfree(tmp); }
};

// the connectivity of an element batch on the device; the square loop's one array moves once
struct ElementDofs
{
    DevIn r, c;
    ElementBatch batch;
    ElementDofs(xsb_matrix *h, int32_t kr, int32_t kc, i64 ncells, const void *rdofs, const void *cdofs,
                const double *Aloc = nullptr)
        : r(h, rdofs, h->isz() * (size_t)kr * (size_t)ncells),
          c(h, square(kr, kc, rdofs, cdofs) ? nullptr : cdofs, h->isz() * (size_t)kc * (size_t)ncells),
          batch{r.ptr, square(kr, kc, rdofs, cdofs) ? r.ptr : c.ptr, Aloc, kr, kc, ncells}
    {
    }
    static bool square(int32_t kr, int32_t kc, const void *rdofs, const void *cdofs) { return rdofs == cdofs && kr == kc; }
};

struct DevOut
{
    xsb_matrix *h;
    void *user;
    void *ptr = nullptr;
    void *tmp = nullptr;
    size_t bytes;
    DevOut(xsb_matrix *h_, void *p, size_t b) : h(h_), user(p), bytes(b)
    {
        if (p == nullptr || b == 0)
            return;
        if (is_device_ptr(p))
            ptr = p;
        else
        {
            tmp = h->dalloc(b);
            ptr = tmp;
        }
    }
    void finish()
    { // enqueue the copy back; caller synchronises
        if (tmp)
            XSB_CUDA(cudaMemcpyAsync(user, tmp, bytes, cudaMemcpyDeviceToHost, h->stream));
    }
    ~DevOut() { h->dfree(tmp); }
};

u64 read_scalar(xsb_matrix *h, int slot)
{
    XSB_CUDA(cudaMemcpyAsync(h->h_scal + slot, h->d_scal + slot, sizeof(u64), cudaMemcpyDeviceToHost, h->stream));
    h->sync();
    return h->h_scal[slot];
}

void write_scalar(xsb_matrix *h, int slot, u64 v)
{
    h->h_scal[slot] = v;
    XSB_CUDA(cudaMemcpyAsync(h->d_scal + slot, h->h_scal + slot, sizeof(u64), cudaMemcpyHostToDevice, h->stream));
}

void check_tid_flavour(xsb_matrix *h, int32_t tid, int32_t flavour)
{
    REQUIRE(tid >= 0 && tid < h->n_tid, XSB_EINVAL, "tid out of range");
    REQUIRE(flavour >= XSB_UPDATE && flavour <= XSB_ASSIGN, XSB_EINVAL, "unknown insertion flavour");
}

// The multi-partition wrapper refuses A[i,j] = v for an entry that is not in the CSC yet
// (genericmtextendablesparsematrixcsc.jl:63-68: error("use rawupdateindex! for new entries ...")).
// Called on the freshly packed records of an assign batch of a handle with several partition buffers.
void check_mt_assign(xsb_matrix *h, const Rec *recs, i64 count)
{
    write_scalar(h, 2, 0);
    count_missing_records(h->stream, recs, count, h->Ls, h->view(), h->idx64, h->base, h->d_scal + 2, h->lc);
    const u64 missing = read_scalar(h, 2);
    REQUIRE(missing == 0, XSB_EILLEGAL,
            "use rawupdateindex! for new entries into a matrix with several partition buffers (" +
                std::to_string(missing) + " assigned positions are not in the CSC); batch rejected");
}

bool runs_eligible(const xsb_matrix *h);

// fixed-capacity exchange: what the unpack kernels found (h_route[2 kMaxRanks ..] was copied and the stream synchronised)
void check_exchange(xsb_matrix *h)
{
    const u64 flags = h->h_route[2 * kMaxRanks];
    REQUIRE((flags & 8ull) == 0, XSB_ESTATE,
            "peer exchange: a rank did not deliver (or take) its block in time (XSB_PEER_TIMEOUT_MS); the ranks are out of step");
    REQUIRE((flags & 32ull) == 0, XSB_ESTATE,
            "a record owned by another rank was staged after xsb_route_pack_peer: it would never reach its owner");
    REQUIRE((flags & 4ull) == 0, XSB_EINVAL, "a received block carries no header: capacities of sender and receiver differ");
    REQUIRE((flags & 2ull) == 0, XSB_ESTATE,
            "a bucket of the exchange did not fit its block: records were cut off; reset! and repeat the step with larger "
            "capacities (or use xsb_route_count / xsb_route_prepare / xsb_route_finish)");
    REQUIRE((flags & 1ull) == 0, XSB_EBOUNDS, "a received record is not owned by this rank");
    if (flags & 16ull)
        h->has_assign = true; // a received record is an A[i,j] = v: ordered fold
    // the old paths need the true sizes of the regions
    h->n_low = (i64)h->h_route[2 * kMaxRanks + 1];
    h->n_high = (i64)h->h_route[2 * kMaxRanks + 2];
}

// flush! on grouped chunks (xsb_runs.cu): the product path.  Returns false -- with the staged records and the
// resident CSC untouched (apart from the in-place grouping of chunks, which keeps every entry's insertions in
// stream order) -- when this flush has to take another path: a stream without column locality, a column too long
// or too rich for one thread.
// The fold is an exact left fold in insertion order, so both summation modes take it alike.
bool runs_flush(xsb_matrix *h, StageTimer *tp, int64_t *nnz_out)
{
    cudaStream_t s = h->stream;
    Stage &st = h->stage[0];
    const i64 count = st.count;
    if (!runs_eligible(h) || !runs_supported(h->L, (u64)count, h->n) || !colfold_supported(h->L, (u64)count, h->n))
        return false;
    Rec *buf = st.buf + st.front;
    // ---- the run index: what the producers published, plus the regions they left in stream order
    if (tp)
        tp->begin(s);
    if (h->runs.dead || !h->runs.ws)
    {
        if (h->runs.ws)
            XSB_CUDA(cudaMemsetAsync(h->runs.ws, 0, 256, s));
        h->runs.nchunks = 0;
        h->runs.sorted_end = 0;
        h->runs.dead = false;
    }
    h->runs_reserve(count);
    RunRegions reg{0xffffffffu, 0xffffffffu};
    i64 bounds[4] = {h->runs.sorted_end, count, count, count};
    if (h->L.ownerbits > 0 || h->nranks > 0)
    { // [own | from lower ranks | from higher ranks]: a chunk never straddles two regions
        const i64 low_end = h->low_end < 0 ? count : h->low_end;
        const i64 own_end = h->routed ? h->own_end : count;
        bounds[1] = std::max(own_end, h->runs.sorted_end);
        bounds[2] = std::max(low_end, bounds[1]);
        reg.own_end = (u32)bounds[1];
        reg.low_end = (u32)bounds[2];
    }
    {
        u64 extra = 0;
        for (int r = 0; r < 3; ++r)
            extra += chunk_sort_chunks((u64)(bounds[r + 1] - bounds[r]));
        if ((u64)h->runs.nchunks + extra > (u64)h->runs.cap_chunks)
        { // many small batches filled the chunk table: rebuild the index from scratch, in whole chunks
            XSB_CUDA(cudaMemsetAsync(h->runs.ws, 0, 256, s));
            h->runs.nchunks = 0;
            h->runs.sorted_end = 0;
            bounds[0] = 0;
        }
    }
    const RunTarget rt = run_target(h->runs.ws, (u64)h->runs.cap_records, h->L);
    h->stats_precounted = h->runs.sorted_end;
    for (int r = 0; r < 3; ++r)
    {
        if (bounds[r + 1] > bounds[r])
        {
            chunk_sort(s, buf, (u64)bounds[r], (u64)bounds[r + 1], rt, h->runs.nchunks, h->lc);
            h->runs.nchunks += chunk_sort_chunks((u64)(bounds[r + 1] - bounds[r]));
        }
    }
    h->runs.sorted_end = count;
    XSB_CUDA(cudaMemcpyAsync(h->h_scal + 4, rt.counters, sizeof(u64), cudaMemcpyDeviceToHost, s));
    if (h->fixed_exchange)
        XSB_CUDA(cudaMemcpyAsync(h->h_route + 2 * kMaxRanks, h->d_route, sizeof(u64) * 3, cudaMemcpyDeviceToHost, s));
    if (tp)
        tp->end(s, &StageTimes::gcount);
    h->sync();
    if (h->fixed_exchange)
        check_exchange(h);
    const u32 npairs = (u32)(h->h_scal[4] & 0xffffffffull);
    const u32 flags = (u32)(h->h_scal[4] >> 32);
    h->stats_pairs = (i64)npairs;
    if (flags != 0u || npairs > rt.cap)
    { // a chunk with too many distinct columns: this stream has no column locality
        if (h->grouping == XSB_GROUPING_AUTO)
            h->grouping_misses++;
        h->runs.dead = true;
        return false;
    }
    // ---- every column's runs into its bucket
    if (tp)
        tp->begin(s);
    void *ws = h->dalloc(runs_workspace_bytes((u64)npairs, h->n));
    runs_bucket(s, rt, h->runs.nchunks, npairs, h->n, h->L, reg, ws, h->lc);
    if (tp)
        tp->end(s, &StageTimes::sort);
    // ---- merge: resident column + runs -> new column
    const i64 nnz_old = h->nnz;
    const size_t ub = (size_t)(nnz_old + count); // entries the new matrix can hold at most
    const size_t rv_bytes = (h->isz() * ub + 255) & ~(size_t)255;
    void *new_colptr = h->dalloc(h->isz() * (size_t)(h->n + 1));
    unsigned char *store = static_cast<unsigned char *>(h->dalloc(rv_bytes + 8 * ub + 32));
    void *new_rowval = store;
    double *new_nzval = reinterpret_cast<double *>(store + rv_bytes);
    const u64 avg = (u64)count / (u64)std::max<i64>(1, h->n);
    const u32 maxlen = (u32)std::max<u64>(1024, 8 * avg);
    int level = h->fold_hint ? runs_level_for(h->fold_hint) : (nnz_old > 0 ? runs_level_for((u32)std::min<i64>(64, 2 * nnz_old / std::max<i64>(1, h->n) + 4))
                                                                           : (avg < 14 ? 0 : (avg < 40 ? 2 : 3)));
    i64 nnz_new = -1;
    bool ok = false;
    if (tp)
        tp->begin(s);
    for (bool first = true;; first = false)
    {
        runs_fold(s, buf, h->L, h->n, h->idx64, h->base, h->view(), ws, npairs, level, maxlen, new_rowval, new_nzval,
                  new_colptr, h->d_scal + 0, reinterpret_cast<u32 *>(h->d_scal + 6), reinterpret_cast<u32 *>(h->d_scal + 7),
                  first, h->has_assign, h->lc);
        XSB_CUDA(cudaMemcpyAsync(h->h_scal + 6, h->d_scal + 6, 2 * sizeof(u64), cudaMemcpyDeviceToHost, s));
        nnz_new = (i64)read_scalar(h, 0);
        const u32 redo = (u32)h->h_scal[6];
        const u32 maxd = (u32)h->h_scal[7];
        if (redo == 0u)
        {
            if (maxd)
                h->fold_hint = maxd;
            ok = true;
            break;
        }
        if ((redo & 6u) || level >= 3)
            break; // a very long column, or one too rich for the largest table
        level = std::max(level + 1, maxd > 0 ? runs_level_for(maxd) : 0); // the next table shape
    }
    if (tp)
        tp->end(s, &StageTimes::fold);
    h->dfree(ws);
    if (!ok)
    {
        h->dfree(new_colptr);
        h->dfree(store);
        h->runs_misses++; // two in a row: this handle's producers stop grouping, its flushes take the other paths
        return false;
    }
    h->runs_misses = 0;
    h->grouping_misses = 0;
    // ---- the new matrix replaces the resident one; the staging buffer stays where it is
    h->dfree(h->colptr);
    h->dfree(h->csc_store);
    h->colptr = new_colptr;
    h->csc_store = store;
    h->csc_store_bytes = rv_bytes + 8 * ub + 32;
    h->rowval = new_rowval;
    h->nzval = new_nzval;
    h->nnz = nnz_new;
    const size_t exact = (h->isz() + 8) * (size_t)nnz_new;
    if (h->csc_store_bytes > exact + h->shrink_surplus_bytes)
        h->shrink_store();
    h->clear_staging(false);
    if (nnz_new != nnz_old)
        h->drop_frozen();
    *nnz_out = nnz_new;
    return true;
}

int32_t do_flush(xsb_matrix *h, int32_t mode, int32_t combine, int64_t *nnz_out, int32_t *pattern_changed)
{
    REQUIRE(mode == XSB_DETERMINISTIC || mode == XSB_FAST, XSB_EINVAL, "unknown summation mode");
    REQUIRE(combine == XSB_COMBINE_SEED || combine == XSB_COMBINE_ADD, XSB_EINVAL, "unknown combine mode");
    const i64 n_ins = h->pending();
    h->drop_half_freeze();
    h->lc.in_flush = 0;
    h->alloc_ms = 0.f;
    std::memset(&h->stats, 0, sizeof(h->stats));
    h->stats.nnz_old = h->nnz;
    h->stats.nnz_new = h->nnz;
    if (n_ins == 0)
    { // flush! is a no-op without new entries: extendable.jl:249
        if (h->nranks > 0)
            h->clear_staging(false); // a rank that staged and received nothing: forget the routing state of this step
        if (nnz_out)
            *nnz_out = h->nnz;
        if (pattern_changed)
            *pattern_changed = 0;
        return XSB_OK;
    }
    REQUIRE(h->nranks == 0 || h->routed, XSB_ESTATE,
            "slab handle: route the staged records (xsb_route_prepare/xsb_route_finish) before flush");
    cudaStream_t s = h->stream;
    StageTimer timer;
    StageTimer *tp = h->profiling ? &timer : nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (tp)
    {
        XSB_CUDA(cudaEventCreate(&e0));
        XSB_CUDA(cudaEventCreate(&e1));
        XSB_CUDA(cudaEventRecord(e0, s));
    }

    const i64 nnz_old = h->nnz;
    h->stats_pairs = 0;
    h->stats_direct = 0;
    h->stats_preagg = 0;
    h->stats_precounted = 0;
    if (combine == XSB_COMBINE_SEED && !(mode == XSB_FAST && h->preagg))
    { // ---- the product path: grouped chunks, records never move, resident CSC merged column by column
        int64_t nnz_runs = 0;
        const i64 foreign_runs = h->foreign + h->n_pad;
        if (runs_flush(h, tp, &nnz_runs))
        {
            h->stats.n_inserted = n_ins - foreign_runs;
            h->stats.nnz_old = nnz_old;
            h->stats.nnz_new = nnz_runs;
            h->stats.column_path = 4;
            h->stats.kernel_launches = h->lc.in_flush;
            h->stats.ms_host_alloc = h->alloc_ms;
            h->stats.group_pairs = h->stats_pairs;
            h->stats.direct_fold = 1;
            h->stats.precounted = n_ins > 0 ? (float)((double)h->stats_precounted / (double)n_ins) : 0.f;
            if (tp)
            {
                XSB_CUDA(cudaEventRecord(e1, s));
                h->sync();
                StageTimes t;
                timer.collect(t);
                cudaEventElapsedTime(&t.total, e0, e1);
                cudaEventDestroy(e0);
                cudaEventDestroy(e1);
                h->stats.ms_total = t.total;
                h->stats.ms_histogram = t.gcount;
                h->stats.ms_group_count = t.gcount;
                h->stats.ms_pair_sort = t.sort;
                h->stats.ms_sort = t.sort;
                h->stats.ms_fold = t.fold;
                h->stats.ms_reduce = t.fold;
            }
            if (nnz_out)
                *nnz_out = nnz_runs;
            if (pattern_changed)
                *pattern_changed = (nnz_runs != nnz_old) ? 1 : 0; // the pattern only ever grows
            return XSB_OK;
        }
        if (tp)
        { // spans of the abandoned attempt stay in the totals of this flush
            h->sync();
        }
    }
    // slab handles keep every region of the buffer chunk aligned: a gap of skipped records follows the old entries
    const i64 front = (h->L.ownerbits > 0 && h->n_tid == 1) ? xsb_matrix::chunk_up(nnz_old) : nnz_old;
    i64 total = front + n_ins; // records the flush works on (shrinks if XSB_FAST pre-aggregates)
    const i64 total_cap = total;
    h->stats_pairs = 0;
    h->stats_direct = 0;
    h->stats_preagg = 0;
    h->stats_precounted = 0;
    REQUIRE((u64)total < (1ull << 40), XSB_EINVAL, "too many staged entries");

    // ---- input buffer A = [old CSC as records | staged records in tid order]
    Rec *A = nullptr;
    bool a_is_stage0 = false;
    if (tp)
        tp->begin(s);
    if (h->n_tid == 1)
    {
        A = h->stage[0].buf; // front was reserved when staging began
        REQUIRE(h->stage[0].front == front && h->stage[0].cap >= total, XSB_ESTATE, "staging buffer out of step");
        a_is_stage0 = true;
    }
    else
    {
        A = static_cast<Rec *>(h->dalloc(sizeof(Rec) * (size_t)total));
        i64 off = nnz_old;
        for (auto &st : h->stage)
        {
            if (st.count)
                XSB_CUDA(cudaMemcpyAsync(A + off, st.buf + st.front, sizeof(Rec) * (size_t)st.count,
                                         cudaMemcpyDeviceToDevice, s));
            off += st.count;
        }
    }
    if (tp)
        tp->end(s, &StageTimes::other);
    if (tp)
        tp->begin(s);
    expand_csc_records(s, h->view(), h->n, h->idx64, h->base, h->L, A, h->lc);
    if (front > nnz_old)
        route_fill_skipped(s, A + nnz_old, front - nnz_old, h->L, h->lc);
    if (tp)
        tp->end(s, &StageTimes::expand);

    Rec *B = static_cast<Rec *>(h->dalloc(sizeof(Rec) * (size_t)total));
    struct
    {
        Rec *p;
        i64 cap;
    } bufs[2] = {{A, a_is_stage0 ? h->stage[0].cap : total_cap}, {B, total_cap}};
    auto cap_of = [&](const Rec *p) { return p == bufs[0].p ? bufs[0].cap : bufs[1].cap; };

    // ---- XSB_FAST: accumulate-on-insert inside windows of the staged stream (xsb_preagg.cu); the
    // partial sums replace the staged records, the old entries ride in front of them as before
    bool preagged = false;
    if (mode == XSB_FAST && !h->has_assign && !h->fixed_exchange && combine == XSB_COMBINE_SEED && h->preagg && h->preagg_misses < 2 &&
        n_ins >= 4096)
    {
        if (tp)
            tp->begin(s);
        XSB_CUDA(cudaMemsetAsync(h->d_scal + 3, 0, sizeof(u64), s));
        if (nnz_old)
            XSB_CUDA(cudaMemcpyAsync(B, A, sizeof(Rec) * (size_t)nnz_old, cudaMemcpyDeviceToDevice, s));
        preaggregate_records(s, A + front, (u64)n_ins, h->L, B + nnz_old, h->d_scal + 3, h->lc);
        if (tp)
            tp->end(s, &StageTimes::preagg);
        const i64 kept = (i64)read_scalar(h, 3);
        h->stats_preagg = kept;
        // a stream that hardly repeats itself inside a window gains nothing: stop trying on this handle
        h->preagg_misses = (kept * 4 > n_ins * 3) ? h->preagg_misses + 1 : 0;
        total = nnz_old + kept;
        std::swap(A, B);
        preagged = true;
    }
    KeyLayout Lf = h->L; // layout the fold sees: partial sums are not tied to a partition
    if (preagged)
        Lf.tidbits = 0;
    const size_t ws_bytes = std::max(sort_workspace_bytes((u64)total), reduce_workspace_bytes((u64)total, h->n));
    void *ws = h->dalloc(ws_bytes);
    // slab handles: records owned (and already received) by other ranks are still in the buffer.  The
    // grouping kernels skip them by their owner bits; every other path first drops them with one
    // stable partition on the owner bits.
    const i64 foreign = h->foreign + h->n_pad;
    if (h->fixed_exchange)
    { // capacity-sized regions: the true sizes (and what the unpack kernels found) are on the device
        XSB_CUDA(cudaMemcpyAsync(h->h_route + 2 * kMaxRanks, h->d_route, sizeof(u64) * 3, cudaMemcpyDeviceToHost, s));
        h->sync();
        check_exchange(h);
    }
    const i64 n_low = h->n_low, n_high = h->n_high;
    bool tomb = h->L.ownerbits > 0 && (foreign > 0 || front > nnz_old || h->fixed_exchange);
    // the fold must meet the records of a column as [old | lower ranks | own | higher ranks]
    ChunkOrder ord{};
    const ChunkOrder *pord = nullptr;
    if (h->L.ownerbits > 0 && !preagged && n_low > 0)
    {
        const i64 W = group_chunk_records();
        const i64 low_end = h->low_end < 0 ? h->stage[0].count : h->low_end;
        ord.c_old = (u32)(front / W);
        ord.c_own = (u32)((front + h->own_end) / W);
        ord.c_low = (u32)((front + low_end + W - 1) / W);
        pord = &ord;
    }
    auto drop_foreign = [&]() {
        if (!tomb)
            return;
        u64 counts[kRadix] = {0};
        partition_records(s, A, B, (u64)total, h->L.ownershift(), h->L.ownerbits, ws, h->lc, counts);
        u64 off = 0;
        for (int r = 0; r < h->rank; ++r)
            off += counts[r];
        const i64 mine = (i64)counts[h->rank];
        const Rec *src = B + off;
        if (preagged || n_low == 0)
        {
            if (mine > 0)
                XSB_CUDA(cudaMemcpyAsync(A, src, sizeof(Rec) * (size_t)mine, cudaMemcpyDeviceToDevice, s));
        }
        else
        { // [old | own | low | high] -> [old | low | own | high]
            const i64 own = mine - nnz_old - n_low - n_high;
            auto cp = [&](i64 dst, i64 from, i64 cnt) {
                if (cnt > 0)
                    XSB_CUDA(cudaMemcpyAsync(A + dst, src + from, sizeof(Rec) * (size_t)cnt, cudaMemcpyDeviceToDevice, s));
            };
            cp(0, 0, nnz_old);
            cp(nnz_old, nnz_old + own, n_low);
            cp(nnz_old + n_low, nnz_old, own);
            cp(nnz_old + n_low + own, nnz_old + own + n_low, n_high);
        }
        total = mine;
        tomb = false;
    };

    void *new_colptr = h->dalloc(h->isz() * (size_t)(h->n + 1));
    Rec *sorted = nullptr, *spare = nullptr;
    void *new_rowval = nullptr;
    double *new_nzval = nullptr;
    void *new_store = nullptr; // allocation that holds rowval|nzval after the flush
    size_t new_store_bytes = 0;
    i64 nnz_new = -1;
    SortPlan plan{};
    int passes_run = 0;
    int path = 0; // 0: (col,row) sort + flat reduction, 2: column sort + hash fold, 3: grouping + hash fold
    if (h->strategy == XSB_STRATEGY_AUTO && colfold_supported(h->L, (u64)total, h->n))
    {
        // ---- sort by column only; the per-column kernel folds duplicates through a hash table
        void *cws = h->dalloc(colfold_workspace_bytes((u64)total, h->n));
        bool grouped = false;
        if (h->grouping != XSB_GROUPING_OFF && (h->grouping == XSB_GROUPING_ON || h->grouping_misses < 2) &&
            group_supported(h->L, (u64)total, h->n))
        { // two-pass grouping through sparse per-chunk column histograms (streams with column locality)
            void *gws = h->dalloc(group_workspace_bytes((u64)total, h->n));
            u32 *nzcol, *nzstart;
            u64 *totals;
            colfold_lists(cws, (u64)total, h->n, &nzcol, &nzstart, &totals);
            int pair_passes = 0;
            u64 npairs = 0;
            grouped = group_by_column(s, A, B, (u64)total, h->n, h->L, gws, ws, nzcol, nzstart, totals, h->h_scal + 4, h->lc,
                                      tp, &pair_passes, &npairs, tomb ? h->L.ownershift() : -1, (u32)h->rank, pord);
            h->dfree(gws);
            h->stats_pairs = (i64)npairs;
            if (grouped)
            {
                sorted = B;
                spare = A;
                passes_run += pair_passes;
                h->grouping_misses = 0;
            }
            else if (h->grouping == XSB_GROUPING_AUTO)
                h->grouping_misses++; // two misses in a row: stop trying on this handle
        }
        if (!grouped)
        {
            drop_foreign();
            colfold_clear_counts(s, cws, (u64)total, h->n);
            plan = make_sort_plan(h->L.low + h->L.rowbits, h->L.colbits);
            sorted = radix_sort_records(s, A, B, (u64)total, plan, ws, h->lc, tp, colfold_counts(cws, (u64)total, h->n),
                                        h->L.low + h->L.rowbits, h->L.colbits);
            passes_run += plan.npasses;
            spare = (sorted == A) ? B : A;
        }
        bool direct = false, lists_ready = grouped;
        if (!h->no_direct_fold && colfold_direct_supported(Lf, combine, !h->has_assign))
        { // one pass: fold every column and write rowval / nzval / colptr in place (the spare buffer)
            new_rowval = spare;
            new_nzval = reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(spare) + 8 * (size_t)total);
            colfold_direct(s, sorted, (u64)total, Lf, h->n, h->idx64, h->base, new_rowval, new_nzval, new_colptr, cws,
                           h->d_scal + 0, reinterpret_cast<u32 *>(h->d_scal + 6), grouped,
                           reinterpret_cast<u32 *>(h->d_scal + 7), h->fold_hint, h->lc, tp);
            XSB_CUDA(cudaMemcpyAsync(h->h_scal + 6, h->d_scal + 6, 2 * sizeof(u64), cudaMemcpyDeviceToHost, s));
            nnz_new = (i64)read_scalar(h, 0);
            const u32 redo = (u32)h->h_scal[6];
            if ((u32)h->h_scal[7])
                h->fold_hint = (u32)h->h_scal[7];
            lists_ready = true;
            if (redo == 0u)
            {
                direct = true;
                new_store = spare;
                new_store_bytes = sizeof(Rec) * (size_t)total;
                path = grouped ? 3 : 2;
                h->stats_direct = 1;
            }
            else if (redo & 6u)
                h->no_direct_fold = true; // long or very rich columns: this handle parks and compacts from now on
        }
        if (!direct)
        {
            colfold_reduce(s, sorted, (u64)total, Lf, combine, !h->has_assign, h->n, h->idx64, h->base, spare,
                           new_colptr, cws, h->d_scal + 0, reinterpret_cast<u32 *>(h->d_scal + 6), lists_ready,
                           reinterpret_cast<u32 *>(h->d_scal + 7), h->fold_hint, h->lc, tp);
            path = grouped ? 3 : 2;
            XSB_CUDA(cudaMemcpyAsync(h->h_scal + 6, h->d_scal + 6, 2 * sizeof(u64), cudaMemcpyDeviceToHost, s));
            nnz_new = (i64)read_scalar(h, 0);
            if ((u32)h->h_scal[7])
                h->fold_hint = (u32)h->h_scal[7]; // distinct rows per column: picks the next flush's table size
            if ((u32)h->h_scal[6] == 0u)
            {
                const size_t rv_bytes = (h->isz() * (size_t)nnz_new + 15) & ~(size_t)15;
                new_store_bytes = rv_bytes + 8 * (size_t)nnz_new;
                new_store = h->dalloc(new_store_bytes);
                new_rowval = new_store;
                new_nzval = reinterpret_cast<double *>(static_cast<unsigned char *>(new_store) + rv_bytes);
                colfold_compact(s, spare, (u64)total, h->n, h->idx64, h->base, new_colptr, new_rowval, new_nzval, cws,
                                h->lc, tp);
                h->dfree(spare); // back to the buffer cache
            }
            else
            { // a group of columns too rich for the in-warp table: finish with the general sort (records are intact)
                A = sorted;
                B = spare;
                path = 0;
            }
        }
        h->dfree(cws);
    }
    if (path == 0)
    {
        drop_foreign();
        // ---- sort by (col,row), then a flat segmented reduction
        plan = make_sort_plan(h->L.low, h->L.sortbits());
        sorted = radix_sort_records(s, A, B, (u64)total, plan, ws, h->lc, tp);
        passes_run += plan.npasses;
        spare = (sorted == A) ? B : A;
        new_rowval = spare;
        new_nzval = reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(spare) + 8 * (size_t)total);
        reduce_emit_csc(s, sorted, (u64)total, h->L, combine, mode, !h->has_assign, h->n, h->idx64, h->base,
                        new_rowval, new_nzval, new_colptr, ws, h->d_scal + 0, h->lc, tp);
        nnz_new = (i64)read_scalar(h, 0);
        new_store = spare;
        new_store_bytes = sizeof(Rec) * (size_t)total;
    }
    const bool column_path = path != 0;

    if (tp)
        tp->begin(s);
    h->dfree(ws);
    h->dfree(h->colptr);
    h->dfree(h->csc_store);
    h->colptr = new_colptr;
    h->csc_store = new_store;
    h->csc_store_bytes = new_store_bytes;
    h->rowval = new_rowval;
    h->nzval = new_nzval;
    h->nnz = nnz_new;

    // The CSC stays in the (duplicate-count sized) ping-pong buffer: copying it into an exact
    // allocation costs 32 B per entry of HBM traffic.  Only a large surplus is given back.
    const size_t exact = (h->isz() + 8) * (size_t)nnz_new;
    if (h->csc_store_bytes > exact + h->shrink_surplus_bytes)
        h->shrink_store();

    // the buffer that held the sorted records is recycled as the next staging buffer
    if (a_is_stage0)
    {
        h->stage[0].buf = sorted;
        h->stage[0].cap = cap_of(sorted);
    }
    else
        h->dfree(sorted);
    h->clear_staging(false);
    if (nnz_new != nnz_old)
        h->drop_frozen();
    if (tp)
        tp->end(s, &StageTimes::other);

    h->stats.n_inserted = n_ins - foreign;
    h->stats.nnz_old = nnz_old;
    h->stats.nnz_new = nnz_new;
    h->stats.sort_passes = passes_run;
    h->stats.sort_bits = column_path ? h->L.colbits : h->L.sortbits();
    h->stats.column_path = path;
    h->stats.kernel_launches = h->lc.in_flush;
    h->stats.ms_host_alloc = h->alloc_ms;
    h->stats.group_pairs = h->stats_pairs;
    h->stats.direct_fold = h->stats_direct;
    h->stats.preagg_records = h->stats_preagg;
    h->stats.precounted = n_ins > 0 ? (float)((double)h->stats_precounted / (double)n_ins) : 0.f;
    if (tp)
    {
        XSB_CUDA(cudaEventRecord(e1, s));
        h->sync();
        StageTimes t;
        timer.collect(t);
        cudaEventElapsedTime(&t.total, e0, e1);
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        h->stats.ms_total = t.total;
        h->stats.ms_expand = t.expand;
        h->stats.ms_histogram = t.histogram + t.gcount;
        h->stats.ms_sort = t.sort + t.gscatter;
        h->stats.ms_reduce = t.reduce + t.fold + t.compact;
        h->stats.ms_group_count = t.gcount;
        h->stats.ms_pair_sort = path == 3 ? t.histogram + t.sort : 0.f;
        h->stats.ms_group_scatter = t.gscatter;
        h->stats.ms_fold = t.fold;
        h->stats.ms_compact = t.compact;
        h->stats.ms_preagg = t.preagg;
        h->stats.ms_colptr = t.colptr;
        h->stats.ms_other = t.other;
    }
    if (nnz_out)
        *nnz_out = nnz_new;
    if (pattern_changed)
        *pattern_changed = (nnz_new != nnz_old) ? 1 : 0; // the pattern only ever grows
    return XSB_OK;
}

// slab handles: fills the staged records up to a whole number of chunks with records the flush skips
void pad_region(xsb_matrix *h)
{
    if (h->L.ownerbits == 0)
        return;
    Stage &st = h->stage[0];
    const i64 end = st.front + st.count;
    const i64 pad = xsb_matrix::chunk_up(end) - end;
    if (pad == 0)
        return;
    h->ensure_stage(0, pad);
    route_fill_skipped(h->stream, st.buf + st.front + st.count, pad, h->L, h->lc);
    st.count += pad;
    h->n_pad += pad;
}

// room for `count` generated records in partition tid; returns where to write them
Rec *begin_emit(xsb_matrix *h, int32_t tid, int32_t flavour, i64 count)
{
    check_tid_flavour(h, tid, flavour);
    REQUIRE(count >= 0, XSB_EINVAL, "negative count");
    REQUIRE(!h->routed, XSB_ESTATE, "routed records are pending: flush before inserting again");
    h->drop_half_freeze();
    h->ensure_stage(tid, count);
    Stage &st = h->stage[tid];
    return st.buf + st.front + st.count;
}

// may this handle's flush work on grouped chunks (xsb_runs.cu)?
bool runs_eligible(const xsb_matrix *h)
{
    return h->n_tid == 1 && h->strategy == XSB_STRATEGY_AUTO && h->grouping != XSB_GROUPING_OFF &&
           (h->grouping == XSB_GROUPING_ON || (h->grouping_misses < 2 && h->runs_misses < 2));
}

// Called after begin_emit: may the producer of the next `count` records of partition `tid` group its chunks
// (xsb_chunk.cuh) and publish their runs?  `chunks` = chunks it will append.  On success *rt / *chunk0 / *pos0
// say where the runs go, the id of the first chunk and the position of the first record.
bool runs_begin(xsb_matrix *h, int32_t tid, i64 count, u32 chunks, RunTarget *rt, u32 *chunk0, u32 *pos0)
{
    if (!h->precount || tid != 0 || !runs_eligible(h) || count <= 0)
        return false;
    Stage &st = h->stage[0];
    if (h->runs.dead || st.count != h->runs.sorted_end)
        return false; // something staged before was not grouped: the flush groups the rest
    if (!runs_supported(h->L, (u64)(st.count + count), h->n))
        return false;
    h->runs_reserve(std::max<i64>(st.cap - st.front, st.count + count));
    if ((u64)h->runs.nchunks + chunks > (u64)h->runs.cap_chunks)
        return false;
    *rt = run_target(h->runs.ws, (u64)h->runs.cap_records, h->L);
    *chunk0 = h->runs.nchunks;
    *pos0 = (u32)st.count;
    return true;
}

void runs_end(xsb_matrix *h, i64 count, u32 chunks)
{
    h->runs.nchunks += chunks;
    h->runs.sorted_end += count;
}

void end_emit(xsb_matrix *h, int32_t tid, int32_t flavour, i64 count)
{
    h->stage[tid].count += count;
    if (flavour == XSB_ASSIGN)
        h->has_assign = true;
}

// the limits of an element batch: kr, kc in [1, 64]; its kr kc ncells calls stay below 2^63
i64 element_calls(int32_t kr, int32_t kc, int64_t ncells)
{
    REQUIRE(kr >= 1 && kr <= 64 && kc >= 1 && kc <= 64, XSB_EINVAL,
            kr == kc ? "element size k must be in [1, 64]" : "element sizes kr and kc must be in [1, 64]");
    REQUIRE(ncells >= 0, XSB_EINVAL, "negative element count");
    REQUIRE(ncells <= INT64_MAX / ((i64)kr * kc), XSB_EINVAL, kr == kc ? "k^2 * ncells overflows" : "kr * kc * ncells overflows");
    return (i64)kr * kc * ncells;
}

// xsb_freeze_pattern / xsb_freeze_elements
void freeze_check(xsb_matrix *h, i64 count)
{
    REQUIRE(count >= 0 && (u64)count < (1ull << 32), XSB_EINVAL, "count must be below 2^32");
    REQUIRE(h->pending() == 0, XSB_ESTATE, "flush! before freezing the pattern");
}

// `lookup(slot)` finds the nzval slot of every call of the stream; the entry -> nzval map is built from them
template <class Lookup> int32_t freeze_impl(xsb_matrix *h, i64 count, Lookup &&lookup)
{
    cudaStream_t s = h->stream;
    i64 *slot = static_cast<i64 *>(h->dalloc(8 * (size_t)count));
    write_scalar(h, 2, 0);
    write_scalar(h, 3, ~0ull);
    lookup(slot);
    const u64 oob = read_scalar(h, 3);
    const u64 missing = read_scalar(h, 2);
    if (oob != ~0ull || missing != 0)
    {
        h->dfree(slot);
        if (oob != ~0ull)
            throw ApiError(XSB_EBOUNDS, "BoundsError: position " + std::to_string(oob) + " is outside the matrix");
        throw ApiError(XSB_EILLEGAL, std::to_string(missing) + " positions are not in the frozen pattern");
    }
    Rec *A = static_cast<Rec *>(h->dalloc(sizeof(Rec) * (size_t)count));
    Rec *B = static_cast<Rec *>(h->dalloc(sizeof(Rec) * (size_t)count));
    void *ws = h->dalloc(sort_workspace_bytes((u64)count));
    slots_to_records(s, slot, count, A, h->lc);
    const SortPlan plan = make_sort_plan(0, ceil_log2(std::max<i64>(h->nnz, 2)));
    Rec *sorted = radix_sort_records(s, A, B, (u64)count, plan, ws, h->lc, nullptr);
    h->f_perm = static_cast<u32 *>(h->dalloc(4 * (size_t)std::max<i64>(count, 1)));
    h->f_segstart = static_cast<u32 *>(h->dalloc(4 * (size_t)(h->nnz + 1)));
    h->f_slot = static_cast<u32 *>(h->dalloc(4 * (size_t)std::max<i64>(count, 1)));
    build_frozen_map(s, sorted, count, h->nnz, h->f_perm, h->f_segstart, h->f_slot, h->lc);
    h->dfree(A);
    h->dfree(B);
    h->dfree(ws);
    h->dfree(slot);
    h->f_count = count;
    h->frozen = true;
    h->sync();
    return XSB_OK;
}

// the calls of a stream frozen across column slabs
void slab_freeze_check(xsb_matrix *h)
{
    REQUIRE(h, XSB_EINVAL, "NULL handle");
    REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
    REQUIRE(h->pending() == 0, XSB_ESTATE, "insertions are pending: flush! first");
}

// xsb_freeze_slab / xsb_freeze_slab_elements: `classify(slot, tags)` resolves the own positions and tags every
// position with its owner; the stable copy-out of the routing (xsb_route.cu, on a layout whose owner field starts at
// bit 32 above the stream index) gathers the foreign ones destination after destination.  Leaves the handle half
// frozen.
template <class Classify> int32_t freeze_slab_impl(xsb_matrix *h, i64 count, int64_t *send_counts, Classify &&classify)
{
    cudaStream_t s = h->stream;
    const size_t room = (size_t)std::max<i64>(count, 1);
    i64 *slot = static_cast<i64 *>(h->dalloc(8 * room));
    Rec *tags = static_cast<Rec *>(h->dalloc(sizeof(Rec) * room));
    write_scalar(h, 2, 0);
    write_scalar(h, 3, ~0ull);
    classify(slot, tags);
    const u64 oob = read_scalar(h, 3);
    const u64 missing = read_scalar(h, 2);
    if (oob != ~0ull || missing != 0)
    {
        h->dfree(slot);
        h->dfree(tags);
        if (oob != ~0ull)
            throw ApiError(XSB_EBOUNDS, "BoundsError: position " + std::to_string(oob) + " of the stream is outside the matrix");
        throw ApiError(XSB_EILLEGAL, std::to_string(missing) + " positions in this rank's columns are not in the frozen pattern");
    }
    KeyLayout Lr = h->L; // owner field at bit 32, the stream index below it
    Lr.low = 32;
    Lr.tidbits = Lr.rowbits = Lr.colbits = 0;
    void *ws = h->dalloc(route_workspace_bytes((u64)room, h->nranks));
    u64 counts[kMaxRanks] = {0};
    route_count(s, tags, (u64)count, Lr, ws, counts, h->lc);
    i64 foreign = 0;
    for (int r = 0; r < h->nranks; ++r)
        if (r != h->rank)
            foreign += (i64)counts[r];
    const size_t froom = (size_t)std::max<i64>(foreign, 1);
    Rec *gathered = static_cast<Rec *>(h->dalloc(sizeof(Rec) * froom));
    route_extract(s, tags, (u64)count, Lr, ws, counts, gathered, h->lc);
    h->fs_send_idx = static_cast<u32 *>(h->dalloc(4 * froom));
    h->fs_send_pos = static_cast<u64 *>(h->dalloc(8 * froom));
    slab_split(s, gathered, foreign, h->fs_send_idx, h->fs_send_pos, h->lc);
    h->dfree(gathered);
    h->dfree(ws);
    h->dfree(tags);
    h->fs_slot = slot;
    for (int r = 0; r < h->nranks; ++r)
    {
        h->fs_send[r] = (i64)counts[r];
        if (send_counts)
            send_counts[r] = (int64_t)counts[r];
    }
    h->fs_foreign = foreign;
    h->f_count = count;
    h->fs_state = 1;
    h->sync();
    return XSB_OK;
}

} // namespace

extern "C" {

int32_t xsb_version(void) { return XSB_VERSION; }

int32_t xsb_device_count(int32_t *count)
{
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        g_err = std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e);
        if (count)
            *count = 0;
        return XSB_ECUDA;
    }
    if (count)
        *count = c;
    return XSB_OK;
}

static int32_t create_impl(int64_t m, int64_t n_global, int32_t nranks, int32_t rank, const int64_t *splits,
                           int32_t val_type, int32_t idx_type, int32_t index_base, int32_t n_tid, int32_t device,
                           xsb_matrix **out)
{
    if (out)
        *out = nullptr;
    xsb_matrix *h = nullptr;
    int32_t rc = guard(nullptr, [&]() -> int32_t {
        REQUIRE(out != nullptr, XSB_EINVAL, "out is NULL");
        REQUIRE(m >= 1 && n_global >= 1, XSB_EINVAL, "matrix dimensions must be >= 1");
        REQUIRE(val_type == XSB_F64, XSB_EINVAL, "only Float64 values are supported");
        REQUIRE(idx_type == XSB_I32 || idx_type == XSB_I64, XSB_EINVAL, "idx_type must be XSB_I32 or XSB_I64");
        REQUIRE(index_base == 0 || index_base == 1, XSB_EINVAL, "index_base must be 0 or 1");
        REQUIRE(n_tid >= 1 && n_tid <= (1 << 16), XSB_EINVAL, "n_tid must be in 1..65536");
        if (idx_type == XSB_I32)
            REQUIRE(m < (1ll << 31) - 1 && n_global < (1ll << 31) - 1, XSB_EINVAL, "dimensions exceed Int32");
        i64 col_begin = 0, n = n_global;
        if (nranks > 0)
        {
            REQUIRE(nranks <= kMaxRanks, XSB_EINVAL, "at most 16 ranks");
            REQUIRE(rank >= 0 && rank < nranks && splits, XSB_EINVAL, "bad rank or NULL splits");
            REQUIRE(n_tid == 1, XSB_EINVAL, "slab handles take one partition buffer per rank");
            REQUIRE(splits[0] == 0 && splits[nranks] == n_global, XSB_EINVAL, "splits must cover [0, n)");
            for (int r = 0; r < nranks; ++r)
                REQUIRE(splits[r] < splits[r + 1], XSB_EINVAL, "every rank must own at least one column");
            col_begin = splits[rank];
            n = splits[rank + 1] - splits[rank];
        }
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
        {
            cudaGetLastError();
            throw ApiError(XSB_ECUDA, "no CUDA device: libxsparse_b200 has no CPU fallback");
        }
        REQUIRE(device >= 0 && device < ndev, XSB_EINVAL, "device ordinal out of range");
        KeyLayout L{};
        L.tidbits = n_tid > 1 ? ceil_log2(n_tid) : 0;
        L.low = 2 + L.tidbits;
        L.rowbits = ceil_log2(m);
        L.colbits = ceil_log2(n);
        if (nranks > 0)
        { // every rank uses the same field widths: a record is in its owner's layout wherever it is staged
            i64 widest = 1;
            for (int r = 0; r < nranks; ++r)
                widest = std::max<i64>(widest, splits[r + 1] - splits[r]);
            L.colbits = ceil_log2(widest);
            L.ownerbits = ceil_log2(nranks);
            L.nranks = nranks;
            L.self = rank;
            for (int r = 0; r <= nranks; ++r)
                L.splits[r] = splits[r];
            L.self_lo = splits[rank];
            L.self_width = (u64)(splits[rank + 1] - splits[rank]);
        }
        KeyLayout Ls = L; // insertion side: global columns in, owner found by pack()
        Ls.cols_global = 1;
        REQUIRE(L.low + L.rowbits + L.colbits + L.ownerbits <= 64, XSB_EINVAL,
                "m*n*n_tid does not fit the 64-bit packed key");
        REQUIRE(L.rowbits <= 32 && L.colbits <= 32 && n_global < (1ll << 32), XSB_EINVAL,
                "dimensions above 2^32 are not supported");
        XSB_CUDA(cudaSetDevice(device));
        h = new xsb_matrix();
        h->m = m;
        h->n = n;
        h->n_global = n_global;
        h->col_begin = col_begin;
        h->nranks = nranks;
        h->rank = rank;
        h->idx64 = idx_type == XSB_I64;
        h->base = index_base;
        h->n_tid = n_tid;
        h->device = device;
        h->L = L;
        h->Ls = Ls;
        h->stage.resize((size_t)n_tid);
        XSB_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        cudaMemPool_t pool;
        XSB_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
        unsigned long long thr = ~0ull; // keep freed blocks cached: flush allocates and frees large buffers
        XSB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
        h->d_scal = static_cast<u64 *>(h->dalloc(sizeof(u64) * 8));
        XSB_CUDA(cudaMallocHost(reinterpret_cast<void **>(&h->h_scal), sizeof(u64) * 8));
        if (nranks > 0)
        {
            h->d_route = static_cast<u64 *>(h->dalloc(sizeof(u64) * 4));
            XSB_CUDA(cudaMemsetAsync(h->d_route, 0, sizeof(u64) * 4, h->stream));
            XSB_CUDA(cudaMallocHost(reinterpret_cast<void **>(&h->h_route), sizeof(u64) * (2 * kMaxRanks + 4)));
        }
        XSB_CUDA(cudaEventCreate(&h->ev0));
        XSB_CUDA(cudaEventCreate(&h->ev1));
        h->set_empty_csc();
        *out = h;
        return XSB_OK;
    });
    if (rc != XSB_OK && h)
    {
        xsb_destroy(h);
        if (out)
            *out = nullptr;
    }
    return rc;
}

int32_t xsb_create(int64_t m, int64_t n, int32_t val_type, int32_t idx_type, int32_t index_base, int32_t n_tid,
                   int32_t device, xsb_matrix **out)
{
    return create_impl(m, n, 0, 0, nullptr, val_type, idx_type, index_base, n_tid, device, out);
}

int32_t xsb_create_slab(int64_t m, int64_t n_global, int32_t n_ranks, int32_t rank, const int64_t *col_splits,
                        int32_t val_type, int32_t idx_type, int32_t index_base, int32_t device, xsb_matrix **out)
{
    if (n_ranks < 1)
    {
        g_err = "n_ranks must be >= 1";
        return XSB_EINVAL;
    }
    return create_impl(m, n_global, n_ranks, rank, col_splits, val_type, idx_type, index_base, 1, device, out);
}

int32_t xsb_slab_info(const xsb_matrix *h, int64_t *col_begin, int64_t *col_end, int64_t *n_global)
{
    if (!h)
        return XSB_EINVAL;
    if (col_begin)
        *col_begin = h->col_begin;
    if (col_end)
        *col_end = h->col_begin + h->n;
    if (n_global)
        *n_global = h->n_global;
    return XSB_OK;
}

// Counts the staged records per owning rank: send_counts[r] = records rank r owns (r == own rank:
// the records that stay).  One read of the keys; nothing moves.
int32_t xsb_route_count(xsb_matrix *h, int64_t *send_counts)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && send_counts, XSB_EINVAL, "NULL argument");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(!h->routed, XSB_ESTATE, "staged records were already routed");
        Stage &st = h->stage[0];
        h->dfree(h->route_ws);
        h->route_ws = nullptr;
        for (int r = 0; r < kMaxRanks; ++r)
            h->route_counts[r] = 0;
        if (st.count > 0 && h->L.ownerbits > 0)
        {
            h->route_ws = h->dalloc(route_workspace_bytes((u64)st.count, h->nranks));
            route_count(h->stream, st.buf + st.front, (u64)st.count, h->L, h->route_ws, h->route_counts, h->lc,
                        h->tileflags);
        }
        else
            h->route_counts[h->rank] = (u64)st.count;
        h->route_counted = st.count;
        for (int r = 0; r < h->nranks; ++r)
            send_counts[r] = (int64_t)h->route_counts[r];
        return XSB_OK;
    });
}

// Copies the staged records owned by OTHER ranks into the caller's send buffer, destination rank
// after destination rank, each bucket in stream order; the rank's own records stay staged where
// they are.  send_counts as in xsb_route_count; capacity = room of the send buffer in records.
int32_t xsb_route_prepare(xsb_matrix *h, void *send_records, int64_t capacity, int64_t *send_counts)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && send_counts, XSB_EINVAL, "NULL argument");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(!h->routed, XSB_ESTATE, "staged records were already routed");
        Stage &st = h->stage[0];
        if (h->route_counted != st.count || (st.count > 0 && h->L.ownerbits > 0 && !h->route_ws))
        {
            const int32_t rc = xsb_route_count(h, send_counts);
            if (rc != XSB_OK)
                return rc;
        }
        i64 foreign = 0;
        for (int r = 0; r < h->nranks; ++r)
        {
            send_counts[r] = (int64_t)h->route_counts[r];
            if (r != h->rank)
                foreign += (i64)h->route_counts[r];
        }
        REQUIRE(capacity >= foreign, XSB_EINVAL,
                "send buffer too small: " + std::to_string(foreign) + " records leave this rank");
        REQUIRE(foreign == 0 || (send_records && is_device_ptr(send_records)), XSB_EINVAL,
                "send buffer must be device memory");
        if (foreign > 0)
            route_extract(h->stream, st.buf + st.front, (u64)st.count, h->L, h->route_ws, h->route_counts,
                          static_cast<Rec *>(send_records), h->lc);
        h->dfree(h->route_ws);
        h->route_ws = nullptr;
        h->route_counted = -1;
        h->foreign = foreign; // they stay behind in the staging buffer; the flush skips them by owner
        h->routed = true;
        pad_region(h);
        h->own_end = st.count;
        h->sync();
        return XSB_OK;
    });
}

// Appends records received from another rank (already in this rank's layout, in the sender's
// stream order) behind what is staged.  Call once per source, in source-rank order.
int32_t xsb_route_finish(xsb_matrix *h, int32_t src_rank, const void *recv_records, int64_t count)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(count >= 0, XSB_EINVAL, "negative count");
        REQUIRE(h->pending() == 0 || h->routed, XSB_ESTATE, "unrouted records are still staged");
        REQUIRE(src_rank >= 0 && src_rank < h->nranks && src_rank != h->rank, XSB_EINVAL, "bad source rank");
        REQUIRE(src_rank > h->last_src, XSB_ESTATE, "sources must be handed over in ascending rank order");
        h->last_src = src_rank;
        if (!h->routed)
        { // nothing was staged on this rank: the own region is empty
            h->ensure_stage(0, 0);
            h->own_end = 0;
        }
        if (src_rank > h->rank && h->low_end < 0)
        { // first source above this rank: the region of the lower ranks is complete
            pad_region(h);
            h->low_end = h->stage[0].count;
        }
        REQUIRE(count == 0 || (recv_records && is_device_ptr(recv_records)), XSB_EINVAL,
                "receive buffer must be device memory");
        if (count > 0)
        {
            h->ensure_stage(0, count);
            Stage &st = h->stage[0];
            write_scalar(h, 1, ~0ull);
            write_scalar(h, 5, 0ull);
            route_check(h->stream, static_cast<const Rec *>(recv_records), count, h->L, h->n, h->d_scal + 1,
                        h->d_scal + 5, h->lc);
            XSB_CUDA(cudaMemcpyAsync(st.buf + st.front + st.count, recv_records, sizeof(Rec) * (size_t)count,
                                     cudaMemcpyDeviceToDevice, h->stream));
            XSB_CUDA(cudaMemcpyAsync(h->h_scal + 5, h->d_scal + 5, sizeof(u64), cudaMemcpyDeviceToHost, h->stream));
            const u64 bad = read_scalar(h, 1);
            if (h->h_scal[5] != 0ull)
                h->has_assign = true; // the received stream holds A[i,j]=v records: ordered fold needed
            REQUIRE(bad == ~0ull, XSB_EBOUNDS,
                    "record " + std::to_string(bad) + " of the received buffer is not owned by this rank");
            st.count += count;
            (src_rank < h->rank ? h->n_low : h->n_high) += count;
        }
        h->routed = true;
        return XSB_OK;
    });
}

// Fixed-capacity exchange, step 1: copies the records other ranks own into one BLOCK per destination rank d != own
// -- a 16-byte header {records of the bucket, magic} followed by caps[d] record slots -- block after block in
// `send_records` (device; room for sum(caps[d] + 1) records).  Nothing is read back: the whole call is stream-ordered.
// A bucket fuller than its block is cut off; the receiving rank's flush reports it (XSB_ESTATE).
namespace
{
// common part of xsb_route_pack / xsb_route_pack_peer: h->h_route[d] holds the address of block d's first slot
void pack_blocks(xsb_matrix *h, const i64 *caps, const PeerFlags &sig)
{
    Stage &st = h->stage[0];
    if (!st.buf)
        h->ensure_stage(0, 0);
    h->dfree(h->route_ws);
    h->route_ws = h->dalloc(route_workspace_bytes((u64)std::max<i64>(st.count, 1), h->nranks));
    route_pack(h->stream, st.buf + st.front, (u64)st.count, h->L, h->route_ws, caps, h->h_route, h->h_route + kMaxRanks, sig,
               h->d_route, h->lc, h->tileflags);
    h->fixed_exchange = true; // the flags of this step are read (and cleared) with the staged records
}

// the own region of the step is complete
void close_own_region(xsb_matrix *h)
{
    Stage &st = h->stage[0];
    h->route_counted = -1;
    h->foreign = 0; // unknown on the host: the flush skips them by their owner bits
    h->routed = true;
    h->fixed_exchange = true;
    pad_region(h);
    h->own_end = st.count;
}

// common part of xsb_route_unpack / xsb_route_unpack_peer: blocks[src] = header of the block from rank src
void unpack_blocks(xsb_matrix *h, const Rec *const *blocks, const i64 *caps)
{
    if (!h->routed)
    { // nothing was staged on this rank: the own region is empty
        h->ensure_stage(0, 0);
        h->own_end = 0;
    }
    h->routed = true;
    h->fixed_exchange = true;
    // flavours of the received records: the unpack kernels raise bit 4 of the flags for A[i,j] = v records;
    // check_exchange (at the flush) turns that into has_assign
    for (int src = 0; src < h->nranks; ++src)
    {
        if (src == h->rank)
        { // the region of the lower ranks is complete
            pad_region(h);
            h->low_end = h->stage[0].count;
            continue;
        }
        const i64 cap = caps[src];
        if (blocks[src])
        { // also for cap == 0: the header must say "no records"
            h->ensure_stage(0, cap);
            Stage &st = h->stage[0];
            route_unpack(h->stream, blocks[src], cap, st.buf + st.front + st.count, h->L, h->n, h->d_route, h->d_route + 1,
                         src < h->rank ? 0 : 1, h->lc);
            st.count += cap;
            (src < h->rank ? h->n_low : h->n_high) += cap;
        }
        h->last_src = src;
    }
    if (h->low_end < 0)
        h->low_end = h->stage[0].count;
}

size_t px_block_records(i64 cap) { return ((size_t)cap + 1 + 15) & ~(size_t)15; }
// byte offset of the block src -> dst (step parity p) in dst's mailbox; total size for src == nranks
size_t px_offset(const i64 *caps, int nranks, int dst, int src, int parity)
{
    size_t off = 512;
    for (int s2 = 0; s2 < nranks; ++s2)
    {
        const i64 cap = caps[dst * nranks + s2];
        if (s2 == dst || cap <= 0)
            continue;
        const size_t bytes = 16 * px_block_records(cap);
        if (s2 == src)
            return off + (size_t)parity * bytes;
        off += 2 * bytes;
    }
    return off;
}
} // namespace

int32_t xsb_route_pack(xsb_matrix *h, void *send_records, const int64_t *caps, int64_t send_capacity)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && caps, XSB_EINVAL, "NULL argument");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(!h->routed, XSB_ESTATE, "staged records were already routed");
        i64 need = 0;
        for (int d = 0; d < h->nranks; ++d)
            if (d != h->rank)
            {
                REQUIRE(caps[d] >= 0, XSB_EINVAL, "negative block capacity");
                need += caps[d] + 1;
            }
        REQUIRE(send_capacity >= need, XSB_EINVAL, "send buffer too small for the blocks");
        REQUIRE(need == 0 || (send_records && is_device_ptr(send_records)), XSB_EINVAL, "send buffer must be device memory");
        Rec *blk = static_cast<Rec *>(send_records);
        for (int d = 0; d < h->nranks; ++d)
        {
            h->h_route[d] = d == h->rank ? 0ull : reinterpret_cast<u64>(blk + 1); // first slot behind the header
            if (d != h->rank)
                blk += caps[d] + 1;
        }
        PeerFlags none{};
        pack_blocks(h, reinterpret_cast<const i64 *>(caps), none);
        close_own_region(h);
        return XSB_OK;
    });
}

// Fixed-capacity exchange, step 2 (after the all-to-all): `recv_records` holds the blocks of the source ranks
// src != own in ascending order, block src = header + caps[src] slots.  Every block becomes a region of caps[src]
// staged records (the bucket's records, then records the flush skips).  Stream-ordered; errors (a record of another
// owner, a bucket that was cut off) surface at xsb_flush.
int32_t xsb_route_unpack(xsb_matrix *h, const void *recv_records, const int64_t *caps)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && caps, XSB_EINVAL, "NULL argument");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(h->pending() == 0 || h->routed, XSB_ESTATE, "unrouted records are still staged");
        REQUIRE(h->last_src < 0, XSB_ESTATE, "records of other ranks were already appended");
        i64 total = 0;
        for (int s2 = 0; s2 < h->nranks; ++s2)
            if (s2 != h->rank)
            {
                REQUIRE(caps[s2] >= 0, XSB_EINVAL, "negative block capacity");
                total += caps[s2];
            }
        REQUIRE(total == 0 || (recv_records && is_device_ptr(recv_records)), XSB_EINVAL, "receive buffer must be device memory");
        const Rec *blocks[kMaxRanks] = {};
        const Rec *blk = static_cast<const Rec *>(recv_records);
        for (int src = 0; src < h->nranks && blk; ++src)
            if (src != h->rank)
            {
                blocks[src] = blk;
                blk += caps[src] + 1;
            }
        unpack_blocks(h, blocks, reinterpret_cast<const i64 *>(caps));
        return XSB_OK;
    });
}

// ------------------------------------------------------------------------------------------------------------
// Peer exchange: the fixed-capacity exchange over NVLink peer memory, without a communication library on the
// records' path.  Setup (collective over the ranks of one node, host side):
//   every rank: xsb_peer_exchange_create(h, caps, handle)   caps[dst * n_ranks + src] = slots of the block src -> dst,
//               the same matrix on every rank; allocates this rank's mailbox and exports it (64-byte CUDA IPC handle)
//   all-gather the handles (any transport: they are plain bytes)
//   every rank: xsb_peer_exchange_connect(h, handles)       maps the mailboxes of the ranks it exchanges blocks with
// Step: xsb_route_pack_peer(h) (the copy-out kernel stores every block into its receiver's mailbox and raises the
// receiver's flag) -> xsb_route_unpack_peer(h) (waits for the flags of this step, takes the blocks, tells the
// senders that their blocks were taken) -> xsb_flush.  Everything is stream-ordered on the handle's stream; two
// blocks per pair (step parity) let a sender run one step ahead of its receiver.  Every rank makes both calls in
// every step.  Teardown: xsb_peer_exchange_disconnect on every rank, a barrier, xsb_peer_exchange_destroy.
// ------------------------------------------------------------------------------------------------------------
int32_t xsb_peer_exchange_create(xsb_matrix *h, const int64_t *caps, void *ipc_handle_out)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && caps, XSB_EINVAL, "NULL argument");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(!h->px.created, XSB_ESTATE, "this handle has a peer exchange already: destroy it first");
        const int nr = h->nranks;
        for (int k = 0; k < nr * nr; ++k)
            REQUIRE(caps[k] >= 0, XSB_EINVAL, "negative block capacity");
        auto &px = h->px;
        std::memcpy(px.caps, caps, sizeof(i64) * (size_t)nr * nr);
        px.box_bytes = px_offset(px.caps, nr, h->rank, nr, 0);
        // cudaMalloc, not the stream-ordered pool: only such memory can be exported to another process
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&px.box), px.box_bytes);
        if (e != cudaSuccess)
        {
            cudaGetLastError();
            px.box = nullptr;
            throw ApiError(XSB_ENOMEM, std::string("mailbox allocation failed: ") + cudaGetErrorString(e));
        }
        XSB_CUDA(cudaMemsetAsync(px.box, 0, px.box_bytes, h->stream));
        XSB_CUDA(cudaStreamSynchronize(h->stream));
        if (ipc_handle_out)
        {
            cudaIpcMemHandle_t ih;
            e = cudaIpcGetMemHandle(&ih, px.box);
            if (e != cudaSuccess)
            {
                cudaGetLastError();
                cudaFree(px.box);
                px.box = nullptr;
                throw ApiError(XSB_ECUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
            }
            static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
            std::memcpy(ipc_handle_out, &ih, 64);
        }
        px.seq = 0;
        px.created = true;
        px.connected = false;
        px.packed = false;
        if (const char *t = std::getenv("XSB_PEER_TIMEOUT_MS"))
            px.timeout_ns = (u64)std::max(1ll, std::atoll(t)) * 1000000ull;
        return XSB_OK;
    });
}

namespace
{
bool px_talks_to(const xsb_matrix *h, int r)
{
    const int nr = h->nranks;
    return r != h->rank && (h->px.caps[r * nr + h->rank] > 0 || h->px.caps[h->rank * nr + r] > 0);
}
} // namespace

int32_t xsb_peer_exchange_connect(xsb_matrix *h, const void *ipc_handles)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && ipc_handles, XSB_EINVAL, "NULL argument");
        REQUIRE(h->px.created && !h->px.connected, XSB_ESTATE, "xsb_peer_exchange_create comes first (once)");
        auto &px = h->px;
        for (int r = 0; r < h->nranks; ++r)
        {
            if (!px_talks_to(h, r))
                continue;
            cudaIpcMemHandle_t ih;
            std::memcpy(&ih, static_cast<const unsigned char *>(ipc_handles) + 64 * (size_t)r, 64);
            void *p = nullptr;
            const cudaError_t e = cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess)
            {
                cudaGetLastError();
                for (int q = 0; q < r; ++q)
                    if (px.peer[q] && px.peer_ipc[q])
                    {
                        cudaIpcCloseMemHandle(px.peer[q]);
                        px.peer[q] = nullptr;
                    }
                throw ApiError(XSB_ECUDA, "cannot map the mailbox of rank " + std::to_string(r) + " (" + cudaGetErrorString(e) +
                                              "): the ranks must be processes on one node whose GPUs have peer access");
            }
            px.peer[r] = static_cast<unsigned char *>(p);
            px.peer_ipc[r] = true;
        }
        px.connected = true;
        return XSB_OK;
    });
}

// ranks that live in ONE process (several handles, one or several GPUs with peer access): no IPC, the mailboxes of
// the other handles are used directly.  peers[r] = handle of rank r (peers[own rank] is ignored).
int32_t xsb_peer_exchange_connect_local(xsb_matrix *h, xsb_matrix *const *peers)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && peers, XSB_EINVAL, "NULL argument");
        REQUIRE(h->px.created && !h->px.connected, XSB_ESTATE, "xsb_peer_exchange_create comes first (once)");
        auto &px = h->px;
        for (int r = 0; r < h->nranks; ++r)
        {
            if (!px_talks_to(h, r))
                continue;
            REQUIRE(peers[r] && peers[r]->px.created && peers[r]->nranks == h->nranks && peers[r]->rank == r, XSB_EINVAL,
                    "peers[r] must be the handle of rank r with a mailbox");
            REQUIRE(std::memcmp(peers[r]->px.caps, px.caps, sizeof(i64) * (size_t)h->nranks * h->nranks) == 0, XSB_EINVAL,
                    "the ranks disagree on the block capacities");
            if (peers[r]->device != h->device)
            {
                int can = 0;
                XSB_CUDA(cudaDeviceCanAccessPeer(&can, h->device, peers[r]->device));
                REQUIRE(can, XSB_ESTATE, "no peer access between the GPUs of two ranks");
                const cudaError_t e = cudaDeviceEnablePeerAccess(peers[r]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                    XSB_CUDA(e);
                cudaGetLastError();
            }
            px.peer[r] = peers[r]->px.box;
            px.peer_ipc[r] = false;
        }
        px.connected = true;
        return XSB_OK;
    });
}

int32_t xsb_peer_exchange_disconnect(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        auto &px = h->px;
        if (!px.created)
            return XSB_OK;
        XSB_CUDA(cudaStreamSynchronize(h->stream));
        for (int r = 0; r < kMaxRanks; ++r)
        {
            if (px.peer[r] && px.peer_ipc[r])
                cudaIpcCloseMemHandle(px.peer[r]);
            px.peer[r] = nullptr;
            px.peer_ipc[r] = false;
        }
        cudaGetLastError();
        px.connected = false;
        return XSB_OK;
    });
}

int32_t xsb_peer_exchange_destroy(xsb_matrix *h)
{
    const int32_t rc = xsb_peer_exchange_disconnect(h);
    if (rc != XSB_OK)
        return rc;
    return guard(h, [&]() -> int32_t {
        auto &px = h->px;
        if (px.box)
            cudaFree(px.box);
        cudaGetLastError();
        px.box = nullptr;
        px.box_bytes = 0;
        px.created = false;
        px.packed = false;
        return XSB_OK;
    });
}

int32_t xsb_route_pack_peer(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(h->px.connected, XSB_ESTATE, "no peer exchange: xsb_peer_exchange_create / _connect come first");
        REQUIRE(!h->routed, XSB_ESTATE, "staged records were already routed");
        REQUIRE(!h->px.packed, XSB_ESTATE, "xsb_route_unpack_peer of the previous step is missing");
        auto &px = h->px;
        const int nr = h->nranks, me = h->rank;
        const u64 seq = ++px.seq;
        const int parity = (int)(seq & 1ull);
        i64 caps_out[kMaxRanks] = {};
        PeerFlags waitf{}, sig{};
        bool any_wait = false;
        for (int d = 0; d < nr; ++d)
        {
            h->h_route[d] = 0ull;
            caps_out[d] = d == me ? 0 : px.caps[d * nr + me];
            if (d == me || caps_out[d] <= 0)
                continue;
            unsigned char *blk = px.peer[d] + px_offset(px.caps, nr, d, me, parity);
            h->h_route[d] = reinterpret_cast<u64>(blk + 16);
            sig.addr[d] = reinterpret_cast<u64>(px.peer[d] + 8 * (size_t)me); // ready[me] of rank d
            sig.value[d] = seq;
            if (seq > 2)
            { // the block of this parity was last used in step seq - 2: d must have taken it
                waitf.addr[d] = reinterpret_cast<u64>(px.box + 8 * (size_t)(kMaxRanks + d)); // done[d], own mailbox
                waitf.value[d] = seq - 2;
                any_wait = true;
            }
        }
        if (any_wait)
            peer_wait(h->stream, waitf, px.timeout_ns, h->d_route, h->lc);
        pack_blocks(h, caps_out, sig);
        px.packed = true;
        px.packed_upto = h->stage[0].count; // insertions may go on: what follows must be this rank's own
        return XSB_OK;
    });
}

int32_t xsb_route_unpack_peer(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(h->px.connected && h->px.packed, XSB_ESTATE, "xsb_route_pack_peer of this step comes first");
        REQUIRE(h->last_src < 0, XSB_ESTATE, "records of other ranks were already appended");
        auto &px = h->px;
        const int nr = h->nranks, me = h->rank;
        const u64 seq = px.seq;
        const int parity = (int)(seq & 1ull);
        i64 caps_in[kMaxRanks] = {};
        const Rec *blocks[kMaxRanks] = {};
        PeerFlags waitf{}, sig{};
        bool any = false;
        for (int s2 = 0; s2 < nr; ++s2)
        {
            caps_in[s2] = s2 == me ? 0 : px.caps[me * nr + s2];
            if (s2 == me || caps_in[s2] <= 0)
                continue;
            blocks[s2] = reinterpret_cast<const Rec *>(px.box + px_offset(px.caps, nr, me, s2, parity));
            waitf.addr[s2] = reinterpret_cast<u64>(px.box + 8 * (size_t)s2); // ready[s2], own mailbox
            waitf.value[s2] = seq;
            sig.addr[s2] = reinterpret_cast<u64>(px.peer[s2] + 8 * (size_t)(kMaxRanks + me)); // done[me] of rank s2
            sig.value[s2] = seq;
            any = true;
        }
        {
            Stage &st = h->stage[0];
            if (st.count > px.packed_upto)
                route_tailcheck(h->stream, st.buf + st.front, (u64)px.packed_upto, (u64)st.count, h->L, h->tileflags, h->d_route,
                                h->lc);
            close_own_region(h);
        }
        if (any)
            peer_wait(h->stream, waitf, px.timeout_ns, h->d_route, h->lc);
        unpack_blocks(h, blocks, caps_in);
        if (any)
            peer_signal(h->stream, sig, h->lc);
        px.packed = false;
        return XSB_OK;
    });
}

int32_t xsb_destroy(xsb_matrix *h)
{
    if (!h)
        return XSB_OK;
    cudaSetDevice(h->device);
    if (h->stream)
        cudaStreamSynchronize(h->stream);
    for (int r = 0; r < kMaxRanks; ++r)
        if (h->px.peer[r] && h->px.peer_ipc[r])
            cudaIpcCloseMemHandle(h->px.peer[r]);
    if (h->px.box)
        cudaFree(h->px.box);
    h->drop_frozen();
    h->drop_blocks();
    h->clear_staging(true);
    h->runs_release();
    h->dfree(h->colptr);
    h->dfree(h->csc_store);
    h->dfree(h->route_ws);
    h->dfree(h->tileflags);
    h->dfree(h->d_scal);
    h->dfree(h->d_route);
    h->release_cache();
    if (h->h_scal)
        cudaFreeHost(h->h_scal);
    if (h->h_route)
        cudaFreeHost(h->h_route);
    if (h->ev0)
        cudaEventDestroy(h->ev0);
    if (h->ev1)
        cudaEventDestroy(h->ev1);
    for (cudaEvent_t e : h->ev_slice)
        if (e)
            cudaEventDestroy(e);
    if (h->copy_stream)
    {
        cudaStreamSynchronize(h->copy_stream);
        cudaStreamDestroy(h->copy_stream);
    }
    if (h->stream)
    {
        cudaStreamSynchronize(h->stream);
        cudaStreamDestroy(h->stream);
    }
    cudaGetLastError();
    delete h;
    return XSB_OK;
}

const char *xsb_last_error(const xsb_matrix *h) { return h ? h->err.c_str() : g_err.c_str(); }

int32_t xsb_reset(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        h->drop_frozen();
        h->drop_blocks();
        h->clear_staging(false);
        h->set_empty_csc();
        return XSB_OK;
    });
}

int32_t xsb_set_csc(xsb_matrix *h, const void *colptr, const void *rowval, const void *nzval)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && colptr, XSB_EINVAL, "NULL argument");
        h->drop_blocks();
        const size_t isz = h->isz();
        // nnz = colptr[n] - base
        unsigned char last[8];
        XSB_CUDA(cudaMemcpy(last, static_cast<const unsigned char *>(colptr) + isz * (size_t)h->n, isz,
                            cudaMemcpyDefault));
        i64 nnz;
        if (h->idx64)
        {
            int64_t v;
            std::memcpy(&v, last, 8);
            nnz = v - h->base;
        }
        else
        {
            int32_t v;
            std::memcpy(&v, last, 4);
            nnz = v - h->base;
        }
        REQUIRE(nnz >= 0, XSB_EINVAL, "colptr[n] is smaller than the index base");
        REQUIRE(nnz == 0 || (rowval && nzval), XSB_EINVAL, "NULL rowval/nzval");
        h->drop_frozen();
        h->clear_staging(false);
        h->dfree(h->colptr);
        h->dfree(h->csc_store);
        h->colptr = h->dalloc(isz * (size_t)(h->n + 1));
        XSB_CUDA(cudaMemcpyAsync(h->colptr, colptr, isz * (size_t)(h->n + 1), cudaMemcpyDefault, h->stream));
        const size_t rv_bytes = (isz * (size_t)nnz + 15) & ~(size_t)15;
        unsigned char *st = static_cast<unsigned char *>(h->dalloc(rv_bytes + 8 * (size_t)nnz));
        if (nnz)
        {
            XSB_CUDA(cudaMemcpyAsync(st, rowval, isz * (size_t)nnz, cudaMemcpyDefault, h->stream));
            XSB_CUDA(cudaMemcpyAsync(st + rv_bytes, nzval, 8 * (size_t)nnz, cudaMemcpyDefault, h->stream));
        }
        h->csc_store = st;
        h->csc_store_bytes = rv_bytes + 8 * (size_t)nnz;
        h->rowval = st;
        h->nzval = reinterpret_cast<double *>(st + rv_bytes);
        h->nnz = nnz;
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_shrink_to_fit(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        h->shrink_store();
        if (h->pending() == 0)
        {
            h->clear_staging(true);
            h->runs_release();
        }
        h->release_cache();
        return XSB_OK;
    });
}

int32_t xsb_size(const xsb_matrix *h, int64_t *m, int64_t *n)
{
    if (!h)
        return XSB_EINVAL;
    if (m)
        *m = h->m;
    if (n)
        *n = h->n;
    return XSB_OK;
}

int32_t xsb_nnz(const xsb_matrix *h, int64_t *nnz)
{
    if (!h || !nnz)
        return XSB_EINVAL;
    *nnz = h->nnz;
    return XSB_OK;
}

int32_t xsb_reserve(xsb_matrix *h, int32_t tid, int64_t count)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(tid >= 0 && tid < h->n_tid, XSB_EINVAL, "tid out of range");
        REQUIRE(count >= 0, XSB_EINVAL, "negative count");
        h->ensure_stage(tid, count);
        return XSB_OK;
    });
}

int32_t xsb_insert_batch(xsb_matrix *h, int32_t tid, const void *I, const void *J, const void *V, int64_t count,
                         int32_t flavour)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        check_tid_flavour(h, tid, flavour);
        REQUIRE(count >= 0, XSB_EINVAL, "negative count");
        if (count == 0)
            return XSB_OK;
        REQUIRE(I && J && V, XSB_EINVAL, "NULL array");
        Rec *dst = begin_emit(h, tid, flavour, count);
        DevIn dI(h, I, h->isz() * (size_t)count), dJ(h, J, h->isz() * (size_t)count), dV(h, V, 8 * (size_t)count);
        write_scalar(h, 1, ~0ull);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0, chunks = 0;
        const bool grouped = runs_begin(h, tid, count, pack_chunks(count), &rt, &chunk0, &pos0);
        if (grouped)
            chunks = pack_records_grouped(h->stream, dI.ptr, dJ.ptr, static_cast<const double *>(dV.ptr), count, h->idx64,
                                          h->base, h->m, h->n_global, h->Ls, (u32)tid, (u32)flavour, dst, h->d_scal + 1,
                                          h->lc, rt, chunk0, pos0, h->stage_flags(tid));
        else
            pack_records(h->stream, dI.ptr, dJ.ptr, static_cast<const double *>(dV.ptr), count, h->idx64, h->base, h->m,
                         h->n_global, h->Ls, (u32)tid, (u32)flavour, dst, h->d_scal + 1, h->lc, h->stage_flags(tid));
        const u64 bad = read_scalar(h, 1);
        if (bad != ~0ull)
        {
            if (grouped)
                h->runs.dead = true; // the rejected batch left runs behind: the index is rebuilt at flush time
            throw ApiError(XSB_EBOUNDS, "BoundsError: entry " + std::to_string(bad) +
                                            " of the batch is outside the matrix; batch rejected");
        }
        if (h->n_tid > 1 && flavour == XSB_ASSIGN)
            check_mt_assign(h, dst, count);
        end_emit(h, tid, flavour, count);
        if (grouped)
            runs_end(h, count, chunks);
        return XSB_OK;
    });
}

int32_t xsb_insert_triplets(xsb_matrix *h, int32_t tid, const xsb_triplet *T, int64_t count, int32_t flavour)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        check_tid_flavour(h, tid, flavour);
        REQUIRE(count >= 0, XSB_EINVAL, "negative count");
        REQUIRE((u64)h->m < (1ull << 32) && (u64)h->n_global < (1ull << 32), XSB_EINVAL,
                "triplets carry 32-bit indices: the matrix needs fewer than 2^32 rows and columns");
        if (count == 0)
            return XSB_OK;
        REQUIRE(T, XSB_EINVAL, "NULL array");
        REQUIRE((reinterpret_cast<uintptr_t>(T) & 15u) == 0, XSB_EINVAL, "triplet array must be 16-byte aligned");
        Rec *dst = begin_emit(h, tid, flavour, count);
        const bool from_host = !is_device_ptr(T);
        write_scalar(h, 1, ~0ull);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0, chunks = 0;
        const bool grouped = runs_begin(h, tid, count, pack_chunks(count), &rt, &chunk0, &pos0);
        // Host triplets go over PCIe straight into the staging buffer and are rewritten in place.  A large batch
        // travels in slices on a second stream, and slice k is packed while slice k + 1 is on the wire: the packing
        // (1.6 ms per 100 M records) disappears behind the transfer.
        constexpr i64 kSlice = (i64)1 << 22; // 4 M records = 64 MB: a whole number of chunks (pack_chunks)
        const bool sliced = from_host && count >= 3 * kSlice;
        if (sliced && !h->copy_stream)
        {
            XSB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
            for (cudaEvent_t &e : h->ev_slice)
                XSB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        if (sliced)
        { // the transfers may not overtake what the handle's stream still does with the staging buffer
            XSB_CUDA(cudaEventRecord(h->ev_slice[2], h->stream));
            XSB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_slice[2], 0));
        }
        const i64 step = sliced ? kSlice : count;
        int k = 0;
        for (i64 off = 0; off < count; off += step, ++k)
        {
            const i64 cnt = std::min(step, count - off);
            const void *src = static_cast<const Rec *>(static_cast<const void *>(T)) + off;
            if (from_host)
            {
                cudaStream_t cs = sliced ? h->copy_stream : h->stream;
                XSB_CUDA(cudaMemcpyAsync(dst + off, src, sizeof(Rec) * (size_t)cnt, cudaMemcpyHostToDevice, cs));
                if (sliced)
                {
                    XSB_CUDA(cudaEventRecord(h->ev_slice[k & 1], cs));
                    XSB_CUDA(cudaStreamWaitEvent(h->stream, h->ev_slice[k & 1], 0));
                }
                src = dst + off;
            }
            StageFlags sf = h->stage_flags(tid);
            sf.pos0 += off;
            if (grouped)
                chunks += pack_triplets_grouped(h->stream, src, cnt, h->base, h->m, h->n_global, h->Ls, (u32)tid, (u32)flavour,
                                                dst + off, h->d_scal + 1, h->lc, rt, chunk0 + pack_chunks(off),
                                                pos0 + (u32)off, sf, off);
            else
                pack_triplets(h->stream, src, cnt, h->base, h->m, h->n_global, h->Ls, (u32)tid, (u32)flavour, dst + off,
                              h->d_scal + 1, h->lc, sf, off);
        }
        const u64 bad = read_scalar(h, 1);
        if (bad != ~0ull)
        {
            if (grouped)
                h->runs.dead = true;
            throw ApiError(XSB_EBOUNDS, "BoundsError: entry " + std::to_string(bad) +
                                            " of the batch is outside the matrix; batch rejected");
        }
        if (h->n_tid > 1 && flavour == XSB_ASSIGN)
            check_mt_assign(h, dst, count);
        end_emit(h, tid, flavour, count);
        if (grouped)
            runs_end(h, count, chunks);
        return XSB_OK;
    });
}

int32_t xsb_insert_elements(xsb_matrix *h, int32_t tid, int32_t k, int64_t ncells, const void *dofs, const double *Aloc,
                            int32_t flavour)
{
    return xsb_insert_elements_rect(h, tid, k, k, ncells, dofs, dofs, Aloc, flavour);
}

int32_t xsb_insert_elements_rect(xsb_matrix *h, int32_t tid, int32_t kr, int32_t kc, int64_t ncells, const void *rdofs,
                                 const void *cdofs, const double *Aloc, int32_t flavour)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        check_tid_flavour(h, tid, flavour);
        const i64 count = element_calls(kr, kc, ncells);
        if (count == 0)
            return XSB_OK;
        REQUIRE(rdofs && cdofs && Aloc, XSB_EINVAL, "NULL array");
        Rec *dst = begin_emit(h, tid, flavour, count);
        DevIn dA(h, Aloc, 8 * (size_t)count);
        const ElementDofs ed(h, kr, kc, ncells, rdofs, cdofs, static_cast<const double *>(dA.ptr));
        const ElementBatch &eb = ed.batch;
        write_scalar(h, 1, ~0ull);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0, chunks = 0;
        const bool grouped = runs_begin(h, tid, count, insert_elements_chunks(kr, kc, ncells), &rt, &chunk0, &pos0);
        if (grouped)
            chunks = insert_elements_grouped(h->stream, eb, h->idx64, h->base, h->m, h->n_global, h->Ls, (u32)tid,
                                             (u32)flavour, dst, h->d_scal + 1, h->lc, h->stage_flags(tid), rt, chunk0, pos0);
        else
            insert_elements(h->stream, eb, h->idx64, h->base, h->m, h->n_global, h->Ls, (u32)tid, (u32)flavour, dst,
                            h->d_scal + 1, h->lc, h->stage_flags(tid));
        const u64 bad = read_scalar(h, 1);
        if (bad != ~0ull)
        {
            if (grouped)
                h->runs.dead = true; // the rejected batch left runs behind: the index is rebuilt at flush time
            const char *what = ElementDofs::square(kr, kc, rdofs, cdofs) ? "a dof" : (bad & 1u) ? "a column dof" : "a row dof";
            throw ApiError(XSB_EBOUNDS, "BoundsError: element " + std::to_string(bad >> 1) + " of the batch has " + what +
                                            " outside the matrix; batch rejected");
        }
        if (h->n_tid > 1 && flavour == XSB_ASSIGN)
            check_mt_assign(h, dst, count);
        end_emit(h, tid, flavour, count);
        if (grouped)
            runs_end(h, count, chunks);
        return XSB_OK;
    });
}

int32_t xsb_pending(const xsb_matrix *h, int64_t *count)
{
    if (!h || !count)
        return XSB_EINVAL;
    *count = h->pending();
    return XSB_OK;
}

int32_t xsb_flush(xsb_matrix *h, int32_t mode, int64_t *nnz_out, int32_t *pattern_changed)
{
    return xsb_flush_ex(h, mode, XSB_COMBINE_SEED, nnz_out, pattern_changed);
}

int32_t xsb_flush_ex(xsb_matrix *h, int32_t mode, int32_t combine, int64_t *nnz_out, int32_t *pattern_changed)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        return do_flush(h, mode, combine, nnz_out, pattern_changed);
    });
}

int32_t xsb_fetch_csc(xsb_matrix *h, void *colptr_out, void *rowval_out, void *nzval_out)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        if (colptr_out)
            XSB_CUDA(cudaMemcpyAsync(colptr_out, h->colptr, h->isz() * (size_t)(h->n + 1), cudaMemcpyDefault,
                                     h->stream));
        if (rowval_out && h->nnz)
            XSB_CUDA(cudaMemcpyAsync(rowval_out, h->rowval, h->isz() * (size_t)h->nnz, cudaMemcpyDefault, h->stream));
        if (nzval_out && h->nnz)
            XSB_CUDA(cudaMemcpyAsync(nzval_out, h->nzval, 8 * (size_t)h->nnz, cudaMemcpyDefault, h->stream));
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_get_values(xsb_matrix *h, const void *I, const void *J, void *V_out, int64_t count)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(count >= 0, XSB_EINVAL, "negative count");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "flush! before reading entries");
        if (count == 0)
            return XSB_OK;
        REQUIRE(I && J && V_out, XSB_EINVAL, "NULL array");
        DevIn dI(h, I, h->isz() * (size_t)count), dJ(h, J, h->isz() * (size_t)count);
        DevOut dV(h, V_out, 8 * (size_t)count);
        i64 *slot = static_cast<i64 *>(h->dalloc(8 * (size_t)count));
        write_scalar(h, 2, 0);
        write_scalar(h, 3, ~0ull);
        lookup_slots(h->stream, h->view(), h->m, h->n, h->idx64, h->base, dI.ptr, dJ.ptr, count, slot, h->d_scal + 2,
                     h->d_scal + 3, h->lc);
        gather_values(h->stream, h->nzval, slot, count, static_cast<double *>(dV.ptr), h->lc);
        dV.finish();
        h->dfree(slot);
        const u64 oob = read_scalar(h, 3);
        REQUIRE(oob == ~0ull, XSB_EBOUNDS, "BoundsError: position " + std::to_string(oob) + " is outside the matrix");
        return XSB_OK;
    });
}

int32_t xsb_zero_values(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        zero_values(h->stream, h->nzval, h->nnz, h->lc);
        return XSB_OK;
    });
}

int32_t xsb_freeze_pattern(xsb_matrix *h, const void *I, const void *J, int64_t count)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        freeze_check(h, count);
        REQUIRE(count == 0 || (I && J), XSB_EINVAL, "NULL array");
        h->drop_frozen();
        DevIn dI(h, I, h->isz() * (size_t)count), dJ(h, J, h->isz() * (size_t)count);
        return freeze_impl(h, count, [&](i64 *slot) {
            lookup_slots(h->stream, h->view(), h->m, h->n, h->idx64, h->base, dI.ptr, dJ.ptr, count, slot, h->d_scal + 2,
                         h->d_scal + 3, h->lc);
        });
    });
}

int32_t xsb_freeze_elements(xsb_matrix *h, int32_t k, int64_t ncells, const void *dofs)
{
    return xsb_freeze_elements_rect(h, k, k, ncells, dofs, dofs);
}

int32_t xsb_freeze_elements_rect(xsb_matrix *h, int32_t kr, int32_t kc, int64_t ncells, const void *rdofs,
                                 const void *cdofs)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        const i64 count = element_calls(kr, kc, ncells);
        freeze_check(h, count);
        REQUIRE(count == 0 || (rdofs && cdofs), XSB_EINVAL, "NULL array");
        h->drop_frozen();
        ElementDofs ed(h, kr, kc, ncells, rdofs, cdofs);
        return freeze_impl(h, count, [&](i64 *slot) {
            lookup_slots_elements(h->stream, h->view(), h->m, h->n, h->idx64, h->base, ed.batch, count, slot,
                                  h->d_scal + 2, h->d_scal + 3, h->lc);
        });
    });
}

static int32_t reassemble_impl(xsb_matrix *h, const void *V, int64_t count, int32_t mode, bool zero_first)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->frozen, XSB_ESTATE, "no frozen pattern");
        REQUIRE(h->fs_state == 0, XSB_ESTATE,
                "the frozen stream spans column slabs: re-assemble with xsb_reassemble_slab_pack / _values");
        REQUIRE(count == h->f_count, XSB_ESIZE, "value count differs from the frozen stream");
        REQUIRE(mode == XSB_DETERMINISTIC || mode == XSB_FAST, XSB_EINVAL, "unknown summation mode");
        if (count == 0)
        {
            if (zero_first)
                zero_values(h->stream, h->nzval, h->nnz, h->lc);
            return XSB_OK;
        }
        REQUIRE(V, XSB_EINVAL, "NULL array");
        DevIn dV(h, V, 8 * (size_t)count);
        if (mode == XSB_DETERMINISTIC)
            reassemble_deterministic(h->stream, static_cast<const double *>(dV.ptr), h->f_perm, h->f_segstart, h->nnz,
                                     h->nzval, zero_first, h->lc);
        else
        {
            if (zero_first)
                zero_values(h->stream, h->nzval, h->nnz, h->lc);
            reassemble_fast(h->stream, static_cast<const double *>(dV.ptr), h->f_slot, count, h->nzval, h->lc);
        }
        return XSB_OK;
    });
}

int32_t xsb_reassemble_values(xsb_matrix *h, const void *V, int64_t count, int32_t mode)
{
    return reassemble_impl(h, V, count, mode, false);
}

int32_t xsb_reassemble_values_zeroed(xsb_matrix *h, const void *V, int64_t count, int32_t mode)
{
    return reassemble_impl(h, V, count, mode, true);
}

int32_t xsb_unfreeze(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        h->drop_frozen();
        return XSB_OK;
    });
}

int32_t xsb_freeze_slab(xsb_matrix *h, const void *I, const void *J, int64_t count, int64_t *send_counts)
{
    return guard(h, [&]() -> int32_t {
        slab_freeze_check(h);
        freeze_check(h, count);
        REQUIRE(count == 0 || (I && J), XSB_EINVAL, "NULL array");
        h->drop_frozen();
        DevIn dI(h, I, h->isz() * (size_t)count), dJ(h, J, h->isz() * (size_t)count);
        return freeze_slab_impl(h, count, send_counts, [&](i64 *slot, Rec *tags) {
            slab_classify(h->stream, h->view(), h->m, h->n_global, h->Ls, h->idx64, h->base, dI.ptr, dJ.ptr, count, slot,
                          tags, h->d_scal + 2, h->d_scal + 3, h->lc);
        });
    });
}

int32_t xsb_freeze_slab_elements(xsb_matrix *h, int32_t k, int64_t ncells, const void *dofs, int64_t *send_counts)
{
    return xsb_freeze_slab_elements_rect(h, k, k, ncells, dofs, dofs, send_counts);
}

int32_t xsb_freeze_slab_elements_rect(xsb_matrix *h, int32_t kr, int32_t kc, int64_t ncells, const void *rdofs,
                                      const void *cdofs, int64_t *send_counts)
{
    return guard(h, [&]() -> int32_t {
        slab_freeze_check(h);
        const i64 count = element_calls(kr, kc, ncells);
        freeze_check(h, count);
        REQUIRE(count == 0 || (rdofs && cdofs), XSB_EINVAL, "NULL array");
        h->drop_frozen();
        ElementDofs ed(h, kr, kc, ncells, rdofs, cdofs);
        return freeze_slab_impl(h, count, send_counts, [&](i64 *slot, Rec *tags) {
            slab_classify_elements(h->stream, h->view(), h->m, h->n_global, h->Ls, h->idx64, h->base, ed.batch, count,
                                   slot, tags, h->d_scal + 2, h->d_scal + 3, h->lc);
        });
    });
}

int32_t xsb_freeze_slab_prepare(xsb_matrix *h, void *send_positions, int64_t capacity)
{
    return guard(h, [&]() -> int32_t {
        slab_freeze_check(h);
        REQUIRE(h->fs_state == 1, XSB_ESTATE, "no slab freeze in progress: xsb_freeze_slab first");
        REQUIRE(capacity >= h->fs_foreign, XSB_EINVAL,
                "send buffer too small: " + std::to_string(h->fs_foreign) + " positions leave this rank");
        REQUIRE(h->fs_foreign == 0 || (send_positions && is_device_ptr(send_positions)), XSB_EINVAL,
                "send buffer must be device memory");
        if (h->fs_foreign > 0)
            XSB_CUDA(cudaMemcpyAsync(send_positions, h->fs_send_pos, 8 * (size_t)h->fs_foreign, cudaMemcpyDeviceToDevice,
                                     h->stream));
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_freeze_slab_finish(xsb_matrix *h, const void *recv_positions, const int64_t *recv_counts)
{
    return guard(h, [&]() -> int32_t {
        slab_freeze_check(h);
        REQUIRE(h->fs_state == 1, XSB_ESTATE, "no slab freeze in progress: xsb_freeze_slab first");
        try
        {
            REQUIRE(recv_counts, XSB_EINVAL, "NULL recv_counts");
            i64 low = 0, high = 0;
            for (int r = 0; r < h->nranks; ++r)
            {
                if (r == h->rank)
                    continue;
                REQUIRE(recv_counts[r] >= 0 && recv_counts[r] < ((i64)1 << 32), XSB_EINVAL, "bad receive count");
                (r < h->rank ? low : high) += recv_counts[r];
            }
            const i64 own = h->f_count, total = low + own + high;
            REQUIRE((u64)total < (1ull << 32), XSB_EINVAL,
                    "received positions plus the own stream must stay below 2^32 (the map indexes values with 32 bits)");
            REQUIRE(low + high == 0 || (recv_positions && is_device_ptr(recv_positions)), XSB_EINVAL,
                    "receive buffer must be device memory");
            cudaStream_t s = h->stream;
            const size_t room = (size_t)std::max<i64>(total, 1);
            Rec *A = static_cast<Rec *>(h->dalloc(sizeof(Rec) * room));
            write_scalar(h, 2, 0);
            write_scalar(h, 3, ~0ull);
            slab_records(s, h->view(), h->m, h->n, h->idx64, h->base, h->fs_slot, own, recv_positions, low, total, A,
                         h->d_scal + 2, h->d_scal + 3, h->lc);
            const u64 oob = read_scalar(h, 3);
            const u64 missing = read_scalar(h, 2);
            if (oob != ~0ull || missing != 0)
            {
                h->dfree(A);
                if (oob != ~0ull)
                    throw ApiError(XSB_EBOUNDS,
                                   "BoundsError: received position " + std::to_string(oob) + " is outside this rank's slab");
                throw ApiError(XSB_EILLEGAL, std::to_string(missing) + " received positions are not in the frozen pattern");
            }
            // foreign own positions carry slot nnz: they sort behind every real slot and stay out of the map
            const i64 nmap = total - h->fs_foreign;
            Rec *B = static_cast<Rec *>(h->dalloc(sizeof(Rec) * room));
            void *ws = h->dalloc(sort_workspace_bytes((u64)total));
            const SortPlan plan = make_sort_plan(0, ceil_log2(std::max<i64>(h->nnz + 1, 2)));
            Rec *sorted = radix_sort_records(s, A, B, (u64)total, plan, ws, h->lc, nullptr);
            h->f_perm = static_cast<u32 *>(h->dalloc(4 * (size_t)std::max<i64>(nmap, 1)));
            h->f_segstart = static_cast<u32 *>(h->dalloc(4 * (size_t)(h->nnz + 1)));
            h->f_slot = static_cast<u32 *>(h->dalloc(4 * room));
            XSB_CUDA(cudaMemsetAsync(h->f_slot, 0xff, 4 * room, s)); // kNoSlot where build_frozen_map writes nothing
            build_frozen_map(s, sorted, nmap, h->nnz, h->f_perm, h->f_segstart, h->f_slot, h->lc);
            h->dfree(A);
            h->dfree(B);
            h->dfree(ws);
            h->dfree(h->fs_slot);
            h->dfree(h->fs_send_pos);
            h->fs_slot = nullptr;
            h->fs_send_pos = nullptr;
            for (int r = 0; r < h->nranks; ++r)
                h->fs_recv[r] = r == h->rank ? 0 : (i64)recv_counts[r];
            h->fs_low = low;
            h->fs_total = total;
            h->frozen = true;
            h->fs_state = 2;
            h->sync();
        }
        catch (...)
        {
            h->drop_frozen();
            throw;
        }
        return XSB_OK;
    });
}

int32_t xsb_frozen_slab_counts(const xsb_matrix *hc, int64_t *send_counts, int64_t *recv_counts)
{
    xsb_matrix *h = const_cast<xsb_matrix *>(hc);
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->nranks > 0, XSB_ESTATE, "not a slab handle");
        REQUIRE(h->fs_state == 2, XSB_ESTATE, "no frozen slab stream");
        for (int r = 0; r < h->nranks; ++r)
        {
            if (send_counts)
                send_counts[r] = h->fs_send[r];
            if (recv_counts)
                recv_counts[r] = h->fs_recv[r];
        }
        return XSB_OK;
    });
}

namespace
{
void slab_step_check(xsb_matrix *h, int64_t count)
{
    slab_freeze_check(h);
    REQUIRE(h->fs_state == 2, XSB_ESTATE,
            h->fs_state == 1 ? "the slab freeze is not complete: xsb_freeze_slab_finish first" : "no frozen slab stream");
    REQUIRE(count == h->f_count, XSB_ESIZE, "value count differs from the frozen stream");
}
} // namespace

int32_t xsb_reassemble_slab_pack(xsb_matrix *h, const double *V, int64_t count, double *send_values)
{
    return guard(h, [&]() -> int32_t {
        slab_step_check(h, count);
        if (h->fs_foreign == 0)
            return XSB_OK;
        REQUIRE(V, XSB_EINVAL, "NULL array");
        REQUIRE(send_values && is_device_ptr(send_values), XSB_EINVAL, "send buffer must be device memory");
        DevIn dV(h, V, 8 * (size_t)count);
        slab_pack_values(h->stream, static_cast<const double *>(dV.ptr), h->fs_send_idx, h->fs_foreign, send_values, h->lc);
        return XSB_OK;
    });
}

int32_t xsb_reassemble_slab_values(xsb_matrix *h, const double *V, int64_t count, const double *recv_values, int32_t mode,
                                   int32_t zero_first)
{
    return guard(h, [&]() -> int32_t {
        slab_step_check(h, count);
        REQUIRE(mode == XSB_DETERMINISTIC || mode == XSB_FAST, XSB_EINVAL, "unknown summation mode");
        const i64 nrecv = h->fs_total - h->f_count;
        REQUIRE(count == 0 || V, XSB_EINVAL, "NULL array");
        REQUIRE(nrecv == 0 || recv_values, XSB_EINVAL, "NULL receive buffer");
        DevIn dV(h, V, 8 * (size_t)count), dR(h, recv_values, 8 * (size_t)nrecv);
        const SlabValues sv{static_cast<const double *>(dR.ptr), (u32)h->fs_low, (u32)h->f_count};
        const double *v = static_cast<const double *>(dV.ptr);
        if (mode == XSB_DETERMINISTIC)
            reassemble_deterministic(h->stream, v, h->f_perm, h->f_segstart, h->nnz, h->nzval, zero_first != 0, h->lc, &sv);
        else
        {
            if (zero_first)
                zero_values(h->stream, h->nzval, h->nnz, h->lc);
            reassemble_fast(h->stream, v, h->f_slot, h->fs_total, h->nzval, h->lc, &sv);
        }
        return XSB_OK;
    });
}

int32_t xsb_mark_dirichlet(xsb_matrix *h, double penalty, uint8_t *marker_out)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && marker_out, XSB_EINVAL, "NULL argument");
        REQUIRE(h->m == h->n, XSB_ESIZE, "Dirichlet passes need a square matrix");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "flush! first");
        DevOut dM(h, marker_out, (size_t)h->n);
        mark_dirichlet(h->stream, h->view(), h->n, h->idx64, h->base, penalty, static_cast<unsigned char *>(dM.ptr),
                       h->lc);
        dM.finish();
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_eliminate_dirichlet(xsb_matrix *h, const uint8_t *marker)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && marker, XSB_EINVAL, "NULL argument");
        REQUIRE(h->m == h->n, XSB_ESIZE, "Dirichlet passes need a square matrix");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "flush! first");
        DevIn dM(h, marker, (size_t)h->n);
        eliminate_dirichlet(h->stream, h->view(), h->n, h->idx64, h->base, static_cast<const unsigned char *>(dM.ptr),
                            h->lc);
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_mul(xsb_matrix *h, const void *x, void *y)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && x && y, XSB_EINVAL, "NULL argument");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "staged insertions are pending: flush first");
        REQUIRE(h->nnz < (1ll << 32) && h->m < (1ll << 32) - 1 && h->n < (1ll << 32), XSB_EINVAL,
                "matrix too large for the 32-bit row-major map");
        cudaStream_t s = h->stream;
        if (!h->csr_map)
        { // once per pattern
            h->csr_map = static_cast<u32 *>(h->dalloc(csr_map_bytes(h->m, h->nnz)));
            const size_t cnt = (size_t)std::max<i64>(h->nnz, 1);
            Rec *ta = static_cast<Rec *>(h->dalloc(sizeof(Rec) * cnt));
            Rec *tb = static_cast<Rec *>(h->dalloc(sizeof(Rec) * cnt));
            void *ws = h->dalloc(sort_workspace_bytes((u64)cnt));
            build_csr_map(s, h->view(), h->m, h->n, h->idx64, h->base, ta, tb, ws, h->csr_map, h->lc);
            h->dfree(ws);
            h->dfree(tb);
            h->dfree(ta);
        }
        DevIn dx(h, x, sizeof(double) * (size_t)h->n);
        DevOut dy(h, y, sizeof(double) * (size_t)h->m);
        csr_mul(s, h->csr_map, h->m, h->nnz, h->nzval, static_cast<const double *>(dx.ptr), static_cast<double *>(dy.ptr),
                h->lc);
        dy.finish();
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_pattern_hash(xsb_matrix *h, uint64_t *hash_out)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && hash_out, XSB_EINVAL, "NULL argument");
        pattern_hash(h->stream, h->view(), h->n, h->idx64, h->d_scal + 4, h->lc);
        *hash_out = read_scalar(h, 4);
        return XSB_OK;
    });
}

int32_t xsb_pattern_equal(xsb_matrix *a, xsb_matrix *b, int32_t *equal_out)
{
    if (!a || !b || !equal_out)
        return XSB_EINVAL;
    if (a == b)
    {
        *equal_out = 1;
        return XSB_OK;
    }
    // lock both handles in address order (two threads comparing the same pair the other way round must not deadlock)
    xsb_matrix *first = a < b ? a : b, *second = a < b ? b : a;
    std::lock_guard<std::recursive_mutex> l1(first->mu), l2(second->mu);
    return guard(a, [&]() -> int32_t {
        REQUIRE(a->pending() == 0 && b->pending() == 0, XSB_ESTATE, "flush! both matrices first");
        if (a->m != b->m || a->n != b->n || a->nnz != b->nnz)
        {
            *equal_out = 0;
            return XSB_OK;
        }
        if (a->device != b->device)
        { // no common address space to compare in: equal fingerprints (64-bit, both patterns 0-based would be needed)
            REQUIRE(a->base == b->base && a->idx64 == b->idx64, XSB_EINVAL,
                    "handles on different devices must share index type and base");
            write_scalar(a, 4, 0);
            pattern_hash(a->stream, a->view(), a->n, a->idx64, a->d_scal + 4, a->lc);
            const u64 ha = read_scalar(a, 4);
            XSB_CUDA(cudaSetDevice(b->device));
            write_scalar(b, 4, 0);
            pattern_hash(b->stream, b->view(), b->n, b->idx64, b->d_scal + 4, b->lc);
            const u64 hb = read_scalar(b, 4);
            XSB_CUDA(cudaSetDevice(a->device));
            *equal_out = ha == hb;
            return XSB_OK;
        }
        b->sync(); // b's arrays are read on a's stream
        write_scalar(a, 4, 0);
        pattern_diff(a->stream, a->view(), a->idx64, a->base, b->view(), b->idx64, b->base, a->n, a->d_scal + 4, a->lc);
        *equal_out = read_scalar(a, 4) == 0ull;
        return XSB_OK;
    });
}

namespace {
// rowval / nzval of `nnz` entries in one store from the handle's cache, as the flush lays them out
void *alloc_store(xsb_matrix *h, i64 nnz, size_t *bytes, void **rowval, double **nzval)
{
    const size_t rv_bytes = (h->isz() * (size_t)nnz + 15) & ~(size_t)15;
    *bytes = rv_bytes + 8 * (size_t)nnz;
    unsigned char *st = static_cast<unsigned char *>(h->dalloc(*bytes));
    *rowval = st;
    *nzval = reinterpret_cast<double *>(st + rv_bytes);
    return st;
}

void check_result_nnz(const xsb_matrix *h, u64 nnz)
{
    REQUIRE(h->idx64 || nnz + (u64)h->base <= (u64)INT32_MAX, XSB_EINVAL,
            "the result has " + std::to_string(nnz) + " entries, more than Int32 indices can address");
}
} // namespace

int32_t xsb_add(xsb_matrix *a, xsb_matrix *b, int32_t op, xsb_matrix **out)
{
    if (out)
        *out = nullptr;
    if (!a || !b || !out)
    {
        g_err = "NULL argument";
        return XSB_EINVAL;
    }
    // lock both handles in address order (two threads adding the same pair the other way round must not deadlock)
    xsb_matrix *first = a < b ? a : b, *second = a < b ? b : a;
    std::lock_guard<std::recursive_mutex> l1(first->mu), l2(second->mu);
    return guard(a, [&]() -> int32_t {
        REQUIRE(op == XSB_OP_ADD || op == XSB_OP_SUB, XSB_EINVAL, "op must be XSB_OP_ADD or XSB_OP_SUB");
        REQUIRE(a->nranks == 0 && b->nranks == 0, XSB_ESTATE, "+ and - work on whole matrices, not on column slabs");
        REQUIRE(a->block_size == 0 && b->block_size == 0, XSB_ESTATE, "+ and - do not take a pointblock result");
        REQUIRE(a->pending() == 0 && b->pending() == 0, XSB_ESTATE, "flush! both matrices first");
        REQUIRE(a->m == b->m && a->n == b->n, XSB_ESIZE,
                "DimensionMismatch: dimensions must match: a has dims (" + std::to_string(a->m) + ", " +
                    std::to_string(a->n) + "), b has dims (" + std::to_string(b->m) + ", " + std::to_string(b->n) + ")");
        REQUIRE(a->idx64 == b->idx64 && a->base == b->base, XSB_EINVAL, "A and B must share index type and base");
        REQUIRE(a->device == b->device, XSB_EINVAL, "A and B must live on the same device");
        xsb_matrix *c = nullptr;
        const int32_t rc = create_impl(a->m, a->n, 0, 0, nullptr, XSB_F64, a->idx64 ? XSB_I64 : XSB_I32, a->base, 1,
                                       a->device, &c);
        if (rc != XSB_OK)
            throw ApiError(rc, "+/-: " + g_err);
        try
        {
            a->sync(); // A and B are read on C's stream
            b->sync();
            const CscView va = a->view(), vb = b->view();
            const int alg = op == XSB_OP_ADD ? kAlgAdd : kAlgSub;
            void *ws = c->dalloc(merge_workspace_bytes(va.nnz, vb.nnz));
            merge_count(c->stream, alg, va, &vb, a->n, a->idx64, a->base, ws, c->lc);
            XSB_CUDA(cudaMemcpyAsync(c->h_scal, ws, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
            c->sync();
            const u64 nnz = c->h_scal[0];
            check_result_nnz(c, nnz);
            c->dfree(c->csc_store);
            c->csc_store = alloc_store(c, (i64)nnz, &c->csc_store_bytes, &c->rowval, &c->nzval);
            merge_write(c->stream, alg, va, &vb, a->n, a->idx64, a->base, ws, c->colptr, c->rowval, c->nzval, c->lc);
            c->nnz = (i64)nnz;
            c->dfree(ws);
            c->sync();
        }
        catch (...)
        {
            xsb_destroy(c);
            XSB_CUDA(cudaSetDevice(a->device));
            throw;
        }
        *out = c;
        return XSB_OK;
    });
}

int32_t xsb_dropzeros(xsb_matrix *h, int64_t *nnz_out, int32_t *pattern_changed)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "staged insertions are pending: flush first");
        REQUIRE(h->block_size == 0, XSB_ESTATE, "dropzeros! does not take a pointblock result");
        const CscView v = h->view();
        void *ws = h->dalloc(merge_workspace_bytes(v.nnz, 0));
        try
        {
            merge_count(h->stream, kAlgKeep, v, nullptr, h->n, h->idx64, h->base, ws, h->lc);
            XSB_CUDA(cudaMemcpyAsync(h->h_scal, ws, sizeof(u64), cudaMemcpyDeviceToHost, h->stream));
            h->sync();
            const i64 nnz = (i64)h->h_scal[0];
            if (nnz != h->nnz)
            {
                void *colptr = h->dalloc(h->isz() * (size_t)(h->n + 1));
                size_t bytes = 0;
                void *rowval = nullptr;
                double *nzval = nullptr;
                void *store = alloc_store(h, nnz, &bytes, &rowval, &nzval);
                merge_write(h->stream, kAlgKeep, v, nullptr, h->n, h->idx64, h->base, ws, colptr, rowval, nzval, h->lc);
                h->dfree(h->colptr);
                h->dfree(h->csc_store);
                h->colptr = colptr;
                h->csc_store = store;
                h->csc_store_bytes = bytes;
                h->rowval = rowval;
                h->nzval = nzval;
                h->drop_frozen(); // the frozen maps (plain or slab), a half-made slab freeze and the csr_map
                h->sync();
            }
            h->dfree(ws);
            if (nnz_out)
                *nnz_out = nnz;
            if (pattern_changed)
                *pattern_changed = nnz != v.nnz ? 1 : 0;
            h->nnz = nnz;
        }
        catch (...)
        {
            h->dfree(ws);
            throw;
        }
        return XSB_OK;
    });
}

int32_t xsb_pointblock(xsb_matrix *h, int32_t blocksize, xsb_matrix **out)
{
    if (out)
        *out = nullptr;
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && out, XSB_EINVAL, "NULL argument");
        REQUIRE(blocksize >= 1, XSB_EINVAL, "blocksize must be >= 1");
        REQUIRE(h->nranks == 0, XSB_ESTATE, "pointblock works on a whole matrix, not on a column slab");
        REQUIRE(h->pending() == 0, XSB_ESTATE, "flush! before pointblock");
        const i64 bs = blocksize;
        const i64 nb = h->n / bs; // nblock = n / blocksize, extendable.jl:299
        REQUIRE(nb >= 1, XSB_ESIZE, "blocksize exceeds the matrix size");
        xsb_matrix *b = nullptr;
        const int32_t rc = create_impl(nb, nb, 0, 0, nullptr, XSB_F64, h->idx64 ? XSB_I64 : XSB_I32, h->base, 1,
                                       h->device, &b);
        if (rc != XSB_OK)
            throw ApiError(rc, "pointblock: " + g_err);
        try
        {
            h->sync(); // the pattern handle works on its own stream
            if (h->nnz > 0)
            {
                Rec *dst = begin_emit(b, 0, XSB_RAW, h->nnz);
                write_scalar(b, 1, ~0ull);
                pointblock_emit(b->stream, h->view(), h->n, h->idx64, h->base, bs, nb, b->Ls, dst, b->d_scal + 1,
                                b->lc);
                const u64 bad = read_scalar(b, 1);
                if (bad != ~0ull)
                    throw ApiError(XSB_EBOUNDS, "BoundsError: entry " + std::to_string(bad) +
                                                    " of the matrix falls outside the " + std::to_string(nb) + "x" +
                                                    std::to_string(nb) + " block matrix");
                end_emit(b, 0, XSB_RAW, h->nnz);
                int64_t nnzb = 0;
                int32_t changed = 0;
                const int32_t frc = do_flush(b, XSB_DETERMINISTIC, XSB_COMBINE_SEED, &nnzb, &changed);
                if (frc != XSB_OK)
                    throw ApiError(frc, "pointblock: " + b->err);
            }
            b->block_size = (int)bs;
            const size_t nbytes = sizeof(double) * (size_t)b->nnz * (size_t)(bs * bs);
            b->blocks = static_cast<double *>(b->dalloc(nbytes));
            if (b->nnz > 0)
            {
                XSB_CUDA(cudaMemsetAsync(b->blocks, 0, nbytes, b->stream));
                write_scalar(b, 1, ~0ull);
                pointblock_fill(b->stream, h->view(), h->n, h->idx64, h->base, bs, b->view(), b->blocks,
                                b->d_scal + 1, b->lc);
                const u64 lost = read_scalar(b, 1);
                REQUIRE(lost == ~0ull, XSB_EINVAL, "pointblock: entry without a block (internal error)");
            }
            b->sync();
        }
        catch (...)
        {
            xsb_destroy(b);
            XSB_CUDA(cudaSetDevice(h->device));
            throw;
        }
        *out = b;
        return XSB_OK;
    });
}

int32_t xsb_block_size(const xsb_matrix *hb, int32_t *blocksize)
{
    if (!hb || !blocksize)
        return XSB_EINVAL;
    *blocksize = hb->block_size;
    return XSB_OK;
}

int32_t xsb_fetch_blocks(xsb_matrix *hb, void *blocks_out)
{
    return guard(hb, [&]() -> int32_t {
        REQUIRE(hb && blocks_out, XSB_EINVAL, "NULL argument");
        REQUIRE(hb->blocks != nullptr && hb->block_size > 0, XSB_ESTATE, "not a result of xsb_pointblock");
        const size_t nbytes = sizeof(double) * (size_t)hb->nnz * (size_t)hb->block_size * (size_t)hb->block_size;
        if (nbytes)
            XSB_CUDA(cudaMemcpyAsync(blocks_out, hb->blocks, nbytes, cudaMemcpyDefault, hb->stream));
        hb->sync();
        return XSB_OK;
    });
}

int32_t xsb_stream_count_fdrand(int64_t nx, int64_t ny, int64_t nz, int64_t *count)
{
    if (!count || nx < 1 || ny < 1 || nz < 1)
        return XSB_EINVAL;
    *count = fdrand_prefix(nx, ny, nz, nx * ny * nz);
    return XSB_OK;
}

int32_t xsb_stream_count_p1fem(int64_t nxn, int64_t nyn, int64_t nzn, int64_t *count)
{
    if (!count || nxn < 2 || nyn < 2 || nzn < 2)
        return XSB_EINVAL;
    *count = 20 * 6 * (nxn - 1) * (nyn - 1) * (nzn - 1);
    return XSB_OK;
}

int32_t xsb_stream_count_blockrd(int64_t nx, int64_t ny, int64_t nz, int32_t ns, int64_t *count)
{
    if (!count || nx < 1 || ny < 1 || nz < 1 || ns < 1)
        return XSB_EINVAL;
    *count = blockrd_count(nx, ny, nz, ns);
    return XSB_OK;
}

int32_t xsb_emit_fdrand_range(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz, uint64_t seed,
                              int32_t ones, int32_t flavour, int64_t l_begin, int64_t l_end)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(nx >= 1 && ny >= 1 && nz >= 1, XSB_EINVAL, "grid dimensions must be >= 1");
        const i64 N = nx * ny * nz;
        REQUIRE(h->m == N && h->n_global == N, XSB_ESIZE, "Matrix size mismatch"); // sprand.jl:66-68
        REQUIRE(0 <= l_begin && l_begin <= l_end && l_end <= N, XSB_EINVAL, "bad node range");
        const i64 count = fdrand_prefix(nx, ny, nz, l_end) - fdrand_prefix(nx, ny, nz, l_begin);
        Rec *dst = begin_emit(h, tid, flavour, count);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0;
        if (runs_begin(h, tid, count, emit_fdrand_chunks(l_begin, l_end), &rt, &chunk0, &pos0))
        {
            const u32 chunks = emit_fdrand_grouped(h->stream, nx, ny, nz, seed, ones, h->Ls, (u32)tid, (u32)flavour, l_begin,
                                                   l_end, dst, h->lc, h->stage_flags(tid), rt, chunk0, pos0);
            end_emit(h, tid, flavour, count);
            runs_end(h, count, chunks);
            return XSB_OK;
        }
        emit_fdrand(h->stream, nx, ny, nz, seed, ones, h->Ls, (u32)tid, (u32)flavour, l_begin, l_end, dst, h->lc,
                    h->stage_flags(tid));
        end_emit(h, tid, flavour, count);
        return XSB_OK;
    });
}

int32_t xsb_emit_fdrand(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz, uint64_t seed, int32_t ones,
                        int32_t flavour)
{
    return xsb_emit_fdrand_range(h, tid, nx, ny, nz, seed, ones, flavour, 0, nx * ny * nz);
}

int32_t xsb_emit_p1fem_range(xsb_matrix *h, int32_t tid, int64_t nxn, int64_t nyn, int64_t nzn, int32_t flavour,
                             int64_t cz_begin, int64_t cz_end)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(nxn >= 2 && nyn >= 2 && nzn >= 2, XSB_EINVAL, "mesh needs at least 2 nodes per direction");
        const i64 N = nxn * nyn * nzn;
        REQUIRE(h->m == N && h->n_global == N, XSB_ESIZE, "Matrix size mismatch");
        REQUIRE(0 <= cz_begin && cz_begin <= cz_end && cz_end <= nzn - 1, XSB_EINVAL, "bad cube-layer range");
        const i64 count = 20 * 6 * (nxn - 1) * (nyn - 1) * (cz_end - cz_begin);
        Rec *dst = begin_emit(h, tid, flavour, count);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0;
        if (runs_begin(h, tid, count, emit_p1fem_chunks(nxn, nyn, cz_begin, cz_end), &rt, &chunk0, &pos0))
        {
            const u32 chunks = emit_p1fem_grouped(h->stream, nxn, nyn, nzn, h->Ls, (u32)tid, (u32)flavour, cz_begin, cz_end,
                                                  dst, h->lc, h->stage_flags(tid), rt, chunk0, pos0);
            end_emit(h, tid, flavour, count);
            runs_end(h, count, chunks);
            return XSB_OK;
        }
        emit_p1fem(h->stream, nxn, nyn, nzn, h->Ls, (u32)tid, (u32)flavour, cz_begin, cz_end, dst, h->lc,
                   h->stage_flags(tid));
        end_emit(h, tid, flavour, count);
        return XSB_OK;
    });
}

int32_t xsb_emit_p1fem(xsb_matrix *h, int32_t tid, int64_t nxn, int64_t nyn, int64_t nzn, int32_t flavour)
{
    return xsb_emit_p1fem_range(h, tid, nxn, nyn, nzn, flavour, 0, nzn - 1);
}

int32_t xsb_emit_blockrd(xsb_matrix *h, int32_t tid, int64_t nx, int64_t ny, int64_t nz, int32_t ns, uint64_t seed,
                         int32_t flavour)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        REQUIRE(nx >= 1 && ny >= 1 && nz >= 1 && ns >= 1 && ns <= 16, XSB_EINVAL, "bad grid or species count");
        const i64 N = nx * ny * nz * ns;
        REQUIRE(h->m == N && h->n_global == N, XSB_ESIZE, "Matrix size mismatch");
        const i64 count = blockrd_count(nx, ny, nz, ns);
        Rec *dst = begin_emit(h, tid, flavour, count);
        RunTarget rt;
        u32 chunk0 = 0, pos0 = 0;
        const u32 want = emit_blockrd_chunks(nx, ny, nz, ns);
        if (want > 0 && runs_begin(h, tid, count, want, &rt, &chunk0, &pos0))
        {
            const u32 chunks = emit_blockrd_grouped(h->stream, nx, ny, nz, ns, seed, h->Ls, (u32)tid, (u32)flavour, dst,
                                                    h->lc, h->stage_flags(tid), rt, chunk0, pos0);
            end_emit(h, tid, flavour, count);
            runs_end(h, count, chunks);
            return XSB_OK;
        }
        emit_blockrd(h->stream, nx, ny, nz, ns, seed, h->Ls, (u32)tid, (u32)flavour, dst, h->lc, h->stage_flags(tid));
        end_emit(h, tid, flavour, count);
        return XSB_OK;
    });
}

int32_t xsb_debug_fetch_staged(xsb_matrix *h, int32_t tid, void *I, void *J, void *V, int32_t *flavour,
                               int64_t capacity, int64_t *count)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && count, XSB_EINVAL, "NULL argument");
        REQUIRE(tid >= 0 && tid < h->n_tid, XSB_EINVAL, "tid out of range");
        const Stage &st = h->stage[tid];
        *count = st.count;
        if (!I || !J || !V)
            return XSB_OK;
        REQUIRE(capacity >= st.count, XSB_EINVAL, "capacity too small");
        if (st.count == 0)
            return XSB_OK;
        const size_t c = (size_t)st.count;
        DevOut dI(h, I, h->isz() * c), dJ(h, J, h->isz() * c), dV(h, V, 8 * c), dF(h, flavour, 4 * c);
        unpack_records(h->stream, st.buf + st.front, st.count, h->idx64, h->base, h->routed ? h->L : h->Ls, dI.ptr, dJ.ptr,
                       static_cast<double *>(dV.ptr), static_cast<int *>(dF.ptr), h->lc);
        dI.finish();
        dJ.finish();
        dV.finish();
        dF.finish();
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_synchronize(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        h->sync();
        return XSB_OK;
    });
}

int32_t xsb_get_stream(xsb_matrix *h, void **stream_out)
{
    if (!h || !stream_out)
        return XSB_EINVAL;
    *stream_out = h->stream;
    return XSB_OK;
}

int32_t xsb_timer_start(xsb_matrix *h)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h, XSB_EINVAL, "NULL handle");
        XSB_CUDA(cudaEventRecord(h->ev0, h->stream));
        return XSB_OK;
    });
}

int32_t xsb_timer_stop(xsb_matrix *h, float *ms_out)
{
    return guard(h, [&]() -> int32_t {
        REQUIRE(h && ms_out, XSB_EINVAL, "NULL argument");
        XSB_CUDA(cudaEventRecord(h->ev1, h->stream));
        XSB_CUDA(cudaEventSynchronize(h->ev1));
        XSB_CUDA(cudaEventElapsedTime(ms_out, h->ev0, h->ev1));
        return XSB_OK;
    });
}

int32_t xsb_set_strategy(xsb_matrix *h, int32_t strategy)
{
    if (!h || (strategy != XSB_STRATEGY_AUTO && strategy != XSB_STRATEGY_FULLSORT))
        return XSB_EINVAL;
    h->strategy = strategy;
    return XSB_OK;
}

int32_t xsb_set_grouping(xsb_matrix *h, int32_t grouping)
{
    if (!h || grouping < XSB_GROUPING_AUTO || grouping > XSB_GROUPING_ON)
        return XSB_EINVAL;
    h->grouping = grouping;
    h->grouping_misses = 0;
    h->runs_misses = 0;
    return XSB_OK;
}

int32_t xsb_set_precount(xsb_matrix *h, int32_t enable)
{
    if (!h)
        return XSB_EINVAL;
    h->precount = enable != 0;
    return XSB_OK;
}

int32_t xsb_set_preaggregation(xsb_matrix *h, int32_t enable)
{
    if (!h)
        return XSB_EINVAL;
    h->preagg = enable != 0;
    h->preagg_misses = 0;
    return XSB_OK;
}

int32_t xsb_set_profiling(xsb_matrix *h, int32_t enable)
{
    if (!h)
        return XSB_EINVAL;
    h->profiling = enable != 0;
    return XSB_OK;
}

int32_t xsb_get_flush_stats(const xsb_matrix *h, xsb_flush_stats *out)
{
    if (!h || !out)
        return XSB_EINVAL;
    *out = h->stats;
    return XSB_OK;
}

int32_t xsb_kernel_launches(const xsb_matrix *h, int64_t *count)
{
    if (!h || !count)
        return XSB_EINVAL;
    *count = h->lc.total;
    return XSB_OK;
}

} // extern "C"
