// Host side of the TAD engine: C ABI (include/theia_tad.h), job queue, workspace, phase
// orchestration.  One worker thread per context runs jobs FIFO on one CUDA stream; callers
// (the controller's workers, pkg/controller/util.go:43) only enqueue and poll.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "../../include/theia_tad.h"
#include "tad_kernels.h"
#include "tad_nccl.h"

using namespace tad;

namespace {

struct DevBuf {            // grow-only device buffer (ensure()); freed with the context that owns it
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;               // owns its allocation
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
};

struct PinnedBlock {
    void *p = nullptr;
    size_t cap = 0;
};

constexpr int kMaxEvents = 24;
constexpr int kMaxChunks = 16;          // host-resident input is copied and histogrammed in chunks
constexpr int kMaxRanks = 8;
constexpr int kMaxXChunks = kMaxSeg / kMaxRanks;   // exchange chunks: scatter of chunk c+1 overlaps the all-to-all of chunk c
constexpr int kTotalStages = 6;   // ingest, partition, exchange, group, detect, egress

// Layout of the scratch words (u64) of `small` (device, 4096 bytes) and `h_small` (pinned, kSmallWords).  An all-gather
// sends from one slot and receives one entry per rank at another.  Each slot names the phase that owns it.
enum SmallSlot : int {
    kSlotSend = 0,            // agree on rows, gather16: this rank's entry of the all-gather
    kSlotSegRows = 0,         // exact multi-GPU partition: rows of each (source rank, chunk) segment in the owned range
    kSlotRows = 8,            // agree on rows: every rank's row count
    kSlotGather16 = 16,       // gather16 (exported-buffer handles, largest shard): 16 words per rank
    kSlotOvf = 32,            // optimistic peer pull: every rank's overflow count
    kSlotFront = 40,          // exact peer pull: rows in front of the owned range in each source's partition
    kSlotBarrier = 48,        // barrier(): the word every rank sends
    kSlotBarrierRecv = 56,    // barrier(): the words every rank receives
    kSlotSendLo = 64,         // exact multi-GPU partition (host only): kMaxRanks + 1 send boundaries per exchange chunk
    kSmallWords = 256,
};
static_assert(kSlotSegRows + kMaxSeg <= kSlotFront, "segment rows and the rows in front of the owned range overlap");
static_assert(kSlotFront + kMaxRanks <= kSlotBarrier, "the rows in front of the owned range overlap the barrier");
static_assert(kSlotSendLo + kMaxXChunks * (kMaxRanks + 1) <= kSmallWords, "send boundaries overrun h_small");

// ---- NUMA placement of pinned host memory --------------------------------------------------------------------------
// On a two-socket box half of the GPUs hang off each socket; a pinned buffer on the wrong socket makes every H2D / D2H
// copy cross the inter-socket link, and eight ranks doing that at once is what held the 8-GPU end-to-end rate down in
// round 1.  Pinned allocations therefore happen with the calling thread temporarily confined to the CPUs of the GPU's
// NUMA node (the driver touches the pages inside cudaHostAlloc: first touch = local), with a PREFERRED memory policy on
// top where the container allows set_mempolicy.  TAD_NUMA=0 switches all of it off.
struct NumaInfo {
    int node = -1;
    cpu_set_t cpus;
    bool ok = false;
};

NumaInfo numa_of_device(int device)
{
    NumaInfo ni;
    CPU_ZERO(&ni.cpus);
    if (const char *e = getenv("TAD_NUMA")) if (atoi(e) == 0) return ni;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return ni; }
    for (char *p = bus; *p; p++) if (*p >= 'A' && *p <= 'Z') *p = (char)(*p - 'A' + 'a');
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    if (!f) return ni;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    if (node < 0) return ni;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return ni;
    char list[4096] = {0};
    if (!fgets(list, sizeof(list), f)) list[0] = 0;
    fclose(f);
    int n = 0;
    for (char *p = list; *p && *p != '\n';) {          // "0-31,64-95"
        char *end = nullptr;
        long a = strtol(p, &end, 10), b = a;
        if (end == p) break;
        if (*end == '-') { p = end + 1; b = strtol(p, &end, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int)c, &ni.cpus); n++; }
        p = *end == ',' ? end + 1 : end;
    }
    // only CPUs this process may use anyway
    cpu_set_t allowed;
    if (sched_getaffinity(0, sizeof(allowed), &allowed) == 0) {
        n = 0;
        for (int c = 0; c < CPU_SETSIZE; c++) {
            if (CPU_ISSET(c, &ni.cpus) && !CPU_ISSET(c, &allowed)) CPU_CLR(c, &ni.cpus);
            if (CPU_ISSET(c, &ni.cpus)) n++;
        }
    }
    ni.node = node;
    ni.ok = n > 0;
    return ni;
}

// Scope guard: the calling thread runs on (and prefers memory of) the GPU's NUMA node while it is alive.
struct NumaScope {
    cpu_set_t saved;
    bool restore = false, policy = false;
    explicit NumaScope(const NumaInfo &ni)
    {
        if (!ni.ok) return;
        if (sched_getaffinity(0, sizeof(saved), &saved) != 0) return;
        if (sched_setaffinity(0, sizeof(ni.cpus), &ni.cpus) == 0) restore = true;
#ifdef SYS_set_mempolicy
        unsigned long mask[16] = {0};
        if (ni.node < (int)(sizeof(mask) * 8)) {
            mask[ni.node / (8 * sizeof(unsigned long))] |= 1ul << (ni.node % (8 * sizeof(unsigned long)));
            policy = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof(mask) * 8) == 0;
        }
#endif
    }
    ~NumaScope()
    {
#ifdef SYS_set_mempolicy
        if (policy) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
#endif
        if (restore) sched_setaffinity(0, sizeof(saved), &saved);
    }
};

double now_ms()
{
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

}  // namespace

struct tad_job {
    tad_ctx *ctx = nullptr;
    tad_job_spec spec{};
    std::vector<uint32_t> ns_ignore;
    tad_columns cols{};
    std::mutex mu;
    std::condition_variable cv;
    tad_status st{};
    std::atomic<int> cancel{0};
    PinnedBlock result_block;
    tad_rows rows{};
    double t_submit = 0;
};

struct tad_ctx {
    tad_config cfg{};
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev[kMaxEvents]{};
    cudaEvent_t chunk_ev[kMaxChunks]{};
    cudaEvent_t start_ev = nullptr;
    cudaEvent_t x_ev[kMaxXChunks + 1]{};
    int exchange_chunks = kMaxXChunks;
    bool exchange_chunks_forced = false;     // TAD_EXCHANGE_CHUNKS given: use it at every world size
    uint64_t exchange_min_rows = 1u << 22;   // below this the exchange is not worth chunking (TAD_EXCHANGE_MIN_ROWS)
    std::mutex mu;
    std::condition_variable cv;
    std::deque<tad_job *> queue;
    std::thread worker;
    bool stop = false;
    int debug_logb = -1;
    int debug_target = 0;      // TAD_GROUP_TARGET: mean rows per bucket (tuning)
    // device workspace (grow-only, reused across jobs; jobs are serialized by the worker)
    DevBuf d_col[10], hist, offsets, cursor, big_list, big_base, cls_list, csr_p, stats, part, csr_v, csr_t, nsb, npb, sbase, outb, ns_ignore, spill,
        dbx, dbi, exch, scan_sync, small, hist_all, seg_off, seg_total, entries, ar_y, ar_pred, ar_lam, ovf;
    int optimistic = 1;      // TAD_OPTIMISTIC=0: always the exact (histogram + scan + scatter) partition
    unsigned long long *h_small = nullptr;   // pinned, kSmallWords x u64 (layout: SmallSlot)
    uint32_t scan_epoch = 0;
    uint32_t *h_stats = nullptr;   // pinned readback of the device scalars
    std::mutex pool_mu;
    std::vector<PinnedBlock> pinned_pool;
    NcclComm nccl;
    NumaInfo numa;                                  // NUMA node of the GPU: pinned buffers and the worker thread live there
    // multi-GPU optimistic partition + peer pull (DESIGN.md section 6): every rank scatters into fixed-capacity slots of an
    // exported buffer (arrival counters in front, slots behind), the peers map it (CUDA IPC) and the owner's group kernel
    // pulls its bucket segments over NVLink -- no histogram pass, no all-to-all, no receive buffer.
    int peer_pull = 1;                              // TAD_PEER_PULL=0: always the exact partition + NCCL all-to-all
    int sort_classes = 0;                           // TAD_SORT_CLASSES=1: capacity-class bucket lists sorted by bucket before the group phase
    DevBuf sortb;
    size_t x_budget = 72ull << 30;                  // largest exported slot buffer (TAD_SLOT_BUDGET_GB); beyond it: exact partition
    DevBuf xbuf;                                    // exported: [counters: B x u32, padded][slots: B x slot x Row32]
    void *peer_x[kMaxRanks]{};                      // peers' xbuf mapped into this process
    bool peers_mapped = false;
    size_t x_agreed = 0;                            // exported size all ranks agreed on at the last (re)mapping
    DevBuf xcnt, xtotal;                            // per-source counts / totals of the owned bucket range
};

namespace {

const char *kErrNames[] = {"ok", "invalid argument", "CUDA error", "out of memory", "NCCL error", "illegal state",
                           "cancelled", "unsupported", "internal error"};

struct JobFail {
    int code;
    char msg[256];
};

[[noreturn]] void fail(int code, const char *fmt, ...)
{
    JobFail f;
    f.code = code;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(f.msg, sizeof(f.msg), fmt, ap);
    va_end(ap);
    throw f;
}

#define CU(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            fail(_e == cudaErrorMemoryAllocation ? TAD_ERR_NOMEM : TAD_ERR_CUDA, "%s: %s (%s:%d)", #expr, \
                 cudaGetErrorString(_e), __FILE__, __LINE__);                                            \
    } while (0)

void *ensure(DevBuf &b, size_t bytes)      // returns b.p
{
    if (bytes <= b.cap) return b.p;
    if (b.p) CU(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = bytes + bytes / 16 + 256;
    want = (want + 255) & ~size_t(255);
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = (bytes + 255) & ~size_t(255);
        CU(cudaMalloc(&b.p, want));
    }
    b.cap = want;
    return b.p;
}

PinnedBlock take_pinned(tad_ctx *ctx, size_t bytes)
{
    {
        std::lock_guard<std::mutex> lk(ctx->pool_mu);
        int best = -1;
        for (size_t i = 0; i < ctx->pinned_pool.size(); i++)
            if (ctx->pinned_pool[i].cap >= bytes && (best < 0 || ctx->pinned_pool[i].cap < ctx->pinned_pool[best].cap))
                best = (int)i;
        if (best >= 0) {
            PinnedBlock b = ctx->pinned_pool[best];
            ctx->pinned_pool.erase(ctx->pinned_pool.begin() + best);
            return b;
        }
    }
    PinnedBlock b;
    b.cap = (bytes + bytes / 8 + 4095) & ~size_t(4095);
    NumaScope numa(ctx->numa);
    CU(cudaHostAlloc(&b.p, b.cap, cudaHostAllocDefault));
    return b;
}

void give_pinned(tad_ctx *ctx, PinnedBlock b)
{
    if (!b.p) return;
    std::lock_guard<std::mutex> lk(ctx->pool_mu);
    ctx->pinned_pool.push_back(b);
}

void set_progress(tad_job *job, int state, int completed)
{
    std::lock_guard<std::mutex> lk(job->mu);
    job->st.state = state;
    job->st.completed_stages = completed;
}

int pick_logb(const tad_ctx *ctx, uint64_t rows)
{
    if (ctx->debug_logb >= 0) return ctx->debug_logb;
    // mean bucket ~ 0.375 * capacity: connection sizes are lumpy, so leave head-room
    // 4 ranks and more: twice the rows per bucket -- half as many, twice as large pieces for the peer pull (group phase at N = 8:
    // 6.3 -> 5.0 ms, at N = 4: 4.4 -> 4.2 ms; profiles/r02/ab8_summary.txt, ab9_summary.txt); every rank derives the same value
    // from the same world size
    uint64_t target = (uint64_t)kGroupTarget * (ctx->cfg.world_size >= 4 ? 2 : 1);
    if (ctx->debug_target > 0) target = (uint64_t)ctx->debug_target;
    int logb = 0;
    while (logb < 22 && (rows >> logb) > target) logb++;
    return logb;
}

size_t col_bytes(int idx, uint64_t rows)
{
    static const size_t w[10] = {4, 4, 2, 2, 1, 4, 4, 8, 4, 4};
    return w[idx] * rows;
}

void *col_ptr(const tad_columns &c, int idx)
{
    switch (idx) {
    case 0: return c.src_ip;
    case 1: return c.dst_ip;
    case 2: return c.src_port;
    case 3: return c.dst_port;
    case 4: return c.proto;
    case 5: return c.flow_start;
    case 6: return c.flow_end;
    case 7: return c.value;
    case 8: return c.src_ns;
    default: return c.dst_ns;
    }
}

struct OutLayout {
    size_t off[11];
    size_t total;
};
// src_ip dst_ip flow_start flow_end (u32) | stddev algo_calc throughput (f64) | ports (u16) | proto anomaly (u8)
OutLayout out_layout(uint64_t cap)
{
    OutLayout L;
    size_t o = 0;
    auto add = [&](int i, size_t w) {
        L.off[i] = o;
        o += (w * cap + 255) & ~size_t(255);
    };
    add(0, 8); add(1, 8); add(2, 8);          // stddev, algo_calc, throughput
    add(3, 4); add(4, 4); add(5, 4); add(6, 4);  // src_ip, dst_ip, flow_start, flow_end
    add(7, 2); add(8, 2);                      // src_port, dst_port
    add(9, 1); add(10, 1);                     // proto, anomaly
    L.total = o;
    return L;
}

OutCols out_cols(void *base, const OutLayout &L)
{
    char *b = static_cast<char *>(base);
    OutCols o;
    o.stddev = reinterpret_cast<double *>(b + L.off[0]);
    o.algo_calc = reinterpret_cast<double *>(b + L.off[1]);
    o.throughput = reinterpret_cast<double *>(b + L.off[2]);
    o.src_ip = reinterpret_cast<uint32_t *>(b + L.off[3]);
    o.dst_ip = reinterpret_cast<uint32_t *>(b + L.off[4]);
    o.flow_start = reinterpret_cast<uint32_t *>(b + L.off[5]);
    o.flow_end = reinterpret_cast<uint32_t *>(b + L.off[6]);
    o.src_port = reinterpret_cast<uint16_t *>(b + L.off[7]);
    o.dst_port = reinterpret_cast<uint16_t *>(b + L.off[8]);
    o.proto = reinterpret_cast<uint8_t *>(b + L.off[9]);
    o.anomaly = reinterpret_cast<uint8_t *>(b + L.off[10]);
    return o;
}

void nccl_ok(int rc) { if (rc) fail(TAD_ERR_NCCL, "%s", nccl_last_error()); }

// Barrier of all ranks on the job stream (an 8-byte all-gather).  Returns the NCCL status.
int barrier(tad_ctx *ctx)
{
    unsigned long long *d = static_cast<unsigned long long *>(ctx->small.p);
    return nccl_allgather(&ctx->nccl, d + kSlotBarrier, d + kSlotBarrierRecv, 8, ctx->stream);
}

// What a partition path leaves for the group phase: where the rows of each owned bucket are, and the row counts.
struct Partition {
    SegDesc seg{};
    SeriesEntry *entries = nullptr;
    uint64_t kept = 0, owned = 0;          // rows of this rank that passed the filters / rows of its bucket range
    const Row32 *ovf_rows = nullptr;       // single-GPU optimistic partition: rows that found their slot full
    uint32_t n_ovf = 0;
    bool sync_at_end = false;              // peers read this rank's exported rows: meet them before the next job
};

// One job on the worker thread.  run_job calls the phases in order; the members are what the phases share.
struct JobRun {
    tad_ctx *const ctx;
    tad_job *const job;
    const tad_job_spec &sp;
    const cudaStream_t st;
    const uint64_t R;                      // rows of this rank
    const bool host_input;
    const int world, me;
    int nchunks = 1;                       // H2D chunks of host input
    const void *dcol[10]{};                // device columns (the caller's own when device-resident)
    ColPtrs c{};
    RowFilter f{};
    uint32_t *d_stats = nullptr;
    unsigned long long *d_small = nullptr;     // layout: SmallSlot
    uint64_t R_total = 0;                  // rows of all ranks
    int logB = 0;                          // B global buckets; this rank owns the Bl buckets from b_lo on
    uint32_t B = 0, Bl = 0, b_lo = 0;
    uint32_t slotM = 0;                    // multi-GPU optimistic partition: slot rows per (bucket, source rank)
    size_t x_cnt_bytes = 0;                // exported buffer: arrival counters in front of the rows
    uint32_t *hist = nullptr, *offsets = nullptr, *cursor = nullptr, *big_list = nullptr, *big_base = nullptr;
    uint32_t *cls_list = nullptr, *nsb = nullptr, *npb = nullptr;
    uint64_t *csr_v = nullptr;             // grouped series (CSR) and series base per bucket
    uint32_t *csr_t = nullptr, *csr_p = nullptr, *sbase = nullptr;
    uint64_t launches = 0;
    int nev = 0, ev_phase[kMaxEvents];

    JobRun(tad_ctx *ctx_, tad_job *job_)
        : ctx(ctx_), job(job_), sp(job_->spec), st(ctx_->stream), R(job_->cols.rows),
          host_input(job_->cols.mem != TAD_MEM_DEVICE && R > 0), world(ctx_->cfg.world_size), me(ctx_->cfg.rank) {}
    // event closing `phase`
    void mark(int phase) { if (nev < kMaxEvents) { CU(cudaEventRecord(ctx->ev[nev], st)); ev_phase[nev++] = phase; } }
    void check_cancel() { if (job->cancel.load()) fail(TAD_ERR_CANCELLED, "job cancelled"); }
    void read_stats()             // device scalars -> ctx->h_stats
    {
        CU(cudaMemcpyAsync(ctx->h_stats, d_stats, ST_COUNT * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    void allgather(const void *send, void *recv, size_t bytes) { nccl_ok(nccl_allgather(&ctx->nccl, send, recv, bytes, st)); }
    SeriesEntry *use_entries(uint64_t owned) { return (SeriesEntry *)ensure(ctx->entries, (owned ? owned : 1) * sizeof(SeriesEntry)); }
    const Row32 *peer_rows(int r) const      // the rows of rank r's exported buffer (this rank's own for r == me)
    {
        return reinterpret_cast<const Row32 *>(static_cast<const char *>(r == me ? ctx->xbuf.p : ctx->peer_x[r]) + x_cnt_bytes);
    }
    uint64_t split(int k, int n) const       // first row of piece k of n (k = n: R); keeps every column 16-byte aligned
    {
        if (k <= 0 || k >= n) return k <= 0 ? 0 : R;
        const uint64_t v = ((R * (uint64_t)k / n) + 15) & ~uint64_t(15);
        return v < R ? v : R;
    }
    ColPtrs offset_cols(uint64_t lo) const   // the device columns from row lo on
    {
        auto at = [&](int i) { return dcol[i] ? static_cast<const char *>(dcol[i]) + col_bytes(i, lo) : nullptr; };
        ColPtrs ck;
        ck.src_ip = (const uint32_t *)at(0); ck.dst_ip = (const uint32_t *)at(1);
        ck.src_port = (const uint16_t *)at(2); ck.dst_port = (const uint16_t *)at(3);
        ck.proto = (const uint8_t *)at(4); ck.flow_start = (const uint32_t *)at(5);
        ck.flow_end = (const uint32_t *)at(6); ck.value = (const uint64_t *)at(7);
        ck.src_ns = (const uint32_t *)at(8); ck.dst_ns = (const uint32_t *)at(9);
        return ck;
    }
    // First pass over the input: launch(cols, rows) on each H2D chunk once it has landed (host input; the copy and the
    // overlapped pass are accounted as TAD_PHASE_H2D), or once on the device-resident columns.
    template <class Launch>
    void over_input(int phase_if_device, Launch launch)
    {
        if (host_input) {
            for (int k = 0; k < nchunks; k++) {
                const uint64_t lo = split(k, nchunks), hi = split(k + 1, nchunks);
                CU(cudaStreamWaitEvent(st, ctx->chunk_ev[k], 0));
                if (hi <= lo) continue;
                CU(launch(offset_cols(lo), hi - lo)); launches++;
            }
            mark(TAD_PHASE_H2D);
        } else {
            CU(launch(c, R)); launches += R ? 1 : 0;
            mark(phase_if_device);
        }
    }

    // ---- ingest: host columns -> device (device-resident columns are used in place) -------
    // Host input is copied in chunks on a second stream; the bucket histogram is additive, so the
    // histogram of chunk i runs while chunk i+1 is still on the PCIe bus.
    void ingest()
    {
        CU(cudaSetDevice(ctx->cfg.device));
        set_progress(job, TAD_STATE_RUNNING, 0);
        d_stats = (uint32_t *)ensure(ctx->stats, 64 * sizeof(uint32_t));
        CU(cudaMemsetAsync(d_stats, 0, 64 * sizeof(uint32_t), st));
        if (!ctx->scan_sync.p) CU(cudaMemsetAsync(ensure(ctx->scan_sync, scan_sync_bytes()), 0, scan_sync_bytes(), st));
        const tad_columns &hc = job->cols;
        for (int i = 0; i < 10; i++) {
            void *src = col_ptr(hc, i);
            if (src && R > 0) dcol[i] = hc.mem == TAD_MEM_DEVICE ? src : ensure(ctx->d_col[i], col_bytes(i, R));
        }
        if (host_input)            // ~8M rows (232 MB) per chunk
            nchunks = (int)std::min<uint64_t>(kMaxChunks, (R + (8u << 20) - 1) / (8u << 20));
        mark(-1);
        if (host_input) {
            CU(cudaEventRecord(ctx->start_ev, st));
            CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->start_ev, 0));   // workspace of the previous job is free
            for (int k = 0; k < nchunks; k++) {
                const uint64_t lo = split(k, nchunks), hi = split(k + 1, nchunks);
                for (int i = 0; i < 10 && hi > lo; i++)
                    if (dcol[i])
                        CU(cudaMemcpyAsync((char *)dcol[i] + col_bytes(i, lo), (const char *)col_ptr(hc, i) + col_bytes(i, lo),
                                           col_bytes(i, hi - lo), cudaMemcpyHostToDevice, ctx->copy_stream));
                CU(cudaEventRecord(ctx->chunk_ev[k], ctx->copy_stream));
            }
        }
        c = offset_cols(0);
        f.start_time = sp.start_time; f.end_time = sp.end_time;
        if (!job->ns_ignore.empty() && (c.src_ns || c.dst_ns)) {
            ensure(ctx->ns_ignore, job->ns_ignore.size() * 4);
            CU(cudaMemcpyAsync(ctx->ns_ignore.p, job->ns_ignore.data(), job->ns_ignore.size() * 4, cudaMemcpyHostToDevice, st));
            f.n_ns_ignore = (uint32_t)job->ns_ignore.size();
            f.ns_ignore = static_cast<const uint32_t *>(ctx->ns_ignore.p);
        }
    }
    // ---- agree on the rows of the table, pick the buckets (the same global count on every rank) ----------------------
    void pick_buckets()
    {
        R_total = R;
        d_small = (unsigned long long *)ensure(ctx->small, 4096);
        if (world > 1 && sp.global_rows) {
            R_total = sp.global_rows;      // the host counted the table: no start-of-job collective, no host sync
        } else if (world > 1) {
            ctx->h_small[kSlotSend] = R;
            CU(cudaMemcpyAsync(d_small + kSlotSend, ctx->h_small + kSlotSend, 8, cudaMemcpyHostToDevice, st));
            allgather(d_small + kSlotSend, d_small + kSlotRows, 8);
            CU(cudaMemcpyAsync(ctx->h_small, d_small + kSlotRows, 8 * world, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            mark(TAD_PHASE_SYNC);          // arrival skew of the ranks at job start (avoided when the host passes global_rows)
            R_total = 0;
            for (int r = 0; r < world; r++) R_total += ctx->h_small[r];
        }
        logB = pick_logb(ctx, R_total);
        int logW = 0;
        while ((1 << logW) < world) logW++;
        if (logB < logW) logB = logW;
        B = 1u << logB;                 // global buckets
        Bl = B >> logW;                 // buckets owned by one rank
        b_lo = Bl * (uint32_t)me;
        slotM = std::max<uint32_t>(256u, (uint32_t)kGroupCap / (uint32_t)world);
        x_cnt_bytes = (((size_t)B * 4) + 65535) & ~size_t(65535);
        hist = (uint32_t *)ensure(ctx->hist, (size_t)B * 4);
        offsets = (uint32_t *)ensure(ctx->offsets, ((size_t)B + 1) * 4);
        cursor = (uint32_t *)ensure(ctx->cursor, (size_t)B * 4);
        big_list = (uint32_t *)ensure(ctx->big_list, (size_t)B * 4);
        big_base = (uint32_t *)ensure(ctx->big_base, ((size_t)B + 1) * 4);
        cls_list = (uint32_t *)ensure(ctx->cls_list, (size_t)B * 4 * 3);
        nsb = (uint32_t *)ensure(ctx->nsb, (size_t)Bl * 4);
        npb = (uint32_t *)ensure(ctx->npb, (size_t)Bl * 4);
        // part[] (exact partition: 32 B per local row) is not needed when the multi-GPU optimistic path runs out of the exported
        // slot buffer; the exact multi-GPU branch allocates it on demand
        if (world == 1) ensure(ctx->part, (R ? R : 1) * sizeof(Row32));
        CU(cudaMemsetAsync(nsb, 0, (size_t)Bl * 4, st));
        CU(cudaMemsetAsync(npb, 0, (size_t)Bl * 4, st));
    }
    // ---- partition: an optimistic path where it applies; where it falls back, the exact path for the world size
    Partition partition()
    {
        Partition p;
        if (world == 1 && ctx->optimistic && R > 0 && (uint64_t)B * kGroupCap * sizeof(Row32) <= (64ull << 30) &&
            local_slots(p))
            return p;
        const size_t x_need = x_cnt_bytes + (size_t)B * slotM * sizeof(Row32);
        if (world > 1 && ctx->peer_pull && ctx->optimistic && R_total > 0 && (uint64_t)B * slotM <= (1ull << 31) &&
            x_need <= ctx->x_budget && peer_slots(p, x_need))
            return p;
        return world == 1 ? exact_local() : exact_multi();
    }
    // ---- single GPU, optimistic partition: no histogram pass.  Bucket b owns a fixed slot of kGroupCap rows; a
    // row that finds its slot full goes to the overflow list, and such buckets take the spill path.  With host input
    // the scatter of H2D chunk i runs while chunk i+1 is on the bus.  Falls back to the exact two-pass partition
    // when the overflow list fills up (heavily skewed tables).
    bool local_slots(Partition &p)
    {
        constexpr uint32_t kSlot = kGroupCap;      // = the largest shared-memory class: overflow is as rare as a spill was
        const uint64_t ovf_cap = std::max<uint64_t>(1u << 20, R / 32);
        Row32 *part = (Row32 *)ensure(ctx->part, (uint64_t)B * kSlot * sizeof(Row32));
        Row32 *ovf = (Row32 *)ensure(ctx->ovf, ovf_cap * sizeof(Row32));
        CU(cudaMemsetAsync(cursor, 0, (size_t)B * 4, st));
        mark(-1);
        over_input(TAD_PHASE_SCATTER, [&](const ColPtrs &ck, uint64_t n) {
            return launch_scatter(st, ck, n, f, logB, cursor, part, kSlot, ovf, (uint32_t)ovf_cap, d_stats + ST_OVF);
        });
        // arrival counts -> (virtual) bucket offsets, capacity-class lists, list of over-full buckets
        CU(launch_bucket_scan(st, cursor, offsets, hist /* unused cursor copy */, B, kSlot, big_list, big_base, cls_list,
                              d_stats, ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        mark(TAD_PHASE_SCAN);
        read_stats();
        if (ctx->h_stats[ST_OVF] <= ovf_cap) {
            p.n_ovf = ctx->h_stats[ST_OVF];
            p.ovf_rows = ovf;
            p.kept = p.owned = ctx->h_stats[ST_KEPT];
            p.seg.nseg = 1; p.seg.base[0] = part; p.seg.off[0] = offsets; p.seg.stride = kSlot;
            p.entries = use_entries(p.owned);
            return true;
        }
        CU(cudaMemsetAsync(d_stats, 0, 64 * sizeof(uint32_t), st));      // discard; redo exactly
        return false;
    }
    // ---- exported buffer + peer mappings (multi-GPU peer pull) -----------------------------------------------------------
    void gather16()        // blocking 128-byte all-gather through pinned memory (rare: regrow, exact-path row counts)
    {
        CU(cudaMemcpyAsync(d_small + kSlotSend, ctx->h_small + kSlotSend, 16 * 8, cudaMemcpyHostToDevice, st));
        allgather(d_small + kSlotSend, d_small + kSlotGather16, 16 * 8);
        CU(cudaMemcpyAsync(ctx->h_small + kSlotGather16, d_small + kSlotGather16, 16 * 8 * world, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    // Every rank calls this with the SAME `need` in the same job (it depends only on values all ranks share), so all ranks
    // regrow together: unmap, barrier (nobody maps a buffer that is about to be freed), reallocate, exchange the IPC
    // handles, map.  First job or a larger table only.
    void ensure_exported(size_t need)
    {
        // the decision must be the same on every rank: it is taken on the size the ranks last agreed on, not on the local
        // capacity (which may differ when one rank's allocation fell back to the exact size under memory pressure)
        if (need <= ctx->x_agreed && ctx->peers_mapped) return;
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        for (int r = 0; r < world; r++)
            if (ctx->peer_x[r]) { CU(cudaIpcCloseMemHandle(ctx->peer_x[r])); ctx->peer_x[r] = nullptr; }
        ctx->peers_mapped = false;
        memset(ctx->h_small + kSlotSend, 0, 16 * 8);
        gather16();
        ensure(ctx->xbuf, need);
        cudaIpcMemHandle_t mine;
        CU(cudaIpcGetMemHandle(&mine, ctx->xbuf.p));
        memset(ctx->h_small + kSlotSend, 0, 16 * 8);
        ctx->h_small[kSlotSend] = ctx->xbuf.cap;
        memcpy(ctx->h_small + kSlotSend + 2, &mine, sizeof(mine));
        gather16();
        for (int r = 0; r < world; r++) {
            if (r == me) continue;
            cudaIpcMemHandle_t h;
            memcpy(&h, ctx->h_small + kSlotGather16 + 16 * r + 2, sizeof(h));
            if (ctx->h_small[kSlotGather16 + 16 * r] < need) fail(TAD_ERR_INTERNAL, "rank %d exports a smaller partition buffer", r);
            cudaError_t e = cudaIpcOpenMemHandle(&ctx->peer_x[r], h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                cudaGetLastError();
                ctx->peer_x[r] = nullptr;
                fail(TAD_ERR_CUDA, "cannot map the partition buffer of rank %d (%s); set TAD_PEER_PULL=0 on every rank to "
                                   "exchange rows through NCCL instead", r, cudaGetErrorString(e));
            }
        }
        ctx->peers_mapped = true;
        ctx->x_agreed = need;
    }
    // ---- several GPUs, optimistic partition + peer pull ---------------------------------------------------------------
    // Every rank scatters its rows into fixed-capacity slots of ALL global buckets (slot = kGroupCap / world rows: a
    // source holds 1/world of a bucket on average) inside a buffer its peers have mapped with CUDA IPC.  One 8-byte
    // all-gather after the scatter is the barrier "every rank's slots are complete" and carries the overflow counts: if
    // any slot overflowed anywhere, all ranks take the exact path (same decision everywhere: it is made on the
    // gathered data).  Otherwise each rank reads the arrival counters of its bucket range out of the peers' buffers and
    // its group kernel pulls the rows themselves, segment by segment, with the bulk copies it issues anyway.
    bool peer_slots(Partition &p, size_t x_need)
    {
        ensure_exported(x_need);
        uint32_t *xcursor = static_cast<uint32_t *>(ctx->xbuf.p);
        Row32 *xpart = reinterpret_cast<Row32 *>(static_cast<char *>(ctx->xbuf.p) + x_cnt_bytes);
        uint32_t *xcnt = (uint32_t *)ensure(ctx->xcnt, (size_t)Bl * 4 * world);
        uint32_t *xtotal = (uint32_t *)ensure(ctx->xtotal, (size_t)Bl * 4);
        CU(cudaMemsetAsync(xcursor, 0, (size_t)B * 4, st));
        mark(-1);
        over_input(TAD_PHASE_SCATTER, [&](const ColPtrs &ck, uint64_t n) {
            return launch_scatter(st, ck, n, f, logB, xcursor, xpart, slotM, nullptr, 0, d_stats + ST_OVF);
        });
        // barrier + overflow agreement: {overflow rows, -} of every rank
        allgather(d_stats + ST_OVF, d_small + kSlotOvf, 8);
        mark(TAD_PHASE_SYNC);
        PeerCounters pc{};
        for (int r = 0; r < world; r++) pc.p[r] = r == me ? xcursor : static_cast<const uint32_t *>(ctx->peer_x[r]);
        CU(launch_gather_counts(st, pc, world, b_lo, Bl, slotM, xcnt, xtotal, xcursor, B, d_stats + ST_LOCALKEPT)); launches += 2;
        mark(TAD_PHASE_EXCHANGE);
        CU(launch_bucket_scan(st, xtotal, offsets, cursor, Bl, kGroupCap, big_list, big_base, cls_list, d_stats,
                              ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        mark(TAD_PHASE_SCAN);
        CU(cudaMemcpyAsync(ctx->h_small + kSlotOvf, d_small + kSlotOvf, 8 * world, cudaMemcpyDeviceToHost, st));
        read_stats();
        check_cancel();
        uint64_t any_ovf = 0;
        for (int r = 0; r < world; r++) any_ovf += (uint32_t)ctx->h_small[kSlotOvf + r];
        if (any_ovf == 0) {
            p.sync_at_end = true;       // peers may still read this rank's slots: no rank starts its next job before all are done
            p.kept = ctx->h_stats[ST_LOCALKEPT];
            p.owned = ctx->h_stats[ST_KEPT];
            p.seg.nseg = world; p.seg.stride = slotM; p.seg.b_lo = b_lo;
            for (int r = 0; r < world; r++) { p.seg.base[r] = peer_rows(r); p.seg.off[r] = xcnt + (size_t)r * Bl; }
            p.entries = use_entries(p.owned);
            return true;
        }
        CU(cudaMemsetAsync(d_stats, 0, 64 * sizeof(uint32_t), st));      // discard; redo exactly (every rank does)
        return false;
    }
    // ---- single GPU, exact partition: histogram, scan, scatter; also the fallback of the optimistic one -----------------
    Partition exact_local()
    {
        Row32 *part = (Row32 *)ctx->part.p;
        CU(cudaMemsetAsync(hist, 0, (size_t)B * 4, st));
        mark(-1);
        over_input(TAD_PHASE_HIST, [&](const ColPtrs &ck, uint64_t n) { return launch_hist(st, ck, n, f, logB, hist); });
        CU(launch_bucket_scan(st, hist, offsets, cursor, B, (uint32_t)kGroupCap, big_list, big_base, cls_list, d_stats,
                              ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        mark(TAD_PHASE_SCAN);
        CU(launch_scatter(st, c, R, f, logB, cursor, part)); launches += R ? 1 : 0;
        mark(TAD_PHASE_SCATTER);
        read_stats();
        Partition p;
        p.kept = p.owned = ctx->h_stats[ST_KEPT];
        p.seg.nseg = 1; p.seg.base[0] = part; p.seg.off[0] = offsets;
        p.entries = reinterpret_cast<SeriesEntry *>(part);      // in place over the staged bucket rows
        return p;
    }
    // ---- multi GPU, exact partition: K row chunks; chunk c is sent over NVLink (comm stream) while chunk c+1 is scattered ------
    // chunked (overlapped) exchange pays off at N = 2 (measured 11.5 -> 9.6 ms); at N >= 4 the NVLink all-to-all is
    // longer than the scatter it could hide behind and the extra segments cost the group kernel more than is won
    // With peer pull (default) the exact partition is written into the EXPORTED buffer and the owners' group kernels read
    // their segments straight out of the peers' copies: no receive buffer, no all-to-all (and no chunking: K = 1).
    Partition exact_multi()
    {
        const bool pull = ctx->peer_pull != 0;
        const int K = pull ? 1 : (R >= ctx->exchange_min_rows && (world == 2 || ctx->exchange_chunks_forced)) ? ctx->exchange_chunks : 1;
        const int NS = world * K;                              // segments: (source rank, chunk)
        Row32 *part;
        if (pull) {
            // the exported buffer must hold the largest shard: the ranks agree on it (blocking 128-byte all-gather; this path
            // is the fallback for skewed or very large tables, where a host sync more does not matter)
            memset(ctx->h_small + kSlotSend, 0, 16 * 8);
            ctx->h_small[kSlotSend] = R;
            gather16();
            uint64_t max_rows = 1;
            for (int r = 0; r < world; r++) max_rows = std::max<uint64_t>(max_rows, ctx->h_small[kSlotGather16 + 16 * r]);
            ensure_exported(x_cnt_bytes + max_rows * sizeof(Row32));
            part = reinterpret_cast<Row32 *>(static_cast<char *>(ctx->xbuf.p) + x_cnt_bytes);
        } else {
            part = (Row32 *)ensure(ctx->part, (R ? R : 1) * sizeof(Row32));
        }
        hist = (uint32_t *)ensure(ctx->hist, (size_t)B * 4 * K);
        offsets = (uint32_t *)ensure(ctx->offsets, ((size_t)B + 1) * 4 * K);
        cursor = (uint32_t *)ensure(ctx->cursor, (size_t)B * 4 * K);
        uint32_t *hist_all = (uint32_t *)ensure(ctx->hist_all, (size_t)B * 4 * NS);
        uint32_t *seg_off = (uint32_t *)ensure(ctx->seg_off, ((size_t)Bl + 1) * 4 * NS);
        uint32_t *seg_total = (uint32_t *)ensure(ctx->seg_total, (size_t)Bl * 4);
        CU(cudaMemsetAsync(hist, 0, (size_t)B * 4 * K, st));
        if (host_input)
            for (int k = 0; k < nchunks; k++) CU(cudaStreamWaitEvent(st, ctx->chunk_ev[k], 0));
        mark(TAD_PHASE_H2D);
        for (int cx = 0; cx < K; cx++) {
            const uint64_t lo = split(cx, K), hi = split(cx + 1, K);
            if (hi > lo) { CU(launch_hist(st, offset_cols(lo), hi - lo, f, logB, hist + (size_t)cx * B)); launches++; }
        }
        mark(TAD_PHASE_HIST);
        for (int cx = 0; cx < K; cx++) {
            CU(launch_bucket_scan(st, hist + (size_t)cx * B, offsets + (size_t)cx * (B + 1), cursor + (size_t)cx * B, B, 0xffffffffu,
                                  big_list, big_base, nullptr, d_stats, ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        }
        mark(TAD_PHASE_SCAN);
        // every rank learns every (rank, chunk) histogram: segment offsets of the owned bucket range, receive sizes
        allgather(hist, hist_all, (size_t)B * 4 * K);
        CU(launch_segment_scan(st, hist_all, B, b_lo, Bl, NS, seg_off, seg_total, d_small + kSlotSegRows,
                               pull ? d_small + kSlotFront : nullptr)); launches += 2;
        CU(cudaMemcpyAsync(ctx->h_small + kSlotSegRows, d_small + kSlotSegRows, 8 * NS, cudaMemcpyDeviceToHost, st));
        if (pull) CU(cudaMemcpyAsync(ctx->h_small + kSlotFront, d_small + kSlotFront, 8 * NS, cudaMemcpyDeviceToHost, st));
        for (int cx = 0; cx < K; cx++)        // send boundaries of chunk cx: offsets_cx[p * Bl], p = 0..world
            CU(cudaMemcpy2DAsync(ctx->h_small + kSlotSendLo + cx * (kMaxRanks + 1), 8, offsets + (size_t)cx * (B + 1), (size_t)Bl * 4, 4,
                                 world + 1, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        check_cancel();
        const unsigned long long *seg_rows = ctx->h_small + kSlotSegRows;
        SegDesc seg{};
        uint64_t kept = 0, owned = 0;
        bool sync_at_end = false;
        uint64_t recv_off[kMaxSeg], recv_total = 0, send_lo[kMaxXChunks][kMaxRanks + 1] = {};
        for (int sgi = 0; sgi < NS; sgi++) {
            recv_off[sgi] = recv_total;
            if (sgi / K != me) recv_total += seg_rows[sgi] * 32;
            owned += seg_rows[sgi];
        }
        for (int cx = 0; cx < K; cx++) {
            for (int p = 0; p <= world; p++) send_lo[cx][p] = (uint32_t)ctx->h_small[kSlotSendLo + cx * (kMaxRanks + 1) + p];
            kept += send_lo[cx][world];
        }
        if (owned >= (1ull << 32) - 1) fail(TAD_ERR_INVALID_ARG, "more than 2^32-2 rows owned by one GPU after the exchange");
        if (pull) {
            // peer pull: the owners' group kernels read their segments out of the exported partitions
            CU(launch_scatter(st, c, R, f, logB, cursor, part)); launches += R ? 1 : 0;
            mark(TAD_PHASE_SCATTER);
            nccl_ok(barrier(ctx));              // every rank's exact partition is complete
            mark(TAD_PHASE_SYNC);
            seg.nseg = world;
            for (int r = 0; r < world; r++) {
                seg.base[r] = peer_rows(r) + ctx->h_small[kSlotFront + r];   // rows in front of my range
                seg.off[r] = seg_off + (size_t)r * (Bl + 1);
            }
            sync_at_end = true;
        } else {
            // NCCL all-to-all (TAD_PEER_PULL=0): chunk cx is sent on the copy stream while chunk cx+1 is scattered
            cudaStream_t cs = ctx->copy_stream;
            ensure(ctx->exch, recv_total ? recv_total : 32);
            for (int cx = 0; cx < K; cx++) {
                const uint64_t lo = split(cx, K), hi = split(cx + 1, K);
                if (hi > lo) { CU(launch_scatter(st, offset_cols(lo), hi - lo, f, logB, cursor + (size_t)cx * B, part + lo)); launches++; }
                CU(cudaEventRecord(ctx->x_ev[cx], st));
                CU(cudaStreamWaitEvent(cs, ctx->x_ev[cx], 0));
                uint64_t so[kMaxRanks], sb[kMaxRanks], ro[kMaxRanks], rb[kMaxRanks];
                for (int p = 0; p < world; p++) {
                    so[p] = (lo + send_lo[cx][p]) * 32;
                    sb[p] = (send_lo[cx][p + 1] - send_lo[cx][p]) * 32;
                    ro[p] = recv_off[p * K + cx];
                    rb[p] = seg_rows[p * K + cx] * 32;
                }
                nccl_ok(nccl_alltoallv(&ctx->nccl, part, so, sb, ctx->exch.p, ro, rb, cs));
            }
            mark(TAD_PHASE_SCATTER);
            CU(cudaEventRecord(ctx->x_ev[K], cs));
            CU(cudaStreamWaitEvent(st, ctx->x_ev[K], 0));
            seg.nseg = NS;
            for (int sgi = 0; sgi < NS; sgi++) {
                const int r = sgi / K, cx = sgi % K;
                seg.base[sgi] = r == me ? part + split(cx, K) + send_lo[cx][me]
                                        : reinterpret_cast<const Row32 *>((const char *)ctx->exch.p + recv_off[sgi]);
                seg.off[sgi] = seg_off + (size_t)sgi * (Bl + 1);
            }
        }
        // final (virtual) bucket offsets of the owned range, oversized-bucket list, capacity-class lists
        CU(launch_bucket_scan(st, seg_total, offsets, cursor, Bl, kGroupCap, big_list, big_base, cls_list, d_stats,
                              ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        mark(TAD_PHASE_EXCHANGE);           // = the part of the exchange NOT hidden behind the scatter
        read_stats();
        return Partition{seg, use_entries(owned), kept, owned, nullptr, 0, sync_at_end};
    }
    // ---- group (+ spill) ------------------------------------------------------------------
    void group(const Partition &p, uint32_t n_big, uint64_t big_rows)
    {
        const uint64_t cap_rows = p.owned ? p.owned : 1;
        csr_v = (uint64_t *)ensure(ctx->csr_v, cap_rows * 8 + 64);       // + one sector: the direct detector reads whole 32-byte sectors
        csr_t = (uint32_t *)ensure(ctx->csr_t, cap_rows * 4);
        if (sp.algo == TAD_ALGO_DBSCAN) csr_p = (uint32_t *)ensure(ctx->csr_p, cap_rows * 4);
        mark(-1);
        int l = 0;
        const uint32_t n_cls[3] = {ctx->h_stats[ST_NCLS0], ctx->h_stats[ST_NCLS1], ctx->h_stats[ST_NCLS2]};
        if (ctx->sort_classes) {
            // class lists in ascending bucket order: concurrently running CTAs then touch neighbouring slots / csr stretches
            ensure(ctx->sortb, sort_lists_scratch_bytes(Bl));
            int bits = 1;
            while ((1u << bits) < Bl && bits < 32) bits++;
            for (int k = 0; k < 3; k++)
                if (n_cls[k] > 1) { CU(sort_bucket_list(st, cls_list + (size_t)k * Bl, n_cls[k], bits, ctx->sortb.p, ctx->sortb.cap)); launches += 3; }
        }
        CU(launch_group(st, p.seg, p.entries, offsets, Bl, cls_list, n_cls, csr_v, csr_t, csr_p, nsb, npb, sp.reducer, &l));
        launches += l;
        mark(TAD_PHASE_GROUP);
        if (n_big) {
            ensure(ctx->spill, spill_scratch_bytes(big_rows));
            l = 0;
            CU(run_spill(st, p.seg, p.entries, offsets, big_list, big_base, n_big, big_rows, ctx->spill.p, ctx->spill.cap, csr_v,
                         csr_t, nsb, npb, sp.reducer, &l, p.ovf_rows, p.n_ovf));
            launches += l;
            mark(TAD_PHASE_SPILL);
        }
    }
    // ---- series scan: series base per bucket; series and point counts -> h_stats ------------
    void series_scan(uint64_t owned)
    {
        sbase = (uint32_t *)ensure(ctx->sbase, sbase_words(Bl, owned ? owned : 1) * 4);   // + bucket hint per 32 series
        CU(launch_series_scan(st, nsb, npb, sbase, Bl, d_stats, ctx->scan_sync.p, ++ctx->scan_epoch)); launches++;
        read_stats();
    }
    // ---- detect: result rows into the device buffer of layout L; returns their count --------
    uint64_t detect(const Partition &p, uint32_t S, uint64_t points, OutLayout &L)
    {
        const uint64_t cap_rows = p.owned ? p.owned : 1;
        const bool emit_all = (sp.flags & TAD_FLAG_EMIT_ALL) != 0;
        uint64_t out_cap = emit_all ? points : (points / 8 + (1u << 16));
        if (out_cap > points) out_cap = points;
        if (out_cap == 0) out_cap = 1;
        uint64_t out_rows = 0;
        for (int attempt = 0; attempt < 3; attempt++) {
            L = out_layout(out_cap);
            ensure(ctx->outb, L.total);
            const OutCols oc = out_cols(ctx->outb.p, L);
            CU(cudaMemsetAsync(d_stats + ST_OUTCOUNT, 0, 4, st));
            mark(-1);
            if (sp.algo == TAD_ALGO_EWMA) {
                CU(launch_detect_ewma(st, p.entries, offsets, sbase, Bl, S, csr_v, csr_t, oc, (uint32_t)out_cap, d_stats, emit_all));
                launches += S ? 1 : 0;
            } else if (sp.algo == TAD_ALGO_DBSCAN) {
                ensure(ctx->dbx, cap_rows * 4);         // prefix count of core points, per point slot
                ensure(ctx->dbi, cap_rows);             // noise flag, per point slot
                CU(launch_detect_dbscan(st, p.entries, offsets, sbase, Bl, S, csr_v, csr_t, csr_p, (uint32_t *)ctx->dbx.p,
                                        (uint8_t *)ctx->dbi.p, oc, (uint32_t)out_cap, d_stats, emit_all));
                launches += S ? 1 : 0;
            } else if (sp.algo == TAD_ALGO_ARIMA) {
                ensure(ctx->ar_y, cap_rows * 8);
                ensure(ctx->ar_pred, cap_rows * 8);
                ensure(ctx->ar_lam, ((size_t)S + 1) * 8);
                CU(launch_detect_arima(st, p.entries, offsets, sbase, Bl, S, csr_v, csr_t, (double *)ctx->ar_y.p,
                                       (double *)ctx->ar_pred.p, (double *)ctx->ar_lam.p, attempt == 0, oc, (uint32_t)out_cap,
                                       d_stats, emit_all));
                launches += S ? (attempt == 0 ? 3 : 1) : 0;
            } else {
                fail(TAD_ERR_UNSUPPORTED, "algorithm %d is not implemented by this build", sp.algo);
            }
            mark(TAD_PHASE_DETECT);
            read_stats();
            out_rows = ctx->h_stats[ST_OUTCOUNT];
            if (out_rows <= out_cap) break;
            out_cap = out_rows;                 // capacity guess too small: rerun detect (idempotent)
            if (attempt == 2) fail(TAD_ERR_INTERNAL, "result capacity did not converge");
        }
        return out_rows;
    }
    // ---- egress: result rows -> pinned host memory -------------------------------------------
    void egress(const OutLayout &L, uint64_t out_rows)
    {
        mark(-1);
        static const size_t w[11] = {8, 8, 8, 4, 4, 4, 4, 2, 2, 1, 1};
        OutLayout HL = out_layout(out_rows ? out_rows : 1);
        job->result_block = take_pinned(ctx, HL.total);
        char *hb = static_cast<char *>(job->result_block.p);
        const char *db = static_cast<const char *>(ctx->outb.p);
        for (int i = 0; i < 11 && out_rows; i++)
            CU(cudaMemcpyAsync(hb + HL.off[i], db + L.off[i], w[i] * out_rows, cudaMemcpyDeviceToHost, st));
        OutCols ho = out_cols(hb, HL);
        job->rows.rows = out_rows;
        job->rows.src_ip = ho.src_ip; job->rows.dst_ip = ho.dst_ip;
        job->rows.src_port = ho.src_port; job->rows.dst_port = ho.dst_port;
        job->rows.proto = ho.proto; job->rows.flow_start = ho.flow_start; job->rows.flow_end = ho.flow_end;
        job->rows.stddev = ho.stddev; job->rows.algo_calc = ho.algo_calc; job->rows.throughput = ho.throughput;
        job->rows.anomaly = ho.anomaly;
        mark(TAD_PHASE_D2H);
        CU(cudaStreamSynchronize(st));
    }
    // ---- status: counts, phase times; the job is COMPLETED ---------------------------------------
    void report(const Partition &p, uint32_t S, uint64_t points, uint64_t out_rows, uint64_t big_rows)
    {
        double phase_ms[TAD_NPHASES] = {0};
        float total = 0;
        for (int i = 1; i < nev; i++) {
            if (ev_phase[i] < 0) continue;
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, ctx->ev[i - 1], ctx->ev[i]));
            phase_ms[ev_phase[i]] += ms;
        }
        // device span excludes the H2D/D2H copies: first partition event .. last detect event
        int first_k = -1, last_k = -1;
        for (int i = 0; i < nev; i++) {
            if ((ev_phase[i] == TAD_PHASE_HIST || ev_phase[i] == TAD_PHASE_H2D || ev_phase[i] == TAD_PHASE_SCATTER) && first_k < 0)
                first_k = i - 1;
            if (ev_phase[i] == TAD_PHASE_DETECT || (ev_phase[i] == TAD_PHASE_SYNC && last_k >= 0)) last_k = i;
        }
        if (first_k >= 0 && last_k > first_k) CU(cudaEventElapsedTime(&total, ctx->ev[first_k], ctx->ev[last_k]));
        std::lock_guard<std::mutex> lk(job->mu);
        tad_status &s = job->st;
        s.rows_in = R; s.rows_kept = p.kept; s.rows_owned = p.owned;
        s.points = points; s.series = S; s.result_rows = out_rows; s.spill_rows = big_rows;
        s.gpu_launches = launches; s.device_ms = total;
        for (int i = 0; i < TAD_NPHASES; i++) s.phase_ms[i] = phase_ms[i];
        s.total_ms = now_ms() - job->t_submit;
        s.completed_stages = kTotalStages; s.state = TAD_STATE_COMPLETED;
        job->cv.notify_all();     // last touch of `job` by the worker (tad_release may free it now)
    }
};

void run_job(tad_ctx *ctx, tad_job *job)
{
    JobRun run(ctx, job);
    run.ingest();
    run.pick_buckets();
    const Partition p = run.partition();
    run.check_cancel();
    const uint32_t n_big = ctx->h_stats[ST_NBIG];
    const uint64_t big_rows = ctx->h_stats[ST_BIGROWS];
    set_progress(job, TAD_STATE_RUNNING, 3);    // ingest, partition, exchange
    run.group(p, n_big, big_rows);
    run.series_scan(p.owned);
    run.check_cancel();
    const uint32_t S = ctx->h_stats[ST_SERIES];
    const uint64_t points = ctx->h_stats[ST_POINTS];
    set_progress(job, TAD_STATE_RUNNING, 4);
    OutLayout L{};
    const uint64_t out_rows = run.detect(p, S, points, L);
    run.check_cancel();
    set_progress(job, TAD_STATE_RUNNING, 5);
    if (p.sync_at_end) {
        // end-of-job barrier of the peer-pull paths: my slots and counters may be overwritten (next job) only after every
        // peer's group kernel has read them; its wait is the ranks' arrival skew, accounted as TAD_PHASE_SYNC
        run.mark(-1);
        nccl_ok(barrier(ctx));
        run.mark(TAD_PHASE_SYNC);
    }
    run.egress(L, out_rows);
    run.report(p, S, points, out_rows, big_rows);
}

void worker_main(tad_ctx *ctx)
{
    if (ctx->numa.ok) sched_setaffinity(0, sizeof(ctx->numa.cpus), &ctx->numa.cpus);      // this thread only
    cudaSetDevice(ctx->cfg.device);
    for (;;) {
        tad_job *job = nullptr;
        {
            std::unique_lock<std::mutex> lk(ctx->mu);
            ctx->cv.wait(lk, [&] { return ctx->stop || !ctx->queue.empty(); });
            if (ctx->queue.empty()) return;       // stop requested and drained
            job = ctx->queue.front();
            ctx->queue.pop_front();
        }
        try {
            if (job->cancel.load()) fail(TAD_ERR_CANCELLED, "job cancelled");
            run_job(ctx, job);
        } catch (const JobFail &f) {
            // nothing of this job may still be reading the caller's columns once it is reported FAILED
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamSynchronize(ctx->stream);
            cudaGetLastError();
            std::lock_guard<std::mutex> lk(job->mu);
            job->st.state = TAD_STATE_FAILED;
            job->st.error = f.code;
            snprintf(job->st.err_msg, sizeof(job->st.err_msg), "%s", f.msg);
            job->st.total_ms = now_ms() - job->t_submit;
            job->cv.notify_all();
        }
    }
}

int validate(const tad_job_spec *spec, const tad_columns *cols, char *msg, size_t n)
{
    if (spec->algo != TAD_ALGO_EWMA && spec->algo != TAD_ALGO_ARIMA && spec->algo != TAD_ALGO_DBSCAN) {
        // controller.go:527-529
        snprintf(msg, n, "invalid request: Throughput Anomaly Detector algorithm type should be 'EWMA' or 'ARIMA' or 'DBSCAN'");
        return TAD_ERR_INVALID_ARG;
    }
    if (spec->reducer != TAD_REDUCE_MAX && spec->reducer != TAD_REDUCE_SUM) {
        snprintf(msg, n, "invalid request: reducer should be max or sum");
        return TAD_ERR_INVALID_ARG;
    }
    if (spec->start_time && spec->end_time && spec->end_time <= spec->start_time) {
        // controller.go:535-539
        snprintf(msg, n, "invalid request: EndInterval should be after StartInterval");
        return TAD_ERR_INVALID_ARG;
    }
    if (cols->rows && (!cols->flow_end || !cols->value)) {
        snprintf(msg, n, "invalid request: flow_end and value columns are required");
        return TAD_ERR_INVALID_ARG;
    }
    if (cols->rows && spec->start_time && !cols->flow_start) {
        // flowStartSeconds >= start filters on the flow_start KEY column; a job whose key has none (the external / svc
        // aggregated modes, anomaly_detection.py:568-571) applies that bound on the host, where the column lives
        snprintf(msg, n, "invalid request: start_time needs the flow_start column");
        return TAD_ERR_INVALID_ARG;
    }
    if (cols->rows >= (1ull << 32) - 1) {
        snprintf(msg, n, "invalid request: at most 2^32-2 rows per GPU");
        return TAD_ERR_INVALID_ARG;
    }
    if (cols->mem != TAD_MEM_HOST && cols->mem != TAD_MEM_DEVICE) {
        snprintf(msg, n, "invalid request: bad column memory kind");
        return TAD_ERR_INVALID_ARG;
    }
    if (spec->n_ns_ignore && !spec->ns_ignore) {
        snprintf(msg, n, "invalid request: ns_ignore is NULL");
        return TAD_ERR_INVALID_ARG;
    }
    return TAD_OK;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int tad_abi_version(void) { return TAD_ABI_VERSION; }

int tad_get_unique_id(void *out, size_t bytes)
{
    if (!out || bytes < 128) return TAD_ERR_INVALID_ARG;
    return nccl_get_unique_id(out, bytes) == 0 ? TAD_OK : TAD_ERR_NCCL;
}

const char *tad_strerror(int err)
{
    const int i = -err;
    if (i < 0 || i > 8) return "unknown error";
    return kErrNames[i];
}

int tad_init(const tad_config *cfg, tad_ctx **out)
{
    if (!cfg || !out) return TAD_ERR_INVALID_ARG;
    if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) return TAD_ERR_INVALID_ARG;
    if (cfg->world_size > kMaxRanks || (cfg->world_size & (cfg->world_size - 1))) return TAD_ERR_INVALID_ARG;   // 1, 2, 4, 8
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        fprintf(stderr, "theia_tad: no CUDA device is available; this library has no CPU fallback\n");
        return TAD_ERR_CUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) return TAD_ERR_INVALID_ARG;
    if (cudaSetDevice(cfg->device) != cudaSuccess) return TAD_ERR_CUDA;
    tad_ctx *ctx = new tad_ctx();
    ctx->cfg = *cfg;
    ctx->cfg.nccl_unique_id = nullptr;
    if (const char *e = getenv("TAD_DEBUG_LOGB")) ctx->debug_logb = atoi(e);
    if (const char *e = getenv("TAD_GROUP_TARGET")) ctx->debug_target = atoi(e);
    ctx->numa = numa_of_device(cfg->device);
    NumaScope numa_scope(ctx->numa);
    bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < kMaxChunks; i++) ok = cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->start_ev, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && i <= kMaxXChunks; i++) ok = cudaEventCreateWithFlags(&ctx->x_ev[i], cudaEventDisableTiming) == cudaSuccess;
    if (const char *e = getenv("TAD_OPTIMISTIC")) ctx->optimistic = atoi(e);
    // defaults = the fastest measured configuration per world size (DESIGN.md section 6): peer pull everywhere, the exact fallback
    // pulled as well, capacity-class lists sorted by bucket from 4 ranks on (locality of the small remote reads)
    ctx->peer_pull = 1;
    ctx->sort_classes = cfg->world_size >= 4 ? 1 : 0;
    if (const char *e = getenv("TAD_PEER_PULL")) ctx->peer_pull = atoi(e);
    if (const char *e = getenv("TAD_SORT_CLASSES")) ctx->sort_classes = atoi(e);
    if (const char *e = getenv("TAD_SLOT_BUDGET_GB")) ctx->x_budget = (size_t)strtoull(e, nullptr, 10) << 30;
    if (const char *e = getenv("TAD_EXCHANGE_MIN_ROWS")) ctx->exchange_min_rows = strtoull(e, nullptr, 10);
    if (getenv("TAD_EXCHANGE_CHUNKS")) ctx->exchange_chunks_forced = true;
    if (const char *e = getenv("TAD_EXCHANGE_CHUNKS")) ctx->exchange_chunks = atoi(e) < 1 ? 1 : (atoi(e) > kMaxXChunks ? kMaxXChunks : atoi(e));
    for (int i = 0; ok && i < kMaxEvents; i++) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    ok = ok && cudaHostAlloc((void **)&ctx->h_stats, 64 * sizeof(uint32_t), cudaHostAllocDefault) == cudaSuccess;
    ok = ok && cudaHostAlloc((void **)&ctx->h_small, kSmallWords * sizeof(unsigned long long), cudaHostAllocDefault) == cudaSuccess;
    if (!ok) {
        tad_shutdown(ctx);      // releases whatever was created
        return TAD_ERR_CUDA;
    }
    if (cfg->world_size > 1) {
        int rc = nccl_comm_init(&ctx->nccl, cfg->world_size, cfg->rank, cfg->nccl_unique_id, cfg->nccl_unique_id_bytes);
        if (rc != 0) {
            tad_shutdown(ctx);
            return TAD_ERR_NCCL;
        }
    }
    ctx->worker = std::thread(worker_main, ctx);
    *out = ctx;
    return TAD_OK;
}

void tad_shutdown(tad_ctx *ctx)
{
    if (!ctx) return;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->stop = true;
    }
    ctx->cv.notify_all();
    if (ctx->worker.joinable()) ctx->worker.join();
    cudaSetDevice(ctx->cfg.device);
    if (ctx->peers_mapped && ctx->nccl.comm && ctx->small.p && ctx->stream) {
        // an exported buffer must outlive every peer's mapping of it: unmap, meet the peers, only then free (delete ctx)
        for (int r = 0; r < kMaxRanks; r++)
            if (ctx->peer_x[r]) { cudaIpcCloseMemHandle(ctx->peer_x[r]); ctx->peer_x[r] = nullptr; }
        if (barrier(ctx) == 0) cudaStreamSynchronize(ctx->stream);
        ctx->peers_mapped = false;
    }
    nccl_comm_destroy(&ctx->nccl);
    for (auto &b : ctx->pinned_pool) cudaFreeHost(b.p);
    if (ctx->h_stats) cudaFreeHost(ctx->h_stats);
    if (ctx->h_small) cudaFreeHost(ctx->h_small);
    for (int i = 0; i < kMaxEvents; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < kMaxChunks; i++)
        if (ctx->chunk_ev[i]) cudaEventDestroy(ctx->chunk_ev[i]);
    if (ctx->start_ev) cudaEventDestroy(ctx->start_ev);
    for (int i = 0; i <= kMaxXChunks; i++)
        if (ctx->x_ev[i]) cudaEventDestroy(ctx->x_ev[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;      // frees the device workspace
}

int tad_alloc_columns(tad_ctx *ctx, uint64_t capacity, int32_t mem, tad_columns *cols)
{
    if (!ctx || !cols || (mem != TAD_MEM_HOST && mem != TAD_MEM_DEVICE)) return TAD_ERR_INVALID_ARG;
    memset(cols, 0, sizeof(*cols));
    cols->capacity = capacity;
    cols->mem = mem;
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return TAD_ERR_CUDA;
    NumaScope numa_scope(ctx->numa);
    void **slots[8] = {(void **)&cols->src_ip, (void **)&cols->dst_ip, (void **)&cols->src_port, (void **)&cols->dst_port,
                       (void **)&cols->proto, (void **)&cols->flow_start, (void **)&cols->flow_end, (void **)&cols->value};
    for (int i = 0; i < 8; i++) {
        const size_t bytes = ((col_bytes(i, capacity ? capacity : 1)) + 255) & ~size_t(255);
        cudaError_t e = mem == TAD_MEM_HOST ? cudaHostAlloc(slots[i], bytes, cudaHostAllocDefault) : cudaMalloc(slots[i], bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            tad_free_columns(ctx, cols);
            return TAD_ERR_NOMEM;
        }
    }
    return TAD_OK;
}

int tad_alloc_ns_columns(tad_ctx *ctx, tad_columns *cols)
{
    if (!ctx || !cols || !cols->capacity) return TAD_ERR_INVALID_ARG;
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return TAD_ERR_CUDA;
    NumaScope numa_scope(ctx->numa);
    void **slots[2] = {(void **)&cols->src_ns, (void **)&cols->dst_ns};
    for (int i = 0; i < 2; i++) {
        if (*slots[i]) continue;
        const size_t bytes = (cols->capacity * 4 + 255) & ~size_t(255);
        cudaError_t e = cols->mem == TAD_MEM_HOST ? cudaHostAlloc(slots[i], bytes, cudaHostAllocDefault) : cudaMalloc(slots[i], bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return TAD_ERR_NOMEM;
        }
    }
    return TAD_OK;
}

int tad_free_columns(tad_ctx *ctx, tad_columns *cols)
{
    if (!ctx || !cols) return TAD_ERR_INVALID_ARG;
    cudaSetDevice(ctx->cfg.device);
    for (int i = 0; i < 10; i++) {
        void *p = col_ptr(*cols, i);
        if (!p) continue;
        if (cols->mem == TAD_MEM_HOST) cudaFreeHost(p); else cudaFree(p);
    }
    memset(cols, 0, sizeof(*cols));
    return TAD_OK;
}

int tad_submit(tad_ctx *ctx, const tad_job_spec *spec, const tad_columns *cols, tad_job **out)
{
    if (!ctx || !spec || !cols || !out) return TAD_ERR_INVALID_ARG;
    tad_job *job = new tad_job();
    job->ctx = ctx;
    job->spec = *spec;
    job->spec.id[sizeof(job->spec.id) - 1] = 0;
    job->cols = *cols;
    job->t_submit = now_ms();
    job->st.total_stages = kTotalStages;
    *out = job;
    char msg[200];
    int rc = validate(spec, cols, msg, sizeof(msg));
    if (rc != TAD_OK) {
        // like the controller (controller.go:505-514): illegal arguments are terminal FAILED, never retried
        job->st.state = TAD_STATE_FAILED;
        job->st.error = rc;
        snprintf(job->st.err_msg, sizeof(job->st.err_msg), "error in creating AnomalyDetector: %s", msg);
        return rc;
    }
    if (spec->n_ns_ignore) job->ns_ignore.assign(spec->ns_ignore, spec->ns_ignore + spec->n_ns_ignore);
    job->spec.ns_ignore = nullptr;
    job->st.state = TAD_STATE_SCHEDULED;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->stop) {
            job->st.state = TAD_STATE_FAILED;
            job->st.error = TAD_ERR_STATE;
            snprintf(job->st.err_msg, sizeof(job->st.err_msg), "context is shutting down");
            return TAD_ERR_STATE;
        }
        ctx->queue.push_back(job);
    }
    ctx->cv.notify_one();
    return TAD_OK;
}

int tad_poll(tad_job *job, tad_status *status)
{
    if (!job || !status) return TAD_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(job->mu);
    *status = job->st;
    return TAD_OK;
}

int tad_wait(tad_job *job, int64_t timeout_ms, tad_status *status)
{
    if (!job) return TAD_ERR_INVALID_ARG;
    std::unique_lock<std::mutex> lk(job->mu);
    auto done = [&] { return job->st.state == TAD_STATE_COMPLETED || job->st.state == TAD_STATE_FAILED; };
    if (timeout_ms < 0) {
        while (!done()) job->cv.wait_for(lk, std::chrono::milliseconds(50));
    } else {
        const double deadline = now_ms() + (double)timeout_ms;
        while (!done() && now_ms() < deadline) job->cv.wait_for(lk, std::chrono::milliseconds(1));
    }
    if (status) *status = job->st;
    return TAD_OK;
}

int tad_result(tad_job *job, tad_rows *rows)
{
    if (!job || !rows) return TAD_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> lk(job->mu);
    if (job->st.state != TAD_STATE_COMPLETED) return TAD_ERR_STATE;
    *rows = job->rows;
    return TAD_OK;
}

int tad_cancel(tad_job *job)
{
    if (!job) return TAD_ERR_INVALID_ARG;
    job->cancel.store(1);
    return TAD_OK;
}

int tad_release(tad_job *job)
{
    if (!job) return TAD_ERR_INVALID_ARG;
    {
        std::unique_lock<std::mutex> lk(job->mu);
        const int s = job->st.state;
        if (s == TAD_STATE_SCHEDULED || s == TAD_STATE_RUNNING) {
            job->cancel.store(1);
            while (!(job->st.state == TAD_STATE_COMPLETED || job->st.state == TAD_STATE_FAILED))
                job->cv.wait_for(lk, std::chrono::milliseconds(1));
        }
    }
    give_pinned(job->ctx, job->result_block);
    delete job;
    return TAD_OK;
}

}  // extern "C"
