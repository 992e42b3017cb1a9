// engine.cu — host side of the B200 scan engine behind include/vsb200.h.
//
// Owns device residency of a column shard (the GPU counterpart of table_context.preloaded,
// /root/reference/src/sqlite-vector.c:126-137, filled by vector_quantize_preload :1338-1404),
// launches the sm_100a kernels in scan_kernels.cuh and finishes each query with the reference's
// k-slot algorithm (:1808-1817, :2022-2069, :2145-2152) over the few hundred surviving candidates.
// No CPU fallback: if CUDA is unavailable every entry point returns VSB_ENODEV.
#include "../../include/vsb200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "scan_kernels.cuh"
#include "batch_kernels.cuh"
#include "quant_kernels.cuh"

using namespace vsb;

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};
int g_opt_stage_bytes = 16384; // upper bound of one warp tile (ring stage); 12 KB tiles x 2 stages measured best (99% of HBM peak)
int g_opt_direct = 0;          // 1: force the no-staging kernel
int g_opt_ring_bytes = 0;      // 0: use all shared memory left
int g_opt_no_batch = 0;        // 1: never take the tensor-core batch path
int g_opt_batch_debug = 0;     // 1: print per-stage timings of the batch path to stderr (serialises the stages)
int g_opt_batch_m0 = 128;      // batch path: rows refined exhaustively before the first tensor-core level
int g_opt_merge_stream = 1;    // process exchange, batched queries: wait + merge + copy back on their own stream (overlaps the next batch's levels)
int g_opt_batch_growth = 8;    // batch path: each tensor-core level covers rows [m, growth*m) (capped by k, see batch_growth)
int g_opt_fuse_mb = 0;         // > 0: vsb_scan_submit_group fuses a group into ONE scan launch when one query's scan reads less than this
                               // many MB (measured per query on one GPU: 84.0 -> 76.9 us at 0.48 GB; 2 GPUs: 285 -> 271 us at 1.92 GB).
                               // Off by default: a persistent 8-query launch leaves the NCCL all-gather of the previous group no SM until
                               // it ends (2 GPUs: the step-vs-scan gap grew from 3 to 14 us per query), not yet measured at 8 GPUs.
int g_opt_balance = 1;         // 1: adaptive row partition of the single-query scan (per-CTA speeds feed the next partition)
int g_opt_epi_chunk = 1;       // 1: integer tensor-core epilogue tests 32-column chunks (max score vs weakest bound) before any per-column work
int g_opt_epi2 = 4;            // epilogue shape of tc_scan_kernel (see launch_tc_mc): 4 = 16 epilogue warps where that variant exists (integer kinds, 256-query tiles), else 8; 2 = 8 warps; 0 = 4 warps
int g_opt_time_kernels = 0;    // 1: bracket every kernel launch with CUDA events (bench.py roofline leg)
int g_opt_scan_streams = 2;    // 2: consecutive scan launches alternate between two streams, so the CTAs of launch i+1 take over each SM
                               // as soon as the CTA of launch i on it exits (one scan CTA fits per SM): no grid-wide drain between
                               // launches, per-SM speed differences turn into an earlier start of the next query.  1: one stream.
int g_opt_push_mode = 1;       // exchange: 1 (default) = a small kernel on the exchange stream pushes a finished group's heads; 0 = the filter's last block pushes its head itself (fused: costs ~2 us per query with 8 targets, profiles/r02j)
int g_opt_push_repeat = 1;     // experiment: push every exchange target this many times (see exchange_fill_push)
int g_opt_xwait_ms = 2000;     // exchange: how long the receiving side waits for a peer's head before it reports an error

// cudaFuncSetAttribute costs ~1 us per call; the dynamic shared memory limit of a kernel only ever needs to grow
int set_smem_limit(const void *fn, size_t bytes) {
    static std::mutex mu;
    static std::vector<std::pair<const void *, size_t>> seen;     // per process; devices are identical B200s
    std::lock_guard<std::mutex> lk(mu);
    int dev = 0;
    cudaGetDevice(&dev);
    const void *key = (const void *)((uintptr_t)fn ^ ((uintptr_t)dev << 56));
    for (auto &e : seen)
        if (e.first == key) {
            if (e.second >= bytes) return 0;
            cudaError_t r = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (r == cudaSuccess) e.second = bytes;
            return (int)r;
        }
    cudaError_t r = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (r == cudaSuccess) r = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (r == cudaSuccess) seen.emplace_back(key, bytes);
    return (int)r;
}

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(e_ == cudaErrorMemoryAllocation ? VSB_ENOMEM : VSB_ECUDA, "%s failed: %s (%s:%d)", \
                        #call, cudaGetErrorString(e_), __FILE__, __LINE__);                                \
    } while (0)

int elem_size(int vtype) {
    switch (vtype) {
    case VSB_F32: return 4;
    case VSB_F16: case VSB_BF16: return 2;
    case VSB_U8: case VSB_I8: return 1;
    }
    return 0;
}

constexpr size_t kStageBuf = 32u << 20;  // pinned staging buffers for preload (two of them)
constexpr int kOutCap = 1 << 16;         // survivor capacity per query (mapped pinned)
constexpr int kMaxK = 256;               // candidate path; larger k uses the all-distances path
constexpr int kSlots = 32;               // result slots: queries in flight (the sharded exchange moves groups of them; a rank may have at most
                                         // kSlots / 2 queries in flight so that a peer never overwrites a gather row that is still being read)

// result block of one query, written by filter_kernel into DEVICE memory and fetched with one async copy:
//   head = the result head (layout in scan_kernels.cuh) with room for the first kFirstFetch survivors (kHeadBytes, what travels)
//   tail = the (rare) survivors beyond kFirstFetch, fetched by a second copy.
// The heads of all slots are ONE contiguous allocation (slot s at s * kHeadBytes), so a launcher can all-gather the
// heads of a group of consecutive slots with a single collective.  (Zero-copy writes of ~300 scattered 8-byte records
// over PCIe made the filter kernel 5x slower than writing to HBM and copying once.)
constexpr int kFirstFetch = 1024;
constexpr size_t kHeadBytes = kResHdrBytes + sizeof(uint2) * kFirstFetch;

// scan workspace of ONE query (per-stream k-lists / CTA lists, in-CTA bounds, candidate logs): written by scan_kernel,
// read by filter_kernel
struct QWork {
    float *d_lists = nullptr, *d_tlocal = nullptr;
    uint2 *d_logs = nullptr;
    int *d_counts = nullptr;
};
// One launch scans up to kMaxGroup independent queries back to back (scan_kernel); a Work holds their workspaces plus what
// is per launch.  Two Works alternate so that the filters of launch i (filter stream) overlap the scan of launch i+1.
struct Work {
    QWork q[kMaxGroup];
    long long *d_bounds = nullptr;   // [CTAs + 1] adaptive tile partition used by the NEXT scan on this workspace
    unsigned *d_cta_time = nullptr;  // [CTAs] cycles each scan CTA took (written by scan_kernel, read by filter_kernel)
    long long bounds_tiles = -1;     // total tiles the bounds were laid out for (-1: not initialised)
    cudaEvent_t scanned = nullptr;   // scan stream: the scan that filled this workspace has finished
    cudaEvent_t drained = nullptr;   // filter stream: the filters that read this workspace have finished
    bool in_use = false;
};
constexpr int kWorks = 4;

struct Slot {
    uint8_t *d_res = nullptr, *h_res = nullptr;      // this slot's head inside vsb_index::d_heads / h_heads
    uint2 *d_out = nullptr;                          // first kFirstFetch survivors (inside the head)
    uint2 *h_tail = nullptr, *d_tail = nullptr;      // survivors kFirstFetch.. (inside vsb_index::d_tails / h_tails)
    int2 *d_table = nullptr;
    int *d_hdr = nullptr;
    uint8_t *h_query = nullptr, *d_query = nullptr;  // pinned staging + device copy of the query
    int *d_ctrl = nullptr;
    cudaEvent_t done = nullptr;   // recorded after the result block of this slot has been copied to the host
    int seq = 0;
};

}  // namespace

struct vsb_index {
    int device = 0, vtype = 0, dim = 0, esize = 0, pitch = 0;
    long long cap = 0, n = 0, first_seq = 0;
    uint8_t *d_vec = nullptr;
    bool implicit_ids = true;
    std::vector<int64_t> h_rowids;
    cudaStream_t stream = nullptr;
    uint8_t *stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    int stage_next = 0;
    int num_sms = 0, max_smem = 0;
    cudaStream_t fstream = nullptr;   // filter + result copy of a query; `stream` carries staging, scans and the batch path
    // streamed mode (corpus larger than the device budget, SURVEY §8 f3): the column lives in pinned host memory and passes
    // through two device windows of win_rows rows; every window is scanned like a shard while the next one is copied
    bool streamed = false;
    uint8_t *h_arena = nullptr;       // [cap][pitch] pinned
    uint8_t *d_win[2] = {nullptr, nullptr};
    long long win_rows = 0;
    cudaStream_t cstream = nullptr;   // window copies
    cudaEvent_t win_copied[2] = {nullptr, nullptr}, win_scanned[2] = {nullptr, nullptr};
    long long st_stream_bytes = 0, st_stream_us = 0;
    cudaStream_t stream2 = nullptr;   // second scan stream (option scan_streams = 2): single-query scans alternate between the two
    cudaStream_t xstream = nullptr;   // exchange: flag wait + copy of the gathered heads to the host
    int snext = 0;
    struct Exchange *xch = nullptr;   // peer-memory exchange (multi-GPU), see exchange.inc
    // scan workspaces
    int ws_kcap = 0, ws_logcap = 0, ws_streams = 0, ws_next = 0;
    Work work[kWorks];
    Slot slot[kSlots];
    uint8_t *d_heads = nullptr, *h_heads = nullptr;   // kSlots x kHeadBytes
    uint8_t *d_tails = nullptr, *h_tails = nullptr;   // kSlots x (kOutCap - kFirstFetch) x uint2
    bool slots_ready = false;
    float *d_dist_all = nullptr;
    int last_slot = -1, last_metric = 0;
    // optional per-kernel event timing (vsb_profile_read)
    std::vector<cudaEvent_t> prof_ev;   // quadruples: before scan, after scan (scan stream), before filter, after filter (filter stream)
    std::vector<int> prof_kind;         // 1 = scan only, 2 = scan + filter
    std::vector<int> prof_nq;           // queries scanned by the timed launch
    size_t prof_used = 0;
    unsigned prof_tick = 0;
    size_t dev_bytes = 0;
    long long st_queries = 0, st_survivors = 0, st_fallbacks = 0, st_last_survivors = 0;
    long long st_batches = 0, st_batch_cands = 0, st_batch_kept = 0, st_tc_us = 0, st_tc_rows = 0, st_batch_us = 0;
    void *batch = nullptr;   // BatchWs (tensor-core batch path workspace)
};

namespace {

// ------------------------------------------------------------------ kernel dispatch
using ScanFn = void (*)(const ScanParams);
template <int VT, int MC, bool D>
ScanFn fn_of() { return scan_kernel<VT, MC, D>; }

ScanFn pick_kernel(int vtype, int mc, bool direct) {
#define ROW(VT)                                                                                                   \
    case VT:                                                                                                      \
        switch (mc) {                                                                                             \
        case MC_L2: return direct ? fn_of<VT, MC_L2, true>() : fn_of<VT, MC_L2, false>();                         \
        case MC_COS: return direct ? fn_of<VT, MC_COS, true>() : fn_of<VT, MC_COS, false>();                      \
        case MC_DOT: return direct ? fn_of<VT, MC_DOT, true>() : fn_of<VT, MC_DOT, false>();                      \
        case MC_L1: return direct ? fn_of<VT, MC_L1, true>() : fn_of<VT, MC_L1, false>();                         \
        }                                                                                                         \
        break;
    switch (vtype) {
        ROW(T_F32) ROW(T_F16) ROW(T_BF16) ROW(T_U8) ROW(T_I8)
    }
#undef ROW
    return nullptr;
}

int metric_class(int metric, int *root) {
    *root = 0;
    switch (metric) {
    case VSB_L2: *root = 1; return MC_L2;
    case VSB_SQUARED_L2: return MC_L2;
    case VSB_COSINE: return MC_COS;
    case VSB_DOT: return MC_DOT;
    case VSB_L1: return MC_L1;
    }
    return -1;
}

struct Plan {
    bool direct;
    int log2P, wtile_bytes, nsw;
    size_t smem;
};

// choose lanes-per-row, ring depth and shared-memory size for (pitch, kcap)
Plan make_plan(const vsb_index *ix, int kcap) {
    Plan pl{};
    const int pitch = ix->pitch;
    int log2P = 0;
    while (log2P < 5 && (32 >> log2P) * (long long)pitch > g_opt_stage_bytes) ++log2P;
    const size_t fixed = kBarrierBytes + (((size_t)2 * pitch + (size_t)2 * kWarps * kcap * 4 + 127) & ~(size_t)127);   // 2 query + 2 list buffers
    size_t avail = (size_t)ix->max_smem > fixed ? (size_t)ix->max_smem - fixed : 0;
    if (g_opt_ring_bytes > 0 && (size_t)g_opt_ring_bytes < avail) avail = (size_t)g_opt_ring_bytes;
    const size_t wtile = (size_t)(32 >> log2P) * pitch;
    // leave room on the SM for one filter block of the previous query (it runs beside the scan CTA, see launch_scan_group)
    const size_t reserve = filter_fast_smem(ix->num_sms) + 3072;
    if (kcap > 0 && kcap <= 32 && avail > reserve && (avail - reserve) / kWarps / (wtile ? wtile : 1) >= 2) avail -= reserve;
    int nsw = (int)(avail / kWarps / (wtile ? wtile : 1));
    if (nsw > kMaxStages) nsw = kMaxStages;
    pl.direct = g_opt_direct || nsw < 2;
    if (pl.direct) {
        pl.log2P = 5;  // a whole warp per row, coalesced 16-byte loads straight from HBM
        pl.wtile_bytes = pitch;
        pl.nsw = 1;
        pl.smem = fixed;
    } else {
        pl.log2P = log2P;
        pl.wtile_bytes = (int)wtile;
        pl.nsw = nsw;
        pl.smem = fixed + (size_t)kWarps * nsw * wtile;
    }
    return pl;
}

void free_slots(vsb_index *ix) {
    if (ix->slot[0].h_query) cudaFreeHost(ix->slot[0].h_query);     // slot 0 holds the base of the shared allocations
    if (ix->slot[0].d_query) cudaFree(ix->slot[0].d_query);
    if (ix->slot[0].d_ctrl) cudaFree(ix->slot[0].d_ctrl);
    for (int i = 0; i < kSlots; ++i) {
        Slot &s = ix->slot[i];
        if (s.done) cudaEventDestroy(s.done);
        s = Slot();
    }
    if (ix->h_heads) cudaFreeHost(ix->h_heads);
    if (ix->d_heads) cudaFree(ix->d_heads);
    if (ix->h_tails) cudaFreeHost(ix->h_tails);
    if (ix->d_tails) cudaFree(ix->d_tails);
    ix->h_heads = nullptr; ix->d_heads = nullptr; ix->h_tails = nullptr; ix->d_tails = nullptr;
    ix->slots_ready = false;
}

int ensure_slots_alloc(vsb_index *ix) {
    const size_t tail_bytes = sizeof(uint2) * (size_t)(kOutCap - kFirstFetch);
    CU(cudaMalloc((void **)&ix->d_heads, kHeadBytes * kSlots));
    CU(cudaMemset(ix->d_heads, 0, kHeadBytes * kSlots));
    CU(cudaHostAlloc((void **)&ix->h_heads, kHeadBytes * kSlots, cudaHostAllocDefault));
    memset(ix->h_heads, 0, kHeadBytes * kSlots);
    CU(cudaMalloc((void **)&ix->d_tails, tail_bytes * kSlots));
    CU(cudaHostAlloc((void **)&ix->h_tails, tail_bytes * kSlots, cudaHostAllocDefault));
    uint8_t *hq = nullptr, *dq = nullptr;                      // query staging of all slots: one pinned + one device allocation
    int *dc = nullptr;
    CU(cudaHostAlloc((void **)&hq, (size_t)ix->pitch * kSlots, cudaHostAllocDefault));
    ix->slot[0].h_query = hq;
    CU(cudaMalloc((void **)&dq, (size_t)ix->pitch * kSlots));
    ix->slot[0].d_query = dq;
    CU(cudaMalloc((void **)&dc, sizeof(int) * 4 * kSlots));
    ix->slot[0].d_ctrl = dc;
    CU(cudaMemset(dc, 0, sizeof(int) * 4 * kSlots));
    for (int i = 0; i < kSlots; ++i) {
        Slot &s = ix->slot[i];
        s.d_res = ix->d_heads + kHeadBytes * i;
        s.h_res = ix->h_heads + kHeadBytes * i;
        s.d_tail = (uint2 *)(ix->d_tails + tail_bytes * i);
        s.h_tail = (uint2 *)(ix->h_tails + tail_bytes * i);
        s.d_hdr = (int *)s.d_res;
        s.d_table = (int2 *)(s.d_res + kHdrBytes);
        s.d_out = (uint2 *)(s.d_res + kResHdrBytes);
        s.h_query = hq + (size_t)ix->pitch * i;
        s.d_query = dq + (size_t)ix->pitch * i;
        s.d_ctrl = dc + 4 * i;
        CU(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
    return VSB_OK;
}

int ensure_slots(vsb_index *ix) {
    if (ix->slots_ready) return VSB_OK;
    const int rc = ensure_slots_alloc(ix);
    if (rc != VSB_OK) { free_slots(ix); return rc; }   // a half-built slot set must not be reused (g_err keeps the CUDA message)
    ix->slots_ready = true;
    return VSB_OK;
}

// the device buffers of all scan workspaces (their events stay)
void free_workspaces(vsb_index *ix) {
    ix->ws_kcap = 0;
    for (Work &w : ix->work) {
        for (QWork &q : w.q) {
            cudaFree(q.d_lists); cudaFree(q.d_logs); cudaFree(q.d_counts); cudaFree(q.d_tlocal);
            q = QWork();
        }
        cudaFree(w.d_bounds); cudaFree(w.d_cta_time);
        w.d_bounds = nullptr; w.d_cta_time = nullptr;
        w.bounds_tiles = -1;
        w.in_use = false;
    }
}

int ensure_workspace(vsb_index *ix, int k) {
    const int kcap = (k + 31) & ~31;
    const int logcap = std::max(256, 12 * k);
    const int streams = ix->num_sms * kWarps;
    if (ix->ws_kcap >= kcap && ix->ws_logcap >= logcap && ix->ws_streams == streams) return VSB_OK;
    CU(cudaStreamSynchronize(ix->stream));       // queries in flight still use the old workspaces
    CU(cudaStreamSynchronize(ix->stream2));
    CU(cudaStreamSynchronize(ix->fstream));
    free_workspaces(ix);
    for (Work &w : ix->work) {
        for (QWork &q : w.q) {
            CU(cudaMalloc((void **)&q.d_lists, sizeof(float) * (size_t)streams * kcap));
            CU(cudaMalloc((void **)&q.d_logs, sizeof(uint2) * (size_t)streams * logcap));
            CU(cudaMalloc((void **)&q.d_counts, sizeof(int) * (size_t)streams));
            CU(cudaMalloc((void **)&q.d_tlocal, sizeof(float) * (size_t)streams));
        }
        CU(cudaMalloc((void **)&w.d_bounds, sizeof(long long) * (size_t)(ix->num_sms + 1)));
        CU(cudaMalloc((void **)&w.d_cta_time, sizeof(unsigned) * (size_t)ix->num_sms));
        if (!w.scanned) CU(cudaEventCreateWithFlags(&w.scanned, cudaEventDisableTiming));
        if (!w.drained) CU(cudaEventCreateWithFlags(&w.drained, cudaEventDisableTiming));
    }
    ix->ws_kcap = kcap; ix->ws_logcap = logcap; ix->ws_streams = streams;
    return VSB_OK;
}

unsigned exchange_next_seq(vsb_index *ix, int slot);
int merge_blocks_strided(const uint8_t *blocks, int world, size_t stride, const int64_t *first_seq, int k, int64_t *out_rowids, double *out_dist);
void exchange_free(vsb_index *ix);
int exchange_fill_push(vsb_index *ix, PushParams *pp);

// launches ONE scan kernel for nq independent queries (device pointers, pitch bytes each) on ix->stream and, when k > 0,
// one filter launch (grid.y = nq) on ix->fstream.  slots[g] receives query g's result.
// fetch: copy the slots' heads to pinned host memory afterwards (false when the heads are all-gathered on the device)
// ss: the scan stream of this launch (next_scan_stream); push: the filter also pushes each head into the exchange targets
// view_vec / view_n: scan these rows instead of the resident column (the windows of a streamed index)
int launch_scan_group(vsb_index *ix, int metric, const uint8_t *const *d_queries, int nq, int k, Slot *const *slots, float *d_dist_all,
                      bool fetch, cudaStream_t ss, bool push = false, const uint8_t *view_vec = nullptr, long long view_n = -1) {
    const uint8_t *scan_vec = view_vec ? view_vec : ix->d_vec;
    const long long scan_n = view_vec ? view_n : ix->n;
    if (!scan_vec) return fail(VSB_EINVAL, "this entry point needs a resident (not streamed) index");
    int root = 0;
    const int mc = metric_class(metric, &root);
    if (mc < 0) return fail(VSB_EINVAL, "unknown distance metric %d", metric);
    if (nq < 1 || nq > kMaxGroup) return fail(VSB_EINVAL, "a launch scans 1..%d queries", kMaxGroup);
    // per-launch list stride: the workspace may have been sized by an earlier, larger k (ensure_workspace never shrinks), but
    // the scan's list layout, the filter's FAST/generic choice and its shared-memory layout all follow THIS query's k
    const int kcap = k > 0 ? ((k + 31) & ~31) : 0;
    if (kcap > ix->ws_kcap) return fail(VSB_EINVAL, "scan workspace too small for k = %d", k);
    const Plan pl = make_plan(ix, kcap);
    ScanFn fn = pick_kernel(ix->vtype, mc, pl.direct);
    if (!fn) return fail(VSB_EINVAL, "unsupported vector type %d", ix->vtype);
    // max-shared carve-out for the scan AND the filter kernel: kernels that want different L1/shared splits cannot share
    // an SM, and the filter blocks of launch i are meant to run beside the scan CTAs of launch i+1
    CU((cudaError_t)set_smem_limit((const void *)fn, pl.smem));

    // the scan runs on its scan stream (ss), the filter (+ result copy) on ix->fstream: while the filters of this launch walk the
    // k-lists and compact the candidate logs, the scan of the next launch is already streaming the shard (the filter
    // blocks are small enough to sit on the SMs beside the scan CTAs).  The two workspaces alternate.
    Work *wk = nullptr;
    if (k > 0) {
        wk = &ix->work[ix->ws_next];
        ix->ws_next = (ix->ws_next + 1) % kWorks;
        if (wk->in_use) CU(cudaStreamWaitEvent(ss, wk->drained, 0));   // its previous filters must have read it
    }
    // adaptive partition (k <= 32 path only: that filter kernel maintains it): equal shares to start with
    const long long rpw = 32 >> pl.log2P;
    const long long total_tiles = (scan_n + rpw - 1) / rpw;
    const bool balance = wk != nullptr && g_opt_balance && kcap == 32 && total_tiles >= 64ll * ix->num_sms;
    if (balance && wk->bounds_tiles != total_tiles) {
        std::vector<long long> b((size_t)ix->num_sms + 1);
        for (int c = 0; c <= ix->num_sms; ++c) b[(size_t)c] = (total_tiles * c) / ix->num_sms;
        CU(cudaMemcpyAsync(wk->d_bounds, b.data(), sizeof(long long) * b.size(), cudaMemcpyHostToDevice, ss));   // pageable: staged before return
        CU(cudaMemsetAsync(wk->d_cta_time, 0, sizeof(unsigned) * (size_t)ix->num_sms, ss));
        wk->bounds_tiles = total_tiles;
    }
    ScanParams p{};
    p.vec = scan_vec;
    p.n = scan_n;
    p.pitch = ix->pitch;
    p.nc = ix->pitch / 16;
    p.log2P = pl.log2P;
    p.wtile_bytes = pl.wtile_bytes;
    p.nsw = pl.nsw;
    p.root = root;
    p.k = k;
    p.kcap = kcap;
    p.logcap = ix->ws_logcap;
    p.nq = nq;
    for (int g = 0; g < nq; ++g) {
        ScanQuery &q = p.q[g];
        q.query = d_queries[g];
        q.lists = wk ? wk->q[g].d_lists : nullptr;
        q.tlocal = wk ? wk->q[g].d_tlocal : nullptr;
        q.logs = wk ? wk->q[g].d_logs : nullptr;
        q.counts = wk ? wk->q[g].d_counts : nullptr;
        q.ctrl = slots ? slots[g]->d_ctrl : nullptr;
        q.dist_all = d_dist_all;
    }
    p.bounds = balance ? wk->d_bounds : nullptr;
    p.cta_time = balance ? wk->d_cta_time : nullptr;
    cudaEvent_t *pev = nullptr;
    if (g_opt_time_kernels > 0 && (ix->prof_tick++ % g_opt_time_kernels) == 0) {   // time_kernels = N: every N-th launch
        if (ix->prof_used + 4 > ix->prof_ev.size()) {
            for (int i = 0; i < 4; ++i) {
                cudaEvent_t e;
                CU(cudaEventCreate(&e));
                ix->prof_ev.push_back(e);
            }
        }
        pev = &ix->prof_ev[ix->prof_used];
        ix->prof_used += 4;
        ix->prof_kind.push_back(k > 0 ? 2 : 1);
        ix->prof_nq.push_back(nq);
        CU(cudaEventRecord(pev[0], ss));
    }
    fn<<<ix->num_sms, kThreads, pl.smem, ss>>>(p);
    CU(cudaGetLastError());
    ++g_launches;
    if (pev) CU(cudaEventRecord(pev[1], ss));
    if (k > 0) {
        CU(cudaEventRecord(wk->scanned, ss));
        CU(cudaStreamWaitEvent(ix->fstream, wk->scanned, 0));
        FilterParams f{};
        if (push) {
            const int rc = exchange_fill_push(ix, &f.push);
            if (rc) return rc;
            if (g_opt_push_mode == 1) f.push.ntargets = 0;      // the heads are pushed by push_heads_kernel (exchange_push); src / world still label the header
        }
        f.S = ix->ws_streams;
        f.k = k;
        f.kcap = kcap;
        f.logcap = ix->ws_logcap;
        f.headcap = kFirstFetch;
        f.outcap = kOutCap;
        f.nq = nq;
        const bool fast = (kcap == 32) && filter_fast_smem(f.S / kWarps) + 2048 <= (size_t)ix->max_smem;
        const int fw = filter_warps(fast);
        const int nblocks = (f.S + fw - 1) / fw;
        if (nblocks > kTableCap) return fail(VSB_ERANGE, "too many filter blocks (%d)", nblocks);
        for (int g = 0; g < nq; ++g) {
            FilterQuery &q = f.q[g];
            Slot *slot = slots[g];
            q.lists = wk->q[g].d_lists;
            q.tlocal = wk->q[g].d_tlocal;
            q.logs = wk->q[g].d_logs;
            q.counts = wk->q[g].d_counts;
            q.out = slot->d_out;
            q.out_tail = slot->d_tail;
            q.table = slot->d_table;
            q.hdr = slot->d_hdr;
            q.ctrl = slot->d_ctrl;
            q.seqno = ++slot->seq;
            q.xslot = (int)(slot - ix->slot);
            q.xseq = push ? exchange_next_seq(ix, q.xslot) : 0u;
        }
        f.bounds = balance ? wk->d_bounds : nullptr;
        f.cta_time = wk->d_cta_time;
        f.total_tiles = total_tiles;
        if (pev) CU(cudaEventRecord(pev[2], ix->fstream));
        const dim3 grid((unsigned)nblocks, (unsigned)nq);
        if (fast) {
            const size_t fsm = filter_fast_smem(f.S / kWarps);
            CU((cudaError_t)set_smem_limit((const void *)filter_kernel<true>, fsm));
            filter_kernel<true><<<grid, fw * 32, fsm, ix->fstream>>>(f);
        } else {
            const size_t fsm = sizeof(float) * ((size_t)2 * kFilterWarps * kcap + (size_t)f.S + 32);
            CU((cudaError_t)set_smem_limit((const void *)filter_kernel<false>, fsm));
            filter_kernel<false><<<grid, fw * 32, fsm, ix->fstream>>>(f);
        }
        CU(cudaGetLastError());
        ++g_launches;
        if (pev) CU(cudaEventRecord(pev[3], ix->fstream));
        CU(cudaEventRecord(wk->drained, ix->fstream));
        wk->in_use = true;
        if (fetch) {   // the heads of consecutive slots are contiguous: one copy when the group's slots are
            bool contiguous = true;
            for (int g = 1; g < nq; ++g) contiguous = contiguous && slots[g]->d_res == slots[g - 1]->d_res + kHeadBytes;
            if (contiguous) CU(cudaMemcpyAsync(slots[0]->h_res, slots[0]->d_res, kHeadBytes * (size_t)nq, cudaMemcpyDeviceToHost, ix->fstream));
            else
                for (int g = 0; g < nq; ++g) CU(cudaMemcpyAsync(slots[g]->h_res, slots[g]->d_res, kHeadBytes, cudaMemcpyDeviceToHost, ix->fstream));
        }
        for (int g = 0; g < nq; ++g) CU(cudaEventRecord(slots[g]->done, ix->fstream));
    }
    return VSB_OK;
}

// single-query scans alternate between two streams (option scan_streams, see g_opt_scan_streams)
cudaStream_t next_scan_stream(vsb_index *ix) {
    if (g_opt_scan_streams < 2) return ix->stream;
    ix->snext ^= 1;
    return ix->snext ? ix->stream2 : ix->stream;
}

inline int64_t rowid_of(const vsb_index *ix, uint32_t local) {
    return ix->implicit_ids ? (int64_t)(ix->first_seq + (long long)local + 1) : ix->h_rowids[local];
}

// ------------------------------------------------------------------ the reference's k-slot algorithm
inline int first_max(const double *v, int n) {  // first index of the maximum, strict '>' (:2022-2049)
    int b = 0;
    for (int i = 1; i < n; ++i)
        if (v[i] > v[b]) b = i;
    return b;
}
// the k slots of one query: started with the max_index carried over from the previous query, offered the candidates in scan
// order, finished into the sorted result
struct SlotReplay {
    int k, mi;
    double *dist;
    int64_t *ids;
    SlotReplay(int k_, int max_index, double *dist_, int64_t *ids_) : k(k_), mi(max_index), dist(dist_), ids(ids_) {   // :1808-1813
        for (int i = 0; i < k; ++i) { dist[i] = std::numeric_limits<double>::infinity(); ids[i] = 0; }
        if (mi < 0 || mi >= k) mi = 0;
    }
    void offer(float d, int64_t id) {  // :2102-2106 / :2145-2152
        if ((double)d < dist[mi]) {
            dist[mi] = (double)d;
            ids[mi] = id;
            mi = first_max(dist, k);
        }
    }
    void offer_bits(uint32_t bits, int64_t id) {   // a candidate's distance as the GPU stored it
        float d;
        memcpy(&d, &bits, 4);
        offer(d, id);
    }
    int finish() {  // exchange sort + INF trim (:2051-2069, :1816-1817); returns the used slots
        const double inf = std::numeric_limits<double>::infinity();
        int unused = 0;
        for (int i = 0; i + 1 < k; ++i) {
            if (dist[i] == inf) ++unused;
            for (int j = i + 1; j < k; ++j)
                if (dist[j] < dist[i]) { std::swap(dist[i], dist[j]); std::swap(ids[i], ids[j]); }
        }
        if (dist[k - 1] == inf) ++unused;
        return k - unused;
    }
};

// ------------------------------------------------------------------ result heads on the host (layout in scan_kernels.cuh)
// survivors that a head carries itself (a head whose kHdrHeadcap is unset or out of range: kFirstFetch)
inline int head_cap(const int *hdr) {
    const int c = hdr[kHdrHeadcap];
    return (c > 0 && c <= kFirstFetch) ? c : kFirstFetch;
}

// walks the survivors of a result head in scan order: visit(distance bits, local row).  Survivors beyond the head's headcap
// are read from tail (nullptr when the head holds them all).  Returns how many were visited.
template <class Visit>
int visit_head(const uint8_t *head, const uint2 *tail, Visit visit) {
    const int *hdr = (const int *)head;
    const int2 *table = (const int2 *)(head + kHdrBytes);
    const uint2 *out = (const uint2 *)(head + kResHdrBytes);
    const int headcap = head_cap(hdr), nblocks = hdr[kHdrBlocks];
    int n = 0;
    for (int b = 0; b < nblocks; ++b) {
        const int2 t = table[b];
        for (int i = 0; i < t.y; ++i, ++n) {
            const int at = t.x + i;
            const uint2 c = at < headcap ? out[at] : tail[at - headcap];
            visit(c.x, c.y);
        }
    }
    return n;
}

// gather the survivors of a finished slot in scan order; returns count or <0
int gather_survivors(vsb_index *ix, Slot *slot, std::vector<uint2> &out, bool *overflow) {
    *overflow = false;
    const int *hdr = (const int *)slot->h_res;
    if (hdr[kHdrSeq] != slot->seq) return fail(VSB_ECUDA, "scan result header not published (seq %d != %d)", hdr[kHdrSeq], slot->seq);
    if (hdr[kHdrFlags]) { *overflow = true; return 0; }
    const int total = hdr[kHdrTotal], headcap = head_cap(hdr);
    if (total > headcap) {  // rare: fetch the tail of the survivor list
        if (cudaMemcpyAsync(slot->h_tail, slot->d_tail, sizeof(uint2) * (size_t)(total - headcap),
                            cudaMemcpyDeviceToHost, ix->fstream) != cudaSuccess ||
            cudaStreamSynchronize(ix->fstream) != cudaSuccess)
            return fail(VSB_ECUDA, "fetching %d survivors failed: %s", total, cudaGetErrorString(cudaGetLastError()));
    }
    out.clear();
    out.reserve((size_t)total);
    const int n = visit_head(slot->h_res, slot->h_tail, [&](uint32_t bits, uint32_t row) { out.push_back(make_uint2(bits, row)); });
    ix->st_queries++;
    ix->st_survivors += n;
    ix->st_last_survivors = n;
    return n;
}

int stage_query(vsb_index *ix, Slot *slot, const void *query, cudaStream_t ss) {
    const int qbytes = ix->dim * ix->esize;
    memcpy(slot->h_query, query, (size_t)qbytes);
    if (ix->pitch > qbytes) memset(slot->h_query + qbytes, 0, (size_t)(ix->pitch - qbytes));
    CU(cudaMemcpyAsync(slot->d_query, slot->h_query, (size_t)ix->pitch, cudaMemcpyHostToDevice, ss));
    return VSB_OK;
}

// ---- streamed index: the window loop.  Window w (rows [w * win_rows, ...)) is copied into d_win[w & 1] on the copy stream
// while window w-1 is being scanned; a window is scanned exactly like a shard (scan + filter into a result slot), its survivors
// carry window-local rows.  visit(w, first_row, rows, slot) is called in window order once the slot's head is on the host.
template <class Launch, class Visit>
int stream_windows(vsb_index *ix, int depth, Launch launch, Visit visit) {
    const long long W = (ix->n + ix->win_rows - 1) / ix->win_rows;
    const auto t0 = std::chrono::steady_clock::now();
    long long next_visit = 0;
    for (long long w = 0; w < W; ++w) {
        const int b = (int)(w & 1);
        const long long r0 = w * ix->win_rows, rows = std::min(ix->win_rows, ix->n - r0);
        if (w >= 2) CU(cudaStreamWaitEvent(ix->cstream, ix->win_scanned[b], 0));       // the scan of window w-2 has read this buffer
        CU(cudaMemcpyAsync(ix->d_win[b], ix->h_arena + (size_t)r0 * ix->pitch, (size_t)rows * ix->pitch, cudaMemcpyHostToDevice, ix->cstream));
        CU(cudaEventRecord(ix->win_copied[b], ix->cstream));
        CU(cudaStreamWaitEvent(ix->stream, ix->win_copied[b], 0));
        while (w - next_visit >= depth) {                                                // free the slot this window will use
            const int rc = visit(next_visit, next_visit * ix->win_rows, std::min(ix->win_rows, ix->n - next_visit * ix->win_rows), (int)(next_visit % depth));
            if (rc) return rc;
            ++next_visit;
        }
        const int rc = launch(w, ix->d_win[b], rows, (int)(w % depth));
        if (rc) return rc;
        CU(cudaEventRecord(ix->win_scanned[b], ix->stream));
        ix->st_stream_bytes += rows * ix->pitch;
    }
    for (; next_visit < W; ++next_visit) {
        const int rc = visit(next_visit, next_visit * ix->win_rows, std::min(ix->win_rows, ix->n - next_visit * ix->win_rows), (int)(next_visit % depth));
        if (rc) return rc;
    }
    ix->st_stream_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return VSB_OK;
}

// all distances of a streamed index (stream modules, k > 256, overflow fallback)
int streamed_scan_all(vsb_index *ix, int metric, const uint8_t *d_query, float *out_dist) {
    if (!ix->d_dist_all) {
        CU(cudaMalloc((void **)&ix->d_dist_all, sizeof(float) * 2 * (size_t)ix->win_rows));
        ix->dev_bytes += sizeof(float) * 2 * (size_t)ix->win_rows;
    }
    return stream_windows(ix, 2,
        [&](long long, const uint8_t *vec, long long rows, int s) {
            return launch_scan_group(ix, metric, &d_query, 1, 0, nullptr, ix->d_dist_all + (size_t)s * ix->win_rows, false, ix->stream, false, vec, rows);
        },
        [&](long long, long long r0, long long rows, int s) {
            // distances of window w sit in half s of d_dist_all; the copy is ordered behind that window's scan on the same stream
            CU(cudaMemcpyAsync(out_dist + r0, ix->d_dist_all + (size_t)s * ix->win_rows, sizeof(float) * (size_t)rows, cudaMemcpyDeviceToHost, ix->stream));
            CU(cudaStreamSynchronize(ix->stream));
            return (int)VSB_OK;
        });
}

// candidates of a streamed index: every window's survivors, in scan order, rows made column-global
int streamed_candidates(vsb_index *ix, int metric, const uint8_t *d_query, int k, std::vector<uint2> &cands, bool *overflow) {
    cands.clear();
    *overflow = false;
    const int depth = 4;                                  // result slots 0..3 rotate over the windows
    std::vector<uint2> part;
    return stream_windows(ix, depth,
        [&](long long, const uint8_t *vec, long long rows, int s) {
            Slot *slot = &ix->slot[s];
            return launch_scan_group(ix, metric, &d_query, 1, k, &slot, nullptr, true, ix->stream, false, vec, rows);
        },
        [&](long long, long long r0, long long, int s) {
            Slot *slot = &ix->slot[s];
            CU(cudaEventSynchronize(slot->done));
            bool ovf = false;
            const int n = gather_survivors(ix, slot, part, &ovf);
            if (n < 0) return n;
            if (ovf) *overflow = true;
            for (const uint2 &c : part) cands.push_back(make_uint2(c.x, c.y + (uint32_t)r0));
            return (int)VSB_OK;
        });
}

// the all-distances path (k > kMaxK, a candidate overflow, vsb_scan_all): stages a host query on slot 0 and computes the
// distance of every row, resident or streamed, into dist (scan order)
int query_all_distances(vsb_index *ix, int metric, const void *query, std::vector<float> &dist) {
    CU(cudaSetDevice(ix->device));
    int rc = ensure_slots(ix);
    if (rc) return rc;
    rc = stage_query(ix, &ix->slot[0], query, ix->stream);
    if (rc) return rc;
    const uint8_t *d_query = ix->slot[0].d_query;
    dist.resize((size_t)ix->n);
    if (ix->streamed) return streamed_scan_all(ix, metric, d_query, dist.data());
    if (!ix->d_dist_all) {
        CU(cudaMalloc((void **)&ix->d_dist_all, sizeof(float) * (size_t)std::max<long long>(ix->cap, 1)));
        ix->dev_bytes += sizeof(float) * (size_t)ix->cap;
    }
    rc = launch_scan_group(ix, metric, &d_query, 1, 0, nullptr, ix->d_dist_all, true, ix->stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(dist.data(), ix->d_dist_all, sizeof(float) * (size_t)ix->n, cudaMemcpyDeviceToHost, ix->stream));
    CU(cudaStreamSynchronize(ix->stream));
    return VSB_OK;
}

// one query, host in / candidates out (sorted by scan order).  Falls back to the all-distances kernel when the
// candidate log overflowed or k is larger than the candidate path supports (still GPU-computed distances).
int query_candidates(vsb_index *ix, int metric, const void *query, int k, std::vector<uint2> &cands) {
    CU(cudaSetDevice(ix->device));
    int rc = ensure_slots(ix);
    if (rc) return rc;
    bool overflow = (k > kMaxK);
    if (!overflow) {
        Slot *slot = &ix->slot[ix->streamed ? kSlots - 1 : 0];   // streamed: slots 0..3 rotate over the windows, the query is parked in the last one
        rc = stage_query(ix, slot, query, ix->stream);
        if (rc) return rc;
        rc = ensure_workspace(ix, k);
        if (rc) return rc;
        if (ix->streamed) {
            rc = streamed_candidates(ix, metric, slot->d_query, k, cands, &overflow);
            if (rc) return rc;
        } else {
            const uint8_t *dq = slot->d_query;
            rc = launch_scan_group(ix, metric, &dq, 1, k, &slot, nullptr, true, ix->stream);
            if (rc) return rc;
            CU(cudaEventSynchronize(slot->done));
            const int n = gather_survivors(ix, slot, cands, &overflow);
            if (n < 0) return n;
        }
    }
    if (!overflow) return VSB_OK;
    ix->st_fallbacks++;
    std::vector<float> dist;
    rc = query_all_distances(ix, metric, query, dist);
    if (rc) return rc;
    cands.resize((size_t)ix->n);
    for (long long i = 0; i < ix->n; ++i) {
        uint32_t bits;
        memcpy(&bits, &dist[(size_t)i], 4);
        cands[(size_t)i] = make_uint2(bits, (uint32_t)i);
    }
    return VSB_OK;
}

int check_index(const vsb_index *ix) {
    if (!ix) return fail(VSB_EINVAL, "null index");
    return VSB_OK;
}

// scan + filter launches for a group of independent queries (query j at queries + j * query_stride; slots first_slot ..).
// push: the heads also travel to the exchange targets (peer memory), see exchange.inc
int submit_group(vsb_index *ix, int metric, const void *queries, int64_t query_stride, int nq, int query_on_device, int k, int fetch,
                 int first_slot, bool push) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!queries || k <= 0 || k > kMaxK) return fail(VSB_EINVAL, "bad scan arguments (k must be 1..%d)", kMaxK);
    if (nq <= 0 || first_slot < 0 || first_slot + nq > kSlots) return fail(VSB_EINVAL, "bad slot group [%d, %d)", first_slot, first_slot + nq);
    CU(cudaSetDevice(ix->device));
    int rc = ensure_slots(ix);
    if (rc) return rc;
    rc = ensure_workspace(ix, k);
    if (rc) return rc;
    const bool fuse = (double)ix->n * ix->pitch < (double)g_opt_fuse_mb * 1048576.0;
    const int per_launch = fuse ? kMaxGroup : 1;          // small shards: one scan launch per kMaxGroup queries
    for (int g0 = 0; g0 < nq; g0 += per_launch) {
        const int m = std::min(per_launch, nq - g0);
        const uint8_t *dq[kMaxGroup];
        Slot *sl[kMaxGroup];
        cudaStream_t ss = next_scan_stream(ix);
        for (int j = 0; j < m; ++j) {
            Slot *slot = &ix->slot[first_slot + g0 + j];
            const uint8_t *q = (const uint8_t *)queries + (size_t)(g0 + j) * (size_t)query_stride;
            if (!query_on_device) {
                if (slot->seq > 0) CU(cudaEventSynchronize(slot->done));   // the slot's pinned staging buffer is free again
                rc = stage_query(ix, slot, q, ss);
                if (rc) return rc;
                q = slot->d_query;
            }
            dq[j] = q;
            sl[j] = slot;
        }
        rc = launch_scan_group(ix, metric, dq, m, k, sl, nullptr, fetch != 0, ss, push);
        if (rc) return rc;
        ix->last_slot = first_slot + g0 + m - 1;
        ix->last_metric = metric;
    }
    return VSB_OK;
}

}  // namespace

#include "batch_host.inc"
#include "exchange.inc"
#include "quantize.inc"

// ====================================================================== C ABI
extern "C" {

int vsb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *vsb_last_error(void) { return g_err.c_str(); }

const char *vsb_backend_name(void) {
    static std::once_flag once;
    static char name[160];
    std::call_once(once, [] {
        int n = vsb_device_count();
        if (n <= 0) { snprintf(name, sizeof name, "CUDA sm_100a (no device)"); return; }
        cudaDeviceProp pr{};
        cudaGetDeviceProperties(&pr, 0);
        snprintf(name, sizeof name, "CUDA sm_100a (%s x%d, cc %d.%d)", pr.name, n, pr.major, pr.minor);
    });
    return name;
}

int64_t vsb_kernel_launches(void) { return g_launches.load(); }

int vsb_set_option(const char *name, int value) {
    int *p = nullptr;
    if (!strcmp(name, "stage_bytes")) p = &g_opt_stage_bytes;
    else if (!strcmp(name, "direct")) p = &g_opt_direct;
    else if (!strcmp(name, "ring_bytes")) p = &g_opt_ring_bytes;
    else if (!strcmp(name, "time_kernels")) p = &g_opt_time_kernels;
    else if (!strcmp(name, "no_batch")) p = &g_opt_no_batch;
    else if (!strcmp(name, "epi2")) p = &g_opt_epi2;
    else if (!strcmp(name, "epi_chunk")) p = &g_opt_epi_chunk;
    else if (!strcmp(name, "balance")) p = &g_opt_balance;
    else if (!strcmp(name, "fuse_mb")) p = &g_opt_fuse_mb;
    else if (!strcmp(name, "batch_m0")) p = &g_opt_batch_m0;
    else if (!strcmp(name, "batch_growth")) p = &g_opt_batch_growth;
    else if (!strcmp(name, "merge_stream")) p = &g_opt_merge_stream;
    else if (!strcmp(name, "batch_debug")) p = &g_opt_batch_debug;
    else if (!strcmp(name, "scan_streams")) p = &g_opt_scan_streams;
    else if (!strcmp(name, "xwait_ms")) p = &g_opt_xwait_ms;
    else if (!strcmp(name, "push_repeat")) p = &g_opt_push_repeat;
    else if (!strcmp(name, "push_mode")) p = &g_opt_push_mode;
    if (!p) return fail(VSB_EINVAL, "unknown option %s", name);
    if (value < 0) return fail(VSB_EINVAL, "option %s: values are non-negative", name);   // so that a negative return is always an error
    int old = *p;
    *p = value;
    return old;
}

static int index_create(vsb_index **out, int device, int vtype, int dim, int64_t capacity_rows, int64_t first_seq, int64_t window_rows);

int vsb_index_create(vsb_index **out, int device, int vtype, int dim, int64_t capacity_rows, int64_t first_seq) {
    return index_create(out, device, vtype, dim, capacity_rows, first_seq, 0);
}

int vsb_index_create_streamed(vsb_index **out, int device, int vtype, int dim, int64_t capacity_rows, int64_t first_seq, int64_t window_rows) {
    if (window_rows <= 0) return fail(VSB_EINVAL, "window_rows must be positive");
    return index_create(out, device, vtype, dim, capacity_rows, first_seq, window_rows);
}

int vsb_index_is_streamed(const vsb_index *ix) { return ix && ix->streamed ? 1 : 0; }

static int index_create(vsb_index **out, int device, int vtype, int dim, int64_t capacity_rows, int64_t first_seq, int64_t window_rows) {
    if (!out) return fail(VSB_EINVAL, "out is null");
    *out = nullptr;
    const int es = elem_size(vtype);
    if (!es) return fail(VSB_EINVAL, "unknown vector type %d", vtype);
    if (dim <= 0) return fail(VSB_EINVAL, "dimension must be positive");
    if (capacity_rows < 0 || capacity_rows > 0xFFFFFFF0ll) return fail(VSB_EINVAL, "capacity_rows out of range");
    int ndev = vsb_device_count();
    if (ndev <= 0) return fail(VSB_ENODEV, "no CUDA device available (this build has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(VSB_EINVAL, "device %d out of range (have %d)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp pr{};
    CU(cudaGetDeviceProperties(&pr, device));
    if (pr.major < 9) return fail(VSB_ENODEV, "device %s (cc %d.%d) lacks TMA bulk copies; sm_100a required", pr.name, pr.major, pr.minor);
    vsb_index *ix = new (std::nothrow) vsb_index();
    if (!ix) return fail(VSB_ENOMEM, "out of host memory");
    ix->device = device; ix->vtype = vtype; ix->dim = dim; ix->esize = es;
    ix->pitch = (dim * es + 15) & ~15;
    ix->cap = capacity_rows; ix->first_seq = first_seq;
    ix->num_sms = pr.multiProcessorCount;
    ix->max_smem = (int)pr.sharedMemPerBlockOptin;
    cudaError_t e = cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->fstream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->xstream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        if (ix->stream) cudaStreamDestroy(ix->stream);
        if (ix->stream2) cudaStreamDestroy(ix->stream2);
        if (ix->fstream) cudaStreamDestroy(ix->fstream);
        delete ix;
        return fail(VSB_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    size_t bytes = (size_t)std::max<long long>(capacity_rows, 1) * ix->pitch + 1024;
    if (window_rows > 0) {
        // streamed: the column stays in pinned host memory, two windows on the device
        ix->streamed = true;
        ix->win_rows = std::min<long long>(std::max<long long>(window_rows, 32), std::max<long long>(capacity_rows, 32));
        e = cudaHostAlloc((void **)&ix->h_arena, bytes, cudaHostAllocDefault);
        const size_t wb = (size_t)ix->win_rows * ix->pitch + 1024;
        for (int b = 0; b < 2 && e == cudaSuccess; ++b) {
            e = cudaMalloc((void **)&ix->d_win[b], wb);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->win_copied[b], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->win_scanned[b], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->cstream, cudaStreamNonBlocking);
        bytes = 2 * wb;
    } else {
        e = cudaMalloc((void **)&ix->d_vec, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        const std::string why = cudaGetErrorString(e);
        vsb_index_free(ix);
        return fail(VSB_ENOMEM, "allocating %zu bytes for the %s column failed: %s", bytes, window_rows > 0 ? "streamed" : "resident", why.c_str());
    }
    ix->dev_bytes = bytes;
    *out = ix;
    return VSB_OK;
}

static int stage_acquire(vsb_index *ix, int *which) {
    const int b = ix->stage_next;
    if (!ix->stage[b]) {
        CU(cudaHostAlloc((void **)&ix->stage[b], kStageBuf, cudaHostAllocDefault));
        CU(cudaEventCreateWithFlags(&ix->stage_ev[b], cudaEventDisableTiming));
    } else {
        CU(cudaEventSynchronize(ix->stage_ev[b]));  // previous copy out of this buffer finished
    }
    ix->stage_next ^= 1;
    *which = b;
    return VSB_OK;
}

// switches ix from implicit rowids (first_seq + row + 1) to an explicit list, filled in for the rows appended so far
static void materialise_ids(vsb_index *ix) {
    if (!ix->implicit_ids) return;
    ix->h_rowids.resize((size_t)ix->n);
    for (long long i = 0; i < ix->n; ++i) ix->h_rowids[(size_t)i] = ix->first_seq + i + 1;
    ix->implicit_ids = false;
}

// src_stride: bytes between rows in host memory; src_off: offset of the vector inside a row
static int append_rows(vsb_index *ix, const uint8_t *src, size_t src_stride, size_t src_off, const int64_t *rowids,
                       bool ids_inline, int64_t nrows) {
    if (nrows < 0) return fail(VSB_EINVAL, "negative row count");
    if (ix->n + nrows > ix->cap) return fail(VSB_ERANGE, "index capacity exceeded (%lld + %lld > %lld)", ix->n, (long long)nrows, ix->cap);
    CU(cudaSetDevice(ix->device));
    const size_t rowbytes = (size_t)ix->dim * ix->esize;
    const size_t pitch = (size_t)ix->pitch;
    if (ids_inline || rowids != nullptr) materialise_ids(ix);
    if (pitch > kStageBuf) return fail(VSB_ERANGE, "row pitch %zu exceeds the %zu-byte staging buffer", pitch, (size_t)kStageBuf);
    const int64_t per_buf = (int64_t)(kStageBuf / pitch);
    for (int64_t done = 0; done < nrows;) {
        // a streamed index takes all rows straight into its pinned arena; a resident one goes through the staging buffers
        const int64_t m = ix->streamed ? nrows : std::min<int64_t>(per_buf, nrows - done);
        int b = 0;
        uint8_t *dst;
        if (ix->streamed) {
            dst = ix->h_arena + (size_t)ix->n * pitch;
        } else {
            const int rc = stage_acquire(ix, &b);
            if (rc) return rc;
            dst = ix->stage[b];
        }
        for (int64_t r = 0; r < m; ++r) {
            const uint8_t *row = src + (size_t)(done + r) * src_stride;
            memcpy(dst + (size_t)r * pitch, row + src_off, rowbytes);
            if (pitch > rowbytes) memset(dst + (size_t)r * pitch + rowbytes, 0, pitch - rowbytes);
            if (ids_inline) {
                uint64_t v = 0;  // little-endian int64 rowid in front of the vector (INT64_FROM_INT8PTR, :86-94)
                for (int i = 7; i >= 0; --i) v = (v << 8) | row[i];
                ix->h_rowids.push_back((int64_t)v);
            }
        }
        if (!ix->streamed) {
            CU(cudaMemcpyAsync(ix->d_vec + (size_t)(ix->n + done) * pitch, dst, (size_t)m * pitch, cudaMemcpyHostToDevice, ix->stream));
            CU(cudaEventRecord(ix->stage_ev[b], ix->stream));
        }
        done += m;
    }
    if (!ids_inline) {
        if (rowids) ix->h_rowids.insert(ix->h_rowids.end(), rowids, rowids + nrows);
        else if (!ix->implicit_ids)
            for (int64_t r = 0; r < nrows; ++r) ix->h_rowids.push_back(ix->first_seq + ix->n + r + 1);
    }
    ix->n += nrows;
    return VSB_OK;
}

int vsb_index_append_dense(vsb_index *ix, const void *vectors, const int64_t *rowids, int64_t nrows) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!vectors && nrows > 0) return fail(VSB_EINVAL, "vectors is null");
    return append_rows(ix, (const uint8_t *)vectors, (size_t)ix->dim * ix->esize, 0, rowids, false, nrows);
}

int vsb_index_append_quant_chunk(vsb_index *ix, const void *chunk, int64_t nrows) {
    if (check_index(ix)) return VSB_EINVAL;
    if (ix->esize != 1) return fail(VSB_EINVAL, "quantized chunks need a UINT8/INT8 index");
    if (!chunk && nrows > 0) return fail(VSB_EINVAL, "chunk is null");
    return append_rows(ix, (const uint8_t *)chunk, (size_t)ix->dim + 8, 8, nullptr, true, nrows);
}

int vsb_index_append_device(vsb_index *ix, const void *d_vectors, const int64_t *d_rowids, int64_t nrows) {
    if (check_index(ix)) return VSB_EINVAL;
    if (nrows < 0 || ix->n + nrows > ix->cap) return fail(VSB_ERANGE, "index capacity exceeded");
    if (ix->streamed) return fail(VSB_EINVAL, "a streamed index takes host rows (vsb_index_append_dense / _quant_chunk)");
    CU(cudaSetDevice(ix->device));
    const size_t rowbytes = (size_t)ix->dim * ix->esize;
    if ((size_t)ix->pitch != rowbytes)
        CU(cudaMemsetAsync(ix->d_vec + (size_t)ix->n * ix->pitch, 0, (size_t)nrows * ix->pitch, ix->stream));
    CU(cudaMemcpy2DAsync(ix->d_vec + (size_t)ix->n * ix->pitch, (size_t)ix->pitch, d_vectors, rowbytes, rowbytes, (size_t)nrows,
                         cudaMemcpyDeviceToDevice, ix->stream));
    if (d_rowids) {
        materialise_ids(ix);
        ix->h_rowids.resize((size_t)(ix->n + nrows));
        CU(cudaMemcpyAsync(ix->h_rowids.data() + ix->n, d_rowids, sizeof(int64_t) * (size_t)nrows, cudaMemcpyDeviceToHost, ix->stream));
    } else if (!ix->implicit_ids) {
        for (int64_t r = 0; r < nrows; ++r) ix->h_rowids.push_back(ix->first_seq + ix->n + r + 1);
    }
    CU(cudaStreamSynchronize(ix->stream));
    ix->n += nrows;
    return VSB_OK;
}

int vsb_index_finalize(vsb_index *ix) {
    if (check_index(ix)) return VSB_EINVAL;
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamSynchronize(ix->stream));
    for (int b = 0; b < 2; ++b) {  // the staging buffers are only needed while loading
        if (ix->stage[b]) { cudaFreeHost(ix->stage[b]); ix->stage[b] = nullptr; }
        if (ix->stage_ev[b]) { cudaEventDestroy(ix->stage_ev[b]); ix->stage_ev[b] = nullptr; }
    }
    return VSB_OK;
}

int64_t vsb_index_rows(const vsb_index *ix) { return ix ? ix->n : 0; }
int64_t vsb_index_device_bytes(const vsb_index *ix) { return ix ? (int64_t)ix->dev_bytes : 0; }
int vsb_index_query_pitch(const vsb_index *ix) { return ix ? ix->pitch : 0; }
int64_t vsb_index_stat(const vsb_index *ix, const char *name) {
    if (!ix || !name) return -1;
    if (!strcmp(name, "queries")) return ix->st_queries;
    if (!strcmp(name, "survivors")) return ix->st_survivors;
    if (!strcmp(name, "last_survivors")) return ix->st_last_survivors;
    if (!strcmp(name, "fallbacks")) return ix->st_fallbacks;
    if (!strcmp(name, "batches")) return ix->st_batches;
    if (!strcmp(name, "batch_cands")) return ix->st_batch_cands;
    if (!strcmp(name, "batch_kept")) return ix->st_batch_kept;
    if (!strcmp(name, "tc_us")) return ix->st_tc_us;
    if (!strcmp(name, "batch_us")) return ix->st_batch_us;
    if (!strcmp(name, "tc_rows")) return ix->st_tc_rows;
    if (!strcmp(name, "stream_bytes")) return ix->st_stream_bytes;
    if (!strcmp(name, "stream_us")) return ix->st_stream_us;
    if (!strcmp(name, "fetch_bytes")) return (long long)kHeadBytes;
    if (!strcmp(name, "slots")) return kSlots;
    if (!strcmp(name, "filter_blocks")) return (ix->num_sms * kWarps + kFilterWarpsFast - 1) / kFilterWarpsFast;
    return -1;
}
void *vsb_index_stream(vsb_index *ix) { return ix ? (void *)ix->fstream : nullptr; }

void vsb_index_free(vsb_index *ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    if (ix->stream2) cudaStreamSynchronize(ix->stream2);
    if (ix->fstream) cudaStreamSynchronize(ix->fstream);
    if (ix->xstream) cudaStreamSynchronize(ix->xstream);
    exchange_free(ix);
    for (int b = 0; b < 2; ++b) {
        if (ix->stage[b]) cudaFreeHost(ix->stage[b]);
        if (ix->stage_ev[b]) cudaEventDestroy(ix->stage_ev[b]);
    }
    free_slots(ix);
    free_workspaces(ix);
    for (Work &w : ix->work) {
        if (w.scanned) cudaEventDestroy(w.scanned);
        if (w.drained) cudaEventDestroy(w.drained);
    }
    if (ix->d_dist_all) cudaFree(ix->d_dist_all);
    if (ix->d_vec) cudaFree(ix->d_vec);
    if (ix->h_arena) cudaFreeHost(ix->h_arena);
    for (int b = 0; b < 2; ++b) {
        if (ix->d_win[b]) cudaFree(ix->d_win[b]);
        if (ix->win_copied[b]) cudaEventDestroy(ix->win_copied[b]);
        if (ix->win_scanned[b]) cudaEventDestroy(ix->win_scanned[b]);
    }
    if (ix->cstream) cudaStreamDestroy(ix->cstream);
    for (cudaEvent_t e : ix->prof_ev) cudaEventDestroy(e);
    batch_free(ix);
    if (ix->fstream) cudaStreamDestroy(ix->fstream);
    if (ix->xstream) cudaStreamDestroy(ix->xstream);
    if (ix->stream2) cudaStreamDestroy(ix->stream2);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
}

int vsb_scan_topk(vsb_index *ix, int metric, const void *queries, int nq, int k, int64_t *out_rowids, double *out_dist,
                  int *out_counts, int *max_index) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!queries || nq < 0 || k < 0) return fail(VSB_EINVAL, "bad scan arguments");
    if (k == 0) {  // k == 0 yields an empty result (src/sqlite-vector.c:1795-1796)
        for (int b = 0; b < nq; ++b) if (out_counts) out_counts[b] = 0;
        return VSB_OK;
    }
    if (!out_rowids || !out_dist) return fail(VSB_EINVAL, "output buffers are null");
    const size_t qbytes = (size_t)ix->dim * ix->esize;
    if (batch_supported(ix, metric, nq, k)) {   // tensor-core path; every query starts from a fresh cursor (max_index 0)
        const auto t0 = std::chrono::steady_clock::now();
        int rc = batch_scan(ix, metric, queries, nq, k, out_rowids, out_dist, out_counts);
        ix->st_batch_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        if (rc == VSB_OK) return VSB_OK;
        if (rc != VSB_ERANGE) return rc;
        ix->st_fallbacks++;                      // capacity exceeded: per-query path below
    }
    std::vector<uint2> cands;
    int mi = max_index ? *max_index : 0;
    for (int b = 0; b < nq; ++b) {
        if (nq > 1) mi = 0;                      // batches: independent queries, like B separate cursors
        int rc = query_candidates(ix, metric, (const uint8_t *)queries + (size_t)b * qbytes, k, cands);
        if (rc) return rc;
        SlotReplay s(k, mi, out_dist + (size_t)b * k, out_rowids + (size_t)b * k);
        for (const uint2 &c : cands) s.offer_bits(c.x, rowid_of(ix, c.y));
        mi = s.mi;
        const int cnt = s.finish();
        if (out_counts) out_counts[b] = cnt;
    }
    if (max_index && nq == 1) *max_index = mi;
    return VSB_OK;
}

int vsb_scan_all(vsb_index *ix, int metric, const void *query, float *out_dist, int64_t *out_rowids) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!query || !out_dist) return fail(VSB_EINVAL, "bad scan arguments");
    std::vector<float> dist;
    const int rc = query_all_distances(ix, metric, query, dist);
    if (rc) return rc;
    memcpy(out_dist, dist.data(), sizeof(float) * (size_t)ix->n);
    if (out_rowids)
        for (long long i = 0; i < ix->n; ++i) out_rowids[i] = rowid_of(ix, (uint32_t)i);
    return VSB_OK;
}

int vsb_scan_candidates(vsb_index *ix, int metric, const void *queries, int nq, int k, vsb_candidate *out, int cap_per_query,
                        int *out_counts) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!queries || !out || !out_counts || nq < 0 || k <= 0 || cap_per_query <= 0) return fail(VSB_EINVAL, "bad scan arguments");
    const size_t qbytes = (size_t)ix->dim * ix->esize;
    std::vector<uint2> cands;
    for (int b = 0; b < nq; ++b) {
        int rc = query_candidates(ix, metric, (const uint8_t *)queries + (size_t)b * qbytes, k, cands);
        if (rc) return rc;
        if ((int)cands.size() > cap_per_query) {
            // too many to ship: reduce on this shard first (the shard-local replay keeps exactly the rows
            // that survive locally; a superset of what can survive globally is NOT guaranteed by truncation,
            // so instead we report the condition)
            return fail(VSB_ERANGE, "query %d produced %zu candidates (> cap %d)", b, cands.size(), cap_per_query);
        }
        vsb_candidate *o = out + (size_t)b * cap_per_query;
        for (size_t i = 0; i < cands.size(); ++i) {
            memcpy(&o[i].dist, &cands[i].x, 4);
            o[i].rowid = rowid_of(ix, cands[i].y);
            o[i].seq = ix->first_seq + (long long)cands[i].y;
            o[i].reserved = 0;
        }
        out_counts[b] = (int)cands.size();
    }
    return VSB_OK;
}

int vsb_replay_topk(const vsb_candidate *cands, int n, int k, int *max_index, int64_t *out_rowids, double *out_dist) {
    if (k <= 0) return 0;
    if ((!cands && n > 0) || !out_rowids || !out_dist) return fail(VSB_EINVAL, "bad replay arguments");
    SlotReplay s(k, max_index ? *max_index : 0, out_dist, out_rowids);
    for (int i = 0; i < n; ++i) s.offer(cands[i].dist, cands[i].rowid);
    if (max_index) *max_index = s.mi;
    return s.finish();
}

int vsb_debug_read(vsb_index *ix, const char *name, void *out, int64_t bytes) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!name || !out || bytes <= 0) return fail(VSB_EINVAL, "bad debug read arguments");
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamSynchronize(ix->stream));
    CU(cudaStreamSynchronize(ix->stream2));
    CU(cudaStreamSynchronize(ix->fstream));
    const Work &w = ix->work[(ix->ws_next + kWorks - 1) % kWorks];     // the workspace of the most recent query
    const void *src = nullptr;
    size_t have = 0;
    if (!strcmp(name, "cta_time")) { src = w.d_cta_time; have = sizeof(unsigned) * (size_t)ix->num_sms; }
    else if (!strcmp(name, "bounds")) { src = w.d_bounds; have = sizeof(long long) * (size_t)(ix->num_sms + 1); }
    else return fail(VSB_EINVAL, "unknown debug buffer %s", name);
    if (!src) return fail(VSB_EINVAL, "no scan has run yet");
    CU(cudaMemcpy(out, src, std::min<size_t>(have, (size_t)bytes), cudaMemcpyDeviceToHost));
    return (int)std::min<size_t>(have, (size_t)bytes);
}

int vsb_profile_read(vsb_index *ix, double *scan_ms, int *scan_launches, double *filter_ms, int *filter_launches) {
    if (check_index(ix)) return VSB_EINVAL;
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamSynchronize(ix->stream));
    CU(cudaStreamSynchronize(ix->stream2));
    CU(cudaStreamSynchronize(ix->fstream));
    double a = 0, b = 0;
    int na = 0, nb = 0;
    for (size_t i = 0; i < ix->prof_kind.size(); ++i) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, ix->prof_ev[4 * i], ix->prof_ev[4 * i + 1]));
        a += ms; na += ix->prof_nq[i];          // a launch that scans G queries counts as G scans
        if (ix->prof_kind[i] == 2) {
            CU(cudaEventElapsedTime(&ms, ix->prof_ev[4 * i + 2], ix->prof_ev[4 * i + 3]));
            b += ms; nb += ix->prof_nq[i];
        }
    }
    ix->prof_kind.clear();
    ix->prof_nq.clear();
    ix->prof_used = 0;
    if (scan_ms) *scan_ms = a;
    if (scan_launches) *scan_launches = na;
    if (filter_ms) *filter_ms = b;
    if (filter_launches) *filter_launches = nb;
    return VSB_OK;
}

int vsb_scan_submit(vsb_index *ix, int metric, const void *query, int query_on_device, int k, int fetch, int want_slot) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!query || k <= 0 || k > kMaxK) return fail(VSB_EINVAL, "bad scan arguments (k must be 1..%d)", kMaxK);
    if (want_slot >= kSlots) return fail(VSB_EINVAL, "slot %d out of range (have %d)", want_slot, kSlots);
    const int si = want_slot >= 0 ? want_slot : (ix->last_slot + 1) % kSlots;
    const int rc = submit_group(ix, metric, query, 0, 1, query_on_device, k, fetch, si, false);
    return rc ? rc : si;   // slot id (>= 0) for vsb_collect / vsb_result_block
}

int vsb_scan_submit_group(vsb_index *ix, int metric, const void *queries, int64_t query_stride, int nq, int query_on_device, int k,
                          int fetch, int first_slot) {
    return submit_group(ix, metric, queries, query_stride, nq, query_on_device, k, fetch, first_slot, false);
}

int vsb_scan_device_query(vsb_index *ix, int metric, const void *d_query, int k) {
    return vsb_scan_submit(ix, metric, d_query, 1, k, 1, -1);
}

int vsb_result_block(vsb_index *ix, int slot_id, void **d_block, int64_t *bytes) {
    if (check_index(ix)) return VSB_EINVAL;
    if (slot_id < 0 || slot_id >= kSlots) return fail(VSB_EINVAL, "bad slot");
    CU(cudaSetDevice(ix->device));
    int rc = ensure_slots(ix);
    if (rc) return rc;
    if (d_block) *d_block = ix->slot[slot_id].d_res;
    if (bytes) *bytes = (int64_t)kHeadBytes;
    return VSB_OK;
}

int vsb_merge_result_blocks(const void *blocks, int world, int64_t block_stride, const int64_t *first_seq, int k, int64_t *out_rowids,
                            double *out_dist) {
    if (!blocks || world <= 0 || !first_seq || k <= 0 || !out_rowids || !out_dist) return fail(VSB_EINVAL, "bad merge arguments");
    return merge_blocks_strided((const uint8_t *)blocks, world, (size_t)block_stride, first_seq, k, out_rowids, out_dist);
}

int vsb_merge_result_groups(const void *blocks, int world, int64_t rank_stride, int64_t block_stride, int nq, const int64_t *first_seq,
                            int k, int64_t *out_rowids, double *out_dist, int *out_counts) {
    if (!blocks || nq <= 0 || !out_counts) return fail(VSB_EINVAL, "bad merge arguments");
    for (int j = 0; j < nq; ++j) {
        const int cnt = vsb_merge_result_blocks((const uint8_t *)blocks + (size_t)j * (size_t)block_stride, world, rank_stride, first_seq, k,
                                                out_rowids + (size_t)j * k, out_dist + (size_t)j * k);
        if (cnt < 0) return cnt;
        out_counts[j] = cnt;
    }
    return VSB_OK;
}

int vsb_batch_shard_scan(vsb_index *ix, int metric, const void *queries, int nq, int k, void **d_block, int64_t *bytes) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!queries || nq <= 0 || k <= 0 || !d_block || !bytes) return fail(VSB_EINVAL, "bad batch scan arguments");
    if (!batch_supported(ix, metric, nq, k))
        return fail(VSB_ERANGE, "no tensor-core batch path for this shard (type %d, metric %d, %d queries, k %d, %lld rows)", ix->vtype, metric,
                    nq, k, ix->n);
    const auto t0 = std::chrono::steady_clock::now();
    int rc = batch_levels(ix, metric, queries, nq, k, true);
    if (rc) return rc;
    CU(cudaStreamSynchronize(ix->stream));
    rc = batch_check(ix, (BatchWs *)ix->batch);
    if (rc) return rc;
    ix->st_batch_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    BatchWs *w = (BatchWs *)ix->batch;
    *d_block = w->d_acc;
    *bytes = (int64_t)acc_block_bytes(nq, acc_cap_of(k));
    return VSB_OK;
}

int vsb_batch_merge(vsb_index *ix, const void *d_blocks, int world, int64_t block_stride, const int64_t *first_seq, int nq, int k,
                    int64_t *out_seq, double *out_dist, int *out_counts) {
    if (check_index(ix)) return VSB_EINVAL;
    if (!d_blocks || world <= 0 || !first_seq || nq <= 0 || k <= 0 || k > kMaxK || !out_seq || !out_dist)
        return fail(VSB_EINVAL, "bad batch merge arguments");
    if (block_stride < (int64_t)acc_block_bytes(nq, acc_cap_of(k))) return fail(VSB_EINVAL, "block stride smaller than a block");
    const auto t0 = std::chrono::steady_clock::now();
    int rc = batch_merge(ix, d_blocks, world, block_stride, first_seq, nq, k, out_seq, out_dist, out_counts);
    ix->st_batch_us += std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return rc;
}

int vsb_index_lookup_rowids(const vsb_index *ix, const int64_t *seq, int64_t n, int64_t *out) {
    if (!ix || (!seq && n > 0) || (!out && n > 0) || n < 0) return fail(VSB_EINVAL, "bad lookup arguments");
    for (int64_t i = 0; i < n; ++i) {
        const long long local = (long long)seq[i] - ix->first_seq;
        out[i] = (local >= 0 && local < ix->n) ? rowid_of(ix, (uint32_t)local) : 0;
    }
    return VSB_OK;
}

int vsb_collect_last(vsb_index *ix, int k, int64_t *out_rowids, double *out_dist, int *out_count) {
    if (check_index(ix)) return VSB_EINVAL;
    if (ix->last_slot < 0) return fail(VSB_EINVAL, "no device scan was launched");
    return vsb_collect(ix, ix->last_slot, k, out_rowids, out_dist, out_count);
}

int vsb_collect(vsb_index *ix, int slot_id, int k, int64_t *out_rowids, double *out_dist, int *out_count) {
    if (check_index(ix)) return VSB_EINVAL;
    if (slot_id < 0 || slot_id >= kSlots || !ix->slots_ready) return fail(VSB_EINVAL, "bad slot");
    CU(cudaSetDevice(ix->device));
    CU(cudaEventSynchronize(ix->slot[slot_id].done));   // only this query's result; a later launch may still be running
    std::vector<uint2> cands;
    bool overflow = false;
    int n = gather_survivors(ix, &ix->slot[slot_id], cands, &overflow);
    if (n < 0) return n;
    if (overflow) return fail(VSB_ERANGE, "candidate log overflowed; use vsb_scan_topk (host query) for this input");
    SlotReplay s(k, 0, out_dist, out_rowids);
    for (const uint2 &c : cands) s.offer_bits(c.x, rowid_of(ix, c.y));
    const int cnt = s.finish();
    if (out_count) *out_count = cnt;
    return VSB_OK;
}

}  // extern "C"
