// api.cu -- host side of libfuzzb200.so: the C-ABI declared in include/fuzzb200.h.
//
// No CPU search path exists in this file: every search launches the sm_100a kernels of kernels.cuh
// and fails with FZB_E_CUDA when no device is usable.  The only host-side algorithm is the
// O(N log N) consolidation of the (small) match list, which the reference also performs after its
// search (common.py:185-189).
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <dlfcn.h>
#include <sched.h>
#include <unistd.h>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <new>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "ham_kernels.cuh"
#include "lp_kernels.cuh"
#include "post_kernels.cuh"
#include "p2p_kernels.cuh"
#include "batch_kernels.cuh"
#include "sym_kernels.cuh"
#include "seg_kernels.cuh"
#include <unordered_map>
#include "debug_kernels.cuh"

using namespace fzb;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(FZB_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));      \
    } while (0)

extern "C" int fzb_version(void) { return FZB_VERSION; }

extern "C" int fzb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" const char *fzb_last_error(void) { return g_err.c_str(); }

// ------------------------------------------------------------------------------------------------
// NCCL, resolved at run time (the process usually has torch's libnccl.so.2 loaded already)
// ------------------------------------------------------------------------------------------------
struct NcclId {
    char b[FZB_NCCL_ID_BYTES];
};
struct NcclApi {
    int (*GetUniqueId)(NcclId *id) = nullptr;
    int (*CommInitRank)(void **comm, int nranks, NcclId id, int rank) = nullptr;  // ncclUniqueId is passed by value
    int (*AllGather)(const void *send, void *recv, size_t count, int dtype, void *comm, cudaStream_t s) = nullptr;
    int (*CommDestroy)(void *comm) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool ok = false;
};
static NcclApi g_nccl;
static std::string g_nccl_path;  // optional explicit library path (fzb_nccl_set_library)

extern "C" void fzb_nccl_set_library(const char *path) { g_nccl_path = path ? path : ""; }

static int nccl_load() {
    static std::once_flag once;
    std::call_once(once, [] {
        void *lib = nullptr;
        if (!g_nccl_path.empty()) lib = dlopen(g_nccl_path.c_str(), RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return;
        *(void **)&g_nccl.GetUniqueId = dlsym(lib, "ncclGetUniqueId");
        *(void **)&g_nccl.CommInitRank = dlsym(lib, "ncclCommInitRank");
        *(void **)&g_nccl.AllGather = dlsym(lib, "ncclAllGather");
        *(void **)&g_nccl.CommDestroy = dlsym(lib, "ncclCommDestroy");
        *(void **)&g_nccl.GetErrorString = dlsym(lib, "ncclGetErrorString");
        g_nccl.ok = g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllGather && g_nccl.CommDestroy;
    });
    return g_nccl.ok ? FZB_OK : fail(FZB_E_CUDA, "libnccl.so.2 not available: %s", dlerror() ? dlerror() : "missing symbols");
}

static void nccl_comm_destroy(void *comm) {
    if (g_nccl.ok && comm) g_nccl.CommDestroy(comm);
}

#define NCCLCK(call)                                                                                      \
    do {                                                                                                  \
        int r_ = (call);                                                                                  \
        if (r_ != 0)                                                                                      \
            return fail(FZB_E_CUDA, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
    } while (0)

// ------------------------------------------------------------------------------------------------
// handles
// ------------------------------------------------------------------------------------------------
struct fzb_haystack {
    std::recursive_mutex mu;  // one search / upload at a time per handle (HandleLock); recursive: has_near_match and
                              // the windowed exact search call the search entry points on their own handle
    int device = 0;
    uint8_t *d = nullptr;  // H[0] == global position buf_lo
    bool owned = true;
    uint64_t buf_len = 0, buf_lo = 0, global_len = 0, own_lo = 0, own_hi = 0;
    uint64_t padded_len = 0;
    uint64_t capacity = 0;  // bytes allocated at d (owned buffers)
    cudaEvent_t ev_stop = nullptr;
    cudaStream_t stream = nullptr;
    uint32_t *d_bitmap = nullptr;
    uint64_t bitmap_words = 0;
    RawRec *d_out = nullptr;
    uint32_t out_cap = 0;
    uint32_t *d_counters = nullptr;
    // k_post writes these straight into MAPPED pinned host memory (no copy operations per search)
    uint32_t *h_counters = nullptr;  // CNT_COUNT counters
    int64_t *h_fin = nullptr;        // final rows (kPostMax x kFinCols)
    int64_t *d_fin = nullptr;        // device copy of the final rows (input of the multi-GPU reduction)
    uint64_t *d_sorted = nullptr;    // k_post scratch: the sorted canonical keys
    fzb_result *pending = nullptr;   // the last result, while its raw records still sit in d_out only
    bool ev1_recorded = false;
    bool filter_attrs_set = false;
    double coll_prob = -1.0;  // sum_c p_c^2 of the byte distribution (sampled lazily; < 0 = unknown)
    // multi-GPU reduction (FZB_F_GLOBAL): peer-memory world (p2p_kernels.cuh) + NCCL for bootstrap / staged fallback
    bool p2p = false;               // every rank of the world can store into every other rank's receive area
    bool local_world = false;       // the world lives in this process (fzb_comm_init_local): no NCCL
    uint8_t *d_p2p = nullptr;       // my receive area: [2 parities][world] slots + flags
    uint8_t *peer_base[kMaxWorld] = {};
    bool peer_opened[kMaxWorld] = {};
    uint32_t p2p_cap = 4096;        // group rows per slot
    uint64_t slot_bytes = 0, flags_off = 0;
    uint32_t epoch = 0;             // number of FZB_F_GLOBAL searches issued on this handle
    bool counters_clean = false;    // the device counters are all zero (the last search's final kernel left them so)
    uint32_t seq = 0;               // number of search attempts enqueued: the last kernel of each writes it to mapped
                                    // memory as its final store and the host polls for it (wait_done)
    MergeScratch *d_ms = nullptr;
    unsigned long long *d_mscore = nullptr;
    uint32_t *d_mpos = nullptr;
    int64_t *h_grows = nullptr;     // mapped: global final rows of the last global search (16 bytes each)
    uint32_t *h_ghdr = nullptr;     // mapped: status, count, epoch
    void *comm = nullptr;  // ncclComm_t
    int rank = 0, world = 1;
    uint32_t gather_cap = 4096;     // rows per rank in one all-gather slot
    int64_t *d_send = nullptr, *d_recv = nullptr;
    int64_t *h_send = nullptr, *h_recv = nullptr;  // pinned
    uint32_t gather_alloc = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int sm_count = 148;
    uint64_t *d_hits = nullptr;     // dense route: list of confirmed n-gram hits
    uint32_t hits_cap = 0;
    uint32_t *d_glist = nullptr;    // compacted list of marked granules
    uint32_t glist_cap = 0;
    uint32_t *d_scratch = nullptr;  // candidate lists of the LP / generic kernels
    uint64_t scratch_words = 0;
    unsigned long long *d_lplist = nullptr;  // streaming LP route: starts that survived the scan
    uint32_t lplist_cap = 0;
    // single-pass multi-pattern batches (batch_kernels.cuh), allocated on first use
    uint32_t *d_mbits = nullptr;
    uint2 *d_gtab = nullptr;
    uint32_t *d_postings = nullptr, *d_pinfo = nullptr;
    BatchPat *d_bpats = nullptr;
    unsigned long long *d_mset = nullptr;
    WorkItem *d_mwork = nullptr;
    uint32_t mset_slots = 0, mwork_cap = 0;
    unsigned long long *d_mhits = nullptr;  // dense batch pass: (pattern, n-gram, position) hits
    uint32_t mhits_cap = 0;
    ulonglong2 *d_lmlut = nullptr;          // LP batch pass: per-byte pattern-set vectors
    unsigned long long *d_lmlist = nullptr; // ... its survivor list (after the sort: grouped by pattern)
    unsigned long long *d_lmkept = nullptr; // ... the survivors of the exact per-pattern window test
    uint32_t *d_lmhist = nullptr;
    uint32_t lmlist_cap = 0;
    // segmented searches (seg_kernels.cuh), allocated on first use
    uint64_t *d_seg_offsets = nullptr;     // the caller's offsets[count + 1]
    uint32_t *d_seg_cnt = nullptr;         // per segment: raw record counts, then final counts ([2][count])
    uint32_t *d_seg_off = nullptr, *d_seg_cur = nullptr;
    uint32_t *h_seg_cnt = nullptr;         // pinned: host copy of d_seg_cnt
    uint64_t seg_count_cap = 0;
    uint64_t *d_seg_keys = nullptr;        // canonical keys grouped by segment
    uint64_t *h_seg_raw = nullptr, *h_seg_fin = nullptr;  // mapped: sorted raw keys / final keys, segment-major
    uint64_t seg_rec_cap = 0;
    uint32_t *h_seg_hdr = nullptr;         // mapped: record count, overflow flag of the last attempt
    fzb_haystack *seg_ws = nullptr;        // long segments are copied here and searched as whole sequences
};

struct fzb_result {
    std::vector<RawRec> raw;      // filled lazily from the owner's mapped staging buffer (fetch_raw)
    uint32_t raw_n = 0;           // number of raw records
    fzb_haystack *owner = nullptr;  // non-null while raw records / global rows still sit in the owner's mapped buffers
    bool raw_in_stage = false;
    void fetch_raw();
    std::vector<RawRec> fin;
    std::vector<int64_t> hulls;  // (hull_start, hull_end) of the group behind each final match
    bool unconsolidated = false;  // exact / Hamming routes: FINAL is the whole raw list in (start, end, dist) order
    bool have_fin = false;        // fin / hulls are filled
    bool device_post = false;  // the final list came from the device (k_post)
    bool raw_ordered = false;  // raw is already in its reference order
    bool has_global = false;   // FZB_F_GLOBAL: gfin is the global consolidated list of all shards
    bool global_on_device = false;  // ... produced by k_merge; its rows sit in owner->h_grows until fetched
    bool fused_issued = false;      // a k_push / k_merge pair ran for this search
    uint32_t fused_status = 0;      // MS_* of that merge
    uint32_t gcount = 0;
    std::vector<RawRec> gfin;
    int raw_order = 0;         // 0 generation (ngram, idx) / 1 canonical / 2 generic n-grams (5 fields)
    bool segmented = false;    // fzb_search_segments: raw / fin are segment-major, seg_n holds the list lengths
    std::vector<uint64_t> seg_n[2];  // [FZB_RAW] / [FZB_FINAL]: per-segment list lengths
    void order_raw();
    fzb_stats stats{};
};

static uint64_t round_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

// Every entry point that touches a handle's device state (buffer, counters, output area, stream order) holds the
// handle's mutex for the whole call: two threads sharing one resident sequence take turns, like callers of the
// reference under the GIL.  (Results are separate objects; their lazy raw fetch is guarded by g_pending_mutex.)
struct HandleLock {
    std::recursive_mutex *m;
    explicit HandleLock(fzb_haystack *h) : m(h ? &h->mu : nullptr) {
        if (m) m->lock();
    }
    ~HandleLock() {
        if (m) m->unlock();
    }
    HandleLock(const HandleLock &) = delete;
    HandleLock &operator=(const HandleLock &) = delete;
};

// The raw records of the LAST search of a handle stay in its DEVICE output buffer (and the global rows of a
// multi-GPU search in its mapped host buffer) until somebody asks for them (fzb_result_copy), the next search
// on the handle is about to overwrite the buffers, or the handle / the result dies: find_near_matches() only
// needs the consolidated list, and shipping 200 KB of raw records over PCIe behind every search is 1-2 % of a
// 4 GiB scan.  One process-wide mutex guards the result <-> handle link.
static std::mutex g_pending_mutex;

void fzb_result::fetch_raw() {
    std::lock_guard<std::mutex> lock(g_pending_mutex);
    if (!owner) return;
    if (raw_in_stage) {  // the records are still in the owner's device buffer: one D2H copy, now
        raw.resize(raw_n);
        if (raw_n) {
            cudaSetDevice(owner->device);
            if (cudaMemcpyAsync(raw.data(), owner->d_out, (size_t)raw_n * sizeof(RawRec), cudaMemcpyDeviceToHost,
                                owner->stream) != cudaSuccess ||
                cudaStreamSynchronize(owner->stream) != cudaSuccess) {
                cudaGetLastError();
                raw.clear();  // (the handle's context is gone: nothing left to fetch)
                raw_n = 0;
            }
        }
        raw_in_stage = false;
    }
    if (global_on_device) {  // rows: start, (end - start) << 32 | dist
        gfin.resize(gcount);
        for (uint32_t i = 0; i < gcount; i++) {
            const int64_t s0 = owner->h_grows[2 * (size_t)i], v = owner->h_grows[2 * (size_t)i + 1];
            gfin[i].start = s0;
            gfin[i].end = s0 + (v >> 32);
            gfin[i].dist = (int32_t)(v & 0xFFFFFFFF);
            gfin[i].idx = -1;
            gfin[i].ngram = -1;
        }
        global_on_device = false;
    }
    owner->pending = nullptr;
    owner = nullptr;
}

static void detach_pending(fzb_haystack *h) {  // before h->d_out / h->h_grows are overwritten or freed
    fzb_result *r;
    {
        std::lock_guard<std::mutex> lock(g_pending_mutex);
        r = h->pending;
    }
    if (r) r->fetch_raw();
}

static int haystack_common_init(fzb_haystack *h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (auto &e : h->ev) CK(cudaEventCreate(&e));
    CK(cudaEventCreate(&h->ev_stop));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    h->sm_count = prop.multiProcessorCount;
    uint64_t granules = (h->padded_len >> kGranuleShift) + 2;
    h->bitmap_words = round_up((granules + 31) / 32, 32);
    CK(cudaMalloc(&h->d_bitmap, h->bitmap_words * sizeof(uint32_t)));
    CK(cudaMalloc(&h->d_counters, CNT_COUNT * sizeof(uint32_t)));
    const unsigned hflags = cudaHostAllocMapped | cudaHostAllocPortable;
    CK(cudaHostAlloc(&h->h_counters, CNT_COUNT * sizeof(uint32_t), hflags));
    memset(h->h_counters, 0, CNT_COUNT * sizeof(uint32_t));  // the sequence word the host polls must not hold a stale value
    CK(cudaHostAlloc(&h->h_fin, (size_t)kPostMax * kFinCols * sizeof(int64_t), hflags));
    CK(cudaMalloc(&h->d_fin, (size_t)kPostMax * kFinCols * sizeof(int64_t)));
    CK(cudaMalloc(&h->d_sorted, (size_t)kPostMax * sizeof(uint64_t)));
    CK(cudaFuncSetAttribute(k_post, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPostSmem));
    CK(cudaMemset(h->d_bitmap, 0, h->bitmap_words * sizeof(uint32_t)));  // stays all-zero between searches
    h->glist_cap = (uint32_t)std::min<uint64_t>(granules, 1u << 20);
    CK(cudaMalloc(&h->d_glist, (size_t)std::max<uint32_t>(h->glist_cap, 1) * sizeof(uint32_t)));
    h->out_cap = 1u << 16;
    CK(cudaMalloc(&h->d_out, (size_t)h->out_cap * (sizeof(RawRec) + sizeof(uint64_t))));  // records + their keys
    return FZB_OK;
}

static int check_shard(uint64_t buf_len, uint64_t buf_lo, uint64_t global_len, uint64_t own_lo,
                       uint64_t own_hi) {
    if (buf_lo + buf_len > global_len || own_lo > own_hi || own_hi > global_len ||
        (own_lo < own_hi && (own_lo < buf_lo || own_hi > buf_lo + buf_len)))
        return fail(FZB_E_INVALID, "inconsistent shard geometry");
    if (buf_lo % 16 != 0) return fail(FZB_E_INVALID, "buf_lo must be a multiple of 16");
    return FZB_OK;
}

static int alloc_buffer(fzb_haystack *h) {
    h->padded_len = round_up(h->buf_len, 128) + 128;
    CK(cudaSetDevice(h->device));
    CK(cudaMalloc(&h->d, h->padded_len));
    h->capacity = h->padded_len;
    CK(cudaMemset(h->d + h->buf_len, 0, h->padded_len - h->buf_len));
    return FZB_OK;
}

static void p2p_free(fzb_haystack *h);
static void seg_free(fzb_haystack *h);
static int upload_bytes(fzb_haystack *h, uint64_t dst_off, const uint8_t *host, uint64_t n);

extern "C" void fzb_haystack_destroy(fzb_haystack *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    detach_pending(h);
    if (h->owned && h->d) cudaFree(h->d);
    if (h->d_bitmap) cudaFree(h->d_bitmap);
    if (h->d_out) cudaFree(h->d_out);
    if (h->d_counters) cudaFree(h->d_counters);
    if (h->d_scratch) cudaFree(h->d_scratch);
    if (h->d_lplist) cudaFree(h->d_lplist);
    if (h->d_mbits) cudaFree(h->d_mbits);
    if (h->d_gtab) cudaFree(h->d_gtab);
    if (h->d_postings) cudaFree(h->d_postings);
    if (h->d_pinfo) cudaFree(h->d_pinfo);
    if (h->d_bpats) cudaFree(h->d_bpats);
    if (h->d_mset) cudaFree(h->d_mset);
    if (h->d_mwork) cudaFree(h->d_mwork);
    if (h->d_mhits) cudaFree(h->d_mhits);
    if (h->d_lmlut) cudaFree(h->d_lmlut);
    if (h->d_lmlist) cudaFree(h->d_lmlist);
    if (h->d_lmkept) cudaFree(h->d_lmkept);
    if (h->d_lmhist) cudaFree(h->d_lmhist);
    if (h->d_glist) cudaFree(h->d_glist);
    if (h->d_hits) cudaFree(h->d_hits);
    if (h->d_send) cudaFree(h->d_send);
    if (h->d_recv) cudaFree(h->d_recv);
    if (h->h_send) cudaFreeHost(h->h_send);
    if (h->h_recv) cudaFreeHost(h->h_recv);
    if (h->comm) nccl_comm_destroy(h->comm);
    p2p_free(h);
    seg_free(h);
    if (h->h_counters) cudaFreeHost(h->h_counters);
    if (h->h_fin) cudaFreeHost(h->h_fin);
    if (h->d_fin) cudaFree(h->d_fin);
    if (h->d_sorted) cudaFree(h->d_sorted);
    for (auto &e : h->ev)
        if (e) cudaEventDestroy(e);
    if (h->ev_stop) cudaEventDestroy(h->ev_stop);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" int fzb_haystack_create_shard(const uint8_t *host, uint64_t buf_len, uint64_t buf_lo,
                                         uint64_t global_len, uint64_t own_lo, uint64_t own_hi,
                                         int device, fzb_haystack **out) {
    if (!out) return fail(FZB_E_INVALID, "out is NULL");
    *out = nullptr;
    if (!host && buf_len) return fail(FZB_E_INVALID, "host buffer is NULL");
    int rc = check_shard(buf_len, buf_lo, global_len, own_lo, own_hi);
    if (rc) return rc;
    if (fzb_device_count() <= device || device < 0)
        return fail(FZB_E_CUDA, "CUDA device %d not available (%d devices)", device, fzb_device_count());
    fzb_haystack *h = new (std::nothrow) fzb_haystack();
    if (!h) return fail(FZB_E_CUDA, "out of host memory");
    h->device = device;
    h->buf_len = buf_len;
    h->buf_lo = buf_lo;
    h->global_len = global_len;
    h->own_lo = own_lo;
    h->own_hi = own_hi;
    rc = alloc_buffer(h);
    if (rc == FZB_OK) rc = haystack_common_init(h);
    if (rc == FZB_OK && buf_len) rc = upload_bytes(h, 0, host, buf_len);
    if (rc) {
        fzb_haystack_destroy(h);
        return rc;
    }
    *out = h;
    return FZB_OK;
}

extern "C" int fzb_haystack_create(const uint8_t *host, uint64_t n, int device, fzb_haystack **out) {
    return fzb_haystack_create_shard(host, n, 0, n, 0, n, device, out);
}

extern "C" int fzb_haystack_adopt_device(const void *dev_ptr, uint64_t buf_len, uint64_t buf_lo,
                                         uint64_t global_len, uint64_t own_lo, uint64_t own_hi,
                                         int device, fzb_haystack **out) {
    if (!out) return fail(FZB_E_INVALID, "out is NULL");
    *out = nullptr;
    if (!dev_ptr || ((uintptr_t)dev_ptr & 15)) return fail(FZB_E_INVALID, "dev_ptr must be 16-byte aligned");
    int rc = check_shard(buf_len, buf_lo, global_len, own_lo, own_hi);
    if (rc) return rc;
    if (fzb_device_count() <= device || device < 0) return fail(FZB_E_CUDA, "CUDA device %d not available", device);
    fzb_haystack *h = new (std::nothrow) fzb_haystack();
    if (!h) return fail(FZB_E_CUDA, "out of host memory");
    h->device = device;
    h->owned = false;
    h->d = (uint8_t *)dev_ptr;
    h->buf_len = buf_len;
    h->buf_lo = buf_lo;
    h->global_len = global_len;
    h->own_lo = own_lo;
    h->own_hi = own_hi;
    h->padded_len = round_up(buf_len, 128) + 128;
    rc = haystack_common_init(h);
    if (rc) {
        fzb_haystack_destroy(h);
        return rc;
    }
    *out = h;
    return FZB_OK;
}

extern "C" int fzb_haystack_alloc(uint64_t buf_len, uint64_t buf_lo, uint64_t global_len, uint64_t own_lo,
                                  uint64_t own_hi, int device, fzb_haystack **out, void **dev_ptr) {
    if (!out) return fail(FZB_E_INVALID, "out is NULL");
    *out = nullptr;
    int rc = check_shard(buf_len, buf_lo, global_len, own_lo, own_hi);
    if (rc) return rc;
    if (fzb_device_count() <= device || device < 0) return fail(FZB_E_CUDA, "CUDA device %d not available", device);
    fzb_haystack *h = new (std::nothrow) fzb_haystack();
    if (!h) return fail(FZB_E_CUDA, "out of host memory");
    h->device = device;
    h->buf_len = buf_len;
    h->buf_lo = buf_lo;
    h->global_len = global_len;
    h->own_lo = own_lo;
    h->own_hi = own_hi;
    rc = alloc_buffer(h);
    if (rc == FZB_OK) rc = haystack_common_init(h);
    if (rc) {
        fzb_haystack_destroy(h);
        return rc;
    }
    if (dev_ptr) *dev_ptr = h->d;
    *out = h;
    return FZB_OK;
}

extern "C" void fzb_synth_host(uint8_t *dst, uint64_t global_offset, uint64_t n, const uint8_t *alphabet,
                               uint32_t alphabet_len, uint64_t seed) {
    uint64_t i = 0;
    while (i < n) {
        uint64_t g = global_offset + i;
        uint32_t w = synth_word(seed, g / 4, alphabet, alphabet_len);
        for (uint64_t b = g % 4; b < 4 && i < n; b++, i++) dst[i] = (uint8_t)(w >> (8 * b));
    }
}

extern "C" int fzb_haystack_fill_synthetic(fzb_haystack *h, const uint8_t *alphabet, uint32_t alphabet_len,
                                           uint64_t seed) {
    HandleLock handle_lock(h);
    if (!h || !alphabet || alphabet_len == 0 || alphabet_len > 256) return fail(FZB_E_INVALID, "bad arguments");
    if (!h->owned) return fail(FZB_E_INVALID, "cannot fill an adopted buffer");
    CK(cudaSetDevice(h->device));
    uint8_t *d_alpha = nullptr;
    CK(cudaMalloc(&d_alpha, 256));
    CK(cudaMemcpyAsync(d_alpha, alphabet, alphabet_len, cudaMemcpyHostToDevice, h->stream));
    int64_t nwords = (int64_t)(round_up(h->buf_len, 4) / 4);
    k_fill_synth<<<h->sm_count * 8, 256, 0, h->stream>>>(h->d, (int64_t)h->buf_lo, nwords, seed, d_alpha,
                                                        alphabet_len);
    CK(cudaGetLastError());
    // bytes past buf_len must stay zero (the last word may have spilled over)
    if (h->buf_len % 4)
        CK(cudaMemsetAsync(h->d + h->buf_len, 0, 4 - h->buf_len % 4, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaFree(d_alpha));
    h->coll_prob = -1.0;
    return FZB_OK;
}

extern "C" int fzb_haystack_write(fzb_haystack *h, uint64_t global_offset, const uint8_t *src, uint64_t n) {
    HandleLock handle_lock(h);
    if (!h || (!src && n)) return fail(FZB_E_INVALID, "bad arguments");
    if (global_offset < h->buf_lo || global_offset + n > h->buf_lo + h->buf_len)
        return fail(FZB_E_INVALID, "write outside the buffer");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(h->d + (global_offset - h->buf_lo), src, n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FZB_OK;
}

extern "C" int fzb_haystack_read(fzb_haystack *h, uint64_t global_offset, uint8_t *dst, uint64_t n) {
    HandleLock handle_lock(h);
    if (!h || (!dst && n)) return fail(FZB_E_INVALID, "bad arguments");
    if (global_offset < h->buf_lo || global_offset + n > h->buf_lo + h->buf_len)
        return fail(FZB_E_INVALID, "read outside the buffer");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dst, h->d + (global_offset - h->buf_lo), n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FZB_OK;
}

extern "C" uint64_t fzb_haystack_len(const fzb_haystack *h) {
    // under the handle's lock like every other call: a windowed exact search / has_near_match on another thread
    // swaps the geometry (global_len included) for the duration of its view
    HandleLock handle_lock(const_cast<fzb_haystack *>(h));
    return h ? h->global_len : 0;
}

// ------------------------------------------------------------------------------------------------
// Upload of PAGEABLE host memory (what a Python bytes object is).  cudaMemcpy from pageable memory stages through
// the driver's own bounce buffer at 7-10 GB/s on these hosts; page-locking the caller's buffer in place
// (cudaHostRegister) costs more than the copy.  Instead: a ring of three 64 MiB pinned buffers; a small pool of
// host threads copies slice i+1 of the caller's buffer into one of them while the DMA engine moves slice i
// to the device -- the pipeline runs at min(host memcpy bandwidth of the pool, PCIe).
// ------------------------------------------------------------------------------------------------
class CopyPool {
  public:
    static CopyPool &get() {
        static CopyPool *pool = new CopyPool();  // leaked on purpose: no joins at process exit
        return *pool;
    }
    void copy(uint8_t *dst, const uint8_t *src, size_t n) {  // parallel memcpy; returns when all of it is done
        if (n < (8u << 20) || threads_.empty()) {
            memcpy(dst, src, n);
            return;
        }
        {
            std::lock_guard<std::mutex> lock(m_);
            dst_ = dst;
            src_ = src;
            n_ = n;
            next_.store(0);
            pending_ = (int)threads_.size();
            gen_++;
        }
        cv_.notify_all();
        work();  // the caller copies too
        std::unique_lock<std::mutex> lock(m_);
        done_.wait(lock, [&] { return pending_ == 0; });
    }

  private:
    static constexpr size_t kSlice = 2u << 20;
    CopyPool() {
        unsigned want = 16;  // enough to stay ahead of PCIe even when the source pages sit on a remote NUMA node
        if (const char *e = getenv("FZB_UPLOAD_THREADS")) want = (unsigned)std::max(0, atoi(e));
        unsigned hw = std::thread::hardware_concurrency();
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof set, &set) == 0) hw = (unsigned)CPU_COUNT(&set);
        want = std::min(want, hw > 1 ? hw - 1 : 0u);
        for (unsigned i = 0; i < want; i++) {
            threads_.emplace_back([this] { loop(); });
            threads_.back().detach();
        }
    }
    void work() {
        for (;;) {
            const size_t off = next_.fetch_add(kSlice);
            if (off >= n_) return;
            memcpy(dst_ + off, src_ + off, std::min(kSlice, n_ - off));
        }
    }
    void loop() {
        uint64_t seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lock(m_);
                cv_.wait(lock, [&] { return gen_ != seen; });
                seen = gen_;
            }
            work();
            std::lock_guard<std::mutex> lock(m_);
            if (--pending_ == 0) done_.notify_all();
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    uint8_t *dst_ = nullptr;
    const uint8_t *src_ = nullptr;
    size_t n_ = 0;
    std::atomic<size_t> next_{0};
    int pending_ = 0;
    uint64_t gen_ = 0;
};

constexpr int kStageBufs = 3;
constexpr size_t kStageBytes = 64u << 20;
static std::mutex g_stage_mutex;  // one staged upload at a time per process (the ring is shared by all handles)
static uint8_t *g_stage[kStageBufs];

static bool is_pinned_host(const void *p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// host -> h->d + dst_off, n bytes, on h->stream; returns when the caller may reuse `host`
static int upload_bytes(fzb_haystack *h, uint64_t dst_off, const uint8_t *host, uint64_t n) {
    if (n == 0) return FZB_OK;
    if (n < (16u << 20) || is_pinned_host(host)) {
        CK(cudaMemcpyAsync(h->d + dst_off, host, n, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return FZB_OK;
    }
    std::lock_guard<std::mutex> lock(g_stage_mutex);
    for (auto &b : g_stage)
        if (!b) CK(cudaHostAlloc(&b, kStageBytes, cudaHostAllocPortable));
    cudaEvent_t ev[kStageBufs];
    for (auto &e : ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    int rc = FZB_OK;
    uint64_t off = 0;
    for (int i = 0; off < n && rc == FZB_OK; i++, off += kStageBytes) {
        const int b = i % kStageBufs;
        const size_t len = (size_t)std::min<uint64_t>(kStageBytes, n - off);
        cudaError_t e = i >= kStageBufs ? cudaEventSynchronize(ev[b]) : cudaSuccess;  // the DMA out of this buffer is done
        if (e == cudaSuccess) {
            CopyPool::get().copy(g_stage[b], host + off, len);
            e = cudaMemcpyAsync(h->d + dst_off + off, g_stage[b], len, cudaMemcpyHostToDevice, h->stream);
        }
        if (e == cudaSuccess) e = cudaEventRecord(ev[b], h->stream);
        if (e != cudaSuccess) rc = fail(FZB_E_CUDA, "staged upload failed: %s", cudaGetErrorString(e));
    }
    cudaError_t e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess && rc == FZB_OK) rc = fail(FZB_E_CUDA, "staged upload failed: %s", cudaGetErrorString(e));
    for (auto &x : ev) cudaEventDestroy(x);
    return rc;
}

extern "C" int fzb_haystack_upload(fzb_haystack *h, const uint8_t *host, uint64_t n) {
    HandleLock handle_lock(h);
    if (!h || (!host && n)) return fail(FZB_E_INVALID, "bad arguments");
    if (!h->owned) return fail(FZB_E_INVALID, "upload needs an owned handle");
    if (round_up(n, 128) + 128 > h->capacity) return fail(FZB_E_INVALID, "upload larger than the handle's capacity");
    CK(cudaSetDevice(h->device));
    const bool shard = h->buf_lo != 0 || h->global_len != h->buf_len || h->own_lo != 0 || h->own_hi != h->buf_len;
    if (shard) {  // a shard keeps its geometry: the new bytes replace the same window of the global sequence
        if (n != h->buf_len) return fail(FZB_E_INVALID, "a shard upload must supply exactly buf_len bytes");
    } else {
        h->buf_len = h->global_len = h->own_hi = n;
        h->own_lo = 0;
    }
    h->padded_len = round_up(n, 128) + 128;
    h->coll_prob = -1.0;
    CK(cudaMemsetAsync(h->d + n, 0, h->padded_len - n, h->stream));
    return upload_bytes(h, 0, host, n);  // the caller may reuse `host` as soon as we return
}

// Wide-symbol sequences (sym_kernels.cuh): the code units travel to a device scratch chunk by chunk and
// k_reduce_symbols writes one byte per symbol into the handle's buffer.
extern "C" int fzb_haystack_upload_symbols(fzb_haystack *h, const void *host, uint64_t n, uint32_t width,
                                           const uint32_t *alphabet, uint32_t n_alpha) {
    HandleLock handle_lock(h);
    if (!h || (!host && n) || (!alphabet && n_alpha)) return fail(FZB_E_INVALID, "bad arguments");
    if (width != 2 && width != 4) return fail(FZB_E_INVALID, "symbol width must be 2 or 4 bytes");
    if (n_alpha > (uint32_t)kMaxPattern) return fail(FZB_E_UNSUPPORTED, "more than %d distinct pattern symbols", kMaxPattern);
    for (uint32_t i = 1; i < n_alpha; i++)
        if (alphabet[i - 1] >= alphabet[i]) return fail(FZB_E_INVALID, "the alphabet must be strictly ascending");
    if (!h->owned) return fail(FZB_E_INVALID, "upload needs an owned handle");
    if (round_up(n, 128) + 128 > h->capacity) return fail(FZB_E_INVALID, "upload larger than the handle's capacity");
    if (h->buf_lo != 0 || h->global_len != h->buf_len || h->own_lo != 0 || h->own_hi != h->buf_len)
        return fail(FZB_E_INVALID, "symbol uploads replace a whole (unsharded) sequence");
    CK(cudaSetDevice(h->device));
    h->buf_len = h->global_len = h->own_hi = n;
    h->padded_len = round_up(n, 128) + 128;
    h->coll_prob = -1.0;
    CK(cudaMemsetAsync(h->d + n, 0, h->padded_len - n, h->stream));
    if (n == 0) {
        CK(cudaStreamSynchronize(h->stream));
        return FZB_OK;
    }
    constexpr uint64_t kChunk = 16u << 20;  // symbols per chunk (a multiple of 4: the kernel stores 32-bit words)
    const uint64_t chunk = std::min<uint64_t>(kChunk, round_up(n, 4));
    uint8_t *d_tmp = nullptr;   // every operation below is on h->stream: a chunk's copy is ordered behind the
    uint32_t *d_alpha = nullptr;  // reduction of the previous chunk, so one scratch buffer is enough
    int rc = FZB_OK;
    auto cleanup = [&]() {
        if (d_tmp) cudaFree(d_tmp);
        if (d_alpha) cudaFree(d_alpha);
    };
#define SYMCK(call)                                                                                \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail(FZB_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));                 \
            cudaStreamSynchronize(h->stream);                                                      \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    SYMCK(cudaMalloc(&d_alpha, 256 * sizeof(uint32_t)));
    if (n_alpha) SYMCK(cudaMemcpyAsync(d_alpha, alphabet, n_alpha * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    SYMCK(cudaMalloc(&d_tmp, chunk * width));
    const uint8_t *src = static_cast<const uint8_t *>(host);
    for (uint64_t off = 0; off < n; off += chunk) {
        const uint64_t cnt = std::min<uint64_t>(chunk, n - off);
        SYMCK(cudaMemcpyAsync(d_tmp, src + off * width, cnt * width, cudaMemcpyHostToDevice, h->stream));
        const int grid = (int)std::min<uint64_t>((uint64_t)h->sm_count * 8, (cnt / 4 + kSymThreads - 1) / kSymThreads + 1);
        if (width == 4)
            k_reduce_symbols<uint32_t><<<grid, kSymThreads, 0, h->stream>>>(reinterpret_cast<const uint32_t *>(d_tmp), cnt,
                                                                            d_alpha, n_alpha, h->d + off);
        else
            k_reduce_symbols<uint16_t><<<grid, kSymThreads, 0, h->stream>>>(reinterpret_cast<const uint16_t *>(d_tmp), cnt,
                                                                            d_alpha, n_alpha, h->d + off);
        SYMCK(cudaGetLastError());
    }
    SYMCK(cudaStreamSynchronize(h->stream));
#undef SYMCK
    cleanup();
    return FZB_OK;
}

extern "C" void *fzb_host_alloc(uint64_t n) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, n ? n : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        fail(FZB_E_CUDA, "cudaHostAlloc(%llu) failed", (unsigned long long)n);
        return nullptr;
    }
    return p;
}

extern "C" void fzb_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" int fzb_timer_start(fzb_haystack *h) {
    if (!h) return fail(FZB_E_INVALID, "NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev[3], h->stream));
    return FZB_OK;
}

extern "C" int fzb_timer_stop(fzb_haystack *h, double *ms) {
    if (!h || !ms) return fail(FZB_E_INVALID, "NULL argument");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev_stop, h->stream));
    CK(cudaEventSynchronize(h->ev_stop));
    float f = 0.f;
    CK(cudaEventElapsedTime(&f, h->ev[3], h->ev_stop));
    *ms = f;
    return FZB_OK;
}

extern "C" int fzb_nccl_unique_id(uint8_t id[FZB_NCCL_ID_BYTES]) {
    if (!id) return fail(FZB_E_INVALID, "NULL argument");
    int rc = nccl_load();
    if (rc) return rc;
    NcclId nid;
    NCCLCK(g_nccl.GetUniqueId(&nid));
    memcpy(id, nid.b, FZB_NCCL_ID_BYTES);
    return FZB_OK;
}

static int ensure_gather_buffers(fzb_haystack *h, uint32_t cap) {
    if (cap <= h->gather_alloc) return FZB_OK;
    if (h->d_send) cudaFree(h->d_send);
    if (h->d_recv) cudaFree(h->d_recv);
    if (h->h_send) cudaFreeHost(h->h_send);
    if (h->h_recv) cudaFreeHost(h->h_recv);
    h->d_send = h->d_recv = h->h_send = h->h_recv = nullptr;
    h->gather_alloc = 0;
    const size_t slot = (size_t)(cap + 1) * kFinCols * sizeof(int64_t);
    CK(cudaMalloc(&h->d_send, slot));
    CK(cudaMalloc(&h->d_recv, slot * h->world));
    CK(cudaMallocHost(&h->h_send, slot));
    CK(cudaMallocHost(&h->h_recv, slot * h->world));
    h->gather_alloc = cap;
    return FZB_OK;
}

// Receive area + scratch of the peer-memory reduction (p2p_kernels.cuh).
static int p2p_alloc(fzb_haystack *h) {
    if (h->world > kMaxWorld) return fail(FZB_E_UNSUPPORTED, "world sizes above %d are not supported", kMaxWorld);
    CK(cudaSetDevice(h->device));
    h->slot_bytes = ((uint64_t)kHdrWords + (uint64_t)h->p2p_cap * kFinCols) * 8;
    h->flags_off = round_up(2 * (uint64_t)h->world * h->slot_bytes, 256);
    const size_t bytes = h->flags_off + 2 * kMaxWorld * sizeof(uint32_t) + 256;
    if (!h->d_p2p) {
        CK(cudaMalloc(&h->d_p2p, bytes));
        CK(cudaMemset(h->d_p2p, 0, bytes));
        CK(cudaMalloc(&h->d_ms, sizeof(MergeScratch)));
        CK(cudaMemset(h->d_ms, 0, sizeof(MergeScratch)));
        const size_t rows = (size_t)h->world * h->p2p_cap;
        CK(cudaMalloc(&h->d_mscore, rows * sizeof(unsigned long long)));
        CK(cudaMalloc(&h->d_mpos, rows * sizeof(uint32_t)));
        const unsigned hflags = cudaHostAllocMapped | cudaHostAllocPortable;
        CK(cudaHostAlloc(&h->h_grows, rows * 2 * sizeof(int64_t), hflags));
        CK(cudaHostAlloc(&h->h_ghdr, 16 * sizeof(uint32_t), hflags));
        memset(h->h_ghdr, 0, 16 * sizeof(uint32_t));
    }
    return FZB_OK;
}

static void p2p_free(fzb_haystack *h) {
    for (int r = 0; r < kMaxWorld; r++) {
        if (h->peer_opened[r] && h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
        h->peer_opened[r] = false;
        h->peer_base[r] = nullptr;
    }
    if (h->d_p2p) cudaFree(h->d_p2p);
    if (h->d_ms) cudaFree(h->d_ms);
    if (h->d_mscore) cudaFree(h->d_mscore);
    if (h->d_mpos) cudaFree(h->d_mpos);
    if (h->h_grows) cudaFreeHost(h->h_grows);
    if (h->h_ghdr) cudaFreeHost(h->h_ghdr);
    h->d_p2p = nullptr;
    h->d_ms = nullptr;
    h->d_mscore = nullptr;
    h->d_mpos = nullptr;
    h->h_grows = nullptr;
    h->h_ghdr = nullptr;
    h->p2p = false;
}

extern "C" int fzb_haystack_comm_init(fzb_haystack *h, const uint8_t id[FZB_NCCL_ID_BYTES], int rank,
                                      int world_size) {
    if (!h || !id || world_size < 1 || rank < 0 || rank >= world_size) return fail(FZB_E_INVALID, "bad arguments");
    int rc = nccl_load();
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (h->comm) nccl_comm_destroy(h->comm);
    h->comm = nullptr;
    p2p_free(h);
    h->local_world = false;
    NcclId nid;
    memcpy(nid.b, id, FZB_NCCL_ID_BYTES);
    NCCLCK(g_nccl.CommInitRank(&h->comm, world_size, nid, rank));
    h->rank = rank;
    h->world = world_size;
    h->epoch = 0;
    rc = ensure_gather_buffers(h, h->gather_cap);
    if (rc) return rc;
    // Peer-memory world: every rank exports its receive area through CUDA IPC; the handles travel over the
    // fresh NCCL communicator (bootstrap only).  Any failure on any rank (no IPC in this container, no peer
    // access between two GPUs) leaves p2p = false on ALL ranks and FZB_F_GLOBAL searches use the staged path.
    struct Hello {
        cudaIpcMemHandle_t handle;
        int32_t ok, device;
        long long pid;
    };
    static_assert(sizeof(Hello) <= 128, "hello record");
    const size_t rec = 128;
    Hello me{};
    me.ok = world_size <= kMaxWorld && p2p_alloc(h) == FZB_OK &&
            cudaIpcGetMemHandle(&me.handle, h->d_p2p) == cudaSuccess;
    cudaGetLastError();
    me.device = h->device;
    me.pid = (long long)getpid();
    std::vector<uint8_t> all(rec * world_size);
    auto exchange = [&](const void *mine) -> int {  // all-gather one 128-byte record per rank
        memset(h->h_send, 0, rec);
        memcpy(h->h_send, mine, sizeof(Hello));
        CK(cudaMemcpyAsync(h->d_send, h->h_send, rec, cudaMemcpyHostToDevice, h->stream));
        NCCLCK(g_nccl.AllGather(h->d_send, h->d_recv, rec, /*ncclInt8*/ 0, h->comm, h->stream));
        CK(cudaMemcpyAsync(h->h_recv, h->d_recv, rec * world_size, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(all.data(), h->h_recv, rec * world_size);
        return FZB_OK;
    };
    rc = exchange(&me);
    if (rc) return rc;
    bool ok = true;
    for (int r = 0; r < world_size; r++) ok = ok && reinterpret_cast<Hello *>(all.data() + rec * r)->ok;
    if (ok) {
        for (int r = 0; r < world_size && ok; r++) {
            const Hello *peer = reinterpret_cast<const Hello *>(all.data() + rec * r);
            if (r == rank) {
                h->peer_base[r] = h->d_p2p;
            } else {
                void *ptr = nullptr;
                if (cudaIpcOpenMemHandle(&ptr, peer->handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                    cudaGetLastError();
                    ok = false;
                } else {
                    h->peer_base[r] = (uint8_t *)ptr;
                    h->peer_opened[r] = true;
                }
            }
        }
    }
    Hello second{};
    second.ok = ok;
    rc = exchange(&second);  // everybody must have opened everybody
    if (rc) return rc;
    for (int r = 0; r < world_size; r++) ok = ok && reinterpret_cast<Hello *>(all.data() + rec * r)->ok;
    h->p2p = ok;
    if (!ok) {
        for (int r = 0; r < kMaxWorld; r++) {
            if (h->peer_opened[r] && h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
            h->peer_opened[r] = false;
            h->peer_base[r] = nullptr;
        }
    }
    return FZB_OK;
}

extern "C" int fzb_comm_init_local(fzb_haystack **handles, int world_size) {
    if (!handles || world_size < 1 || world_size > kMaxWorld) return fail(FZB_E_INVALID, "bad arguments");
    for (int r = 0; r < world_size; r++)
        if (!handles[r]) return fail(FZB_E_INVALID, "NULL handle");
    for (int r = 0; r < world_size; r++) {
        fzb_haystack *h = handles[r];
        if (h->comm) nccl_comm_destroy(h->comm);
        h->comm = nullptr;
        p2p_free(h);
        h->rank = r;
        h->world = world_size;
        h->epoch = 0;
        h->local_world = true;
        int rc = p2p_alloc(h);
        if (rc) return rc;
    }
    for (int r = 0; r < world_size; r++) {
        fzb_haystack *h = handles[r];
        CK(cudaSetDevice(h->device));
        for (int q = 0; q < world_size; q++) {
            h->peer_base[q] = handles[q]->d_p2p;
            if (handles[q]->device != h->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, h->device, handles[q]->device));
                if (!can) return fail(FZB_E_UNSUPPORTED, "no peer access between devices %d and %d", h->device, handles[q]->device);
                cudaError_t e = cudaDeviceEnablePeerAccess(handles[q]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                    return fail(FZB_E_CUDA, "cudaDeviceEnablePeerAccess failed: %s", cudaGetErrorString(e));
                cudaGetLastError();
            }
        }
        h->p2p = true;
    }
    return FZB_OK;
}

// The same peer-memory world WITHOUT NCCL: the caller all-gathers the 64-byte CUDA IPC handles itself (any transport;
// fuzzysearch_b200.sharding does it over its TCP rendezvous).  Also works for several processes sharing ONE GPU,
// which NCCL refuses.  Such a world has no staged fallback: a shard that overflows a slot makes the search fail on
// every rank (FZB_E_UNSUPPORTED) instead of silently returning a partial list.
extern "C" int fzb_p2p_export(fzb_haystack *h, int rank, int world_size, uint8_t handle[FZB_IPC_HANDLE_BYTES]) {
    if (!h || !handle || world_size < 1 || world_size > kMaxWorld || rank < 0 || rank >= world_size)
        return fail(FZB_E_INVALID, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == FZB_IPC_HANDLE_BYTES, "IPC handle size");
    CK(cudaSetDevice(h->device));
    if (h->comm) nccl_comm_destroy(h->comm);
    h->comm = nullptr;
    p2p_free(h);
    h->rank = rank;
    h->world = world_size;
    h->epoch = 0;
    h->local_world = false;
    int rc = p2p_alloc(h);
    if (rc) return rc;
    cudaIpcMemHandle_t mine;
    CK(cudaIpcGetMemHandle(&mine, h->d_p2p));
    memcpy(handle, &mine, sizeof mine);
    return FZB_OK;
}

extern "C" int fzb_p2p_connect(fzb_haystack *h, const uint8_t *handles) {
    if (!h || !handles || !h->d_p2p) return fail(FZB_E_INVALID, "fzb_p2p_export first");
    CK(cudaSetDevice(h->device));
    for (int r = 0; r < h->world; r++) {
        if (r == h->rank) {
            h->peer_base[r] = h->d_p2p;
            continue;
        }
        cudaIpcMemHandle_t peer;
        memcpy(&peer, handles + (size_t)r * FZB_IPC_HANDLE_BYTES, sizeof peer);
        void *ptr = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&ptr, peer, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            for (int q = 0; q < kMaxWorld; q++) {
                if (h->peer_opened[q] && h->peer_base[q]) cudaIpcCloseMemHandle(h->peer_base[q]);
                h->peer_opened[q] = false;
                h->peer_base[q] = nullptr;
            }
            return fail(FZB_E_CUDA, "cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
        }
        h->peer_base[r] = (uint8_t *)ptr;
        h->peer_opened[r] = true;
    }
    h->p2p = true;
    h->local_world = true;  // (no NCCL communicator behind this world: no staged fallback)
    return FZB_OK;
}

extern "C" void fzb_p2p_disable(fzb_haystack *h) {
    if (h) p2p_free(h);
}

extern "C" int fzb_haystack_p2p_enabled(const fzb_haystack *h) { return h && h->p2p ? 1 : 0; }

// ------------------------------------------------------------------------------------------------
// consolidation (common.py:145-189).  Groups are the connected components of interval overlap
// (SURVEY F11): sort by (start,end), sweep with the running hull end; a match joins the current
// group iff start < hull_end (this also reproduces the reference for empty matches, which never
// overlap anything they merely touch).  Winner = min (dist, -(end-start)), ties -> smallest
// (start,end).  Output sorted by (start,end,dist).
// ------------------------------------------------------------------------------------------------
static void consolidate_recs(std::vector<RawRec> v, std::vector<RawRec> &out, std::vector<int64_t> *hulls = nullptr) {
    out.clear();
    if (hulls) hulls->clear();
    if (v.empty()) return;
    auto canonical = [](const RawRec &a, const RawRec &b) {
        if (a.start != b.start) return a.start < b.start;
        if (a.end != b.end) return a.end < b.end;
        return a.dist < b.dist;
    };
    std::sort(v.begin(), v.end(), canonical);
    RawRec best = v[0];
    int64_t hull_start = v[0].start, hull_end = v[0].end;
    auto better = [](const RawRec &a, const RawRec &b) {  // a strictly better than b
        if (a.dist != b.dist) return a.dist < b.dist;
        int64_t la = a.end - a.start, lb = b.end - b.start;
        if (la != lb) return la > lb;
        if (a.start != b.start) return a.start < b.start;
        return a.end < b.end;
    };
    auto close_group = [&]() {
        out.push_back(best);
        if (hulls) {
            hulls->push_back(hull_start);
            hulls->push_back(hull_end);
        }
    };
    for (size_t i = 1; i < v.size(); i++) {
        if (v[i].start < hull_end) {
            if (better(v[i], best)) best = v[i];
            hull_end = std::max(hull_end, v[i].end);
        } else {
            close_group();
            best = v[i];
            hull_start = v[i].start;
            hull_end = v[i].end;
        }
    }
    close_group();
    // winners come out in group order, which is already (start, end, dist) order: groups are
    // disjoint and ordered, and an empty group at x sorts before a group starting at x
}

extern "C" int64_t fzb_consolidate(const int64_t *start, const int64_t *end, const int32_t *dist, uint64_t n,
                                   int64_t *out_start, int64_t *out_end, int32_t *out_dist) {
    if (n && (!start || !end || !dist)) return fail(FZB_E_INVALID, "NULL input");
    std::vector<RawRec> v(n), o;
    for (uint64_t i = 0; i < n; i++) {
        v[i].start = start[i];
        v[i].end = end[i];
        v[i].dist = dist[i];
        v[i].idx = -1;
        v[i].ngram = -1;
    }
    consolidate_recs(std::move(v), o);
    for (size_t i = 0; i < o.size(); i++) {
        if (out_start) out_start[i] = o[i].start;
        if (out_end) out_end[i] = o[i].end;
        if (out_dist) out_dist[i] = o[i].dist;
    }
    return (int64_t)o.size();
}

extern "C" int64_t fzb_consolidate_groups(const int64_t *start, const int64_t *end, const int32_t *dist, uint64_t n,
                                          int64_t *out_rows) {
    if (n && (!start || !end || !dist || !out_rows)) return fail(FZB_E_INVALID, "NULL input");
    std::vector<RawRec> v(n), o;
    std::vector<int64_t> hulls;
    for (uint64_t i = 0; i < n; i++) {
        v[i].start = start[i];
        v[i].end = end[i];
        v[i].dist = dist[i];
        v[i].idx = -1;
        v[i].ngram = -1;
    }
    consolidate_recs(std::move(v), o, &hulls);
    for (size_t i = 0; i < o.size(); i++) {
        out_rows[5 * i + 0] = o[i].start;
        out_rows[5 * i + 1] = o[i].end;
        out_rows[5 * i + 2] = o[i].dist;
        out_rows[5 * i + 3] = hulls[2 * i];
        out_rows[5 * i + 4] = hulls[2 * i + 1];
    }
    return (int64_t)o.size();
}

extern "C" int64_t fzb_result_group_rows(const fzb_result *r, int64_t *rows, uint64_t max_rows) {
    if (!r || (!rows && max_rows)) return fail(FZB_E_INVALID, "NULL argument");
    const std::vector<RawRec> &v = r->fin;
    if (!r->have_fin || r->hulls.size() != v.size() * 2)
        return fail(FZB_E_INVALID, "result was produced with FZB_F_NO_FINAL");
    const size_t n = std::min<size_t>(v.size(), max_rows);
    for (size_t i = 0; i < n; i++) {
        rows[5 * i + 0] = v[i].start;
        rows[5 * i + 1] = v[i].end;
        rows[5 * i + 2] = v[i].dist;
        rows[5 * i + 3] = r->hulls[2 * i];
        rows[5 * i + 4] = r->hulls[2 * i + 1];
    }
    return (int64_t)v.size();
}

extern "C" int fzb_result_hulls(const fzb_result *r, int64_t *hull_start, int64_t *hull_end) {
    if (!r) return fail(FZB_E_INVALID, "result is NULL");
    // (unconsolidated routes: every match is its own group, hull == the match)
    if (!r->have_fin || r->hulls.size() != r->fin.size() * 2)
        return fail(FZB_E_INVALID, "result was produced with FZB_F_NO_FINAL");
    for (size_t i = 0; i < r->fin.size(); i++) {
        if (hull_start) hull_start[i] = r->hulls[2 * i];
        if (hull_end) hull_end[i] = r->hulls[2 * i + 1];
    }
    return FZB_OK;
}

// Merge per-shard consolidated lists.  Each input row is one GROUP of overlapping matches found by a
// shard: its winner (start, end, dist) and the group's hull [hull_start, hull_end).  Groups of
// different shards that overlap belong to one global group (a group's hull is covered by its
// members, so hulls overlap iff members do), and the winner of a union is the better of the two
// winners -- so the global consolidate_overlapping_matches (common.py:185-189) is the same sweep run
// over the groups instead of the raw matches.
// Global consolidation over per-shard groups.  `runs` = (pointer, count) of each shard's rows, in shard
// order; every run is sorted by hull start and runs only interleave within a halo of their seams, so
// instead of sorting, each seam is fixed with an inplace_merge of the few out-of-order rows around it.
struct GroupRow {
    int64_t s, e, d, hs, he;
};

static void merge_group_runs(const std::vector<std::pair<const int64_t *, uint64_t>> &runs, std::vector<RawRec> &out) {
    uint64_t n = 0;
    for (auto &r : runs) n += r.second;
    std::vector<GroupRow> g;
    g.reserve(n);
    auto less = [](const GroupRow &a, const GroupRow &b) {
        if (a.hs != b.hs) return a.hs < b.hs;
        if (a.he != b.he) return a.he < b.he;
        if (a.s != b.s) return a.s < b.s;
        if (a.e != b.e) return a.e < b.e;
        return a.d < b.d;
    };
    for (auto &r : runs) {
        const size_t seam = g.size();
        for (uint64_t i = 0; i < r.second; i++) {
            const int64_t *q = r.first + 5 * i;
            g.push_back(GroupRow{q[0], q[1], q[2], q[3], q[4]});
        }
        if (!std::is_sorted(g.begin() + seam, g.end(), less)) std::sort(g.begin() + seam, g.end(), less);  // defensive
        if (seam > 0 && seam < g.size() && less(g[seam], g[seam - 1])) {
            auto lo = std::upper_bound(g.begin(), g.begin() + seam, g[seam], less);
            auto hi = std::lower_bound(g.begin() + seam, g.end(), g[seam - 1], less);
            std::inplace_merge(lo, g.begin() + seam, hi, less);
        }
    }
    if (!std::is_sorted(g.begin(), g.end(), less)) std::sort(g.begin(), g.end(), less);  // shards smaller than a halo
    auto better = [](const GroupRow &a, const GroupRow &b) {
        if (a.d != b.d) return a.d < b.d;
        int64_t la = a.e - a.s, lb = b.e - b.s;
        if (la != lb) return la > lb;
        if (a.s != b.s) return a.s < b.s;
        return a.e < b.e;
    };
    out.clear();
    out.reserve(n);
    for (uint64_t i = 0; i < n;) {
        GroupRow best = g[i];
        int64_t hull_end = g[i].he;
        uint64_t j = i + 1;
        while (j < n && g[j].hs < hull_end) {
            if (better(g[j], best)) best = g[j];
            hull_end = std::max(hull_end, g[j].he);
            j++;
        }
        RawRec r;
        r.start = best.s;
        r.end = best.e;
        r.dist = (int32_t)best.d;
        r.idx = -1;
        r.ngram = -1;
        out.push_back(r);
        i = j;
    }
}

static void merge_group_rows(const int64_t *rows, uint64_t n, std::vector<RawRec> &out) {
    // one run per maximal sorted stretch is not known here: treat the input as a single run (sorted if needed)
    std::vector<std::pair<const int64_t *, uint64_t>> runs{{rows, n}};
    merge_group_runs(runs, out);
}

extern "C" int64_t fzb_merge_groups(const int64_t *rows, uint64_t n, int64_t *out_start, int64_t *out_end,
                                    int32_t *out_dist) {
    if (n && !rows) return fail(FZB_E_INVALID, "NULL input");
    std::vector<RawRec> o;
    merge_group_rows(rows, n, o);
    for (size_t i = 0; i < o.size(); i++) {
        if (out_start) out_start[i] = o[i].start;
        if (out_end) out_end[i] = o[i].end;
        if (out_dist) out_dist[i] = o[i].dist;
    }
    return (int64_t)o.size();
}

// The staged (host-buffer) all-gather of group rows: used when the fused one behind the kernels could
// not be trusted on every rank (a rank overflowed a buffer and retried, or its list was too long for
// the on-device consolidation).  Collective: every rank calls it the same number of times.
static int allgather_groups_staged(fzb_haystack *h, const std::vector<int64_t> &rows, std::vector<int64_t> &all,
                                   std::vector<uint64_t> &counts) {
    const uint64_t n = rows.size() / kFinCols;
    for (;;) {
        const uint32_t cap = h->gather_cap;
        int rc = ensure_gather_buffers(h, cap);
        if (rc) return rc;
        const size_t slot_rows = (size_t)cap + 1, slot = slot_rows * kFinCols * sizeof(int64_t);
        h->h_send[0] = (int64_t)n;
        h->h_send[1] = n <= cap;
        h->h_send[2] = h->h_send[3] = h->h_send[4] = 0;
        if (n <= cap && n) memcpy(h->h_send + kFinCols, rows.data(), n * kFinCols * sizeof(int64_t));
        CK(cudaMemcpyAsync(h->d_send, h->h_send, (1 + (n <= cap ? n : 0)) * kFinCols * sizeof(int64_t),
                           cudaMemcpyHostToDevice, h->stream));
        NCCLCK(g_nccl.AllGather(h->d_send, h->d_recv, slot, /*ncclInt8*/ 0, h->comm, h->stream));
        CK(cudaMemcpyAsync(h->h_recv, h->d_recv, slot * h->world, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        uint64_t top = 0;
        for (int r = 0; r < h->world; r++) top = std::max<uint64_t>(top, (uint64_t)h->h_recv[(size_t)r * slot_rows * kFinCols]);
        if (top <= cap) {
            all.clear();
            counts.clear();
            for (int r = 0; r < h->world; r++) {
                const int64_t *base = h->h_recv + (size_t)r * slot_rows * kFinCols;
                all.insert(all.end(), base + kFinCols, base + kFinCols + (size_t)base[0] * kFinCols);
                counts.push_back((uint64_t)base[0]);
            }
            return FZB_OK;
        }
        while (h->gather_cap < top) h->gather_cap *= 2;  // every rank sees the same `top`
    }
}

// ------------------------------------------------------------------------------------------------
// search plumbing
// ------------------------------------------------------------------------------------------------
static void fill_params(const fzb_haystack *h, const uint8_t *pattern, uint32_t m, ScanParams &p) {
    memset(&p, 0, sizeof p);
    p.H = h->d;
    p.buf_lo = (int64_t)h->buf_lo;
    p.buf_len = (int64_t)h->buf_len;
    p.N = (int64_t)h->global_len;
    p.own_lo = (int64_t)h->own_lo;
    p.own_hi = (int64_t)h->own_hi;
    p.bitmap = h->d_bitmap;
    p.glist = h->d_glist;
    p.glist_cap = h->glist_cap;
    p.counters = h->d_counters;
    p.m = (int)m;
    memcpy(p.P, pattern, m);
}

static int check_halo(const fzb_haystack *h, uint64_t halo) {
    uint64_t need_lo = h->own_lo > halo ? h->own_lo - halo : 0;
    uint64_t need_hi = std::min(h->global_len, h->own_hi + halo);
    if (h->own_lo == h->own_hi) return FZB_OK;
    if (h->buf_lo > need_lo || h->buf_lo + h->buf_len < need_hi)
        return fail(FZB_E_INVALID, "shard halo too small: need %llu bytes each side",
                    (unsigned long long)halo);
    return FZB_OK;
}

static int ensure_out_cap(fzb_haystack *h, uint64_t need) {
    if (need <= h->out_cap) return FZB_OK;
    uint64_t cap = h->out_cap;
    while (cap < need) cap *= 2;
    if (cap > (1ull << 27)) return fail(FZB_E_UNSUPPORTED, "more than 2^27 raw matches in one search");
    CK(cudaFree(h->d_out));
    h->d_out = nullptr;
    CK(cudaMalloc(&h->d_out, (size_t)cap * (sizeof(RawRec) + sizeof(uint64_t))));
    h->out_cap = (uint32_t)cap;
    return FZB_OK;
}

// Runs one search attempt after another until the output buffer was large enough.  `enqueue` must
// put EVERY kernel of the search on h->stream (filter included: the verify kernels clear the dirty
// bitmap as they consume it, so a retry has to re-mark it) and may record h->ev[1] after its scan
// kernel.  One attempt = one stream synchronisation and NO copy operation: k_post, enqueued behind the
// emitting kernels, writes the counters, the raw records and the final rows into mapped pinned host
// memory, which the host reads as soon as the stream has drained.

// Completion of a search attempt: its last kernel stores h->seq into mapped pinned memory after everything else
// (fenced at system scope); polling that word returns a few microseconds earlier than cudaStreamSynchronize and
// does not depend on the process's device scheduling flags (another library in the process -- e.g. a framework
// that asked for blocking synchronisation -- would otherwise add its wake-up latency to every search).  Falls back to
// the stream synchronisation if the word does not arrive (a failed launch), which also surfaces the error.
static int wait_done(fzb_haystack *h, const volatile uint32_t *word) {
    const uint32_t want = h->seq;
    for (uint64_t spins = 0; *word != want; spins++) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0xFFF) == 0xFFF) {
            const cudaError_t e = cudaStreamQuery(h->stream);
            if (e == cudaSuccess) break;  // stream drained: the word is there (or the kernel never ran: error below)
            if (e != cudaErrorNotReady) return fail(FZB_E_CUDA, "search failed: %s", cudaGetErrorString(e));
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (*word != want) {
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
        if (*word != want) return fail(FZB_E_CUDA, "search kernels did not complete");
    }
    return FZB_OK;
}

// What k_post should do behind the emitting kernels.
struct PostPlan {
    int mode = 1;         // 0 raw stream only; 1 consolidate_overlapping_matches; 2 final = sorted raw list
    bool global = false;  // FZB_F_GLOBAL: reduce the groups of every shard behind the kernels
};

static void finalize_on_host(fzb_result *res, int mode);

template <class F>
static int run_emitting(fzb_haystack *h, fzb_result *res, F enqueue, PostPlan post = PostPlan()) {
    detach_pending(h);  // k_post is about to overwrite the staging buffer an earlier result may still point at
    for (int attempt = 0; attempt < 8; attempt++) {
        if (!h->counters_clean) CK(cudaMemsetAsync(h->d_counters, 0, CNT_COUNT * sizeof(uint32_t), h->stream));
        h->counters_clean = false;
        CK(cudaEventRecord(h->ev[0], h->stream));
        h->ev1_recorded = false;
        int rc = enqueue();
        if (rc) return rc;
        CK(cudaGetLastError());
        h->seq++;
        PostArgs pa{reinterpret_cast<const uint64_t *>(h->d_out + h->out_cap), h->out_cap, post.mode,
                    h->d_sorted, h->d_fin, h->h_fin, h->h_counters, h->d_counters, h->seq, 0};
        // fused multi-GPU reduction over peer memory (below): k_push reads the counters after k_post, and clears them
        pa.clear = !(post.global && attempt == 0 && h->p2p && !res->fused_issued);
        k_post<<<h->sm_count, kPostThreads, kPostSmem, h->stream>>>(pa);
        CK(cudaGetLastError());
        res->stats.n_launches++;
        // fused multi-GPU reduction over peer memory: exactly one push + merge per search, in the FIRST attempt
        // (a rank that has to retry locally has pushed a header with valid = 0: every rank sees it and all of them
        // take the staged path together)
        const bool fused = post.global && attempt == 0 && h->p2p && !res->fused_issued;
        if (fused) {
            h->epoch++;
            WorldArgs w{};
            w.world = h->world;
            w.rank = h->rank;
            w.epoch = h->epoch;
            w.cap = h->p2p_cap;
            w.slot_bytes = h->slot_bytes;
            w.flags_off = h->flags_off;
            for (int r = 0; r < h->world; r++) w.peer[r] = h->peer_base[r];
            k_push<<<kPushCtas, kPushThreads, 0, h->stream>>>(w, h->d_fin, h->d_counters, post.mode, h->d_ms);
            MergeOut mo{h->d_mscore, h->d_mpos, h->h_grows, h->h_ghdr, h->seq};
            k_merge<<<h->world, kPostThreads, 0, h->stream>>>(w, h->d_ms, mo);
            CK(cudaGetLastError());
            res->stats.n_launches += 2;
        }
        CK(cudaEventRecord(h->ev[2], h->stream));
        rc = wait_done(h, fused ? h->h_ghdr + 7 : h->h_counters + CNT_SEQ);
        if (rc) return rc;
        const uint32_t n = h->h_counters[CNT_OUT];
        res->stats.n_candidates = h->h_counters[CNT_CAND];
        if (fused) {
            res->fused_issued = true;
            res->fused_status = h->h_ghdr[0];
            res->gcount = h->h_ghdr[1];
            if (h->h_ghdr[2] != h->epoch && res->fused_status == MS_OK) res->fused_status = MS_TIMEOUT;
        }
        if (n > h->out_cap) {  // output buffer too small: grow and redo the whole attempt
            rc = ensure_out_cap(h, n);
            if (rc) return rc;
            continue;
        }
        const bool posted = h->h_counters[CNT_POST_DONE] != 0;
        // k_post (or k_push behind it, if the shard was valid) zeroed the device counters on its way out
        h->counters_clean = posted && (!fused || (res->fused_status == MS_OK));
        res->raw.clear();
        res->raw_n = n;
        res->raw_ordered = false;
        if (posted || (res->fused_issued && res->fused_status == MS_OK)) {
            // the raw records are in h->d_out, the global rows in h->h_grows: copied out lazily (fetch_raw)
            std::lock_guard<std::mutex> lock(g_pending_mutex);
            res->raw_in_stage = posted;
            res->owner = h;
            h->pending = res;
        }
        if (!posted && n) {  // list too long for k_post: fetch it, the host orders and consolidates
            res->raw.resize(n);
            CK(cudaMemcpyAsync(res->raw.data(), h->d_out, (size_t)n * sizeof(RawRec), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
        }
        res->fin.clear();
        res->hulls.clear();
        res->have_fin = false;
        res->device_post = false;
        if (post.mode != 0) {
            if (posted) {
                const uint32_t nf = h->h_counters[CNT_NFINAL];
                res->fin.resize(nf);
                res->hulls.resize((size_t)nf * 2);
                for (uint32_t i = 0; i < nf; i++) {
                    res->fin[i].start = h->h_fin[kFinCols * i];
                    res->fin[i].end = h->h_fin[kFinCols * i + 1];
                    res->fin[i].dist = (int32_t)h->h_fin[kFinCols * i + 2];
                    res->fin[i].idx = -1;
                    res->fin[i].ngram = -1;
                    res->hulls[2 * i] = h->h_fin[kFinCols * i + 3];
                    res->hulls[2 * i + 1] = h->h_fin[kFinCols * i + 4];
                }
                res->device_post = true;
            } else {
                finalize_on_host(res, post.mode);
            }
            res->have_fin = true;
        }
        float ms = 0.f;
        while (cudaEventQuery(h->ev[2]) == cudaErrorNotReady) {  // a microsecond behind the polled word
        }
        cudaEventElapsedTime(&ms, h->ev[0], h->ev[2]);
        res->stats.gpu_ms = ms;
        res->stats.filter_ms = ms;
        if (h->ev1_recorded) {
            cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]);
            res->stats.filter_ms = ms;
        }
        return FZB_OK;
    }
    return fail(FZB_E_CUDA, "output buffer kept overflowing");
}

static void sort_generation_order(std::vector<RawRec> &v) {
    std::sort(v.begin(), v.end(), [](const RawRec &a, const RawRec &b) {
        if (a.ngram != b.ngram) return a.ngram < b.ngram;
        return a.idx < b.idx;
    });
}

static void sort_generation_order(std::vector<RawRec> &v);
static void sort_canonical(std::vector<RawRec> &v);

void fzb_result::order_raw() {
    fetch_raw();
    if (raw_ordered) return;
    if (raw_order == 0)
        sort_generation_order(raw);
    else if (raw_order == 1)
        sort_canonical(raw);
    else
        std::sort(raw.begin(), raw.end(), [](const RawRec &a, const RawRec &b) {
            if (a.ngram != b.ngram) return a.ngram < b.ngram;
            if (a.idx != b.idx) return a.idx < b.idx;
            if (a.start != b.start) return a.start < b.start;
            if (a.end != b.end) return a.end < b.end;
            return a.dist < b.dist;
        });
    raw_ordered = true;
}

static void sort_canonical(std::vector<RawRec> &v) {
    std::sort(v.begin(), v.end(), [](const RawRec &a, const RawRec &b) {
        if (a.start != b.start) return a.start < b.start;
        if (a.end != b.end) return a.end < b.end;
        return a.dist < b.dist;
    });
}

// Host twin of k_post for lists it does not take (more than kPostMax records).
static void finalize_on_host(fzb_result *res, int mode) {
    if (mode == 1) {
        consolidate_recs(res->raw, res->fin, &res->hulls);
        return;
    }
    res->fin = res->raw;
    sort_canonical(res->fin);
    res->hulls.resize(res->fin.size() * 2);
    for (size_t i = 0; i < res->fin.size(); i++) {
        res->fin[i].idx = -1;
        res->fin[i].ngram = -1;
        res->hulls[2 * i] = res->fin[i].start;
        res->hulls[2 * i + 1] = res->fin[i].end;
    }
}

static int set_filter_attrs(size_t smem) {
    // per device: the attribute belongs to the function on the current device
    CK(cudaFuncSetAttribute(k_filter_sampled, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CK(cudaFuncSetAttribute(k_filter_dense<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmem));
    CK(cudaFuncSetAttribute(k_filter_dense<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmem));
    CK(cudaFuncSetAttribute(k_filter_dense<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmem));
    CK(cudaFuncSetAttribute(k_filter_dense<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDenseSmem));
    CK(cudaFuncSetAttribute(k_filter_dense2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDense2Smem));
    return FZB_OK;
}

constexpr size_t kFilterSmem = kTblSize + 256 * sizeof(uint32_t);
constexpr int kVerifyCtasPerSm = 8;  // k_verify_lev is latency bound (one DRAM round trip + a dependent chain per granule)

// The q-sample lemma of k_filter_sampled needs floor((m-k-3)/4) >= k+1 aligned words per occurrence.
static bool sampled_filter_applies(uint32_t m, uint32_t k, uint32_t flags) {
    if (flags & FZB_F_FORCE_DENSE) return false;
    if (m < 4 || m < k + 3) return false;
    return (m - k - 3) / 4 >= k + 1;
}

// Byte statistics of the haystack from 16 sampled 4 KiB blocks (once per handle content): the
// collision probability sum_c p_c^2 tells how selective a q-gram test is (1/4 on DNA, ~1/95 on text).
static int sample_collision_prob(fzb_haystack *h) {
    if (h->coll_prob >= 0.0) return FZB_OK;
    const uint64_t blk = 4096, nblk = 16;
    std::vector<uint8_t> buf;
    uint64_t hist[256] = {0}, total = 0;
    if (h->buf_len <= blk * nblk) {
        buf.resize(h->buf_len);
        if (h->buf_len) CK(cudaMemcpy(buf.data(), h->d, h->buf_len, cudaMemcpyDeviceToHost));
    } else {
        buf.resize(blk * nblk);
        for (uint64_t i = 0; i < nblk; i++) {
            const uint64_t off = ((h->buf_len - blk) / (nblk - 1) * i) & ~(uint64_t)15;
            CK(cudaMemcpyAsync(buf.data() + i * blk, h->d + off, blk, cudaMemcpyDeviceToHost, h->stream));
        }
        CK(cudaStreamSynchronize(h->stream));
    }
    for (uint8_t c : buf) hist[c]++;
    total = buf.size();
    double s = 0.0;
    if (total)
        for (int c = 0; c < 256; c++) s += ((double)hist[c] / total) * ((double)hist[c] / total);
    h->coll_prob = total ? s : 1.0;
    return FZB_OK;
}

// The sampled filter is sound whenever the lemma holds, but only SELECTIVE if an aligned word rarely
// equals a pattern 4-gram; otherwise (small alphabets) the dense filter, which finds the n-gram hits
// themselves, marks far fewer granules.  Expected marked-granule fractions decide.
static bool sampled_is_selective(fzb_haystack *h, uint32_t m, uint32_t k, int L, int n_ngrams) {
    if (sample_collision_prob(h) != FZB_OK) return true;
    const double c = h->coll_prob;
    const double span = (2.0 * m + 2.0 * k - L - 3.0) / kGranule + 1.0;       // granules marked per word hit
    const double sampled = std::min(1.0, (m - 3.0) * c * c * c * c * (kGranule / 4.0) * span);
    const double dense = std::min(1.0, n_ngrams * std::pow(c, std::min(L, 8)) * kGranule);
    return sampled <= 0.02 || sampled <= dense;
}

// Enqueue the one pass over the haystack that marks candidate granules; records ev[1] behind it.
static int enqueue_filter(fzb_haystack *h, const ScanParams &p, bool sampled, fzb_result *res) {
    const int64_t nvec = (int64_t)(round_up(h->buf_len, 16) / 16);
    const int64_t ntiles = (nvec + kTileVecs - 1) / kTileVecs;
    // dense route on a low-entropy haystack (about six effective symbols or fewer): index the table with 2-bit codes
    bool two_bit = false;
    if (!sampled && h->buf_len > 0 && sample_collision_prob(h) == FZB_OK) two_bit = h->coll_prob >= 0.15;
    if (ntiles > 0) {
        int per_sm = 4;
        if (two_bit) {
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_filter_dense2, kFilterThreads, kDense2Smem));
            per_sm = std::max(per_sm, 1);
        } else if (!sampled) {  // persistent grid = exactly the resident CTAs of the chosen instantiation
            const void *fn = p.q < 4    ? (const void *)k_filter_dense<0>
                             : p.q == 4 ? (const void *)k_filter_dense<1>
                             : p.q < 8  ? (const void *)k_filter_dense<2>
                                        : (const void *)k_filter_dense<3>;
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kFilterThreads, kDenseSmem));
            per_sm = std::max(per_sm, 1);
        }
        int grid = (int)std::min<int64_t>(ntiles, (int64_t)h->sm_count * per_sm);
        if (sampled)
            k_filter_sampled<<<grid, kFilterThreads, kFilterSmem, h->stream>>>(p, nvec, ntiles);
        else if (two_bit)
            k_filter_dense2<<<grid, kFilterThreads, kDense2Smem, h->stream>>>(p, nvec, ntiles);
        else if (p.q < 4)
            k_filter_dense<0><<<grid, kFilterThreads, kDenseSmem, h->stream>>>(p, nvec, ntiles);
        else if (p.q == 4)
            k_filter_dense<1><<<grid, kFilterThreads, kDenseSmem, h->stream>>>(p, nvec, ntiles);
        else if (p.q < 8)
            k_filter_dense<2><<<grid, kFilterThreads, kDenseSmem, h->stream>>>(p, nvec, ntiles);
        else
            k_filter_dense<3><<<grid, kFilterThreads, kDenseSmem, h->stream>>>(p, nvec, ntiles);
        CK(cudaGetLastError());
        res->stats.n_launches++;
    }
    CK(cudaEventRecord(h->ev[1], h->stream));
    h->ev1_recorded = true;
    return FZB_OK;
}

// n-gram Levenshtein search (also serves exact search as k == 0, L == m)
static int search_lev_ngrams(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t k, uint32_t flags,
                             fzb_result *res, int post_mode) {
    ScanParams p;
    fill_params(h, pattern, m, p);
    p.k = (int)k;
    p.L = (int)(m / (k + 1));
    if (p.L == 0) return fail(FZB_E_NGRAM_ZERO, "the subsequence length must be greater than max_l_dist");
    p.n_ngrams = (int)m / p.L;  // range(0, m-L+1, L)
    int rc = check_halo(h, (uint64_t)m + k);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const bool sampled = sampled_filter_applies(m, k, flags) &&
                         ((flags & FZB_F_FORCE_SAMPLED) || sampled_is_selective(h, m, k, p.L, p.n_ngrams));
    p.q = sampled ? 4 : std::min(p.L, 8);
    res->stats.route = k == 0 ? 0 : (sampled ? 1 : 2);
    res->stats.bytes_scanned = h->buf_len;
    CK(cudaSetDevice(h->device));
    if (!h->filter_attrs_set) {
        rc = set_filter_attrs(kFilterSmem);
        if (rc) return rc;
        h->filter_attrs_set = true;
    }
    // dense route: confirmed n-gram hits go to a list and are verified one lane per hit (the window of a
    // hit must fit a lane's shared-memory slot); the list overflowing triggers one retry in granule mode
    const int vm = verify_mode((int)m, p.L);
    bool use_hits = !sampled && k > 0 && (m + 2 * k + 8 <= (uint32_t)kHitSlotBytes);
    if (use_hits && !h->d_hits) {
        h->hits_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1u << 20, h->capacity / 256), 1u << 28);
        CK(cudaMalloc(&h->d_hits, (size_t)h->hits_cap * sizeof(uint64_t)));
    }
    bool fuse_gather = post_mode != 0 && (flags & FZB_F_GLOBAL) != 0;
    bool bitmap_mode = false;
    if (flags & FZB_F_TINY_LIST) p.glist_cap = std::min(h->glist_cap, 8u);
retry_without_hits:
    p.hits = use_hits ? h->d_hits : nullptr;
    p.hits_cap = use_hits ? ((flags & FZB_F_TINY_LIST) ? std::min(h->hits_cap, 8u) : h->hits_cap) : 0;
    rc = run_emitting(h, res, [&]() -> int {
        int r2 = enqueue_filter(h, p, sampled, res);
        if (r2) return r2;
        if (use_hits) {
            if (vm == 0)
                k_verify_hits<0><<<h->sm_count * 8, kHitThreads, 0, h->stream>>>(p, h->d_out, h->out_cap, h->d_counters);
            else if (vm == 1)
                k_verify_hits<1><<<h->sm_count * 8, kHitThreads, 0, h->stream>>>(p, h->d_out, h->out_cap, h->d_counters);
            else
                k_verify_hits<2><<<h->sm_count * 8, kHitThreads, 0, h->stream>>>(p, h->d_out, h->out_cap, h->d_counters);
            res->stats.n_launches++;
            return FZB_OK;
        }
        {   // one verify launch: the granule work list -- or, second attempt after the list overflowed, the whole bitmap
            const int scan_mode = bitmap_mode ? 1 : 0;
            const int grid = h->sm_count * kVerifyCtasPerSm;
            if (vm == 0)
                k_verify_lev<0><<<grid, kVerifyThreads, 0, h->stream>>>(p, h->bitmap_words, h->d_glist, p.glist_cap,
                                                                        scan_mode, h->d_out, h->out_cap, h->d_counters);
            else if (vm == 1)
                k_verify_lev<1><<<grid, kVerifyThreads, 0, h->stream>>>(p, h->bitmap_words, h->d_glist, p.glist_cap,
                                                                        scan_mode, h->d_out, h->out_cap, h->d_counters);
            else
                k_verify_lev<2><<<grid, kVerifyThreads, 0, h->stream>>>(p, h->bitmap_words, h->d_glist, p.glist_cap,
                                                                        scan_mode, h->d_out, h->out_cap, h->d_counters);
        }
        res->stats.n_launches += 1;
        return FZB_OK;
    }, PostPlan{post_mode, fuse_gather});  // the raw stream's order (n-gram, hit index) is restored lazily
    if (rc) return rc;
    if (!use_hits && !bitmap_mode && h->h_counters[CNT_GRAN] > p.glist_cap) {
        // more marked granules than the work list holds: the verify kernel raised CNT_OVERFLOW and did nothing (so a fused
        // reduction, if any, went out invalid); redo the search with the list switched off, sweeping the bitmap
        bitmap_mode = true;
        fuse_gather = false;
        p.glist_cap = 0;
        res->fetch_raw();
        res->raw.clear();
        res->raw_n = 0;
        res->fin.clear();
        goto retry_without_hits;
    }
    if (use_hits && h->h_counters[CNT_HITS] > p.hits_cap) {
        // the fused all-gather (if any) went out with valid = 0 (k_verify_hits raised CNT_OVERFLOW), so every
        // rank will take finish_global's staged round; the retry itself must not issue another collective
        fuse_gather = false;
        use_hits = false;
        res->fetch_raw();  // unlink from the staging buffer
        res->raw.clear();
        res->raw_n = 0;
        res->fin.clear();
        goto retry_without_hits;
    }
    res->raw_order = 0;
    return FZB_OK;
}

// ------------------------------------------------------------------------------------------------
// LP / generic routes (lp_kernels.cuh)
// ------------------------------------------------------------------------------------------------
static int ensure_scratch(fzb_haystack *h, uint64_t words) {
    if (words <= h->scratch_words) return FZB_OK;
    if (h->d_scratch) CK(cudaFree(h->d_scratch));
    h->d_scratch = nullptr;
    h->scratch_words = 0;
    CK(cudaMalloc(&h->d_scratch, words * sizeof(uint32_t)));
    h->scratch_words = words;
    return FZB_OK;
}

// Runs an LP-style search with growing per-thread candidate capacity until no list overflowed.
// `enqueue(grid, cap)` must put every kernel of one attempt on the stream.
template <class F>
static int run_lp(fzb_haystack *h, fzb_result *res, F enqueue, PostPlan post = PostPlan()) {
    const int grid = h->sm_count * 4;
    const uint64_t threads = (uint64_t)grid * kLpThreads;
    for (int cap = 256; cap <= (1 << 16); cap *= 8) {
        int rc = ensure_scratch(h, threads * 2 * (uint64_t)cap);
        if (rc) return rc;
        rc = run_emitting(h, res, [&]() -> int { return enqueue(grid, cap); }, post);
        if (rc) return rc;
        if (!h->h_counters[CNT_OVERFLOW]) return FZB_OK;
    }
    return fail(FZB_E_UNSUPPORTED, "candidate explosion: more than 65536 live candidates for one start");
}

static int search_lev_lp(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t k, uint32_t flags,
                         fzb_result *res, int post_mode) {
    if (k > 0xFFFF) return fail(FZB_E_UNSUPPORTED, "max_l_dist too large");
    ScanParams p;
    fill_params(h, pattern, m, p);
    p.k = (int)k;
    int rc = check_halo(h, (uint64_t)m + k);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    res->stats.route = 3;
    res->stats.bytes_scanned = h->buf_len;
    // streaming form (k_lp_scan + k_lp_verify) when the look-ahead masks cover the window; the list of surviving
    // starts overflowing (low-entropy data: most starts survive) falls back to the tile kernel
    bool streaming = k < m && m + k <= (uint32_t)kLpsMaxWin && !(flags & FZB_F_FORCE_DENSE) && h->buf_len > 0;
    if (streaming && !h->d_lplist) {
        h->lplist_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1u << 20, h->capacity / 64), 1u << 26);
        CK(cudaMalloc(&h->d_lplist, (size_t)h->lplist_cap * sizeof(unsigned long long)));
    }
    const PostPlan plan{post_mode, post_mode != 0 && (flags & FZB_F_GLOBAL) != 0};
    if (streaming) {
        rc = run_lp(h, res, [&](int grid, int cap) -> int {
            k_lp_scan<<<h->sm_count * 4, kLpsThreads, 0, h->stream>>>(p, h->d_lplist, h->lplist_cap);
            CK(cudaEventRecord(h->ev[1], h->stream));
            h->ev1_recorded = true;
            k_lp_verify<<<grid, kLpThreads, 0, h->stream>>>(p, h->d_lplist, h->lplist_cap, h->d_scratch, cap, h->d_out,
                                                            h->out_cap, h->d_counters);
            res->stats.n_launches += 2;
            return FZB_OK;
        }, plan);
        if (rc) return rc;
        if (h->h_counters[CNT_LPWORK] == 0) {
            res->raw_order = 1;
            return FZB_OK;
        }
        res->fetch_raw();  // list overflow: nothing was verified (and the fused reduction saw an invalid shard)
        res->raw.clear();
        res->raw_n = 0;
        res->fin.clear();
    }
    rc = run_lp(h, res, [&](int grid, int cap) -> int {
        k_lev_lp<<<grid, kLpThreads, 0, h->stream>>>(p, h->d_scratch, cap, h->d_out, h->out_cap, h->d_counters);
        res->stats.n_launches++;
        return FZB_OK;
    }, plan);
    if (rc) return rc;
    res->raw_order = 1;
    return FZB_OK;
}

static int search_generic(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs, uint32_t max_ins,
                          uint32_t max_dels, uint32_t max_l, bool ngrams, uint32_t flags, fzb_result *res,
                          int post_mode) {
    // LP route: every substitution and every deletion consumes a pattern character (so does the "insertion +
    // deletion" pair the reference books when the substitutions are used up, generic_search.py:111-128), hence a
    // live candidate at pattern index j has spent l <= j + n_ins < m + max_ins: a total limit above m + max_ins
    // never binds -- not in `l_dist < max_l_dist` (:101-102), not in the deletion loop's bound (:141), not in the
    // final loop (:172-177) -- and can be lowered to it without changing the raw stream.  (Not so on the n-gram
    // route, where max_l_dist also sets the n-gram length and the windows.)  E.g. max_substitutions=100,
    // max_insertions=1, max_deletions=1 on 20 symbols: 102 -> 21.
    if (!ngrams) max_l = (uint32_t)std::min<uint64_t>(max_l, (uint64_t)m + std::min(max_ins, max_l));
    // the packed candidate of sim_generic keeps 6 bits per counter
    if (max_l > 63) return fail(FZB_E_UNSUPPORTED, "max_l_dist > 63 is not supported by the generic search");
    // no counter can exceed max_l (every operation that increments one costs >= 1), so clamping the
    // per-operation limits to max_l changes nothing (LevenshteinSearchParams does the same, common.py:108-116)
    max_subs = std::min(max_subs, max_l);
    max_ins = std::min(max_ins, max_l);
    max_dels = std::min(max_dels, max_l);
    ScanParams p;
    fill_params(h, pattern, m, p);
    p.k = (int)max_l;
    p.max_subs = (int)max_subs;
    p.max_ins = (int)max_ins;
    p.max_dels = (int)max_dels;
    int rc = check_halo(h, (uint64_t)m + max_l);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    res->stats.bytes_scanned = h->buf_len;
    if (!ngrams) {
        res->stats.route = 6;
        rc = run_lp(h, res, [&](int grid, int cap) -> int {
            k_generic_lp<<<grid, kLpThreads, 0, h->stream>>>(p, h->d_scratch, cap, h->d_out, h->out_cap,
                                                             h->d_counters);
            res->stats.n_launches++;
            return FZB_OK;
        }, PostPlan{post_mode, post_mode != 0 && (flags & FZB_F_GLOBAL) != 0});
        if (rc) return rc;
        res->raw_order = 1;
        return FZB_OK;
    }
    p.L = (int)(m / (max_l + 1));
    if (p.L == 0) return fail(FZB_E_NGRAM_ZERO, "the subsequence length must be greater than max_l_dist");
    p.n_ngrams = (int)m / p.L;
    const bool sampled = sampled_filter_applies(m, max_l, flags) &&
                         ((flags & FZB_F_FORCE_SAMPLED) || sampled_is_selective(h, m, max_l, p.L, p.n_ngrams));
    p.q = sampled ? 4 : std::min(p.L, 8);
    res->stats.route = 5;
    rc = set_filter_attrs(kFilterSmem);
    if (rc) return rc;
    rc = run_lp(h, res, [&](int grid, int cap) -> int {
        int r2 = enqueue_filter(h, p, sampled, res);
        if (r2) return r2;
        k_verify_generic<<<grid, kLpThreads, 0, h->stream>>>(p, h->bitmap_words, h->d_scratch, cap, h->d_out,
                                                             h->out_cap, h->d_counters);
        res->stats.n_launches++;
        return FZB_OK;
    }, PostPlan{post_mode, post_mode != 0 && (flags & FZB_F_GLOBAL) != 0});
    if (rc) return rc;
    res->raw_order = 2;  // n-gram major, hit index, then the window's matches in canonical order
    return FZB_OK;
}

// FZB_F_GLOBAL epilogue of every search entry point: turn the per-shard groups into the global final list.
// Fast path: k_push / k_merge already did it on the device (run_emitting).  Otherwise (no peer-memory world, a
// shard whose list overflowed a buffer, pathological chaining across seams) every rank arrives here and the
// rows go through the staged NCCL all-gather and the host merge.
static int finish_global(fzb_haystack *h, fzb_result *res) {
    if (h->world < 1 || (!h->comm && !h->local_world))
        return fail(FZB_E_INVALID, "FZB_F_GLOBAL needs fzb_haystack_comm_init / fzb_comm_init_local");
    if (res->fused_issued) {
        if (res->fused_status == MS_OK) {
            res->has_global = true;
            res->global_on_device = true;
            return FZB_OK;
        }
        if (res->fused_status == MS_TIMEOUT)
            return fail(FZB_E_CUDA, "multi-GPU reduction timed out waiting for a peer (rank %d of %d)", h->rank, h->world);
    }
    if (h->local_world)
        return fail(FZB_E_UNSUPPORTED, "NCCL-free world: a shard produced more than %u groups (or more than %d raw "
                    "matches); the staged fallback needs an NCCL communicator (fzb_haystack_comm_init)", h->p2p_cap, kPostMax);
    std::vector<int64_t> all;
    std::vector<uint64_t> counts;
    const std::vector<RawRec> &v = res->fin;
    std::vector<int64_t> rows(v.size() * kFinCols);
    for (size_t i = 0; i < v.size(); i++) {
        rows[kFinCols * i + 0] = v[i].start;
        rows[kFinCols * i + 1] = v[i].end;
        rows[kFinCols * i + 2] = v[i].dist;
        rows[kFinCols * i + 3] = res->hulls[2 * i];
        rows[kFinCols * i + 4] = res->hulls[2 * i + 1];
    }
    int rc = allgather_groups_staged(h, rows, all, counts);
    if (rc) return rc;
    if (res->unconsolidated) {  // unconsolidated routes (exact, Hamming): the global list is the sorted union
        res->gfin.resize(all.size() / kFinCols);
        for (size_t i = 0; i < res->gfin.size(); i++) {
            res->gfin[i].start = all[kFinCols * i];
            res->gfin[i].end = all[kFinCols * i + 1];
            res->gfin[i].dist = (int32_t)all[kFinCols * i + 2];
            res->gfin[i].idx = -1;
            res->gfin[i].ngram = -1;
        }
        sort_canonical(res->gfin);
    } else {
        std::vector<std::pair<const int64_t *, uint64_t>> runs;
        uint64_t off = 0;
        for (uint64_t c : counts) {
            runs.push_back({all.data() + off * kFinCols, c});
            off += c;
        }
        merge_group_runs(runs, res->gfin);
    }
    res->gcount = (uint32_t)res->gfin.size();
    res->has_global = true;
    return FZB_OK;
}

static int make_result(fzb_result **out, fzb_result **res) {
    if (!out) return fail(FZB_E_INVALID, "out is NULL");
    *out = nullptr;
    *res = new (std::nothrow) fzb_result();
    if (!*res) return fail(FZB_E_CUDA, "out of host memory");
    return FZB_OK;
}

static int check_pattern(const fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t flags = 0) {
    if (!h) return fail(FZB_E_INVALID, "haystack handle is NULL");
    if ((flags & FZB_F_GLOBAL) && !h->comm && !h->local_world)
        return fail(FZB_E_INVALID, "FZB_F_GLOBAL needs fzb_haystack_comm_init / fzb_comm_init_local on this handle");
    if (!pattern || m == 0) return fail(FZB_E_INVALID, "Given subsequence is empty!");
    if (m > FZB_MAX_PATTERN) return fail(FZB_E_UNSUPPORTED, "pattern longer than %d bytes", FZB_MAX_PATTERN);
    return FZB_OK;
}

extern "C" int fzb_search_levenshtein(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t k,
                                      uint32_t flags, fzb_result **out) {
    HandleLock handle_lock(h);
    fzb_result *res;
    int rc = make_result(out, &res);
    if (rc) return rc;
    rc = check_pattern(h, pattern, m, flags);
    if (rc == FZB_OK) {
        // find_near_matches_levenshtein (levenshtein.py:9-38)
        if (k >= m) k = m;  // every k >= len(pattern) takes the same branch (levenshtein.py:62-65): (i, i, m) for all i
        bool ngrams = (k == 0) || (m / (k + 1) >= 3);
        if (flags & FZB_F_FORCE_NGRAMS) ngrams = true;
        if (flags & FZB_F_FORCE_LP) ngrams = false;
        // LevenshteinSearch.consolidate_matches (levenshtein.py:158-160) also applies when k == 0
        const bool want_final = !(flags & FZB_F_NO_FINAL);
        if (ngrams)
            rc = search_lev_ngrams(h, pattern, m, k, flags, res, want_final ? 1 : 0);
        else
            rc = search_lev_lp(h, pattern, m, k, flags, res, want_final ? 1 : 0);
        if (rc == FZB_OK && want_final && (flags & FZB_F_GLOBAL)) rc = finish_global(h, res);
    }
    if (rc) {
        fzb_result_destroy(res);
        return rc;
    }
    *out = res;
    return FZB_OK;
}

// ------------------------------------------------------------------------------------------------
// Batches: one scan for all the patterns the q-sample lemma covers (batch_kernels.cuh)
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kGtabSlots = 1u << 17;     // gram table (open addressing, <= 50 % full)
constexpr uint32_t kMaxBatchGrams = 60000;    // distinct grams of one pass
constexpr uint32_t kMaxBatchPostings = 1u << 20;
constexpr uint32_t kMaxBatchPats = 4096;      // patterns of one pass

static int ensure_batch_buffers(fzb_haystack *h) {
    if (h->d_mbits) return FZB_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMalloc(&h->d_mbits, (kMultiTblWords + kMulti2Words) * sizeof(uint32_t)));  // first + second level tables
    CK(cudaMalloc(&h->d_gtab, kGtabSlots * sizeof(uint2)));
    CK(cudaMalloc(&h->d_postings, kMaxBatchPostings * sizeof(uint32_t)));
    CK(cudaMalloc(&h->d_pinfo, kMaxBatchPats * sizeof(uint32_t)));
    CK(cudaMalloc(&h->d_bpats, kMaxBatchPats * sizeof(BatchPat)));
    h->mset_slots = 1u << 22;
    h->mwork_cap = 1u << 21;
    CK(cudaMalloc(&h->d_mset, (size_t)h->mset_slots * sizeof(unsigned long long)));
    CK(cudaMemset(h->d_mset, 0, (size_t)h->mset_slots * sizeof(unsigned long long)));
    CK(cudaMalloc(&h->d_mwork, (size_t)h->mwork_cap * sizeof(WorkItem)));
    CK(cudaFuncSetAttribute(k_filter_multi, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMultiSmem));
    return FZB_OK;
}

// One pass over the haystack for the patterns ids[0..cnt): fills out[ids[i]].  Returns FZB_OK, an error, or +1 if
// the pass overflowed a device structure (the caller then searches these patterns one by one).
// dense = false: the q-sample scan (k_filter_multi / k_verify_multi) over the 4-grams of the patterns;
// dense = true: the n-gram-prefix scan at every position (k_filter_mdense / k_verify_mhits).
static int batch_pass(fzb_haystack *h, const uint8_t *patterns, const uint32_t *offsets, const uint32_t *ks,
                      const std::vector<uint32_t> &ids, fzb_result **out, fzb_stats *sum, bool dense) {
    const uint32_t cnt = (uint32_t)ids.size();
    std::vector<BatchPat> pats(cnt);
    std::vector<uint32_t> pinfo(cnt);
    std::unordered_map<uint32_t, std::vector<uint32_t>> grams;
    grams.reserve(cnt * 48);
    for (uint32_t i = 0; i < cnt; i++) {
        const uint32_t id = ids[i], m = offsets[id + 1] - offsets[id], k = ks[id];
        BatchPat &bp = pats[i];
        memset(&bp, 0, sizeof bp);
        memcpy(bp.P, patterns + offsets[id], m);
        bp.m = (int)m;
        bp.k = (int)k;
        bp.L = (int)(m / (k + 1));
        bp.n_ngrams = (int)m / bp.L;
        pinfo[i] = m | (k << 8) | ((uint32_t)bp.L << 16);
        if (dense) {  // key: the first 3 bytes of n-gram j; posting: pattern << 8 | j
            for (int j = 0; j < bp.n_ngrams; j++) {
                uint32_t w = 0;
                memcpy(&w, bp.P + j * bp.L, 3);
                grams[w].push_back((i << 8) | (uint32_t)j);
            }
        } else {
            for (uint32_t o = 0; o + 4 <= m; o++) {
                uint32_t w;
                memcpy(&w, bp.P + o, 4);
                grams[w].push_back((i << 8) | o);
            }
        }
    }
    std::vector<uint32_t> bits(kMultiTblWords + (dense ? 0 : kMulti2Words), 0), postings;
    std::vector<uint2> gtab(kGtabSlots, make_uint2(0, 0));
    for (auto &g : grams) {
        const uint32_t w = g.first, hb = (w * kHashMul) >> (32 - kMultiTblBits);
        bits[hb >> 5] |= 1u << (hb & 31u);
        if (!dense) {
            const uint32_t h2 = multi_hash2(w);
            bits[kMultiTblWords + (h2 >> 5)] |= 1u << (h2 & 31u);
        }
        for (size_t first = 0; first < g.second.size(); first += 255) {
            const uint32_t c = (uint32_t)std::min<size_t>(255, g.second.size() - first);
            uint32_t slot = (w * kGramMul) & (kGtabSlots - 1);
            while (gtab[slot].y != 0u) slot = (slot + 1) & (kGtabSlots - 1);
            gtab[slot] = make_uint2(w, (uint32_t)postings.size() | (c << 24));
            postings.insert(postings.end(), g.second.begin() + first, g.second.begin() + first + c);
        }
    }
    int rc = ensure_batch_buffers(h);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (dense && !h->d_mhits) {
        h->mhits_cap = 1u << 23;
        CK(cudaMalloc(&h->d_mhits, (size_t)h->mhits_cap * sizeof(unsigned long long)));
        CK(cudaFuncSetAttribute(k_filter_mdense, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMdenseSmem));
    }
    detach_pending(h);
    CK(cudaMemcpyAsync(h->d_mbits, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_gtab, gtab.data(), gtab.size() * sizeof(uint2), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_postings, postings.data(), postings.size() * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_pinfo, pinfo.data(), pinfo.size() * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_bpats, pats.data(), pats.size() * sizeof(BatchPat), cudaMemcpyHostToDevice, h->stream));
    MultiParams mp{};
    mp.H = h->d;
    mp.buf_lo = (int64_t)h->buf_lo;
    mp.buf_len = (int64_t)h->buf_len;
    mp.N = (int64_t)h->global_len;
    mp.own_lo = (int64_t)h->own_lo;
    mp.own_hi = (int64_t)h->own_hi;
    mp.bits = h->d_mbits;
    mp.bits2 = dense ? nullptr : h->d_mbits + kMultiTblWords;
    mp.gtab = h->d_gtab;
    mp.gtab_mask = kGtabSlots - 1;
    mp.postings = h->d_postings;
    mp.pinfo = h->d_pinfo;
    mp.set = h->d_mset;
    mp.set_mask = h->mset_slots - 1;
    mp.work = h->d_mwork;
    mp.work_cap = h->mwork_cap;
    mp.counters = h->d_counters;
    const int64_t nvec = (int64_t)(round_up(h->buf_len, 16) / 16);
    const int64_t ntiles = (nvec + kMultiTileVecs - 1) / kMultiTileVecs;
    std::vector<RawRec> raw;
    float gpu_ms = 0.f, filter_ms = 0.f;
    uint32_t n_work = 0;
    for (int attempt = 0;; attempt++) {
        if (attempt == 8) return fail(FZB_E_CUDA, "output buffer kept overflowing");
        h->counters_clean = false;  // (this pass leaves its counters behind)
        CK(cudaMemsetAsync(h->d_counters, 0, CNT_COUNT * sizeof(uint32_t), h->stream));
        CK(cudaEventRecord(h->ev[0], h->stream));
        MdenseParams dp{mp, h->d_bpats, h->d_mhits, h->mhits_cap};
        if (ntiles > 0) {
            const int grid = (int)std::min<int64_t>(ntiles, h->sm_count);
            if (dense)
                k_filter_mdense<<<grid, kMultiThreads, kMdenseSmem, h->stream>>>(dp, nvec, ntiles);
            else
                k_filter_multi<<<grid, kMultiThreads, kMultiSmem, h->stream>>>(mp, nvec, ntiles);
        }
        CK(cudaEventRecord(h->ev[1], h->stream));
        if (dense)
            k_verify_mhits<<<h->sm_count * 8, kMhThreads, 0, h->stream>>>(dp, h->d_out, h->out_cap, h->d_counters);
        else
            k_verify_multi<<<h->sm_count * 8, kVmThreads, 0, h->stream>>>(mp, h->d_bpats, h->d_out, h->out_cap, h->d_counters);
        CK(cudaGetLastError());
        CK(cudaEventRecord(h->ev[2], h->stream));
        uint32_t cnts[CNT_COUNT];
        CK(cudaMemcpyAsync(cnts, h->d_counters, sizeof cnts, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (cnts[CNT_OVERFLOW]) {  // work list / set / hit list too small for this batch: clean up, let the caller go one by one
            if (!dense) CK(cudaMemsetAsync(h->d_mset, 0, (size_t)h->mset_slots * sizeof(unsigned long long), h->stream));
            CK(cudaStreamSynchronize(h->stream));
            return 1;
        }
        const uint32_t n = cnts[CNT_OUT];
        if (n > h->out_cap) {
            rc = ensure_out_cap(h, n);
            if (rc) return rc;
            continue;
        }
        raw.resize(n);
        if (n) {
            CK(cudaMemcpyAsync(raw.data(), h->d_out, (size_t)n * sizeof(RawRec), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
        }
        n_work = cnts[CNT_CAND];
        cudaEventElapsedTime(&gpu_ms, h->ev[0], h->ev[2]);
        cudaEventElapsedTime(&filter_ms, h->ev[0], h->ev[1]);
        break;
    }
    // split by pattern, consolidate each list on the host
    std::vector<uint32_t> per(cnt, 0);
    for (const RawRec &r : raw) per[(uint32_t)r.ngram >> 8]++;
    for (uint32_t i = 0; i < cnt; i++) {
        fzb_result *res = new (std::nothrow) fzb_result();
        if (!res) return fail(FZB_E_CUDA, "out of host memory");
        res->raw.reserve(per[i]);
        res->stats.route = dense ? 2 : 1;
        res->stats.bytes_scanned = i == 0 ? h->buf_len : 0;  // the haystack is read once for the whole pass
        res->stats.gpu_ms = i == 0 ? gpu_ms : 0.0;
        res->stats.filter_ms = i == 0 ? filter_ms : 0.0;
        res->stats.n_candidates = i == 0 ? n_work : 0;
        res->stats.n_launches = i == 0 ? 2 : 0;
        out[ids[i]] = res;
    }
    for (const RawRec &r : raw) {
        RawRec q = r;
        q.ngram = r.ngram & 0xFF;
        out[ids[(uint32_t)r.ngram >> 8]]->raw.push_back(q);
    }
    for (uint32_t i = 0; i < cnt; i++) {
        fzb_result *res = out[ids[i]];
        res->raw_n = (uint32_t)res->raw.size();
        res->raw_order = 0;
        consolidate_recs(res->raw, res->fin, &res->hulls);
        res->have_fin = true;
    }
    sum->gpu_ms += gpu_ms;
    sum->filter_ms += filter_ms;
    sum->bytes_scanned += h->buf_len;
    sum->n_candidates += n_work;
    sum->n_launches += 2;
    return FZB_OK;
}

// One shared scan for up to 64 LP-route patterns (k_lp_scan_multi / k_lp_verify_multi).  Same return convention
// as batch_pass.
static int batch_pass_lp(fzb_haystack *h, const uint8_t *patterns, const uint32_t *offsets, const uint32_t *ks,
                         const std::vector<uint32_t> &ids, fzb_result **out, fzb_stats *sum) {
    const uint32_t cnt = (uint32_t)ids.size();
    std::vector<BatchPat> pats(cnt);
    std::vector<ulonglong2> lut(256, make_ulonglong2(0ull, 0ull));
    std::vector<uint32_t> pm32((size_t)cnt * 256, 0u);
    LpMultiParams lp{};
    int wmax = 0;
    uint32_t kmax = 0;
    for (uint32_t i = 0; i < cnt; i++) {
        const uint32_t id = ids[i], m = offsets[id + 1] - offsets[id], k = ks[id];
        BatchPat &bp = pats[i];
        memset(&bp, 0, sizeof bp);
        memcpy(bp.P, patterns + offsets[id], m);
        bp.m = (int)m;
        bp.k = (int)k;
        bp.L = 0;
        bp.n_ngrams = 0;
        for (uint32_t j = 0; j < m; j++) {
            lut[bp.P[j]].x |= 1ull << i;
            pm32[(size_t)i * 256 + bp.P[j]] |= 1u << j;
        }
        for (uint32_t j = 0; j <= std::min(k, m - 1); j++) lut[bp.P[j]].y |= 1ull << i;
        const uint32_t bias = 32 - (m - k);  // need = m - k in [1, 31]
        for (int b = 0; b < 6; b++)
            if ((bias >> b) & 1u) lp.bias[b] |= 1ull << i;
        wmax = std::max(wmax, (int)(m + k));
        kmax = std::max(kmax, k);
    }
    int rc = ensure_batch_buffers(h);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (!h->d_lmlut) {
        CK(cudaMalloc(&h->d_lmlut, 256 * sizeof(ulonglong2) + 64 * 256 * sizeof(uint32_t)));  // vectors + match masks
        h->lmlist_cap = (uint32_t)std::min<uint64_t>(1u << 26, std::max<uint64_t>(1u << 22, h->capacity / 16));
        CK(cudaMalloc(&h->d_lmlist, (size_t)h->lmlist_cap * sizeof(unsigned long long)));
        CK(cudaMalloc(&h->d_lmkept, (size_t)h->lmlist_cap * sizeof(unsigned long long)));
        CK(cudaMalloc(&h->d_lmhist, 256 * sizeof(uint32_t)));  // per-pattern counts [64] + kept total [1] | cursors [64]
        CK(cudaFuncSetAttribute(k_lp_scan_multi, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLmSmem));
    }
    detach_pending(h);
    CK(cudaMemcpyAsync(h->d_lmlut, lut.data(), 256 * sizeof(ulonglong2), cudaMemcpyHostToDevice, h->stream));
    uint32_t *d_pm32 = reinterpret_cast<uint32_t *>(h->d_lmlut + 256);
    CK(cudaMemcpyAsync(d_pm32, pm32.data(), pm32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_bpats, pats.data(), pats.size() * sizeof(BatchPat), cudaMemcpyHostToDevice, h->stream));
    lp.H = h->d;
    lp.buf_lo = (int64_t)h->buf_lo;
    lp.buf_len = (int64_t)h->buf_len;
    lp.N = (int64_t)h->global_len;
    lp.lut = h->d_lmlut;
    lp.wmax = wmax;
    lp.pats = h->d_bpats;
    lp.pm32 = d_pm32;
    lp.list = h->d_lmlist;
    lp.list_cap = h->lmlist_cap;
    lp.counters = h->d_counters;
    int per_sm = 2;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_lp_scan_multi, kLmThreads, kLmSmem));
    per_sm = std::max(per_sm, 1);
    const int vgrid = h->sm_count * 4, sim_cap = 256;
    rc = ensure_scratch(h, (uint64_t)vgrid * kLpThreads * 2 * sim_cap);
    if (rc) return rc;
    const uint64_t chunk = 256ull << 20;  // starts per scan: bounds the survivor list
    std::vector<RawRec> raw;
    float gpu_ms = 0.f, filter_ms = 0.f;
    uint64_t n_work = 0;
    for (int attempt = 0;; attempt++) {
        if (attempt == 8) return fail(FZB_E_CUDA, "output buffer kept overflowing");
        h->counters_clean = false;
        CK(cudaMemsetAsync(h->d_counters, 0, CNT_COUNT * sizeof(uint32_t), h->stream));
        CK(cudaEventRecord(h->ev[0], h->stream));
        bool overflow = false;
        float scan_ms = 0.f;
        for (uint64_t lo = h->own_lo; lo < h->own_hi && !overflow; lo += chunk) {
            lp.own_lo = (int64_t)lo;
            lp.own_hi = (int64_t)std::min<uint64_t>(h->own_hi, lo + chunk);
            CK(cudaMemsetAsync(h->d_counters + CNT_LMLIST, 0, 2 * sizeof(uint32_t), h->stream));  // list length + flag
            CK(cudaMemsetAsync(h->d_counters + CNT_LMNEXT, 0, sizeof(uint32_t), h->stream));       // verify work counter
            CK(cudaEventRecord(h->ev[1], h->stream));
            k_lp_scan_multi<<<h->sm_count * per_sm, kLmThreads, kLmSmem, h->stream>>>(lp);
            CK(cudaEventRecord(h->ev[2], h->stream));
            // exact per-pattern windows, then a counting sort by pattern: the scan's list becomes the sorted output
            CK(cudaMemsetAsync(h->d_lmhist, 0, 256 * sizeof(uint32_t), h->stream));
            k_lm_refine<<<h->sm_count * 8, kLmSortThreads, 0, h->stream>>>(lp, h->d_lmkept, h->d_lmhist);
            k_lm_scatter<<<h->sm_count * 8, kLmSortThreads, 0, h->stream>>>(h->d_lmkept, h->d_lmhist, h->d_lmhist + 128,
                                                                              h->d_lmlist);
            if (kmax <= 4)
                k_lp_verify_multi<4><<<vgrid, kLpThreads, 0, h->stream>>>(lp, h->d_lmlist, h->d_lmhist, h->d_scratch, sim_cap,
                                                                          h->d_out, h->out_cap, h->d_counters);
            else
                k_lp_verify_multi<8><<<vgrid, kLpThreads, 0, h->stream>>>(lp, h->d_lmlist, h->d_lmhist, h->d_scratch, sim_cap,
                                                                          h->d_out, h->out_cap, h->d_counters);
            CK(cudaGetLastError());
            uint32_t cnts[CNT_COUNT];
            CK(cudaMemcpyAsync(cnts, h->d_counters, sizeof cnts, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            float ms = 0.f;
            cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]);
            scan_ms += ms;
            n_work += cnts[CNT_LMLIST];
            sum->n_launches += 4;
            if (cnts[CNT_LMWORK] || cnts[CNT_OVERFLOW]) overflow = true;  // survivor list / candidate lists too small
        }
        if (overflow) return 1;
        CK(cudaEventRecord(h->ev[2], h->stream));
        uint32_t cnts[CNT_COUNT];
        CK(cudaMemcpyAsync(cnts, h->d_counters, sizeof cnts, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        const uint32_t n = cnts[CNT_OUT];
        if (n > h->out_cap) {
            rc = ensure_out_cap(h, n);
            if (rc) return rc;
            n_work = 0;
            continue;
        }
        raw.resize(n);
        if (n) {
            CK(cudaMemcpyAsync(raw.data(), h->d_out, (size_t)n * sizeof(RawRec), cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
        }
        cudaEventElapsedTime(&gpu_ms, h->ev[0], h->ev[2]);
        filter_ms = scan_ms;
        break;
    }
    for (uint32_t i = 0; i < cnt; i++) {
        fzb_result *res = new (std::nothrow) fzb_result();
        if (!res) return fail(FZB_E_CUDA, "out of host memory");
        res->stats.route = 3;
        res->stats.bytes_scanned = i == 0 ? h->buf_len : 0;  // the haystack is read once for the whole pass
        res->stats.gpu_ms = i == 0 ? gpu_ms : 0.0;
        res->stats.filter_ms = i == 0 ? filter_ms : 0.0;
        res->stats.n_candidates = i == 0 ? n_work : 0;
        out[ids[i]] = res;
    }
    for (const RawRec &r : raw) {
        RawRec q = r;
        q.ngram = r.ngram & 0xFF;
        out[ids[(uint32_t)r.ngram >> 8]]->raw.push_back(q);
    }
    {  // consolidate the lists in parallel (LP patterns on text have tens of thousands of raw matches each)
        const unsigned nthreads = std::min<unsigned>(8, std::max(1u, std::thread::hardware_concurrency()));
        std::atomic<uint32_t> next{0};
        auto work = [&]() {
            for (uint32_t i = next.fetch_add(1); i < cnt; i = next.fetch_add(1)) {
                fzb_result *res = out[ids[i]];
                res->raw_n = (uint32_t)res->raw.size();
                res->raw_order = 1;
                consolidate_recs(res->raw, res->fin, &res->hulls);
                res->have_fin = true;
            }
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < nthreads; t++) pool.emplace_back(work);
        work();
        for (auto &t : pool) t.join();
    }
    sum->gpu_ms += gpu_ms;
    sum->filter_ms += filter_ms;
    sum->bytes_scanned += h->buf_len;
    sum->n_candidates += n_work;
    return FZB_OK;
}

extern "C" int fzb_search_levenshtein_batch(fzb_haystack *h, const uint8_t *patterns, const uint32_t *offsets,
                                            const uint32_t *max_l_dist, uint32_t count, uint32_t flags,
                                            fzb_result **out, fzb_stats *total) {
    HandleLock handle_lock(h);
    if (!h || !out || (count && (!patterns || !offsets || !max_l_dist))) return fail(FZB_E_INVALID, "NULL argument");
    for (uint32_t i = 0; i < count; i++) out[i] = nullptr;
    for (uint32_t i = 0; i < count; i++)
        if (offsets[i + 1] < offsets[i]) return fail(FZB_E_INVALID, "offsets must be non-decreasing");
    fzb_stats sum{};
    auto cleanup = [&]() {
        for (uint32_t j = 0; j < count; j++) {
            if (out[j]) fzb_result_destroy(out[j]);
            out[j] = nullptr;
        }
    };
    // patterns the shared scan can take: n-gram route, q-sample lemma holds, 4-grams selective on this haystack,
    // short enough for the 64-bit match table; no special flags (forced routes, raw-only, multi-GPU reduction)
    std::vector<uint32_t> shared;
    if (flags == 0 && h->buf_len > 0) {
        for (uint32_t i = 0; i < count; i++) {
            const uint32_t m = offsets[i + 1] - offsets[i], k = max_l_dist[i];
            if (m == 0 || m > (uint32_t)kBatchMaxM || k == 0 || k >= m) continue;
            const uint32_t L = m / (k + 1);
            if (L < 3 || !sampled_filter_applies(m, k, 0)) continue;
            if (check_halo(h, (uint64_t)m + k) != FZB_OK) continue;
            if (!sampled_is_selective(h, m, k, (int)L, (int)(m / L))) continue;
            shared.push_back(i);
        }
    }
    size_t done = 0;
    while (done < shared.size()) {  // passes of bounded size (gram table / posting capacity)
        std::vector<uint32_t> ids;
        uint64_t ngr = 0;
        while (done < shared.size() && ids.size() < kMaxBatchPats) {
            const uint32_t m = offsets[shared[done] + 1] - offsets[shared[done]];
            if (ngr + (m - 3) > kMaxBatchGrams) break;
            ngr += m - 3;
            ids.push_back(shared[done++]);
        }
        if (ids.size() < 2) {  // not worth a shared pass
            done -= ids.size();
            break;
        }
        int rc = batch_pass(h, patterns, offsets, max_l_dist, ids, out, &sum, false);
        if (rc < 0) {
            cleanup();
            return rc;
        }
        if (rc > 0) {  // overflow: these patterns fall through to the one-by-one path
            for (uint32_t id : ids)
                if (out[id]) {
                    fzb_result_destroy(out[id]);
                    out[id] = nullptr;
                }
        }
    }
    // the n-gram-route patterns the lemma does not cover share a scan of their own (n-gram prefixes at every position)
    std::vector<uint32_t> dense_ids;
    if (flags == 0 && h->buf_len > 0 && sample_collision_prob(h) == FZB_OK) {
        double expect = 0.0;  // expected prefix hits per haystack position
        uint32_t dense_grams = 0;
        const double c3 = h->coll_prob * h->coll_prob * h->coll_prob;
        for (uint32_t i = 0; i < count && dense_ids.size() < kMaxBatchPats; i++) {
            if (out[i]) continue;
            const uint32_t m = offsets[i + 1] - offsets[i], k = max_l_dist[i];
            if (m == 0 || m > (uint32_t)kBatchMaxM || k == 0 || k >= m) continue;
            const uint32_t L = m / (k + 1);
            if (L < 3 || m - L > 32 || m + 2 * k + 12 > (uint32_t)kMhSlotBytes) continue;
            if (check_halo(h, (uint64_t)m + k) != FZB_OK) continue;
            if (expect + (m / L) * c3 > 0.02) continue;  // (low-entropy text: prefixes hit everywhere -> one by one)
            if (dense_grams + m / L > kMaxBatchGrams) continue;  // prefix table capacity
            expect += (m / L) * c3;
            dense_grams += m / L;
            dense_ids.push_back(i);
        }
    }
    if (dense_ids.size() >= 2) {
        int rc = batch_pass(h, patterns, offsets, max_l_dist, dense_ids, out, &sum, true);
        if (rc < 0) {
            cleanup();
            return rc;
        }
        if (rc > 0)
            for (uint32_t id : dense_ids)
                if (out[id]) {
                    fzb_result_destroy(out[id]);
                    out[id] = nullptr;
                }
    }
    // LP-route patterns (m // (k+1) < 3) share scans of 64 patterns each (bit-sliced window counters)
    std::vector<uint32_t> lp_ids;
    if (flags == 0 && h->buf_len > 0) {
        for (uint32_t i = 0; i < count; i++) {
            if (out[i]) continue;
            const uint32_t m = offsets[i + 1] - offsets[i], k = max_l_dist[i];
            if (m == 0 || k == 0 || k >= m || m / (k + 1) >= 3) continue;
            if (m > 31 || k > 8 || m + k > 31) continue;  // automaton masks / 6-bit window counters
            if (check_halo(h, (uint64_t)m + k) != FZB_OK) continue;
            lp_ids.push_back(i);
        }
    }
    for (size_t first = 0; first + 2 <= lp_ids.size(); first += 64) {
        std::vector<uint32_t> ids(lp_ids.begin() + first, lp_ids.begin() + std::min(lp_ids.size(), first + 64));
        if (ids.size() < 2) break;
        int rc = batch_pass_lp(h, patterns, offsets, max_l_dist, ids, out, &sum);
        if (rc < 0) {
            cleanup();
            return rc;
        }
        if (rc > 0)
            for (uint32_t id : ids)
                if (out[id]) {
                    fzb_result_destroy(out[id]);
                    out[id] = nullptr;
                }
    }
    for (uint32_t i = 0; i < count; i++) {
        if (out[i]) continue;
        int rc = fzb_search_levenshtein(h, patterns + offsets[i], offsets[i + 1] - offsets[i], max_l_dist[i], flags,
                                        &out[i]);
        if (rc) {
            cleanup();
            return rc;
        }
        sum.gpu_ms += out[i]->stats.gpu_ms;
        sum.filter_ms += out[i]->stats.filter_ms;
        sum.bytes_scanned += out[i]->stats.bytes_scanned;
        sum.n_candidates += out[i]->stats.n_candidates;
        sum.n_launches += out[i]->stats.n_launches;
    }
    sum.route = 7;  // batch
    if (total) *total = sum;
    return FZB_OK;
}

extern "C" int fzb_search_exact(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t flags,
                                fzb_result **out) {
    HandleLock handle_lock(h);
    fzb_result *res;
    int rc = make_result(out, &res);
    if (rc) return rc;
    rc = check_pattern(h, pattern, m, flags);
    if (rc == FZB_E_INVALID && h) rc = fail(FZB_E_INVALID, "subsequence must not be empty");
    if (rc == FZB_OK) rc = search_lev_ngrams(h, pattern, m, 0, flags, res, 2);
    if (rc) {
        fzb_result_destroy(res);
        return rc;
    }
    res->unconsolidated = true;  // ExactSearch.consolidate_matches is the base no-op (common.py:198-205)
    if (flags & FZB_F_GLOBAL) {
        rc = finish_global(h, res);
        if (rc) {
            fzb_result_destroy(res);
            return rc;
        }
    }
    *out = res;
    return FZB_OK;
}

// search_exact(subsequence, sequence, start_index, end_index) (search_exact.py:22-56): the occurrences lying wholly
// inside [start, end).  The window is a VIEW of the resident buffer treated like a shard of a sequence that ends
// at `end` (anchors owned from `start`, occurrences clipped at the view's global end), so the bytes outside the
// window are not scanned.
extern "C" int fzb_search_exact_window(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint64_t start,
                                       uint64_t end, uint32_t flags, fzb_result **out) {
    HandleLock handle_lock(h);
    if (!h || !out) return fail(FZB_E_INVALID, "NULL argument");
    *out = nullptr;
    if (flags & FZB_F_GLOBAL) return fail(FZB_E_INVALID, "windowed exact search is per handle");
    if (h->buf_lo != 0 || h->global_len != h->buf_len || h->own_lo != 0 || h->own_hi != h->buf_len)
        return fail(FZB_E_INVALID, "windowed exact search needs a whole (unsharded) sequence");
    // clamp (search_exact.py:29-30): start into [0, n], end into [start, n]
    start = std::min<uint64_t>(start, h->global_len);
    end = std::max<uint64_t>(start, std::min<uint64_t>(end, h->global_len));
    if (end - start < m) {  // no room for an occurrence (also: the empty window): nothing to launch
        int rc0 = check_pattern(h, pattern, m, flags);
        if (rc0 == FZB_E_INVALID) rc0 = fail(FZB_E_INVALID, "subsequence must not be empty");
        if (rc0) return rc0;
        fzb_result *res;
        rc0 = make_result(out, &res);
        if (rc0) return rc0;
        res->unconsolidated = true;
        res->have_fin = true;
        *out = res;
        return FZB_OK;
    }
    struct Geometry {
        uint8_t *d;
        uint64_t buf_len, buf_lo, own_lo, own_hi, padded_len, global_len;
        double coll_prob;
    } const saved{h->d, h->buf_len, h->buf_lo, h->own_lo, h->own_hi, h->padded_len, h->global_len, h->coll_prob};
    // the view starts a halo before the window (the shard geometry check of the search wants one on both sides;
    // the right one ends at the view's global end), on a 128-byte boundary of the buffer
    const uint64_t halo = round_up((uint64_t)m, 128) + 128;
    const uint64_t vlo = (start > halo ? start - halo : 0) / 128 * 128;
    h->d = saved.d + vlo;
    h->buf_lo = vlo;
    h->buf_len = end - vlo;
    h->padded_len = round_up(h->buf_len, 128) + 128;
    h->global_len = end;
    h->own_lo = start;
    h->own_hi = end;
    h->coll_prob = -1.0;
    const int rc = fzb_search_exact(h, pattern, m, flags, out);
    if (rc == FZB_OK && *out) (*out)->fetch_raw();  // the records leave the view's buffers before the geometry changes back
    h->d = saved.d;
    h->buf_len = saved.buf_len;
    h->buf_lo = saved.buf_lo;
    h->own_lo = saved.own_lo;
    h->own_hi = saved.own_hi;
    h->padded_len = saved.padded_len;
    h->global_len = saved.global_len;
    h->coll_prob = saved.coll_prob;
    return rc;
}

// TMA descriptors of the buffer viewed as rows of 128 bytes (k_hamming_count): box 256 rows / 8 rows,
// SWIZZLE_128B, out-of-bounds rows (the halo before row 0, the tail) read as zeros.
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_row_maps(fzb_haystack *h, CUtensorMap *map256, CUtensorMap *map8) {
    // resolved once per process; a function-local static's initialisation is thread-safe (handles of different
    // threads get here concurrently)
    static const EncodeTiledFn encode = []() -> EncodeTiledFn {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
        return (fn && q == cudaDriverEntryPointSuccess) ? (EncodeTiledFn)fn : nullptr;
    }();
    if (!encode) {
        cudaGetLastError();
        return fail(FZB_E_CUDA, "cuTensorMapEncodeTiled not available");
    }
    const cuuint64_t rows = h->padded_len / kHcRowBytes;  // whole rows inside the allocation
    const cuuint64_t dims[2] = {(cuuint64_t)kHcRowBytes, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kHcRowBytes};
    const cuuint32_t estr[2] = {1, 1};
    for (int which = 0; which < 2; which++) {
        const cuuint32_t box[2] = {(cuuint32_t)kHcRowBytes, which == 0 ? 256u : (cuuint32_t)kHcHaloRows};
        CUresult r = encode(which == 0 ? map256 : map8, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, h->d, dims, strides, box,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(FZB_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    }
    return FZB_OK;
}

// Counter layout of k_hamming_count (ham_recur.h).  FZB_HAM_COUNTERS=nibble|sliced overrides the default.
// -> 0 nibble fields / 1 three slices / 2 two slices (thresholds <= 4 only)
static int ham_counter_layout(int threshold) {  // (read per search: a probe can flip it between two searches)
    const char *e = getenv("FZB_HAM_COUNTERS");
    if (e && !strcmp(e, "nibble")) return 0;
    if (e && !strcmp(e, "sliced3")) return 1;
    // measured on 4 GiB of DNA, m = 32, k = 3: 0.881 ms (three slices) vs 0.948 ms (nibble fields)
    return threshold <= 4 ? 2 : 1;
}

extern "C" int fzb_search_hamming(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t k,
                                  uint32_t flags, fzb_result **out) {
    HandleLock handle_lock(h);
    fzb_result *res;
    int rc = make_result(out, &res);
    if (rc) return rc;
    rc = check_pattern(h, pattern, m, flags);
    if (rc == FZB_OK) rc = check_halo(h, m);
    if (rc == FZB_OK) {
        rc = [&]() -> int {
            ScanParams p;
            fill_params(h, pattern, m, p);
            p.k = (int)std::min<uint32_t>(k, m);
            CK(cudaSetDevice(h->device));
            res->stats.route = 4;
            res->stats.bytes_scanned = h->buf_len;
            // counting q-sample filter needs W = floor((m-3)/4) >= k+1 aligned words and 4-bit fields (k <= 7)
            const bool counting = !(flags & FZB_F_FORCE_DENSE) && (int)m >= 4 * p.k + 7 && p.k <= 7 && h->buf_len > 0;
            HamCountParams hp{};
            CUtensorMap map256, map8;
            if (counting) {
                hp.Wc = std::min<int>((int)(m - 3) / 4, 8);
                hp.bias = 8 - (hp.Wc - p.k);
                hp.nrows = (int64_t)(round_up(h->buf_len, kHcRowBytes) / kHcRowBytes);
                int r3 = make_row_maps(h, &map256, &map8);
                if (r3) return r3;
                CK(cudaFuncSetAttribute(k_hamming_count<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHcSmem));
                CK(cudaFuncSetAttribute(k_hamming_count<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHcSmem));
                CK(cudaFuncSetAttribute(k_hamming_count<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHcSmem));
            }
            const int layout = counting ? ham_counter_layout(hp.Wc - p.k) : 0;
            if (layout == 2) hp.bias = 4 - (hp.Wc - p.k);
            bool bitmap_mode = false;
            PostPlan plan{2, (flags & FZB_F_GLOBAL) != 0};  // FINAL == RAW in (start, end, dist) order, ordered by k_post
        retry_bitmap:
            int r2 = run_emitting(h, res, [&]() -> int {
                if (counting) {
                    const int64_t ntiles = (hp.nrows + kHcThreads - 1) / kHcThreads;
                    const int grid = (int)std::min<int64_t>(ntiles, (int64_t)h->sm_count * 2);
                    if (layout == 2)
                        k_hamming_count<2><<<grid, kHcThreads, kHcSmem, h->stream>>>(p, hp, map256, map8);
                    else if (layout == 1)
                        k_hamming_count<1><<<grid, kHcThreads, kHcSmem, h->stream>>>(p, hp, map256, map8);
                    else
                        k_hamming_count<0><<<grid, kHcThreads, kHcSmem, h->stream>>>(p, hp, map256, map8);
                    CK(cudaEventRecord(h->ev[1], h->stream));
                    h->ev1_recorded = true;
                    // one verify launch: the granule work list -- or, after it overflowed, the whole bitmap
                    k_verify_ham<<<h->sm_count * 4, kVerifyThreads, 0, h->stream>>>(
                        p, h->bitmap_words, h->d_glist, p.glist_cap, bitmap_mode ? 1 : 0, h->d_out, h->out_cap,
                        h->d_counters);
                    res->stats.n_launches += 1;
                } else {
                    k_hamming_scan<<<h->sm_count * 8, kHamThreads, 0, h->stream>>>(p, h->d_out, h->out_cap,
                                                                                   h->d_counters);
                }
                res->stats.n_launches++;
                return FZB_OK;
            }, plan);
            if (r2) return r2;
            if (counting && !bitmap_mode && h->h_counters[CNT_GRAN] > p.glist_cap) {  // work list overflowed (see search_lev_ngrams)
                bitmap_mode = true;
                plan.global = false;
                p.glist_cap = 0;
                res->fetch_raw();
                res->raw.clear();
                res->raw_n = 0;
                res->fin.clear();
                goto retry_bitmap;
            }
            res->raw_order = 1;
            return FZB_OK;
        }();
    }
    if (rc) {
        fzb_result_destroy(res);
        return rc;
    }
    res->unconsolidated = true;
    if (flags & FZB_F_GLOBAL) {
        rc = finish_global(h, res);
        if (rc) {
            fzb_result_destroy(res);
            return rc;
        }
    }
    *out = res;
    return FZB_OK;
}

extern "C" int fzb_search_generic(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs,
                                  uint32_t max_ins, uint32_t max_dels, uint32_t max_l, uint32_t flags,
                                  fzb_result **out) {
    HandleLock handle_lock(h);
    fzb_result *res;
    int rc = make_result(out, &res);
    if (rc) return rc;
    rc = check_pattern(h, pattern, m, flags);
    if (rc == FZB_OK) {
        // find_near_matches_generic (generic_search.py:25-54)
        const bool want_final = !(flags & FZB_F_NO_FINAL);
        if (max_l == 0 && !(flags & (FZB_F_FORCE_LP | FZB_F_FORCE_NGRAMS))) {
            rc = search_lev_ngrams(h, pattern, m, 0, flags, res, want_final ? 1 : 0);
        } else {
            bool ngrams = m / (max_l + 1) >= 3;
            if (flags & FZB_F_FORCE_NGRAMS) ngrams = true;
            if (flags & FZB_F_FORCE_LP) ngrams = false;
            rc = search_generic(h, pattern, m, max_subs, max_ins, max_dels, max_l, ngrams, flags, res,
                                want_final ? 1 : 0);
        }
        if (rc == FZB_OK && want_final && (flags & FZB_F_GLOBAL)) rc = finish_global(h, res);
    }
    if (rc) {
        fzb_result_destroy(res);
        return rc;
    }
    *out = res;
    return FZB_OK;
}

// One cached workspace per device for the one-shot call: the analogue of the reference's reusable
// chunk buffer (__init__.py:141-145) -- a call then costs one H2D copy plus the kernels instead of
// a 4 GiB cudaMalloc/cudaFree pair and a dozen small allocations.
static std::mutex g_ws_mutex;
static fzb_haystack *g_ws[64];

extern "C" void fzb_release_workspace(void) {
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    for (auto &h : g_ws) {
        if (h) fzb_haystack_destroy(h);
        h = nullptr;
    }
}

extern "C" int fzb_find_near_matches(const uint8_t *pattern, uint32_t m, const uint8_t *haystack, uint64_t n,
                                     uint32_t max_subs, uint32_t max_ins, uint32_t max_dels, uint32_t max_l,
                                     int device, fzb_result **out) {
    if (!out) return fail(FZB_E_INVALID, "out is NULL");
    *out = nullptr;
    if (device < 0 || device >= 64 || device >= fzb_device_count())
        return fail(FZB_E_CUDA, "CUDA device %d not available (%d devices)", device, fzb_device_count());
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    fzb_haystack *&h = g_ws[device];
    if (!h || round_up(n, 128) + 128 > h->capacity) {
        if (h) fzb_haystack_destroy(h);
        h = nullptr;
        const uint64_t cap = std::max<uint64_t>(n + n / 8, 1u << 20);  // head-room: repeated calls with growing inputs
        int rc = fzb_haystack_alloc(cap, 0, cap, 0, cap, device, &h, nullptr);
        if (rc) return rc;
    }
    int rc = fzb_haystack_upload(h, haystack, n);
    if (rc) return rc;
    // choose_search_class (__init__.py:60-83) on normalised limits
    if (max_l == 0)
        rc = fzb_search_exact(h, pattern, m, 0, out);
    else if (max_ins == 0 && max_dels == 0)
        rc = fzb_search_hamming(h, pattern, m, std::min(max_l, max_subs), 0, out);
    else if (max_l <= std::min(max_subs, std::min(max_ins, max_dels)))
        rc = fzb_search_levenshtein(h, pattern, m, max_l, 0, out);
    else
        rc = fzb_search_generic(h, pattern, m, max_subs, max_ins, max_dels, max_l, 0, out);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// Segmented search: one pattern over the segments [offsets[i], offsets[i+1]) of one resident buffer, each searched as
// a whole sequence (seg_kernels.cuh).  Short segments: one pass of five kernels whatever their number; long ones:
// copied device-to-device into a workspace handle and searched with the single-sequence entry points.
// ------------------------------------------------------------------------------------------------
static void seg_free(fzb_haystack *h) {
    if (h->seg_ws) fzb_haystack_destroy(h->seg_ws);
    h->seg_ws = nullptr;
    if (h->d_seg_offsets) cudaFree(h->d_seg_offsets);
    if (h->d_seg_cnt) cudaFree(h->d_seg_cnt);
    if (h->d_seg_off) cudaFree(h->d_seg_off);
    if (h->d_seg_cur) cudaFree(h->d_seg_cur);
    if (h->h_seg_cnt) cudaFreeHost(h->h_seg_cnt);
    h->d_seg_offsets = nullptr;
    h->d_seg_cnt = h->d_seg_off = h->d_seg_cur = h->h_seg_cnt = nullptr;
    h->seg_count_cap = 0;
    if (h->d_seg_keys) cudaFree(h->d_seg_keys);
    if (h->h_seg_raw) cudaFreeHost(h->h_seg_raw);
    if (h->h_seg_fin) cudaFreeHost(h->h_seg_fin);
    h->d_seg_keys = h->h_seg_raw = h->h_seg_fin = nullptr;
    h->seg_rec_cap = 0;
    if (h->h_seg_hdr) cudaFreeHost(h->h_seg_hdr);
    h->h_seg_hdr = nullptr;
}

static int ensure_seg_buffers(fzb_haystack *h, uint64_t count, uint64_t recs) {
    const unsigned mapped = cudaHostAllocMapped | cudaHostAllocPortable;
    if (!h->h_seg_hdr) CK(cudaHostAlloc(&h->h_seg_hdr, 4 * sizeof(uint32_t), mapped));
    if (count > h->seg_count_cap) {
        if (h->d_seg_offsets) CK(cudaFree(h->d_seg_offsets));
        if (h->d_seg_cnt) CK(cudaFree(h->d_seg_cnt));
        if (h->d_seg_off) CK(cudaFree(h->d_seg_off));
        if (h->d_seg_cur) CK(cudaFree(h->d_seg_cur));
        if (h->h_seg_cnt) CK(cudaFreeHost(h->h_seg_cnt));
        h->d_seg_offsets = nullptr;
        h->d_seg_cnt = h->d_seg_off = h->d_seg_cur = h->h_seg_cnt = nullptr;
        h->seg_count_cap = 0;
        const uint64_t cap = std::max<uint64_t>(count, 1u << 12);
        CK(cudaMalloc(&h->d_seg_offsets, (cap + 1) * sizeof(uint64_t)));
        CK(cudaMalloc(&h->d_seg_cnt, 2 * cap * sizeof(uint32_t)));
        CK(cudaMalloc(&h->d_seg_off, (cap + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&h->d_seg_cur, cap * sizeof(uint32_t)));
        CK(cudaHostAlloc(&h->h_seg_cnt, 2 * cap * sizeof(uint32_t), cudaHostAllocPortable));
        h->seg_count_cap = cap;
    }
    if (recs > h->seg_rec_cap) {
        if (h->d_seg_keys) CK(cudaFree(h->d_seg_keys));
        if (h->h_seg_raw) CK(cudaFreeHost(h->h_seg_raw));
        if (h->h_seg_fin) CK(cudaFreeHost(h->h_seg_fin));
        h->d_seg_keys = h->h_seg_raw = h->h_seg_fin = nullptr;
        h->seg_rec_cap = 0;
        CK(cudaMalloc(&h->d_seg_keys, recs * sizeof(uint64_t)));
        CK(cudaHostAlloc(&h->h_seg_raw, recs * sizeof(uint64_t), mapped));
        CK(cudaHostAlloc(&h->h_seg_fin, recs * sizeof(uint64_t), mapped));
        h->seg_rec_cap = recs;
    }
    return FZB_OK;
}

static RawRec seg_decode(uint64_t key) {  // canonical_key (kernels.cuh) -> record
    RawRec r;
    r.start = (int64_t)(key >> 18);
    r.end = r.start + (int64_t)((key >> 8) & 0x3FFu);
    r.dist = (int32_t)(key & 0xFFu);
    r.idx = -1;
    r.ngram = -1;
    return r;
}

// choose_search_class (__init__.py:60-83) on normalised limits, as fzb_find_near_matches dispatches
static int seg_search_whole(fzb_haystack *w, const uint8_t *pattern, uint32_t m, uint32_t max_subs, uint32_t max_ins,
                            uint32_t max_dels, uint32_t max_l, fzb_result **r) {
    if (max_l == 0) return fzb_search_exact(w, pattern, m, 0, r);
    if (max_ins == 0 && max_dels == 0) return fzb_search_hamming(w, pattern, m, std::min(max_l, max_subs), 0, r);
    if (max_l <= std::min(max_subs, std::min(max_ins, max_dels))) return fzb_search_levenshtein(w, pattern, m, max_l, 0, r);
    return fzb_search_generic(w, pattern, m, max_subs, max_ins, max_dels, max_l, 0, r);
}

// A segment longer than kSegMaxBytes: device-to-device into the workspace handle, searched there as a whole sequence
// (the HBM-speed filters of the single-sequence routes); its lists are appended to res.
static int seg_search_long(fzb_haystack *h, uint64_t lo, uint64_t n, const uint8_t *pattern, uint32_t m,
                           uint32_t max_subs, uint32_t max_ins, uint32_t max_dels, uint32_t max_l, fzb_result *res,
                           uint64_t *n_raw, uint64_t *n_fin) {
    if (!h->seg_ws || round_up(n, 128) + 128 > h->seg_ws->capacity) {
        if (h->seg_ws) fzb_haystack_destroy(h->seg_ws);
        h->seg_ws = nullptr;
        const uint64_t cap = std::max<uint64_t>(n + n / 8, 1u << 20);
        int rc = fzb_haystack_alloc(cap, 0, cap, 0, cap, h->device, &h->seg_ws, nullptr);
        if (rc) return rc;
    }
    fzb_haystack *w = h->seg_ws;
    w->buf_len = w->global_len = w->own_hi = n;
    w->own_lo = 0;
    w->padded_len = round_up(n, 128) + 128;
    w->coll_prob = -1.0;
    CK(cudaMemsetAsync(w->d + n, 0, w->padded_len - n, w->stream));
    CK(cudaMemcpyAsync(w->d, h->d + lo, n, cudaMemcpyDeviceToDevice, w->stream));
    fzb_result *r = nullptr;
    int rc = seg_search_whole(w, pattern, m, max_subs, max_ins, max_dels, max_l, &r);
    if (rc) return rc;
    r->order_raw();
    std::vector<RawRec> raw = r->raw;
    sort_canonical(raw);
    for (RawRec &x : raw) {
        x.idx = -1;
        x.ngram = -1;
    }
    res->raw.insert(res->raw.end(), raw.begin(), raw.end());
    res->fin.insert(res->fin.end(), r->fin.begin(), r->fin.end());
    *n_raw = raw.size();
    *n_fin = r->fin.size();
    res->stats.n_launches += r->stats.n_launches;
    res->stats.n_candidates += r->stats.n_candidates;
    fzb_result_destroy(r);
    return FZB_OK;
}

static int search_segments(fzb_haystack *h, const uint8_t *pattern, uint32_t m, const uint64_t *offsets,
                           uint64_t count, uint32_t max_subs, uint32_t max_ins, uint32_t max_dels, uint32_t max_l,
                           uint32_t flags, fzb_result *res) {
    int rc = check_pattern(h, pattern, m);
    if (rc) return rc;
    if (flags & FZB_F_GLOBAL) return fail(FZB_E_INVALID, "a segmented search is per handle (no FZB_F_GLOBAL)");
    if (h->buf_lo != 0 || h->global_len != h->buf_len || h->own_lo != 0 || h->own_hi != h->buf_len)
        return fail(FZB_E_INVALID, "a segmented search needs a whole (unsharded) sequence");
    if (count > FZB_SEG_MAX_COUNT) return fail(FZB_E_UNSUPPORTED, "more than %u segments in one call", FZB_SEG_MAX_COUNT);
    if (!offsets) return fail(FZB_E_INVALID, "offsets is NULL");
    if (offsets[count] > h->global_len) return fail(FZB_E_INVALID, "offsets[count] beyond the end of the sequence");
    uint64_t short_bytes = 0;
    for (uint64_t i = 0; i < count; i++) {
        if (offsets[i] > offsets[i + 1]) return fail(FZB_E_INVALID, "offsets must not decrease");
        if (offsets[i + 1] - offsets[i] <= (uint64_t)kSegMaxBytes) short_bytes += offsets[i + 1] - offsets[i];
    }
    res->segmented = true;
    res->unconsolidated = max_l == 0 || (max_ins == 0 && max_dels == 0);
    res->raw_ordered = true;  // segment-major, (start, end, dist) within a segment
    res->raw_order = 1;
    res->have_fin = true;
    res->stats.route = 8;
    res->stats.bytes_scanned = short_bytes;
    res->seg_n[FZB_RAW].assign(count, 0);
    res->seg_n[FZB_FINAL].assign(count, 0);
    if (count == 0) return FZB_OK;
    // the route depends on m and the limits only (fzb_search_levenshtein / _hamming / _generic / _exact)
    SegParams sp;
    memset(&sp, 0, sizeof sp);
    memcpy(sp.P, pattern, m);
    sp.m = (int)m;
    int route;
    if (max_l == 0) {
        route = SEG_EXACT;
    } else if (max_ins == 0 && max_dels == 0) {
        route = SEG_HAMMING;
        sp.k = (int)std::min(std::min(max_l, max_subs), m);
    } else if (max_l <= std::min(max_subs, std::min(max_ins, max_dels))) {
        const uint32_t k = std::min(max_l, m);  // every k >= m takes the same branch (levenshtein.py:62-65)
        sp.k = (int)k;
        route = m / (k + 1) >= 3 ? SEG_LEV_NGRAMS : SEG_LEV_LP;
    } else {
        const bool ngrams = m / (max_l + 1) >= 3;
        uint32_t l = max_l;  // the LP clamp and the limits of search_generic
        if (!ngrams) l = (uint32_t)std::min<uint64_t>(l, (uint64_t)m + std::min(max_ins, l));
        if (l > 63) return fail(FZB_E_UNSUPPORTED, "max_l_dist > 63 is not supported by the generic search");
        sp.k = (int)l;
        sp.max_subs = (int)std::min(max_subs, l);
        sp.max_ins = (int)std::min(max_ins, l);
        sp.max_dels = (int)std::min(max_dels, l);
        route = ngrams ? SEG_GEN_NGRAMS : SEG_GEN_LP;
    }
    if (route == SEG_LEV_NGRAMS || route == SEG_GEN_NGRAMS) {
        sp.L = (int)m / (sp.k + 1);
        sp.n_ngrams = (int)m / sp.L;
    }
    const int vm = route == SEG_LEV_NGRAMS ? verify_mode((int)m, sp.L) : 0;
    const bool lp = route == SEG_LEV_LP || route == SEG_GEN_LP || route == SEG_GEN_NGRAMS;
    const int consolidate = res->unconsolidated ? 0 : 1;
    CK(cudaSetDevice(h->device));
    detach_pending(h);  // the records of this search overwrite the output buffer an earlier result may point at
    h->counters_clean = false;
    rc = ensure_seg_buffers(h, count, h->out_cap);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->d_seg_offsets, offsets, (count + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
    sp.H = h->d;
    sp.offsets = h->d_seg_offsets;
    sp.count = (uint32_t)count;
    sp.counters = h->d_counters;
    const int grid = (int)std::min<uint64_t>((uint64_t)h->sm_count * 8, (count + kSegWarps - 1) / kSegWarps);
    const int post_grid = (int)std::min<uint64_t>((uint64_t)h->sm_count * 4, (count + 32 * kSegWarps - 1) / (32 * kSegWarps));
    int cap = lp ? 256 : 0;
    uint32_t n = 0;
    for (int attempt = 0;; attempt++) {
        if (attempt == 16) return fail(FZB_E_CUDA, "output buffer kept overflowing");
        if (lp) {
            rc = ensure_scratch(h, (uint64_t)grid * kSegThreads * 2 * (uint64_t)cap);
            if (rc) return rc;
        }
        rc = ensure_seg_buffers(h, count, h->out_cap);
        if (rc) return rc;
        cudaStream_t st = h->stream;
        CK(cudaMemsetAsync(h->d_counters, 0, CNT_COUNT * sizeof(uint32_t), st));
        CK(cudaMemsetAsync(h->d_seg_cnt, 0, count * sizeof(uint32_t), st));
        CK(cudaEventRecord(h->ev[0], st));
        uint32_t *scr = h->d_scratch;
        switch (route) {
        case SEG_EXACT: k_seg_search<SEG_EXACT, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap); break;
        case SEG_HAMMING: k_seg_search<SEG_HAMMING, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap); break;
        case SEG_LEV_LP: k_seg_search<SEG_LEV_LP, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap); break;
        case SEG_GEN_LP: k_seg_search<SEG_GEN_LP, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap); break;
        case SEG_GEN_NGRAMS: k_seg_search<SEG_GEN_NGRAMS, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap); break;
        default:
            if (vm == 0)
                k_seg_search<SEG_LEV_NGRAMS, 0><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap);
            else if (vm == 1)
                k_seg_search<SEG_LEV_NGRAMS, 1><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap);
            else
                k_seg_search<SEG_LEV_NGRAMS, 2><<<grid, kSegThreads, 0, st>>>(sp, scr, cap, h->d_out, h->out_cap);
        }
        k_seg_hist<<<h->sm_count * 4, kSegSortThreads, 0, st>>>(h->d_out, h->out_cap, h->d_counters, h->d_seg_cnt);
        k_seg_scan<<<1, kPostThreads, 0, st>>>(h->d_seg_cnt, (uint32_t)count, h->d_counters, h->out_cap, h->d_seg_off,
                                               h->d_seg_cur, h->h_seg_hdr);
        k_seg_scatter<<<h->sm_count * 4, kSegSortThreads, 0, st>>>(h->d_out, h->out_cap, h->d_counters, h->d_seg_cur,
                                                                   h->d_seg_keys);
        k_seg_post<<<post_grid, kSegThreads, 0, st>>>(h->d_seg_cnt, h->d_seg_off, (uint32_t)count, h->d_seg_keys,
                                                      h->d_counters, h->out_cap, consolidate, h->d_seg_cnt + count,
                                                      h->h_seg_raw, h->h_seg_fin);
        CK(cudaGetLastError());
        res->stats.n_launches += 5;
        CK(cudaMemcpyAsync(h->h_seg_cnt, h->d_seg_cnt, 2 * count * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(h->ev[2], st));
        CK(cudaStreamSynchronize(st));  // the only synchronisation of an attempt
        n = h->h_seg_hdr[0];
        if (n > h->out_cap) {
            rc = ensure_out_cap(h, n);
            if (rc) return rc;
            continue;
        }
        if (h->h_seg_hdr[1]) {  // an LP candidate list overflowed: more room per lane
            if (cap >= (1 << 16)) return fail(FZB_E_UNSUPPORTED, "candidate explosion: more than 65536 live candidates for one start");
            cap *= 8;
            continue;
        }
        break;
    }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev[0], h->ev[2]);
    res->stats.gpu_ms = res->stats.filter_ms = ms;
    res->stats.n_candidates = count;
    const uint32_t *raw_n = h->h_seg_cnt, *fin_n = h->h_seg_cnt + count;
    res->raw.reserve(n);
    uint64_t off = 0;
    std::vector<RawRec> one;
    for (uint64_t s = 0; s < count; s++) {
        const uint64_t len = offsets[s + 1] - offsets[s];
        if (len > (uint64_t)kSegMaxBytes) {
            rc = seg_search_long(h, offsets[s], len, pattern, m, max_subs, max_ins, max_dels, max_l, res,
                                 &res->seg_n[FZB_RAW][s], &res->seg_n[FZB_FINAL][s]);
            if (rc) return rc;
            continue;
        }
        const uint32_t nr = raw_n[s];
        const size_t r0 = res->raw.size();
        for (uint32_t i = 0; i < nr; i++) res->raw.push_back(seg_decode(h->h_seg_raw[off + i]));
        if (fin_n[s] == kSegNoFinal) {  // too many records for a warp: sorted and consolidated here
            std::sort(res->raw.begin() + r0, res->raw.end(), [](const RawRec &a, const RawRec &b) {
                if (a.start != b.start) return a.start < b.start;
                if (a.end != b.end) return a.end < b.end;
                return a.dist < b.dist;
            });
        }
        if (!consolidate) {
            res->fin.insert(res->fin.end(), res->raw.begin() + r0, res->raw.end());
            res->seg_n[FZB_FINAL][s] = nr;
        } else if (fin_n[s] == kSegNoFinal) {
            consolidate_recs(std::vector<RawRec>(res->raw.begin() + r0, res->raw.end()), one);
            res->fin.insert(res->fin.end(), one.begin(), one.end());
            res->seg_n[FZB_FINAL][s] = one.size();
        } else {
            for (uint32_t g = 0; g < fin_n[s]; g++) res->fin.push_back(seg_decode(h->h_seg_fin[off + g]));
            res->seg_n[FZB_FINAL][s] = fin_n[s];
        }
        res->seg_n[FZB_RAW][s] = nr;
        off += nr;
    }
    res->raw_n = (uint32_t)res->raw.size();
    return FZB_OK;
}

extern "C" int fzb_search_segments(fzb_haystack *h, const uint8_t *pattern, uint32_t m, const uint64_t *offsets,
                                   uint64_t count, uint32_t max_subs, uint32_t max_ins, uint32_t max_dels,
                                   uint32_t max_l_dist, uint32_t flags, fzb_result **out) {
    HandleLock handle_lock(h);
    fzb_result *res;
    int rc = make_result(out, &res);
    if (rc) return rc;
    rc = search_segments(h, pattern, m, offsets, count, max_subs, max_ins, max_dels, max_l_dist, flags, res);
    if (rc) {
        fzb_result_destroy(res);
        return rc;
    }
    *out = res;
    return FZB_OK;
}

extern "C" int fzb_result_segment_counts(const fzb_result *r, int which, uint64_t *counts) {
    if (!r) return fail(FZB_E_INVALID, "result is NULL");
    if (!r->segmented) return fail(FZB_E_INVALID, "not the result of a segmented search");
    const std::vector<uint64_t> &v = r->seg_n[which == FZB_RAW ? FZB_RAW : FZB_FINAL];
    if (!counts && !v.empty()) return fail(FZB_E_INVALID, "counts is NULL");
    std::copy(v.begin(), v.end(), counts);
    return FZB_OK;
}

// ------------------------------------------------------------------------------------------------
// has_near_match: "is there any match?" with early termination.  The reference's has_near_match_* helpers
// (substitutions_only.py:18-34,139-145,218-233; generic_search.py:240-253; _substitutions_only.c:4-17) stop at the
// first hit of a left-to-right scan.  A GPU scans everywhere at once, so the stop is made coarse instead: the
// sequence is searched in chunks of geometrically growing size (64 MiB, 256 MiB, 1 GiB, the rest), each chunk a
// VIEW of the resident buffer searched exactly like a shard (own range = the chunk, halo from its neighbours,
// window clipping at the global ends only -- so the union of the chunks' raw streams is the whole raw stream);
// the call returns after the first chunk that yields a raw match.  A match near the start costs ~0.1 ms
// whatever the length of the sequence; no match at all costs the full scan plus three chunk turn-arounds.
// ------------------------------------------------------------------------------------------------
extern "C" int fzb_has_near_match(fzb_haystack *h, const uint8_t *pattern, uint32_t m, uint32_t max_subs,
                                  uint32_t max_ins, uint32_t max_dels, uint32_t max_l, int *found) {
    HandleLock handle_lock(h);
    if (!h || !found) return fail(FZB_E_INVALID, "NULL argument");
    *found = 0;
    int rc = check_pattern(h, pattern, m, 0);
    if (rc) return rc;
    struct Geometry {
        uint8_t *d;
        uint64_t buf_len, buf_lo, own_lo, own_hi, padded_len;
    } const saved{h->d, h->buf_len, h->buf_lo, h->own_lo, h->own_hi, h->padded_len};
    CK(cudaSetDevice(h->device));
    if (h->buf_len) sample_collision_prob(h);  // byte statistics of the WHOLE buffer (the views reuse them)
    const uint64_t halo = round_up((uint64_t)m + std::min<uint64_t>(max_l, m), 128) + 128;
    uint64_t chunk = 64ull << 20, lo = saved.own_lo;
    if (const char *e = getenv("FZB_HAS_CHUNK_BYTES"))  // testing: chunk seams on small sequences
        chunk = std::max<uint64_t>(128, round_up(strtoull(e, nullptr, 10), 128));
    rc = FZB_OK;
    do {  // (at least one pass: an empty sequence still has its k >= m matches)
        uint64_t hi = std::min(saved.own_hi, round_up(lo + chunk, 128));
        if (saved.own_hi - hi < chunk / 4) hi = saved.own_hi;  // no tiny last chunk
        // view [vlo, vhi) of the buffer: the chunk plus its halo, 128-byte aligned relative to the buffer start
        const uint64_t want_lo = lo > saved.buf_lo + halo ? lo - halo : saved.buf_lo;
        const uint64_t vlo = saved.buf_lo + (want_lo - saved.buf_lo) / 128 * 128;
        const uint64_t vhi = std::min(saved.buf_lo + saved.buf_len, hi + halo);
        h->d = saved.d + (vlo - saved.buf_lo);
        h->buf_lo = vlo;
        h->buf_len = vhi - vlo;
        h->padded_len = round_up(h->buf_len, 128) + 128;
        h->own_lo = lo;
        h->own_hi = hi;
        fzb_result *res = nullptr;
        // choose_search_class (__init__.py:60-83) on normalised limits; raw stream only
        if (max_l == 0)
            rc = fzb_search_exact(h, pattern, m, FZB_F_NO_FINAL, &res);
        else if (max_ins == 0 && max_dels == 0)
            rc = fzb_search_hamming(h, pattern, m, std::min(max_l, max_subs), FZB_F_NO_FINAL, &res);
        else if (max_l <= std::min(max_subs, std::min(max_ins, max_dels)))
            rc = fzb_search_levenshtein(h, pattern, m, max_l, FZB_F_NO_FINAL, &res);
        else
            rc = fzb_search_generic(h, pattern, m, max_subs, max_ins, max_dels, max_l, FZB_F_NO_FINAL, &res);
        if (rc == FZB_OK && fzb_result_count(res, FZB_RAW) > 0) *found = 1;
        if (res) fzb_result_destroy(res);
        lo = hi;
        chunk *= 4;
    } while (rc == FZB_OK && !*found && lo < saved.own_hi);
    h->d = saved.d;
    h->buf_len = saved.buf_len;
    h->buf_lo = saved.buf_lo;
    h->own_lo = saved.own_lo;
    h->own_hi = saved.own_hi;
    h->padded_len = saved.padded_len;
    return rc;
}

extern "C" int fzb_debug_counters(const fzb_haystack *h, uint32_t out[32]) {
    if (!h || !out) return fail(FZB_E_INVALID, "NULL argument");
    memset(out, 0, 32 * sizeof(uint32_t));
    memcpy(out, h->h_counters, CNT_COUNT * sizeof(uint32_t));
    if (h->h_ghdr) memcpy(out + 16, h->h_ghdr, 16 * sizeof(uint32_t));
    return FZB_OK;
}

// ------------------------------------------------------------------------------------------------
// test hook: the expansion routines of the verify kernels on caller-supplied (sub, seq, budget) cases
// ------------------------------------------------------------------------------------------------
extern "C" int fzb_debug_expand(const uint8_t *subs, const uint32_t *sub_off, const uint8_t *seqs,
                                const uint32_t *seq_off, const int32_t *max_l, const int32_t *variant, uint32_t count,
                                int device, int32_t *out) {
    if (count && (!subs || !sub_off || !seqs || !seq_off || !max_l || !variant || !out))
        return fail(FZB_E_INVALID, "NULL argument");
    if (device < 0 || device >= fzb_device_count()) return fail(FZB_E_CUDA, "CUDA device %d not available", device);
    if (count == 0) return FZB_OK;
    for (uint32_t i = 0; i < count; i++) {
        if (sub_off[i + 1] < sub_off[i] || seq_off[i + 1] < seq_off[i]) return fail(FZB_E_INVALID, "bad offsets");
        if (sub_off[i + 1] - sub_off[i] >= (uint32_t)kDbgMax || seq_off[i + 1] - seq_off[i] >= 2u * kDbgMax)
            return fail(FZB_E_UNSUPPORTED, "case %u too long for the debug entry", i);
        if (variant[i] < 0 || variant[i] > 2 || max_l[i] < 0) return fail(FZB_E_INVALID, "bad variant / budget");
    }
    CK(cudaSetDevice(device));
    uint8_t *d_subs = nullptr, *d_seqs = nullptr;
    uint32_t *d_so = nullptr, *d_qo = nullptr;
    int32_t *d_k = nullptr, *d_v = nullptr, *d_out = nullptr;
    const size_t nsub = std::max<size_t>(sub_off[count], 1), nseq = std::max<size_t>(seq_off[count], 1);
    int rc = [&]() -> int {
        CK(cudaMalloc(&d_subs, nsub));
        CK(cudaMalloc(&d_seqs, nseq));
        CK(cudaMalloc(&d_so, (count + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&d_qo, (count + 1) * sizeof(uint32_t)));
        CK(cudaMalloc(&d_k, count * sizeof(int32_t)));
        CK(cudaMalloc(&d_v, count * sizeof(int32_t)));
        CK(cudaMalloc(&d_out, (size_t)count * 8 * sizeof(int32_t)));
        CK(cudaMemcpy(d_subs, subs, sub_off[count], cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_seqs, seqs, seq_off[count], cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_so, sub_off, (count + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_qo, seq_off, (count + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_k, max_l, count * sizeof(int32_t), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_v, variant, count * sizeof(int32_t), cudaMemcpyHostToDevice));
        k_debug_expand<<<count, 32>>>(d_subs, d_so, d_seqs, d_qo, d_k, d_v, d_out);
        CK(cudaGetLastError());
        CK(cudaMemcpy(out, d_out, (size_t)count * 8 * sizeof(int32_t), cudaMemcpyDeviceToHost));
        return FZB_OK;
    }();
    cudaFree(d_subs);
    cudaFree(d_seqs);
    cudaFree(d_so);
    cudaFree(d_qo);
    cudaFree(d_k);
    cudaFree(d_v);
    cudaFree(d_out);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
extern "C" uint64_t fzb_result_count(const fzb_result *r, int which) {
    if (!r) return 0;
    if (which != FZB_RAW && r->has_global) return r->gcount;
    if (which == FZB_RAW) return r->raw_n;
    return r->fin.size();
}

extern "C" int fzb_result_copy(const fzb_result *r, int which, int64_t *start, int64_t *end, int32_t *dist,
                               int32_t *anchor_ngram, int64_t *anchor_idx) {
    if (!r) return fail(FZB_E_INVALID, "result is NULL");
    if (which == FZB_RAW) const_cast<fzb_result *>(r)->order_raw();
    if (which != FZB_RAW && r->has_global) const_cast<fzb_result *>(r)->fetch_raw();  // global rows are fetched lazily
    const std::vector<RawRec> &v = (which != FZB_RAW && r->has_global) ? r->gfin : (which == FZB_RAW ? r->raw : r->fin);
    const bool anchors = (which == FZB_RAW) && (r->stats.route <= 2);
    for (size_t i = 0; i < v.size(); i++) {
        if (start) start[i] = v[i].start;
        if (end) end[i] = v[i].end;
        if (dist) dist[i] = v[i].dist;
        if (anchor_ngram) anchor_ngram[i] = anchors ? v[i].ngram : -1;
        if (anchor_idx) anchor_idx[i] = anchors ? v[i].idx : -1;
    }
    return FZB_OK;
}

extern "C" int fzb_result_stats(const fzb_result *r, fzb_stats *out) {
    if (!r || !out) return fail(FZB_E_INVALID, "NULL argument");
    *out = r->stats;
    return FZB_OK;
}

extern "C" void fzb_result_destroy(fzb_result *r) {
    if (!r) return;
    {
        std::lock_guard<std::mutex> lock(g_pending_mutex);
        if (r->owner) {
            r->owner->pending = nullptr;
            r->owner = nullptr;
        }
    }
    delete r;
}
