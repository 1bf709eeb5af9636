// dgx_api.cu -- libdgx.so: C ABI (include/dgx.h) over the sm_100a kernels.
//
// Host responsibilities only: lane (stream + workspace) management, building the
// small task / list descriptor tables the kernels read, host<->device copies for
// the host-pointer entry points.  No set-operation or decode arithmetic runs on
// the CPU here: if CUDA is unavailable every entry point fails with
// DGX_ERR_NODEV / DGX_ERR_CUDA (the cgo shim then stays on the Go path).
#include "../../include/dgx.h"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <list>
#include <mutex>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "decode_kernel.cuh"
#include "filter_kernel.cuh"
#include "filter_pipe.cuh"
#include "merge_kernel.cuh"
#include "merge_multi.cuh"
#include "merge_tile32.cuh"
#include "probe_kernel.cuh"
#include "compressed_kernel.cuh"
#include "encode_kernel.cuh"
#include "wire.hpp"

using namespace dgx;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(e_ == cudaErrorMemoryAllocation ? DGX_ERR_OOM : DGX_ERR_CUDA,         \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

extern "C" const char* dgx_last_error(void) { return g_err.c_str(); }

// ---------------------------------------------------------------------------
// global state
// ---------------------------------------------------------------------------
struct Stats {
    std::atomic<uint64_t> calls{0}, uids_in{0}, uids_out{0}, h2d{0}, d2h{0}, launches{0};
};
static Stats g_stats;
static std::mutex g_mu;
static int g_device = -1;
static std::vector<dgx_lane*> g_pool;  // idle lanes for the host-pointer entry points
static std::condition_variable g_pool_cv;
static size_t g_lanes_out = 0;     // lanes currently leased
static size_t g_lanes_total = 0;   // lanes in existence (pooled + leased)
constexpr u32 kStreamRatio = 16;       // filter_kernel: stream an oversized slice when it is <= 16 x the live candidates
constexpr u32 kScapMin = 8192, kScapMax = 65536;  // bytes
static int g_filter_pipe = 1;          // DGX_FILTER=v4 selects the non-persistent kernel
static int g_merge_multi = 1;          // DGX_MERGE=tree forces the pairwise merge tree
static int g_merge_ahead = -1;         // DGX_MERGE_AHEAD: L2 prefetch distance in tiles (-1 = 3 x SM count, the resident CTAs; 0 = off)
static u32 g_merge_stride = 10;        // DGX_MERGE_STRIDE: sample gaps per multiway-merge tile (tile ~ 512 x stride values, 7680-slot rounds)
static size_t g_merge_multi_min = size_t(1) << 18;  // DGX_MERGE_MULTI_MIN: totals below this stay on the tree (fewer launches)
static int g_num_sms = 148;
constexpr size_t kPipeSmemMax = 220 * 1024;

// ---------------------------------------------------------------------------
// arenas
// ---------------------------------------------------------------------------
static cudaError_t pinned_alloc(void** p, size_t bytes);  // NUMA-aware cudaMallocHost (below)
static void numa_probe(int device);
// Device scratch: bump allocator, reset at the start of every public op (safe:
// later work on the same stream is ordered after earlier kernels).
struct DevArena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    std::vector<void*> retired;  // old chunks still referenced by queued work
    int alloc(size_t bytes, void** out) {
        bytes = (bytes + 255) & ~size_t(255);
        if (used + bytes > cap) {
            size_t ncap = std::max(cap * 2, used + bytes + (size_t(1) << 20));
            void* nb = nullptr;
            cudaError_t e = cudaMalloc(&nb, ncap);
            if (e != cudaSuccess) return fail(DGX_ERR_OOM, "cudaMalloc(%zu) failed: %s", ncap, cudaGetErrorString(e));
            if (base) retired.push_back(base);  // pointers handed out earlier in this op stay valid
            base = (char*)nb;
            cap = ncap;
            used = 0;
        }
        *out = base + used;
        used += bytes;
        return DGX_OK;
    }
    // Old chunks may still back pointers the current op hands to the host-side epilogue
    // (e.g. the D2H copy after a lane sync), so they are freed in two steps: a lane sync
    // makes them `freeable` (no queued work references them any more), the next op's
    // reset() actually frees them.
    std::vector<void*> freeable;
    void reset() {
        used = 0;
        for (void* p : freeable) cudaFree(p);
        freeable.clear();
    }
    void release_retired() {
        for (void* p : retired) freeable.push_back(p);
        retired.clear();
    }
    void destroy() {
        release_retired();
        for (void* p : freeable) cudaFree(p);
        freeable.clear();
        if (base) cudaFree(base);
        base = nullptr;
        cap = used = 0;
    }
};

// Pinned host staging for descriptor tables: async H2D copies read from it
// later, so it is only recycled at lane sync.
struct HostArena {
    struct Chunk { char* p; size_t cap, used; };
    std::vector<Chunk> chunks;
    int alloc(size_t bytes, void** out) {
        bytes = (bytes + 63) & ~size_t(63);
        if (chunks.empty() || chunks.back().used + bytes > chunks.back().cap) {
            size_t ncap = std::max(bytes, chunks.empty() ? (size_t(1) << 20) : chunks.back().cap * 2);
            void* p = nullptr;
            cudaError_t e = pinned_alloc(&p, ncap);
            if (e != cudaSuccess) return fail(DGX_ERR_OOM, "cudaMallocHost(%zu) failed: %s", ncap, cudaGetErrorString(e));
            chunks.push_back({(char*)p, ncap, 0});
        }
        Chunk& c = chunks.back();
        *out = c.p + c.used;
        c.used += bytes;
        return DGX_OK;
    }
    size_t used_bytes() const {
        size_t t = 0;
        for (const auto& c : chunks) t += c.used;
        return t;
    }
    void reset() {  // keep the largest (last) chunk
        while (chunks.size() > 1) {
            cudaFreeHost(chunks.front().p);
            chunks.erase(chunks.begin());
        }
        if (!chunks.empty()) chunks.back().used = 0;
    }
    void destroy() {
        for (auto& c : chunks) cudaFreeHost(c.p);
        chunks.clear();
    }
};

struct dgx_lane {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    DevArena ws;
    HostArena host;
    int* d_err = nullptr;   // device error flag (out_cap overflow)
    int* h_err = nullptr;   // pinned mirror
    uint64_t* h_word = nullptr;  // pinned scratch for lengths (8 words)
    uint64_t* h_head = nullptr;  // pinned landing zone for the head of a result (kSpecHead values)
    uint64_t launches = 0;
    // "resident lists" mode (dgx_lane_set_resident_inputs): the plan pre-pass of batch i+1 runs on a side stream while
    // the pipeline kernel of batch i is still running; its tables live in two alternating workspaces
    bool resident_inputs = false;
    cudaStream_t side = nullptr;
    DevArena fws[2];
    cudaEvent_t ev_plan[2] = {nullptr, nullptr}, ev_pipe[2] = {nullptr, nullptr};
    int fslot = 0;
    // Buffers the lane's own queued operations write (outputs of filter batches, merges, decodes since the last
    // dgx_lane_sync).  A batch that reads one of them is NOT planned ahead: its pre-pass is ordered behind the main
    // stream, so "decode -> intersect" or chained intersections on a resident-inputs lane stay correct.
    struct OutRange { const char* p; size_t bytes; };
    std::vector<OutRange> outs;
    bool outs_overflow = false;
    cudaEvent_t ev_prod = nullptr;
    void note_output(const void* p, size_t bytes) {
        if (!resident_inputs || !p || !bytes) return;
        for (OutRange& r : outs)
            if (r.p == (const char*)p) { r.bytes = std::max(r.bytes, bytes); return; }
        if (outs.size() >= 32) { outs_overflow = true; return; }
        outs.push_back({(const char*)p, bytes});
    }
    bool reads_own_output(const void* p) const {
        if (outs_overflow) return true;
        for (const OutRange& r : outs)
            if ((const char*)p >= r.p && (const char*)p < r.p + r.bytes) return true;
        return false;
    }
};
// Results up to this many values reach the host in the same round trip as their length.
constexpr size_t kSpecHead = 8192;

// Start of a device-level op on a lane: bind the device, recycle the workspace.  The pinned descriptor
// staging is only recycled at a lane sync (queued H2D copies read from it); a caller that queues thousands
// of ops without ever syncing would grow it without bound, so past a soft cap the op syncs the stream itself.
constexpr size_t kHostArenaSoftCap = size_t(16) << 20;
static int lane_begin_op(dgx_lane* l) {
    CK(cudaSetDevice(l->device));
    if (l->host.used_bytes() > kHostArenaSoftCap) {
        CK(cudaStreamSynchronize(l->stream));
        l->host.reset();
        l->ws.release_retired();
    }
    l->ws.reset();
    return DGX_OK;
}

// Call after every kernel launch on the lane's stream: reports a failed launch and counts the launch.
static int launched(dgx_lane* l) {
    CK(cudaGetLastError());
    l->launches += 1;
    g_stats.launches += 1;
    return DGX_OK;
}

// ---------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------
extern "C" int dgx_init(int device) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_device >= 0) return DGX_OK;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(DGX_ERR_NODEV, "no CUDA device: %s", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= n) return fail(DGX_ERR_ARG, "device %d out of range (%d devices)", device, n);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(DGX_ERR_NODEV, "libdgx is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    CK(cudaFuncSetAttribute(decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(sizeof(DWarpSmem) * D_WARPS)));
    CK(cudaFuncSetAttribute(decode_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(sizeof(DWarpSmem) * D_WARPS)));
    CK(cudaFuncSetAttribute(icw_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(sizeof(DWarpSmem) * D_WARPS)));
    CK(cudaFuncSetAttribute(filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(2 * F_TA * sizeof(u64) + kScapMax)));
    CK(cudaFuncSetAttribute(filter_pipe_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPipeSmemMax));
    CK(cudaFuncSetAttribute(filter_pipe_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPipeSmemMax));
    g_num_sms = prop.multiProcessorCount;
    numa_probe(device);
    if (const char* s = getenv("DGX_FILTER")) g_filter_pipe = (strcmp(s, "v4") != 0);
    CK(cudaFuncSetAttribute(mmerge3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T_SMEM));
    if (const char* s = getenv("DGX_MERGE")) g_merge_multi = (strcmp(s, "tree") != 0);
    if (const char* s = getenv("DGX_MERGE_MULTI_MIN")) g_merge_multi_min = (size_t)atoll(s);
    if (const char* s = getenv("DGX_MERGE_AHEAD")) g_merge_ahead = atoi(s);
    if (const char* s = getenv("DGX_MERGE_STRIDE")) { const int v = atoi(s); if (v >= 1 && v <= 16) g_merge_stride = (u32)v; }
    g_device = device;
    return DGX_OK;
}

extern "C" void dgx_shutdown(void) {
    dgx_cache_clear();
    std::unique_lock<std::mutex> lk(g_mu);
    g_pool_cv.wait(lk, [] { return g_lanes_out == 0; });  // calls in flight keep their lanes until they return
    for (dgx_lane* l : g_pool) dgx_lane_destroy(l);
    g_pool.clear();
    g_lanes_total = 0;
    g_device = -1;
}

extern "C" int dgx_describe(char* buf, size_t n) {
    int rc = dgx_init(-1);
    if (rc != DGX_OK) return rc;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, g_device));
    snprintf(buf, n, "libdgx sm_100a | device %d: %s, %d SMs, %.1f GB | filter tile %d, merge tile %d",
             g_device, prop.name, prop.multiProcessorCount, prop.totalGlobalMem / 1e9, F_TA, M_T);
    return DGX_OK;
}

// Pinned host memory is placed on the NUMA node the GPU hangs off: a DMA from the far socket runs at
// about half the PCIe rate.  While the pages are allocated the calling thread is moved to the GPU's
// node (first touch) and, where the container allows it, the memory policy prefers that node; both
// are restored afterwards and every step is best effort (DGX_NUMA=0 turns it off).
static int g_numa_node = -2;  // -2 unknown, -1 none
static cpu_set_t g_numa_cpus;
static void numa_probe(int device) {
    g_numa_node = -1;
    if (const char* s = getenv("DGX_NUMA")) if (atoi(s) == 0) return;
    char bus[32] = {0}, path[128];
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) return;
    for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    int node = -1;
    if (f) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
    if (node < 0) return;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return;
    CPU_ZERO(&g_numa_cpus);
    int a, b, n = 0;
    while (fscanf(f, "%d", &a) == 1) {
        b = a;
        int c = fgetc(f);
        if (c == '-') { if (fscanf(f, "%d", &b) != 1) b = a; c = fgetc(f); }
        for (int i = a; i <= b && i < CPU_SETSIZE; ++i) { CPU_SET(i, &g_numa_cpus); ++n; }
        if (c != ',') break;
    }
    fclose(f);
    if (n) g_numa_node = node;
}
static cudaError_t pinned_alloc(void** p, size_t bytes) {
    cpu_set_t old;
    bool moved = false, policy = false;
    if (g_numa_node >= 0) {
        if (sched_getaffinity(0, sizeof(old), &old) == 0 && sched_setaffinity(0, sizeof(g_numa_cpus), &g_numa_cpus) == 0) moved = true;
        unsigned long mask[16] = {0};
        if (g_numa_node < 1024) {
            mask[g_numa_node / (8 * sizeof(unsigned long))] |= 1ul << (g_numa_node % (8 * sizeof(unsigned long)));
            policy = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, 1024ul) == 0;
        }
    }
    const cudaError_t e = cudaMallocHost(p, bytes ? bytes : 1);
    if (policy) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
    if (moved) sched_setaffinity(0, sizeof(old), &old);
    return e;
}

extern "C" void* dgx_host_alloc(size_t bytes) {
    if (dgx_init(-1) != DGX_OK) return nullptr;
    void* p = nullptr;
    if (pinned_alloc(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void dgx_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

extern "C" void dgx_get_stats(dgx_stats* out) {
    out->calls = g_stats.calls;
    out->uids_in = g_stats.uids_in;
    out->uids_out = g_stats.uids_out;
    out->h2d_bytes = g_stats.h2d;
    out->d2h_bytes = g_stats.d2h;
    out->kernel_launches = g_stats.launches;
}

extern "C" dgx_lane* dgx_lane_create(int device, void* stream) {
    if (dgx_init(device) != DGX_OK) return nullptr;
    if (device < 0) device = g_device;
    // One device per process (one alpha process per GPU): kernel attributes, the SM count and the
    // host-pointer entry points are bound to the device dgx_init chose.
    if (device != g_device) {
        fail(DGX_ERR_ARG, "libdgx is bound to device %d in this process; lane requested on device %d", g_device, device);
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    dgx_lane* l = new dgx_lane();
    l->device = device;
    if (stream) {
        l->stream = (cudaStream_t)stream;
    } else {
        if (cudaStreamCreateWithFlags(&l->stream, cudaStreamNonBlocking) != cudaSuccess) { delete l; return nullptr; }
        l->own_stream = true;
    }
    if (cudaMalloc(&l->d_err, 256) != cudaSuccess ||
        pinned_alloc((void**)&l->h_err, 4096 + kSpecHead * sizeof(uint64_t)) != cudaSuccess) {
        fail(DGX_ERR_OOM, "lane allocation failed");
        delete l;
        return nullptr;
    }
    l->h_word = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(l->h_err) + 64);
    l->h_head = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(l->h_err) + 4096);
    *l->h_err = 0;
    cudaMemsetAsync(l->d_err, 0, 256, l->stream);
    return l;
}

extern "C" void dgx_lane_destroy(dgx_lane* l) {
    if (!l) return;
    cudaSetDevice(l->device);
    cudaStreamSynchronize(l->stream);
    l->ws.destroy();
    l->host.destroy();
    if (l->d_err) cudaFree(l->d_err);
    if (l->h_err) cudaFreeHost(l->h_err);
    if (l->side) { cudaStreamSynchronize(l->side); cudaStreamDestroy(l->side); }
    for (int i = 0; i < 2; ++i) {
        l->fws[i].destroy();
        if (l->ev_plan[i]) cudaEventDestroy(l->ev_plan[i]);
        if (l->ev_pipe[i]) cudaEventDestroy(l->ev_pipe[i]);
        if (i == 0 && l->ev_prod) cudaEventDestroy(l->ev_prod);
    }
    if (l->own_stream) cudaStreamDestroy(l->stream);
    delete l;
}

extern "C" void* dgx_lane_stream(dgx_lane* l) { return l ? (void*)l->stream : nullptr; }

extern "C" int dgx_lane_set_resident_inputs(dgx_lane* l, int on) {
    if (!l) return fail(DGX_ERR_ARG, "null lane");
    CK(cudaSetDevice(l->device));
    if (on && !l->side) {
        CK(cudaStreamCreateWithFlags(&l->side, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CK(cudaEventCreateWithFlags(&l->ev_plan[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&l->ev_pipe[i], cudaEventDisableTiming));
        }
        CK(cudaEventCreateWithFlags(&l->ev_prod, cudaEventDisableTiming));
    }
    if (!on && l->side) CK(cudaStreamSynchronize(l->side));
    l->resident_inputs = on != 0;
    return DGX_OK;
}
extern "C" uint64_t dgx_lane_launches(const dgx_lane* l) { return l ? l->launches : 0; }

extern "C" int dgx_lane_sync(dgx_lane* l) {
    if (!l) return fail(DGX_ERR_ARG, "null lane");
    CK(cudaSetDevice(l->device));
    CK(cudaMemcpyAsync(l->h_err, l->d_err, sizeof(int), cudaMemcpyDeviceToHost, l->stream));
    CK(cudaStreamSynchronize(l->stream));
    l->host.reset();
    l->ws.release_retired();
    l->outs.clear();
    l->outs_overflow = false;
    if (*l->h_err) {
        *l->h_err = 0;
        CK(cudaMemsetAsync(l->d_err, 0, sizeof(int), l->stream));
        return fail(DGX_ERR_CAP, "result does not fit out_cap");
    }
    return DGX_OK;
}

extern "C" void* dgx_dev_alloc(size_t bytes) {
    if (dgx_init(-1) != DGX_OK) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) { fail(DGX_ERR_OOM, "cudaMalloc(%zu) failed", bytes); return nullptr; }
    return p;
}
extern "C" void dgx_dev_free(void* p) {
    if (p) cudaFree(p);
}
extern "C" int dgx_memcpy_h2d(dgx_lane* l, void* d, const void* h, size_t bytes) {
    if (!l) return fail(DGX_ERR_ARG, "null lane");
    CK(cudaSetDevice(l->device));
    if (bytes) CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, l->stream));
    g_stats.h2d += bytes;
    return DGX_OK;
}
extern "C" int dgx_memcpy_d2h(dgx_lane* l, void* h, const void* d, size_t bytes) {
    if (!l) return fail(DGX_ERR_ARG, "null lane");
    CK(cudaSetDevice(l->device));
    if (bytes) CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, l->stream));
    g_stats.d2h += bytes;
    return DGX_OK;
}

// ---------------------------------------------------------------------------
// filter (intersect / k-way intersect / difference), device level
// ---------------------------------------------------------------------------
struct ListDesc {
    const uint64_t* ptr;
    size_t len;
    const uint64_t* dyn_len;
};

// Queries q own lists [k_off[q], k_off[q+1]).  Results -> d_out / d_out_off.
static int filter_batch_impl(dgx_lane* l, int op, const ListDesc* lists, const size_t* k_off, size_t nq,
                             uint64_t* d_out, size_t out_cap, uint64_t* d_out_off) {
    if (nq == 0) {
        CK(cudaMemsetAsync(d_out_off, 0, sizeof(uint64_t), l->stream));
        return DGX_OK;
    }
    const size_t nlists = k_off[nq] - k_off[0];
    void *h_raw, *d_raw;
    const size_t tasks_b = nq * sizeof(FTask), lists_b = (nlists + 1) * sizeof(FList);
    int rc = l->host.alloc(tasks_b + lists_b, &h_raw);
    if (rc) return rc;
    FTask* ht = (FTask*)h_raw;
    FList* hl = (FList*)((char*)h_raw + tasks_b);
    uint64_t ntiles = 0, uids_in = 0;
    size_t li = 0, kmax = 1;
    for (size_t q = 0; q < nq; ++q) kmax = std::max(kmax, k_off[q + 1] - k_off[q]);
    // batches of single-list queries take filter_kernel
    const bool use_pipe = g_filter_pipe && kmax >= 2;
    // 2-list batches: 1024-value tiles (per-tile overheads over twice the values); wider queries: 512 (filter_pipe.cuh)
    const int pipe_va = kmax <= 2 ? 4 : 2;
    const uint64_t tile_sz = use_pipe ? (uint64_t)p_tile_size(pipe_va) : (uint64_t)F_TA;
    std::vector<size_t> order;
    for (size_t q = 0; q < nq; ++q) {
        const size_t k0 = k_off[q], k1 = k_off[q + 1];
        const size_t k = k1 - k0;
        if (k == 0) return fail(DGX_ERR_ARG, "query %zu has no lists", q);
        kmax = std::max(kmax, k);
        if (op == DGX_OP_DIFFERENCE && k != 2) return fail(DGX_ERR_ARG, "difference takes exactly two lists");
        order.resize(k);
        std::iota(order.begin(), order.end(), k0);
        if (op == DGX_OP_INTERSECT)  // drive from the shortest list (algo/uidlist.go:309-311)
            std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) { return lists[x].len < lists[y].len; });
        ht[q].tile_base = ntiles;
        ht[q].list_first = (u32)li;
        ht[q].k = (u32)k;
        for (size_t i = 0; i < k; ++i) {
            const ListDesc& L = lists[order[i]];
            hl[li].ptr = (const u64*)L.ptr;
            hl[li].len = L.len;
            hl[li].dyn_len = (const u64*)L.dyn_len;
            uids_in += L.len;
            ++li;
        }
        const uint64_t lenA = lists[order[0]].len;
        ntiles += std::max<uint64_t>(1, (lenA + tile_sz - 1) / tile_sz);
    }
    if (ntiles > 0x7fffffffull) return fail(DGX_ERR_ARG, "batch too large (%llu tiles)", (unsigned long long)ntiles);
    const size_t status_b = ntiles * sizeof(u64) + 64;
    // Where the batch's tables live and which stream prepares them.  Normally: the lane's workspace and stream.
    // Resident-inputs lanes: one of two alternating workspaces and the side stream -- descriptor copies, status
    // reset and the plan pre-pass of THIS batch then run while the pipeline kernel of the PREVIOUS batch is still
    // busy (the lists are immutable, so the pre-pass depends on nothing the main stream has queued).
    const bool ahead = l->resident_inputs && use_pipe && l->side;
    const int slot = l->fslot;
    DevArena* ar = &l->ws;
    cudaStream_t pre = l->stream;
    if (ahead) {
        l->fslot ^= 1;
        ar = &l->fws[slot];
        pre = l->side;
        CK(cudaStreamWaitEvent(l->side, l->ev_pipe[slot], 0));  // the pipeline that last read this workspace is done
        bool dep = false;  // a list this lane's own queued work produces: plan it behind that work, not ahead
        for (size_t i = k_off[0]; i < k_off[nq] && !dep; ++i)
            dep = l->reads_own_output(lists[i].ptr) || (lists[i].dyn_len && l->reads_own_output(lists[i].dyn_len));
        if (dep) {
            CK(cudaEventRecord(l->ev_prod, l->stream));
            CK(cudaStreamWaitEvent(l->side, l->ev_prod, 0));
        }
        ar->reset();
    }
    rc = ar->alloc(tasks_b + lists_b + status_b, &d_raw);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d_raw, h_raw, tasks_b + lists_b, cudaMemcpyHostToDevice, pre));
    char* d_status = (char*)d_raw + tasks_b + lists_b;
    CK(cudaMemsetAsync(d_status, 0, status_b, pre));
    FParams P;
    P.tasks = (const FTask*)d_raw;
    P.lists = (const FList*)((char*)d_raw + tasks_b);
    P.ntasks = (u32)nq;
    P.ntiles = (u32)ntiles;
    P.op = op;
    P.stream_ratio = kStreamRatio;
    // staging capacity (bytes): ~1.1 tile-widths of 32-bit keys for every filter list of the widest query
    P.scap_bytes = (u32)std::min<size_t>(32768, std::max<size_t>(kScapMin, (kmax - 1) * 1152 * 4));
    P.out = (u64*)d_out;
    P.out_cap = out_cap;
    P.out_off = (u64*)d_out_off;
    P.status = (u64*)d_status;
    P.ticket = (u32*)(d_status + ntiles * sizeof(u64));
    P.err = l->d_err;
    if (!use_pipe) {
        filter_kernel<<<(unsigned)ntiles, F_NT, 2 * F_TA * sizeof(u64) + P.scap_bytes, l->stream>>>(P);
        if (int e = launched(l)) return e;
    } else {
        // ---- persistent TMA pipeline: plan pre-pass + filter_pipe_kernel ----------------
        void* hp_raw;
        rc = l->host.alloc(nq * sizeof(u64), &hp_raw);
        if (rc) return rc;
        u64* h_pb = (u64*)hp_raw;
        u64 npairs = 0;
        for (size_t q = 0; q < nq; ++q) {
            h_pb[q] = npairs;
            const u64 nt = (q + 1 < nq ? ht[q + 1].tile_base : ntiles) - ht[q].tile_base;
            npairs += nt * (u64)(ht[q].k - 1);
        }
        void *d_pb, *d_plan, *d_tiles;
        rc = ar->alloc(nq * sizeof(u64), &d_pb);
        if (rc) return rc;
        rc = ar->alloc(ntiles * sizeof(PTileEntry), &d_tiles);
        if (rc) return rc;
        rc = ar->alloc((npairs + 1) * sizeof(PPlanEntry), &d_plan);
        if (rc) return rc;
        CK(cudaMemcpyAsync(d_pb, h_pb, nq * sizeof(u64), cudaMemcpyHostToDevice, pre));
        filter_tiles_kernel<<<(unsigned)((ntiles + 255) / 256), 256, 0, pre>>>(P.tasks, P.lists, (const u64*)d_pb, P.ntasks,
                                                                               P.ntiles, (PTileEntry*)d_tiles, (u32)tile_sz);
        if (int e = launched(l)) return e;
        if (npairs) {
            const u64 blocks = (npairs + 255) / 256;
            if (blocks > 0x7fffffffull) return fail(DGX_ERR_ARG, "batch too large");
            filter_plan_kernel<<<(unsigned)blocks, 256, 0, pre>>>(P.tasks, P.lists, (const u64*)d_pb, P.ntasks, npairs,
                                                                  (PPlanEntry*)d_plan, (u32)tile_sz);
            if (int e = launched(l)) return e;
        }
        PParams PP;
        PP.f = P;
        PP.plan_base = (const u64*)d_pb;
        PP.plan = (const PPlanEntry*)d_plan;
        PP.tiles = (const PTileEntry*)d_tiles;
        // wide queries: one tile per ticket keeps the look-back order tight (measured 0.476 vs 0.50 ms on
        // C2); 2-list batches have tiny tiles and amortise the metadata chain over two (measured +4 %)
        PP.grp = kmax >= 4 ? 1u : 2u;
        const size_t nl = std::min<size_t>(std::max<size_t>(kmax - 1, 1), P_MAXL);
        const size_t TA = (size_t)tile_sz;
        // staged slices: ~1.125 tile-widths per filter list; a 2-list batch stages up to 2.25 tile-widths of its one
        // filter list (size ratios beyond that probe the list in HBM, the reference's own Jump / Bin regimes)
        size_t cap = (TA + TA / 8) * nl * (kmax <= 2 ? 2 : 1);
        cap = std::min<size_t>(std::max<size_t>(cap, TA + TA / 8), 9216) & ~size_t(1);
        PP.slice_cap = (u32)cap;
        const size_t smem = ((sizeof(PShared) + 127) & ~size_t(127)) + (1 + P_OS) * TA * sizeof(u64) +
                            P_ST * ((TA + 2) + cap) * sizeof(u64);
        if (smem > kPipeSmemMax) return fail(DGX_ERR_ARG, "pipeline stage too large");
        auto kern = pipe_va == 4 ? filter_pipe_kernel<4> : filter_pipe_kernel<2>;
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, P_NT, smem));
        if (per_sm < 1) return fail(DGX_ERR_CUDA, "filter_pipe_kernel does not fit on an SM");
        PP.nctas = (u32)std::min<u64>((u64)per_sm * (u64)g_num_sms, ntiles);
        if (ahead) {
            CK(cudaEventRecord(l->ev_plan[slot], l->side));
            CK(cudaStreamWaitEvent(l->stream, l->ev_plan[slot], 0));
        }
        kern<<<PP.nctas, P_NT, smem, l->stream>>>(PP);
        if (int e = launched(l)) return e;
        if (ahead) CK(cudaEventRecord(l->ev_pipe[slot], l->stream));
    }
    g_stats.uids_in += uids_in;
    return DGX_OK;
}

extern "C" int dgx_dev_filter_batch(dgx_lane* l, int op, const uint64_t* const* d_lists, const size_t* lens,
                                    const size_t* k_off, size_t nq, uint64_t* d_out, size_t out_cap,
                                    uint64_t* d_out_off) {
    if (!l || (op != DGX_OP_INTERSECT && op != DGX_OP_DIFFERENCE)) return fail(DGX_ERR_ARG, "bad lane/op");
    if (int rc = lane_begin_op(l)) return rc;
    const size_t nlists = nq ? k_off[nq] : 0;
    std::vector<ListDesc> ld(nlists);
    for (size_t i = 0; i < nlists; ++i) ld[i] = {d_lists[i], lens[i], nullptr};
    g_stats.calls += 1;
    const int rc = filter_batch_impl(l, op, ld.data(), k_off, nq, d_out, out_cap, d_out_off);
    l->note_output(d_out, out_cap * sizeof(uint64_t));
    l->note_output(d_out_off, (nq + 1) * sizeof(uint64_t));
    return rc;
}

// ---------------------------------------------------------------------------
// MergeSorted, device level: tree of batched 2-way unions
// ---------------------------------------------------------------------------
static int merge_tree_impl(dgx_lane* l, std::vector<MRef> cur, std::vector<uint64_t> ub, uint64_t total,
                           uint64_t* d_out, size_t out_cap, uint64_t* d_out_len);
static int merge_multi_impl(dgx_lane* l, const std::vector<MRef>& runs, const std::vector<uint64_t>& ub, uint64_t total,
                            uint64_t* d_out, size_t out_cap, uint64_t* d_out_len);
static int merge_runs_impl(dgx_lane* l, const std::vector<MRef>& cur, const std::vector<uint64_t>& ub, uint64_t total,
                           uint64_t* d_out, size_t out_cap, uint64_t* d_out_len);

static int merge_sorted_impl(dgx_lane* l, const ListDesc* lists, size_t k, uint64_t* d_out, size_t out_cap,
                             uint64_t* d_out_len) {
    // nil / empty lists are skipped (algo/uidlist.go:400-403)
    std::vector<MRef> cur;
    std::vector<uint64_t> ub;
    uint64_t total = 0;
    for (size_t i = 0; i < k; ++i) {
        if (lists[i].ptr == nullptr || lists[i].len == 0) continue;
        cur.push_back(MRef{(const u64*)lists[i].ptr, nullptr, (u64)lists[i].len});
        ub.push_back(lists[i].len);
        total += lists[i].len;
    }
    g_stats.uids_in += total;
    if (cur.empty()) {
        CK(cudaMemsetAsync(d_out_len, 0, sizeof(uint64_t), l->stream));
        return DGX_OK;
    }
    if (out_cap < total) return fail(DGX_ERR_CAP, "MergeSorted needs out_cap >= sum(lens) = %llu", (unsigned long long)total);
    return merge_runs_impl(l, cur, ub, total, d_out, out_cap, d_out_len);
}

// Dispatch over the number of runs: the single-pass multiway merge for 3..64 large runs, groups of <= 64 runs merged
// multiway into intermediate runs (whose lengths stay on the device: MRef::off) and merged again for more -- two passes
// over HBM up to 4096 runs instead of ceil(log2 k) -- and the pairwise tree for everything small.
static int merge_runs_impl(dgx_lane* l, const std::vector<MRef>& cur, const std::vector<uint64_t>& ub, uint64_t total,
                           uint64_t* d_out, size_t out_cap, uint64_t* d_out_len) {
    const size_t k = cur.size();
    if (g_merge_multi && k >= 3 && k <= (size_t)MM_K && total >= g_merge_multi_min)
        return merge_multi_impl(l, cur, ub, total, d_out, out_cap, d_out_len);
    const size_t ngroups = (k + MM_K - 1) / MM_K;
    // a multiway call is a dozen launches: grouping pays only when every group is a few times the multiway minimum
    if (!g_merge_multi || k <= (size_t)MM_K || total / ngroups < 4 * g_merge_multi_min)
        return merge_tree_impl(l, cur, ub, total, d_out, out_cap, d_out_len);
    const size_t gsz = (k + ngroups - 1) / ngroups;
    void *d_tmp, *d_pairs;
    int rc = l->ws.alloc(total * sizeof(u64), &d_tmp);
    if (rc) return rc;
    rc = l->ws.alloc(2 * ngroups * sizeof(u64), &d_pairs);
    if (rc) return rc;
    CK(cudaMemsetAsync(d_pairs, 0, 2 * ngroups * sizeof(u64), l->stream));
    std::vector<MRef> next;
    std::vector<uint64_t> nub;
    uint64_t goff = 0;
    for (size_t g = 0; g < ngroups; ++g) {
        const size_t b = g * gsz, e = std::min(k, b + gsz);
        if (b >= e) break;
        std::vector<MRef> part(cur.begin() + b, cur.begin() + e);
        std::vector<uint64_t> pub(ub.begin() + b, ub.begin() + e);
        uint64_t tot = 0;
        for (uint64_t v : pub) tot += v;
        u64* dst = (u64*)d_tmp + goff;
        u64* pair = (u64*)d_pairs + 2 * g;  // {0, length of the group's merged run}
        rc = merge_runs_impl(l, part, pub, tot, (uint64_t*)dst, tot, (uint64_t*)(pair + 1));
        if (rc) return rc;
        next.push_back(MRef{dst, pair, (u64)tot});
        nub.push_back(tot);
        goff += tot;
    }
    return merge_runs_impl(l, next, nub, total, d_out, out_cap, d_out_len);
}

// Pairwise merge tree: ceil(log2 k) passes of merge_kernel.
static int merge_tree_impl(dgx_lane* l, std::vector<MRef> cur, std::vector<uint64_t> ub, uint64_t total,
                           uint64_t* d_out, size_t out_cap, uint64_t* d_out_len) {
    // number of levels; a single list still takes one pass (in-list de-duplication)
    int levels = 0;
    for (size_t n = cur.size(); n > 1; n = (n + 1) / 2) ++levels;
    if (levels == 0) levels = 1;
    void* d_tmp = nullptr;
    int rc;
    if (levels > 1) {
        rc = l->ws.alloc(total * sizeof(u64), &d_tmp);
        if (rc) return rc;
    }
    // plan all levels on the host
    struct Level { std::vector<MTask> tasks; uint64_t ntiles; u64* out; size_t off_index; };
    std::vector<Level> plan(levels);
    size_t off_words = 0, task_count = 0;
    uint64_t tiles_total = 0;
    for (int lv = 0; lv < levels; ++lv) {
        Level& L = plan[lv];
        L.out = ((levels - 1 - lv) % 2 == 0) ? (u64*)d_out : (u64*)d_tmp;
        const size_t n = cur.size();
        const size_t nt = (n + 1) / 2;
        L.tasks.resize(nt);
        L.ntiles = 0;
        L.off_index = off_words;
        std::vector<uint64_t> nub(nt);
        for (size_t t = 0; t < nt; ++t) {
            MTask& T = L.tasks[t];
            T.tile_base = L.ntiles;
            T.a = cur[2 * t];
            uint64_t u = ub[2 * t];
            if (2 * t + 1 < n) { T.b = cur[2 * t + 1]; u += ub[2 * t + 1]; }
            else T.b = MRef{nullptr, nullptr, 0};
            nub[t] = u;
            L.ntiles += std::max<uint64_t>(1, (u + M_T - 1) / M_T);
        }
        if (L.ntiles > 0x7fffffffull) return fail(DGX_ERR_ARG, "merge too large");
        off_words += nt + 1;
        task_count += nt;
        tiles_total += L.ntiles;
        // next level's inputs are slices of this level's compact output (offsets patched below)
        cur.assign(nt, MRef{L.out, nullptr, 0});
        ub = nub;
        for (size_t t = 0; t < nt; ++t) { cur[t].len = nub[t]; cur[t].off = (const u64*)(uintptr_t)(L.off_index + t + 1); }
    }
    // device layout: [off words][tasks][status + tickets]
    const size_t off_b = off_words * sizeof(u64);
    const size_t tasks_b = task_count * sizeof(MTask);
    const size_t status_b = (tiles_total + 2 * levels) * sizeof(u64);
    void *d_raw, *h_raw;
    rc = l->ws.alloc(off_b + tasks_b + status_b, &d_raw);
    if (rc) return rc;
    rc = l->host.alloc(tasks_b, &h_raw);
    if (rc) return rc;
    u64* d_off = (u64*)d_raw;
    MTask* d_tasks = (MTask*)((char*)d_raw + off_b);
    u64* d_status = (u64*)((char*)d_raw + off_b + tasks_b);
    // patch symbolic offsets (index+1 encoded in the pointer) into device addresses
    MTask* ht = (MTask*)h_raw;
    size_t ti = 0;
    for (int lv = 0; lv < levels; ++lv)
        for (MTask T : plan[lv].tasks) {
            if (lv > 0) {
                T.a.off = d_off + ((uintptr_t)T.a.off - 1);
                if (T.b.base) T.b.off = d_off + ((uintptr_t)T.b.off - 1);
            }
            ht[ti++] = T;
        }
    CK(cudaMemcpyAsync(d_tasks, ht, tasks_b, cudaMemcpyHostToDevice, l->stream));
    CK(cudaMemsetAsync(d_status, 0, status_b, l->stream));
    size_t tpos = 0;
    uint64_t spos = 0;
    for (int lv = 0; lv < levels; ++lv) {
        Level& L = plan[lv];
        MParams P;
        P.tasks = d_tasks + tpos;
        P.ntasks = (u32)L.tasks.size();
        P.ntiles = (u32)L.ntiles;
        P.out = L.out;
        P.out_cap = (L.out == (u64*)d_out) ? out_cap : total;
        P.out_off = d_off + L.off_index;
        P.status = d_status + spos;
        P.ticket = (u32*)(d_status + spos + L.ntiles);
        P.err = l->d_err;
        merge_kernel<<<(unsigned)L.ntiles, M_NT, 0, l->stream>>>(P);
        if (int e = launched(l)) return e;
        tpos += L.tasks.size();
        spos += L.ntiles + 2;
    }
    CK(cudaMemcpyAsync(d_out_len, d_off + plan[levels - 1].off_index + 1, sizeof(u64), cudaMemcpyDeviceToDevice, l->stream));
    return DGX_OK;
}

// Single-pass multiway merge (merge_multi.cuh, merge_tile32.cuh) for 3..64 runs.
static int merge_multi_impl(dgx_lane* l, const std::vector<MRef>& runs, const std::vector<uint64_t>& ub, uint64_t total,
                            uint64_t* d_out, size_t out_cap, uint64_t* d_out_len) {
    const size_t k = runs.size();
    // About one sample per 512 values, spread over the runs in proportion to their lengths.  Every stride-th distinct
    // sample becomes a splitter, so a tile is the sum of `stride` sample gaps (~5K values at the default 10,
    // Gamma-distributed instead of exponential) and rarely needs more than one 7680-slot round of mmerge3_kernel.
    const u32 stride = g_merge_stride;
    const uint64_t ntarget = std::min<uint64_t>(std::max<uint64_t>(total / 512, 1), uint64_t(1) << 24);
    std::vector<u32> soff(k + 1, 0);
    for (size_t j = 0; j < k; ++j) soff[j + 1] = soff[j] + (u32)((unsigned __int128)ub[j] * ntarget / total);
    const u32 nsamp = soff[k];
    void *h_raw, *d_raw;
    const size_t runs_b = k * sizeof(MRef), soff_b = (k + 1) * sizeof(u32);
    int rc = l->host.alloc(runs_b + soff_b, &h_raw);
    if (rc) return rc;
    memcpy(h_raw, runs.data(), runs_b);
    memcpy((char*)h_raw + runs_b, soff.data(), soff_b);
    const size_t a_samples = ((runs_b + soff_b + 255) & ~size_t(255));
    const size_t a_split = a_samples + (size_t)(nsamp + 1) * 8;
    const size_t a_nsplit = a_split + (size_t)(nsamp + 1) * 8;
    const size_t a_bounds = a_nsplit + 256;
    const size_t a_tin = a_bounds + (size_t)(nsamp + 2) * k * 8;
    const size_t a_tout = a_tin + (size_t)(nsamp + 2) * 8;
    const size_t a_tcnt = a_tout + (size_t)(nsamp + 3) * 8;
    const size_t a_tlo = ((a_tcnt + (size_t)(nsamp + 2) * 4 + 255) & ~size_t(255));
    const size_t a_end = a_tlo + (size_t)(nsamp + 2) * 8;
    rc = l->ws.alloc(a_end, &d_raw);
    if (rc) return rc;
    void* d_scratch;
    rc = l->ws.alloc(total * sizeof(u64), &d_scratch);
    if (rc) return rc;
    char* d = (char*)d_raw;
    CK(cudaMemcpyAsync(d, h_raw, runs_b + soff_b, cudaMemcpyHostToDevice, l->stream));
    MMParams P;
    P.runs = (const MRef*)d;
    P.k = (u32)k;
    P.samp_off = (const u32*)(d + runs_b);
    P.nsamp = nsamp;
    P.stride = stride;
    P.samples = (u64*)(d + a_samples);
    P.splitters = (u64*)(d + a_split);
    P.nsplit = (const u64*)(d + a_nsplit);
    P.bounds = (u64*)(d + a_bounds);
    P.tile_in = (u64*)(d + a_tin);
    P.tile_out = (u64*)(d + a_tout);
    P.tile_cnt = (u32*)(d + a_tcnt);
    P.scratch = (u64*)d_scratch;
    P.out = (u64*)d_out;
    P.out_cap = out_cap;
    P.out_len = (u64*)d_out_len;
    P.err = l->d_err;
    const u32 max_tiles = nsamp / stride + 1;
    P.nbs = max_tiles + 1;
    P.tile_lo = (u64*)(d + a_tlo);
    P.ahead = g_merge_ahead < 0 ? 3u * (u32)g_num_sms : (u32)g_merge_ahead;
    if (nsamp) {
        msample_kernel<<<(nsamp + 255) / 256, 256, 0, l->stream>>>(P);
        if (int e = launched(l)) return e;
        // the sample runs are sorted: the merge tree (with de-duplication) yields the distinct splitters
        std::vector<MRef> sruns;
        std::vector<uint64_t> sub;
        for (size_t j = 0; j < k; ++j) {
            const u32 sj = soff[j + 1] - soff[j];
            if (!sj) continue;
            sruns.push_back(MRef{P.samples + soff[j], nullptr, (u64)sj});
            sub.push_back(sj);
        }
        rc = merge_tree_impl(l, sruns, sub, nsamp, (uint64_t*)P.splitters, nsamp, (uint64_t*)(d + a_nsplit));
        if (rc) return rc;
    } else {
        CK(cudaMemsetAsync(d + a_nsplit, 0, 8, l->stream));
    }
    const uint64_t nb = (uint64_t)(max_tiles + 1) * k;
    mplan2_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    mmerge3_kernel<<<max_tiles, T_NT, T_SMEM, l->stream>>>(P);
    if (int e = launched(l)) return e;
    mscan_kernel<<<1, 1024, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    mcompact_kernel<<<max_tiles, 256, 0, l->stream>>>(P);
    return launched(l);
}

extern "C" int dgx_dev_merge_sorted(dgx_lane* l, const uint64_t* const* d_lists, const size_t* lens, size_t k,
                                    uint64_t* d_out, size_t out_cap, uint64_t* d_out_len) {
    if (!l) return fail(DGX_ERR_ARG, "null lane");
    if (int rc = lane_begin_op(l)) return rc;
    std::vector<ListDesc> ld(k);
    for (size_t i = 0; i < k; ++i) ld[i] = {d_lists[i], lens[i], nullptr};
    g_stats.calls += 1;
    const int rc = merge_sorted_impl(l, ld.data(), k, d_out, out_cap, d_out_len);
    l->note_output(d_out, out_cap * sizeof(uint64_t));
    l->note_output(d_out_len, sizeof(uint64_t));
    return rc;
}

// ---------------------------------------------------------------------------
// UidPack decode, device level
// ---------------------------------------------------------------------------
struct dgx_dev_pack {
    DPack pk;
    void* d_mem = nullptr;
    size_t bytes = 0;
    size_t exact_len = 0;
    uint32_t block_size = 0;
};

// Device layout of a pack: [base u64 | delta_off u64 (n+1) | uid_off u64 (n+1) | num u32 | pad to 16]
// followed by the delta bytes (16-byte aligned, 48 readable bytes of slack for the 16-byte TMA granule and
// the 17-byte group reads).  The metadata image is assembled in pinned staging memory so that a pack
// crosses PCIe as TWO copies (metadata, deltas) and the k packs of a query as 1 + k: small copies cost
// several microseconds of DMA set-up each and used to outweigh the bytes.
struct PackLayout {
    size_t nb, dbytes, o_doff, o_uoff, o_num, meta_bytes, dpad;
};
static PackLayout pack_layout(const dgx_pack_view* v) {
    PackLayout L;
    L.nb = v ? v->nblocks : 0;
    L.dbytes = L.nb ? (size_t)v->delta_off[L.nb] : 0;
    L.o_doff = L.nb * 8;
    L.o_uoff = L.o_doff + (L.nb + 1) * 8;
    L.o_num = L.o_uoff + (L.nb + 1) * 8;
    L.meta_bytes = (L.o_num + L.nb * 4 + 15) & ~size_t(15);
    L.dpad = ((L.dbytes + 15) & ~size_t(15)) + 48;
    return L;
}
// Validates the block table of v and writes its uid_off table (nblocks + 1 words) to h_uoff.
static int pack_scan_blocks(const dgx_pack_view* v, uint64_t* h_uoff, uint64_t* exact_len, uint32_t* max_num_out) {
    const size_t nb = v ? v->nblocks : 0;
    uint64_t acc = 0;
    uint32_t max_num = 0;
    for (size_t i = 0; i < nb; ++i) {
        h_uoff[i] = acc;  // uid_off: exclusive prefix of NumUids, every block's output offset
        const uint32_t num = v->num_uids[i];
        acc += num;
        max_num = std::max(max_num, num);
        // The kernels trust the block table: offsets must ascend and every block must hold at least
        // the 5-byte minimum of each group its NumUids needs (ceil((n-1)/4), codec.go:76-96).  A pack
        // that fails this is refused (the shim stays on the Go path) instead of being walked.
        const uint64_t b0 = v->delta_off[i], b1 = v->delta_off[i + 1];
        const uint64_t need = num > 1 ? 5ull * ((uint64_t)(num + 2) / 4) : 0;
        if (b1 < b0 || b1 - b0 < need)
            return fail(DGX_ERR_ARG, "malformed UidPack: block %zu has %lld delta bytes, NumUids %u needs >= %llu",
                        i, (long long)(b1 - b0), num, (unsigned long long)need);
    }
    h_uoff[nb] = acc;
    *exact_len = acc;
    *max_num_out = max_num;
    return DGX_OK;
}
// Writes the metadata image at h (L.meta_bytes) and validates the block table.
static int pack_fill_meta(const dgx_pack_view* v, const PackLayout& L, char* h, uint64_t* exact_len, uint32_t* max_num) {
    const size_t nb = L.nb;
    if (int rc = pack_scan_blocks(v, (uint64_t*)(h + L.o_uoff), exact_len, max_num)) return rc;
    if (nb) {
        memcpy(h, v->base, nb * 8);
        memcpy(h + L.o_doff, v->delta_off, (nb + 1) * 8);
        memcpy(h + L.o_num, v->num_uids, nb * 4);
    } else {
        memset(h + L.o_doff, 0, 8);
    }
    return DGX_OK;
}
static void pack_point(dgx_dev_pack* out, const dgx_pack_view* v, const PackLayout& L, char* d_meta, char* d_deltas,
                       uint64_t exact_len, uint32_t max_num) {
    out->pk.nblocks = L.nb;
    out->pk.base = (const u64*)d_meta;
    out->pk.delta_off = (const u64*)(d_meta + L.o_doff);
    out->pk.uid_off = (const u64*)(d_meta + L.o_uoff);
    out->pk.num = (const u32*)(d_meta + L.o_num);
    out->pk.deltas = (const unsigned char*)d_deltas;
    out->pk.max_num = max_num;
    out->bytes = L.meta_bytes + L.dpad;
    out->exact_len = exact_len;
    out->block_size = v ? v->block_size : 0;
}

// One pack -> one device allocation (cudaMalloc when arena == nullptr: the caller owns out->d_mem).
static int pack_upload_impl(dgx_lane* l, const dgx_pack_view* v, void* d_mem_or_null, DevArena* arena,
                            dgx_dev_pack* out) {
    const PackLayout L = pack_layout(v);
    const size_t total = L.meta_bytes + L.dpad;
    void* d_mem = d_mem_or_null;
    int rc;
    if (!d_mem) {
        if (arena) { rc = arena->alloc(total, &d_mem); if (rc) return rc; }
        else {
            cudaError_t e = cudaMalloc(&d_mem, total);
            if (e != cudaSuccess) return fail(DGX_ERR_OOM, "cudaMalloc(%zu) failed: %s", total, cudaGetErrorString(e));
            out->d_mem = d_mem;  // owned by *out from here on, also when a later step fails
        }
    }
    void* h_raw;
    rc = l->host.alloc(L.meta_bytes, &h_raw);
    if (rc) return rc;
    uint64_t exact = 0;
    uint32_t max_num = 0;
    rc = pack_fill_meta(v, L, (char*)h_raw, &exact, &max_num);
    if (rc) return rc;
    char* d = (char*)d_mem;
    CK(cudaMemcpyAsync(d, h_raw, L.meta_bytes, cudaMemcpyHostToDevice, l->stream));
    if (L.dbytes) CK(cudaMemcpyAsync(d + L.meta_bytes, v->deltas, L.dbytes, cudaMemcpyHostToDevice, l->stream));
    g_stats.h2d += L.meta_bytes + L.dbytes;
    pack_point(out, v, L, d, d + L.meta_bytes, exact, max_num);
    out->d_mem = d_mem;
    return DGX_OK;
}

// The k packs of one call into the lane's workspace: one copy for all metadata images, one per pack
// for its delta bytes (straight from the caller's memory).  views[i] == nullptr entries are skipped.
// Flat image of a pack (dgx_pack_image_size / dgx_pack_image_view): [base u64 x nb | delta_off u64 x (nb+1) |
// num_uids u32 x nb | pad to 16 | deltas | pad to 16].  A shim that flattens pb.UidPack.Blocks into pinned staging
// memory writes this directly; images written back to back travel as ONE DMA transfer.
static size_t image_meta_bytes(size_t nb) { return (nb * 8 + (nb + 1) * 8 + nb * 4 + 15) & ~size_t(15); }
static bool view_is_image(const dgx_pack_view* v) {
    const size_t nb = v->nblocks;
    const char* b = (const char*)v->base;
    if (!b || (reinterpret_cast<uintptr_t>(b) & 15u)) return false;
    return (const char*)v->delta_off == b + nb * 8 && (const char*)v->num_uids == b + nb * 8 + (nb + 1) * 8 &&
           (const char*)v->deltas == b + image_meta_bytes(nb);
}
static size_t view_image_bytes(const dgx_pack_view* v) {
    return image_meta_bytes(v->nblocks) + (((size_t)v->delta_off[v->nblocks] + 15) & ~size_t(15));
}
// All packs of the call are images laid out back to back: one copy for the images, one for the uid_off tables.
static int packs_upload_run(dgx_lane* l, const dgx_pack_view* const* views, size_t k, dgx_dev_pack* outs, bool* done) {
    *done = false;
    const char* start = nullptr;
    const char* next = nullptr;
    size_t uoff_bytes = 0;
    for (size_t i = 0; i < k; ++i) {
        const dgx_pack_view* v = views[i];
        if (!v) continue;
        if (v->nblocks == 0 || !view_is_image(v)) return DGX_OK;
        if (!start) start = (const char*)v->base;
        else if ((const char*)v->base != next) return DGX_OK;
        next = (const char*)v->base + view_image_bytes(v);
        uoff_bytes += (v->nblocks + 1) * sizeof(uint64_t);
    }
    if (!start) return DGX_OK;
    const size_t run = (size_t)(next - start);
    void *d_img, *d_uoff, *h_uoff;
    int rc = l->ws.alloc(run + 64, &d_img);
    if (rc) return rc;
    rc = l->ws.alloc(uoff_bytes, &d_uoff);
    if (rc) return rc;
    rc = l->host.alloc(uoff_bytes, &h_uoff);
    if (rc) return rc;
    size_t uo = 0;
    for (size_t i = 0; i < k; ++i) {
        const dgx_pack_view* v = views[i];
        if (!v) continue;
        const size_t nb = v->nblocks;
        uint64_t exact = 0;
        uint32_t max_num = 0;
        rc = pack_scan_blocks(v, (uint64_t*)((char*)h_uoff + uo), &exact, &max_num);
        if (rc) return rc;
        char* d = (char*)d_img + ((const char*)v->base - start);
        dgx_dev_pack& P = outs[i];
        P.pk.nblocks = nb;
        P.pk.base = (const u64*)d;
        P.pk.delta_off = (const u64*)(d + nb * 8);
        P.pk.num = (const u32*)(d + nb * 8 + (nb + 1) * 8);
        P.pk.deltas = (const unsigned char*)(d + image_meta_bytes(nb));
        P.pk.uid_off = (const u64*)((char*)d_uoff + uo);
        P.pk.max_num = max_num;
        P.d_mem = nullptr;
        P.bytes = view_image_bytes(v);
        P.exact_len = exact;
        P.block_size = v->block_size;
        uo += (nb + 1) * sizeof(uint64_t);
    }
    CK(cudaMemcpyAsync(d_img, start, run, cudaMemcpyHostToDevice, l->stream));
    CK(cudaMemcpyAsync(d_uoff, h_uoff, uoff_bytes, cudaMemcpyHostToDevice, l->stream));
    g_stats.h2d += run + uoff_bytes;
    *done = true;
    return DGX_OK;
}

static int packs_upload_ws(dgx_lane* l, const dgx_pack_view* const* views, size_t k, dgx_dev_pack* outs) {
    {
        bool done = false;
        int rc0 = packs_upload_run(l, views, k, outs, &done);
        if (rc0 || done) return rc0;
    }
    std::vector<PackLayout> Ls(k);
    size_t meta_total = 0, del_total = 0;
    for (size_t i = 0; i < k; ++i) {
        if (!views[i]) continue;
        Ls[i] = pack_layout(views[i]);
        meta_total += Ls[i].meta_bytes;
        del_total += Ls[i].dpad;
    }
    if (meta_total == 0) return DGX_OK;
    void *d_raw, *h_raw;
    int rc = l->ws.alloc(meta_total + del_total, &d_raw);
    if (rc) return rc;
    rc = l->host.alloc(meta_total, &h_raw);
    if (rc) return rc;
    char* d_meta = (char*)d_raw;
    char* d_del = (char*)d_raw + meta_total;
    char* h = (char*)h_raw;
    size_t mo = 0, dof = 0;
    for (size_t i = 0; i < k; ++i) {
        if (!views[i]) continue;
        uint64_t exact = 0;
        uint32_t max_num = 0;
        rc = pack_fill_meta(views[i], Ls[i], h + mo, &exact, &max_num);
        if (rc) return rc;
        pack_point(&outs[i], views[i], Ls[i], d_meta + mo, d_del + dof, exact, max_num);
        outs[i].d_mem = nullptr;  // workspace memory: not owned
        mo += Ls[i].meta_bytes;
        dof += Ls[i].dpad;
    }
    CK(cudaMemcpyAsync(d_meta, h, meta_total, cudaMemcpyHostToDevice, l->stream));
    for (size_t i = 0; i < k; ++i)
        if (views[i] && Ls[i].dbytes)
            CK(cudaMemcpyAsync((void*)outs[i].pk.deltas, views[i]->deltas, Ls[i].dbytes, cudaMemcpyHostToDevice, l->stream));
    for (size_t i = 0; i < k; ++i)
        if (views[i]) g_stats.h2d += Ls[i].meta_bytes + Ls[i].dbytes;
    return DGX_OK;
}

extern "C" int dgx_dev_pack_upload(dgx_lane* l, const dgx_pack_view* v, dgx_dev_pack** out) {
    if (!l || !out) return fail(DGX_ERR_ARG, "null argument");
    CK(cudaSetDevice(l->device));
    dgx_dev_pack* pk = new dgx_dev_pack();
    int rc = pack_upload_impl(l, v, nullptr, nullptr, pk);
    // the pinned uid_off staging must outlive the async copy
    if (rc == DGX_OK && cudaStreamSynchronize(l->stream) != cudaSuccess) rc = fail(DGX_ERR_CUDA, "pack upload failed");
    if (rc) { dgx_dev_pack_free(pk); return rc; }
    *out = pk;
    return DGX_OK;
}
extern "C" void dgx_dev_pack_free(dgx_dev_pack* pk) {
    if (!pk) return;
    if (pk->d_mem) cudaFree(pk->d_mem);
    delete pk;
}
extern "C" size_t dgx_dev_pack_exact_len(const dgx_dev_pack* pk) { return pk ? pk->exact_len : 0; }
extern "C" size_t dgx_dev_pack_bytes(const dgx_dev_pack* pk) { return pk ? pk->bytes : 0; }

static int decode_impl(dgx_lane* l, const DPack& pk, uint64_t seek, uint64_t* d_out, size_t out_cap,
                       uint64_t* d_out_len) {
    void* d_seek;
    int rc = l->ws.alloc(sizeof(DSeek), &d_seek);
    if (rc) return rc;
    decode_seek_kernel<<<1, 32, 0, l->stream>>>(pk, seek, (DSeek*)d_seek, (u64*)d_out_len, out_cap, l->d_err);
    if (int e = launched(l)) return e;
    if (pk.nblocks) {
        const uint64_t warps = (pk.nblocks + D_BPW - 1) / D_BPW;
        const uint64_t ctas = (warps + D_WARPS - 1) / D_WARPS;
        decode_kernel<<<(unsigned)ctas, D_NT, sizeof(DWarpSmem) * D_WARPS, l->stream>>>(pk, (const DSeek*)d_seek, (u64*)d_out, out_cap);
        if (int e = launched(l)) return e;
    }
    return DGX_OK;
}

extern "C" int dgx_dev_decode(dgx_lane* l, const dgx_dev_pack* pk, uint64_t seek, uint64_t* d_out, size_t out_cap,
                              uint64_t* d_out_len) {
    if (!l || !pk) return fail(DGX_ERR_ARG, "null argument");
    if (int rc = lane_begin_op(l)) return rc;
    g_stats.calls += 1;
    g_stats.uids_in += pk->exact_len;
    const int rc = decode_impl(l, pk->pk, seek, d_out, out_cap, d_out_len);
    l->note_output(d_out, out_cap * sizeof(uint64_t));
    l->note_output(d_out_len, sizeof(uint64_t));
    return rc;
}

// ---------------------------------------------------------------------------
// host-pointer entry points
// ---------------------------------------------------------------------------
// Lanes of the host-pointer entry points.  The pool is bounded: at most kMaxLanes lanes exist (each keeps a stream,
// its workspace and pinned staging at their high-water mark), a caller beyond that waits for one to come back --
// hundreds of cgo goroutines cannot pin hundreds of arenas in HBM.  A lane whose workspace grew past kLaneTrimBytes is
// shrunk when it is returned (it is idle then: every host-pointer call ends with a stream sync).
constexpr size_t kMaxLanes = 32;
constexpr size_t kLaneTrimBytes = size_t(4) << 30;
struct LaneLease {
    dgx_lane* l = nullptr;
    int rc = DGX_OK;
    LaneLease() {
        rc = dgx_init(-1);
        if (rc) return;
        bool create = false;
        {
            std::unique_lock<std::mutex> lk(g_mu);
            g_pool_cv.wait(lk, [] { return !g_pool.empty() || g_lanes_total < kMaxLanes; });
            if (!g_pool.empty()) { l = g_pool.back(); g_pool.pop_back(); }
            else { create = true; g_lanes_total += 1; }
            g_lanes_out += 1;
        }
        if (create) {
            l = dgx_lane_create(g_device, nullptr);
            if (!l) {
                rc = fail(DGX_ERR_CUDA, "cannot create lane: %s", g_err.c_str());
                std::lock_guard<std::mutex> lk(g_mu);
                g_lanes_total -= 1;
                g_lanes_out -= 1;
                g_pool_cv.notify_all();
                return;
            }
        }
        cudaSetDevice(l->device);
        l->ws.reset();
    }
    ~LaneLease() {
        if (!l) return;
        if (l->ws.cap > kLaneTrimBytes) {  // idle (synchronised) lane: give a one-off large workspace back
            cudaStreamSynchronize(l->stream);
            l->ws.destroy();
        }
        std::lock_guard<std::mutex> lk(g_mu);
        g_pool.push_back(l);
        g_lanes_out -= 1;
        g_pool_cv.notify_all();
    }
};

static int upload_list(dgx_lane* l, const uint64_t* h, size_t n, uint64_t** d) {
    void* p;
    int rc = l->ws.alloc((n + 2) * sizeof(uint64_t), &p);
    if (rc) return rc;
    if (n) CK(cudaMemcpyAsync(p, h, n * sizeof(uint64_t), cudaMemcpyHostToDevice, l->stream));
    g_stats.h2d += n * sizeof(uint64_t);
    *d = (uint64_t*)p;
    return DGX_OK;
}

// Result to the host in ONE round trip when it is short: the length word and the first kSpecHead
// values (fewer if the device buffer is smaller) are copied speculatively before the sync; only a
// longer result pays a second copy for its tail.  d_cap = values allocated behind d_out.
static int finish_to_host(dgx_lane* l, const uint64_t* d_len, const uint64_t* d_out, size_t d_cap, uint64_t* out,
                          size_t out_cap, size_t* out_len) {
    const size_t head = std::min(std::min(d_cap, out_cap), kSpecHead);
    CK(cudaMemcpyAsync(l->h_word, d_len, sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    if (head) CK(cudaMemcpyAsync(l->h_head, d_out, head * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    int rc = dgx_lane_sync(l);
    if (rc) return rc;
    const uint64_t n = l->h_word[0];
    if (n > out_cap) return fail(DGX_ERR_CAP, "result (%llu) does not fit out_cap (%zu)", (unsigned long long)n, out_cap);
    if (n) memcpy(out, l->h_head, std::min<size_t>(n, head) * sizeof(uint64_t));
    if (n > head) {
        CK(cudaMemcpyAsync(out + head, d_out + head, (n - head) * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaStreamSynchronize(l->stream));
    }
    g_stats.d2h += std::max<uint64_t>(n, head) * sizeof(uint64_t) + 8;
    g_stats.uids_out += n;
    if (out_len) *out_len = (size_t)n;
    return DGX_OK;
}

static int filter_host(int op, const uint64_t* const* lists, const size_t* lens, size_t k, uint64_t* out,
                       size_t out_cap, size_t* out_len) {
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    std::vector<ListDesc> ld(k);
    size_t cap = SIZE_MAX;
    for (size_t i = 0; i < k; ++i) {
        uint64_t* d;
        int rc = upload_list(l, lists[i], lens[i], &d);
        if (rc) return rc;
        ld[i] = {d, lens[i], nullptr};
        if (op == DGX_OP_INTERSECT) cap = std::min(cap, lens[i]);
    }
    if (op == DGX_OP_DIFFERENCE) cap = lens[0];
    void *d_out, *d_off;
    int rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc(2 * sizeof(uint64_t), &d_off);
    if (rc) return rc;
    const size_t k_off[2] = {0, k};
    rc = filter_batch_impl(l, op, ld.data(), k_off, 1, (uint64_t*)d_out, cap, (uint64_t*)d_off);
    if (rc) return rc;
    return finish_to_host(l, (uint64_t*)d_off + 1, (uint64_t*)d_out, cap, out, out_cap, out_len);
}

extern "C" int dgx_intersect2(const uint64_t* u, size_t n, const uint64_t* v, size_t m, uint64_t* out,
                              size_t out_cap, size_t* out_len) {
    const uint64_t* lists[2] = {u, v};
    const size_t lens[2] = {n, m};
    return filter_host(DGX_OP_INTERSECT, lists, lens, 2, out, out_cap, out_len);
}

extern "C" int dgx_intersect_sorted(const uint64_t* const* lists, const size_t* lens, size_t k, uint64_t* out,
                                    size_t out_cap, size_t* out_len) {
    if (k == 0) {  // IntersectSorted of no lists is the empty list (algo/uidlist.go:298-300)
        if (out_len) *out_len = 0;
        return DGX_OK;
    }
    return filter_host(DGX_OP_INTERSECT, lists, lens, k, out, out_cap, out_len);
}

extern "C" int dgx_difference(const uint64_t* u, size_t n, const uint64_t* v, size_t m, uint64_t* out,
                              size_t out_cap, size_t* out_len) {
    const uint64_t* lists[2] = {u, v};
    const size_t lens[2] = {n, m};
    return filter_host(DGX_OP_DIFFERENCE, lists, lens, 2, out, out_cap, out_len);
}

extern "C" int dgx_merge_sorted(const uint64_t* const* lists, const size_t* lens, size_t k, uint64_t* out,
                                size_t out_cap, size_t* out_len) {
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    std::vector<ListDesc> ld(k);
    size_t total = 0;
    for (size_t i = 0; i < k; ++i) {
        if (lists[i] == nullptr || lens[i] == 0) { ld[i] = {nullptr, 0, nullptr}; continue; }
        uint64_t* d;
        int rc = upload_list(l, lists[i], lens[i], &d);
        if (rc) return rc;
        ld[i] = {d, lens[i], nullptr};
        total += lens[i];
    }
    void *d_out, *d_len;
    int rc = l->ws.alloc((total + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc(64, &d_len);
    if (rc) return rc;
    rc = merge_sorted_impl(l, ld.data(), k, (uint64_t*)d_out, total, (uint64_t*)d_len);
    if (rc) return rc;
    return finish_to_host(l, (uint64_t*)d_len, (uint64_t*)d_out, total, out, out_cap, out_len);
}

extern "C" int dgx_decode(const dgx_pack_view* p, uint64_t seek, uint64_t* out, size_t out_cap, size_t* out_len) {
    if (!p || p->nblocks == 0) {  // nil / empty pack decodes to the empty list (codec/codec.go:445-446)
        if (out_len) *out_len = 0;
        return DGX_OK;
    }
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    dgx_dev_pack pk;
    int rc = pack_upload_impl(l, p, nullptr, &l->ws, &pk);
    if (rc) return rc;
    g_stats.uids_in += pk.exact_len;
    void *d_out, *d_len;
    rc = l->ws.alloc((pk.exact_len + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc(64, &d_len);
    if (rc) return rc;
    rc = decode_impl(l, pk.pk, seek, (uint64_t*)d_out, pk.exact_len, (uint64_t*)d_len);
    if (rc) return rc;
    return finish_to_host(l, (uint64_t*)d_len, (uint64_t*)d_out, pk.exact_len, out, out_cap, out_len);
}

extern "C" int dgx_decode_intersect_sorted(const dgx_pack_view* p, uint64_t seek, const uint64_t* const* lists,
                                           const size_t* lens, size_t k, uint64_t* out, size_t out_cap,
                                           size_t* out_len) {
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    std::vector<ListDesc> ld(k + 1);
    int rc;
    size_t cap = SIZE_MAX;
    for (size_t i = 0; i < k; ++i) {
        uint64_t* d;
        rc = upload_list(l, lists[i], lens[i], &d);
        if (rc) return rc;
        ld[i + 1] = {d, lens[i], nullptr};
        cap = std::min(cap, lens[i]);
    }
    void *d_dec = nullptr, *d_len;
    rc = l->ws.alloc(64, &d_len);
    if (rc) return rc;
    size_t exact = 0;
    if (p && p->nblocks) {
        dgx_dev_pack pk;
        rc = pack_upload_impl(l, p, nullptr, &l->ws, &pk);
        if (rc) return rc;
        exact = pk.exact_len;
        rc = l->ws.alloc((exact + 2) * sizeof(uint64_t), &d_dec);
        if (rc) return rc;
        rc = decode_impl(l, pk.pk, seek, (uint64_t*)d_dec, exact, (uint64_t*)d_len);
        if (rc) return rc;
    } else {
        rc = l->ws.alloc(16, &d_dec);
        if (rc) return rc;
        CK(cudaMemsetAsync(d_len, 0, 8, l->stream));
    }
    g_stats.uids_in += exact;
    ld[0] = {(const uint64_t*)d_dec, exact, (const uint64_t*)d_len};
    cap = std::min(cap, exact);
    void *d_out, *d_off;
    rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc(2 * sizeof(uint64_t), &d_off);
    if (rc) return rc;
    const size_t k_off[2] = {0, k + 1};
    rc = filter_batch_impl(l, DGX_OP_INTERSECT, ld.data(), k_off, 1, (uint64_t*)d_out, cap, (uint64_t*)d_off);
    if (rc) return rc;
    return finish_to_host(l, (uint64_t*)d_off + 1, (uint64_t*)d_out, cap, out, out_cap, out_len);
}

// algo.IntersectCompressedWith on the device (compressed_kernel.cuh): v-ranges of the blocks, decode +
// probe of the touched blocks in shared memory, order-preserving compaction of v.
static int icw_impl(dgx_lane* l, const dgx_dev_pack& pk, uint64_t after, const uint64_t* d_v, size_t m,
                    uint64_t* d_out, size_t out_cap, uint64_t* d_len) {
    const size_t nb = pk.pk.nblocks;
    if (nb == 0 || m == 0) {
        CK(cudaMemsetAsync(d_len, 0, sizeof(uint64_t), l->stream));
        return DGX_OK;
    }
    const size_t tiles = (m + CP_TILE - 1) / CP_TILE;
    const size_t b_rng = ((2 * nb * sizeof(u32)) + 15) & ~size_t(15);
    const size_t b_keep = (m + 15) & ~size_t(15);
    const size_t b_stat = tiles * sizeof(u64) + 64;
    void* d_raw;
    int rc = l->ws.alloc(b_rng + b_keep + b_stat, &d_raw);
    if (rc) return rc;
    CK(cudaMemsetAsync(d_raw, 0, b_rng + b_keep + b_stat, l->stream));
    IcwParams P;
    P.pk = pk.pk;
    P.v = (const u64*)d_v;
    P.m = m;
    P.after = after;
    P.vlo = (u32*)d_raw;
    P.vhi = P.vlo + nb;
    P.keep = (unsigned char*)d_raw + b_rng;
    // search the shorter side's elements in the longer side (the reference's linVsBinRatio idea, :49-59)
    if (m < nb) icw_ranges_by_v_kernel<<<(unsigned)((m + 255) / 256), 256, 0, l->stream>>>(P);
    else icw_ranges_by_block_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    const uint64_t warps = (nb + D_BPW - 1) / D_BPW;
    icw_probe_kernel<<<(unsigned)((warps + D_WARPS - 1) / D_WARPS), D_NT, sizeof(DWarpSmem) * D_WARPS, l->stream>>>(P);
    if (int e = launched(l)) return e;
    CompactParams C;
    C.v = (const u64*)d_v;
    C.keep = P.keep;
    C.m = m;
    C.out = (u64*)d_out;
    C.out_cap = out_cap;
    C.out_len = (u64*)d_len;
    C.status = (u64*)((char*)d_raw + b_rng + b_keep);
    C.ticket = (u32*)((char*)d_raw + b_rng + b_keep + tiles * sizeof(u64));
    C.err = l->d_err;
    compact_kernel<<<(unsigned)tiles, CP_NT, 0, l->stream>>>(C);
    if (int e = launched(l)) return e;
    g_stats.uids_in += pk.exact_len + m;
    return DGX_OK;
}

struct PackLease;
static int intersect_compressed_host(const dgx_pack_ref& ref, uint64_t after_uid, const uint64_t* v, size_t m,
                                     uint64_t* out, size_t out_cap, size_t* out_len);

extern "C" int dgx_intersect_compressed(const dgx_pack_view* p, uint64_t after_uid, const uint64_t* v, size_t m,
                                        uint64_t* out, size_t out_cap, size_t* out_len) {
    const dgx_pack_ref ref = {p, 0, 0};
    return intersect_compressed_host(ref, after_uid, v, m, out, out_cap, out_len);
}
extern "C" int dgx_intersect_compressed_ref(const dgx_pack_ref* ref, uint64_t after_uid, const uint64_t* v, size_t m,
                                            uint64_t* out, size_t out_cap, size_t* out_len) {
    if (!ref) return fail(DGX_ERR_ARG, "null ref");
    return intersect_compressed_host(*ref, after_uid, v, m, out, out_cap, out_len);
}

// ---------------------------------------------------------------------------
// HBM-resident pack cache + IntersectSorted over packs
// ---------------------------------------------------------------------------
// Production holds posting lists as UidPacks (posting.List.plist.Pack, posting/list.go:1795-1800) and
// decodes them per query.  Here a pack crosses PCIe compressed (about 1.5 B/UID instead of 8) and is
// expanded on the device; a pack the caller names with (key, version) -- immutable bytes, e.g. the hash
// of its Badger key and the commit timestamp of the layer -- stays in HBM in its compressed form and
// later calls skip the copy.  Eviction is LRU by bytes; entries in use by a running call are pinned.
static size_t pack_device_bytes(const dgx_pack_view* v) {
    const PackLayout L = pack_layout(v);
    return L.meta_bytes + L.dpad;
}

struct CacheKey {
    uint64_t key, version;
    bool operator==(const CacheKey& o) const { return key == o.key && version == o.version; }
};
struct CacheKeyHash {
    size_t operator()(const CacheKey& k) const {
        uint64_t h = k.key * 0x9E3779B97F4A7C15ull ^ (k.version + 0x7F4A7C15ull + (k.key << 6) + (k.key >> 2));
        return (size_t)(h ^ (h >> 29));
    }
};
struct CacheEntry {
    CacheKey id;
    dgx_dev_pack pk;
    cudaEvent_t ready = nullptr;  // recorded after the upload: other streams wait on it before reading
    int refs = 0;
    std::list<CacheEntry*>::iterator lru;
};
static std::mutex g_cache_mu;
static std::unordered_map<CacheKey, CacheEntry*, CacheKeyHash> g_cache;
static std::list<CacheEntry*> g_cache_lru;  // front = most recently used
static size_t g_cache_bytes = 0;
static size_t g_cache_max = size_t(32) << 30;  // DGX_CACHE_BYTES / dgx_cache_configure
static bool g_cache_env_read = false;
static dgx_cache_stats g_cache_stats = {0, 0, 0, 0, 0, 0};

static void cache_free_entry(CacheEntry* e) {
    // refs == 0: every call that used the entry has synchronised its stream, nothing queued reads it
    if (e->pk.d_mem) cudaFree(e->pk.d_mem);
    if (e->ready) cudaEventDestroy(e->ready);
    g_cache_bytes -= e->pk.bytes;
    delete e;
}
// g_cache_mu held.  Drops least-recently-used idle entries until `extra` more bytes fit.
static void cache_make_room(size_t extra) {
    auto it = g_cache_lru.end();
    while (g_cache_bytes + extra > g_cache_max && it != g_cache_lru.begin()) {
        --it;
        CacheEntry* e = *it;
        if (e->refs > 0) continue;
        it = g_cache_lru.erase(it);
        g_cache.erase(e->id);
        cache_free_entry(e);
        g_cache_stats.evictions += 1;
    }
}

extern "C" int dgx_cache_configure(size_t max_bytes) {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    g_cache_env_read = true;
    g_cache_max = max_bytes;
    cache_make_room(0);
    return DGX_OK;
}
extern "C" void dgx_cache_clear(void) {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    const size_t keep = g_cache_max;
    g_cache_max = 0;
    cache_make_room(0);
    g_cache_max = keep;
}
extern "C" void dgx_cache_get_stats(dgx_cache_stats* out) {
    if (!out) return;
    std::lock_guard<std::mutex> lk(g_cache_mu);
    *out = g_cache_stats;
    out->bytes = g_cache_bytes;
    out->entries = g_cache.size();
    out->max_bytes = g_cache_max;
}

// A pack made available to lane `l`: from the cache (entry != nullptr, one reference held) or copied
// into the lane's workspace for this call only.
struct PackLease {
    dgx_dev_pack pk;
    CacheEntry* entry = nullptr;
};
static void pack_release(PackLease& pl) {
    if (!pl.entry) return;
    std::lock_guard<std::mutex> lk(g_cache_mu);
    pl.entry->refs -= 1;
    pl.entry = nullptr;
}
static int pack_acquire(dgx_lane* l, const dgx_pack_ref& ref, PackLease* out, bool* deferred) {
    *deferred = false;
    const dgx_pack_view* v = ref.pack;
    if (ref.key != 0) {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        if (!g_cache_env_read) {
            g_cache_env_read = true;
            if (const char* s = getenv("DGX_CACHE_BYTES")) g_cache_max = (size_t)strtoull(s, nullptr, 10);
        }
        const CacheKey id{ref.key, ref.version};
        auto it = g_cache.find(id);
        if (it != g_cache.end()) {
            CacheEntry* e = it->second;
            e->refs += 1;
            g_cache_lru.erase(e->lru);
            g_cache_lru.push_front(e);
            e->lru = g_cache_lru.begin();
            g_cache_stats.hits += 1;
            CK(cudaStreamWaitEvent(l->stream, e->ready, 0));
            out->pk = e->pk;
            out->entry = e;
            return DGX_OK;
        }
        g_cache_stats.misses += 1;
        const size_t bytes = pack_device_bytes(v);
        if (v && bytes <= g_cache_max) {
            cache_make_room(bytes);
            if (g_cache_bytes + bytes <= g_cache_max) {
                CacheEntry* e = new CacheEntry();
                e->id = id;
                // the enqueue (a handful of async copies) happens under the lock so that a second caller
                // asking for the same pack finds the recorded event, never a half-built entry
                int rc = pack_upload_impl(l, v, nullptr, nullptr, &e->pk);
                if (rc == DGX_OK && (cudaEventCreateWithFlags(&e->ready, cudaEventDisableTiming) != cudaSuccess ||
                                     cudaEventRecord(e->ready, l->stream) != cudaSuccess))
                    rc = fail(DGX_ERR_CUDA, "cache event failed");
                if (rc) {
                    if (e->pk.d_mem) cudaFree(e->pk.d_mem);
                    if (e->ready) cudaEventDestroy(e->ready);
                    delete e;
                    return rc;
                }
                e->refs = 1;
                g_cache_bytes += e->pk.bytes;
                g_cache_lru.push_front(e);
                e->lru = g_cache_lru.begin();
                g_cache.emplace(id, e);
                out->pk = e->pk;
                out->entry = e;
                return DGX_OK;
            }
        }
        // does not fit (cache disabled, pack larger than the cache, everything pinned): one-shot copy
    }
    *deferred = true;  // copied into the lane's workspace together with the call's other one-shot packs
    return DGX_OK;
}

// Decode every pack of `pls` in full, side by side, with one launch; d_lists[i] receives pack i.
static int decode_batch_impl(dgx_lane* l, const PackLease* pls, size_t k, uint64_t** d_lists) {
    void *h_raw, *d_raw;
    int rc = l->host.alloc(k * sizeof(DJob), &h_raw);
    if (rc) return rc;
    rc = l->ws.alloc(k * sizeof(DJob), &d_raw);
    if (rc) return rc;
    DJob* hj = (DJob*)h_raw;
    u64 warps = 0;
    u32 nj = 0;
    for (size_t i = 0; i < k; ++i) {
        void* d;
        rc = l->ws.alloc((pls[i].pk.exact_len + 2) * sizeof(uint64_t), &d);
        if (rc) return rc;
        d_lists[i] = (uint64_t*)d;
        if (pls[i].pk.pk.nblocks == 0) continue;
        hj[nj].pk = pls[i].pk.pk;
        hj[nj].out = (u64*)d;
        hj[nj].warp_base = warps;
        warps += (pls[i].pk.pk.nblocks + D_BPW - 1) / D_BPW;
        ++nj;
        g_stats.uids_in += pls[i].pk.exact_len;
    }
    if (nj == 0) return DGX_OK;
    CK(cudaMemcpyAsync(d_raw, h_raw, nj * sizeof(DJob), cudaMemcpyHostToDevice, l->stream));
    const u64 ctas = (warps + D_WARPS - 1) / D_WARPS;
    if (ctas > 0x7fffffffull) return fail(DGX_ERR_ARG, "packs too large for one decode launch");
    decode_batch_kernel<<<(unsigned)ctas, D_NT, sizeof(DWarpSmem) * D_WARPS, l->stream>>>((const DJob*)d_raw, nj, warps);
    if (int e = launched(l)) return e;
    return DGX_OK;
}

extern "C" int dgx_intersect_sorted_packed(const dgx_pack_ref* refs, size_t k, uint64_t* out, size_t out_cap,
                                           size_t* out_len) {
    if (out_len) *out_len = 0;
    if (k == 0) return DGX_OK;  // IntersectSorted of no lists (algo/uidlist.go:298-300)
    if (!refs) return fail(DGX_ERR_ARG, "null refs");
    for (size_t i = 0; i < k; ++i)  // a nil / empty pack decodes to the empty list: the intersection is empty
        if (!refs[i].pack || refs[i].pack->nblocks == 0) return DGX_OK;
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    std::vector<PackLease> pls(k);
    std::vector<uint64_t*> d_lists(k, nullptr);
    int rc = DGX_OK;
    size_t got = 0;
    std::vector<const dgx_pack_view*> oneshot(k, nullptr);
    for (; got < k && rc == DGX_OK; ++got) {
        bool deferred = false;
        rc = pack_acquire(l, refs[got], &pls[got], &deferred);
        if (deferred) oneshot[got] = refs[got].pack;
    }
    if (rc == DGX_OK) {
        std::vector<dgx_dev_pack> up(k);
        rc = packs_upload_ws(l, oneshot.data(), k, up.data());
        for (size_t i = 0; i < k && rc == DGX_OK; ++i)
            if (oneshot[i]) pls[i].pk = up[i];
    }
    if (rc == DGX_OK) rc = decode_batch_impl(l, pls.data(), k, d_lists.data());
    size_t cap = SIZE_MAX;
    void *d_out = nullptr, *d_off = nullptr;
    if (rc == DGX_OK) {
        std::vector<ListDesc> ld(k);
        for (size_t i = 0; i < k; ++i) {
            ld[i] = {d_lists[i], pls[i].pk.exact_len, nullptr};
            cap = std::min(cap, pls[i].pk.exact_len);
        }
        rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
        if (rc == DGX_OK) rc = l->ws.alloc(2 * sizeof(uint64_t), &d_off);
        const size_t k_off[2] = {0, k};
        if (rc == DGX_OK) rc = filter_batch_impl(l, DGX_OP_INTERSECT, ld.data(), k_off, 1, (uint64_t*)d_out, cap, (uint64_t*)d_off);
    }
    if (rc == DGX_OK) rc = finish_to_host(l, (uint64_t*)d_off + 1, (uint64_t*)d_out, cap, out, out_cap, out_len);
    else cudaStreamSynchronize(l->stream);  // nothing queued may outlive the references released below
    for (size_t i = 0; i < got; ++i) pack_release(pls[i]);
    return rc;
}

static int intersect_compressed_host(const dgx_pack_ref& ref, uint64_t after_uid, const uint64_t* v, size_t m,
                                     uint64_t* out, size_t out_cap, size_t* out_len) {
    if (out_len) *out_len = 0;
    if (ref.pack == nullptr) return DGX_OK;  // `if pack == nil { return }` (algo/uidlist.go:34-36): o is left untouched
    if (m >= (size_t(1) << 32)) {             // v-ranges are 32-bit: beyond that, decode from the seek and filter
        const uint64_t* lists[1] = {v};
        const size_t lens[1] = {m};
        return dgx_decode_intersect_sorted(ref.pack, after_uid, lists, lens, 1, out, out_cap, out_len);
    }
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    PackLease pl;
    bool deferred = false;
    int rc = pack_acquire(l, ref, &pl, &deferred);
    if (rc == DGX_OK && deferred) rc = pack_upload_impl(l, ref.pack, nullptr, &l->ws, &pl.pk);
    uint64_t* d_v = nullptr;
    void *d_out = nullptr, *d_len = nullptr;
    if (rc == DGX_OK) rc = upload_list(l, v, m, &d_v);
    if (rc == DGX_OK) rc = l->ws.alloc((m + 2) * sizeof(uint64_t), &d_out);
    if (rc == DGX_OK) rc = l->ws.alloc(64, &d_len);
    if (rc == DGX_OK) rc = icw_impl(l, pl.pk, after_uid, d_v, m, (uint64_t*)d_out, m, (uint64_t*)d_len);
    if (rc == DGX_OK) rc = finish_to_host(l, (uint64_t*)d_len, (uint64_t*)d_out, m, out, out_cap, out_len);
    else cudaStreamSynchronize(l->stream);
    pack_release(pl);
    return rc;
}

// Decoder.Seek / SeekToBlock / LinearSeek / Next / UnpackBlock for one call (codec/codec.go:154-384), on the device.
extern "C" int dgx_pack_seek(const dgx_pack_view* p, int kind, uint64_t uid, int whence, size_t block_idx,
                             uint64_t* out, size_t out_cap, size_t* out_len, size_t* block_idx_after) {
    if (out_len) *out_len = 0;
    if (block_idx_after) *block_idx_after = 0;
    if (!p || p->nblocks == 0) return DGX_OK;  // nil pack: every seek returns an empty slice
    if (kind < SK_SEEK || kind > SK_UNPACK || (whence != 0 && whence != 1)) return fail(DGX_ERR_ARG, "bad seek kind / whence");
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    dgx_dev_pack pk;
    int rc = pack_upload_impl(l, p, nullptr, &l->ws, &pk);
    if (rc) return rc;
    void *d_out, *d_meta;
    const size_t cap = std::max<size_t>(pk.pk.max_num, 1);
    rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc(64, &d_meta);
    if (rc) return rc;
    SeekParams S;
    S.pk = pk.pk;
    S.uid = uid;
    S.whence = whence;
    S.kind = kind;
    S.block_idx = block_idx;
    S.out = (u64*)d_out;
    S.out_meta = (u64*)d_meta;
    pack_seek_kernel<<<1, 32, 0, l->stream>>>(S);
    if (int e = launched(l)) return e;
    CK(cudaMemcpyAsync(l->h_word, d_meta, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    CK(cudaMemcpyAsync(l->h_head, d_out, std::min(cap, kSpecHead) * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    rc = dgx_lane_sync(l);
    if (rc) return rc;
    const uint64_t n = l->h_word[0];
    if (block_idx_after) *block_idx_after = (size_t)l->h_word[1];
    if (n > out_cap) return fail(DGX_ERR_CAP, "block (%llu uids) does not fit out_cap (%zu)", (unsigned long long)n, out_cap);
    if (n > kSpecHead) {
        CK(cudaMemcpyAsync(out, d_out, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaStreamSynchronize(l->stream));
    } else if (n) {
        memcpy(out, l->h_head, n * sizeof(uint64_t));
    }
    if (out_len) *out_len = (size_t)n;
    return DGX_OK;
}

// ---------------------------------------------------------------------------
// codec.Encode on the device, packed set operations
// ---------------------------------------------------------------------------
extern "C" size_t dgx_pack_image_size(size_t nblocks, size_t delta_bytes) {
    return image_meta_bytes(nblocks) + ((delta_bytes + 15) & ~size_t(15));
}
extern "C" int dgx_pack_image_view(void* image, uint32_t block_size, size_t nblocks, size_t delta_bytes, dgx_pack_view* view) {
    (void)delta_bytes;
    if (!image || !view || (reinterpret_cast<uintptr_t>(image) & 15u)) return fail(DGX_ERR_ARG, "image must be 16-byte aligned");
    char* b = (char*)image;
    view->block_size = block_size;
    view->nblocks = nblocks;
    view->base = (const uint64_t*)b;
    view->delta_off = (const uint64_t*)(b + nblocks * 8);
    view->num_uids = (const uint32_t*)(b + nblocks * 8 + (nblocks + 1) * 8);
    view->deltas = (const uint8_t*)(b + image_meta_bytes(nblocks));
    return DGX_OK;
}

extern "C" void dgx_encode_bound(size_t n, uint32_t block_size, size_t* nblocks_cap, size_t* delta_cap) {
    const size_t B = block_size ? block_size : 1;
    // a sorted list crosses a multiple of 2^32 rarely: room for 64 extra (short) blocks; dgx_encode reports the
    // exact need with DGX_ERR_CAP when a list has more upper-word changes than that
    const size_t nb = n ? (n + B - 1) / B + 64 : 0;
    if (nblocks_cap) *nblocks_cap = nb;
    if (delta_cap) *delta_cap = 17 * (n / 4 + nb + 1);  // every group is at most 17 bytes
}

struct EncOut {           // device arrays of one encoded pack (workspace memory)
    u64* base; u32* num; u64* delta_off; unsigned char* deltas; u64* counts;
    size_t nblocks_cap, delta_cap;
};
// Encodes d_u[0..n) (n from *d_n when d_n != nullptr, at most n) into workspace arrays.
static int encode_impl(dgx_lane* l, const uint64_t* d_u, size_t n, const uint64_t* d_n, uint32_t block_size,
                       size_t nblocks_cap, size_t delta_cap, EncOut* out) {
    const size_t tiles_a = std::max<size_t>(1, (n + EN_TILE - 1) / EN_TILE);
    const size_t tiles_b = std::max<size_t>(1, (nblocks_cap + EN_TILE - 1) / EN_TILE);
    // workspace: [counts 8w | tickets | err][status_a][status_b] zeroed; seg arrays, block arrays
    const size_t z_bytes = 128 + (tiles_a + tiles_b) * sizeof(u64);
    void *d_z, *d_seg, *d_blk, *d_del;
    int rc = l->ws.alloc(z_bytes, &d_z);
    if (rc) return rc;
    const size_t seg_cap = std::min<size_t>(n, nblocks_cap) + 2;  // more segments than blocks cannot fit anyway
    rc = l->ws.alloc(2 * seg_cap * sizeof(u64), &d_seg);
    if (rc) return rc;
    rc = l->ws.alloc((nblocks_cap + 1) * (4 * sizeof(u64) + sizeof(u32)) + 64, &d_blk);
    if (rc) return rc;
    rc = l->ws.alloc(delta_cap + 64, &d_del);
    if (rc) return rc;
    CK(cudaMemsetAsync(d_z, 0, z_bytes, l->stream));
    EncParams P;
    P.u = (const u64*)d_u;
    P.n = n;
    P.n_dyn = (const u64*)d_n;
    P.bsz = block_size ? block_size : 1;
    P.counts = (u64*)d_z;
    P.ticket = (u32*)((char*)d_z + 64);
    P.err = (int*)((char*)d_z + 96);
    P.status = (u64*)((char*)d_z + 128);
    u64* status_b = P.status + tiles_a;
    P.seg_start = (u64*)d_seg;
    P.seg_cap = seg_cap;
    P.seg_blk = P.seg_start + seg_cap;
    P.nblocks_cap = nblocks_cap;
    char* bp = (char*)d_blk;
    P.base = (u64*)bp; bp += (nblocks_cap + 1) * sizeof(u64);
    P.blk_start = (u64*)bp; bp += (nblocks_cap + 1) * sizeof(u64);
    P.blk_bytes = (u64*)bp; bp += (nblocks_cap + 1) * sizeof(u64);
    P.delta_off = (u64*)bp; bp += (nblocks_cap + 1) * sizeof(u64);
    P.num = (u32*)bp;
    P.deltas = (unsigned char*)d_del;
    P.delta_cap = delta_cap;
    // a list with more segments than seg_cap cannot be encoded into nblocks_cap blocks: the segment pass would
    // overrun its array, so it is bounded by the same capacity check (segments <= blocks)
    enc_segments_kernel<<<(unsigned)tiles_a, EN_NT, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    enc_segscan_kernel<<<1, 1024, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    const size_t warp_ctas = std::max<size_t>(1, (nblocks_cap * 32 + 255) / 256);
    enc_sizes_kernel<<<(unsigned)warp_ctas, 256, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    scan_u64_kernel<<<(unsigned)tiles_b, EN_NT, 0, l->stream>>>(P.blk_bytes, P.delta_off, P.counts + 1, nblocks_cap, status_b,
                                                               P.ticket + 1, P.counts + 2);
    if (int e = launched(l)) return e;
    enc_write_kernel<<<(unsigned)warp_ctas, 256, 0, l->stream>>>(P);
    if (int e = launched(l)) return e;
    out->base = P.base; out->num = P.num; out->delta_off = P.delta_off; out->deltas = P.deltas; out->counts = P.counts;
    out->nblocks_cap = nblocks_cap; out->delta_cap = delta_cap;
    return DGX_OK;
}

// counts + arrays of an encoded pack to the caller's arrays.  *nblocks / *delta_bytes: capacity in, size out.
static int encode_to_host(dgx_lane* l, const EncOut& E, uint32_t block_size, uint64_t* base, uint32_t* num_uids,
                          uint64_t* delta_off, uint8_t* deltas, size_t* nblocks, size_t* delta_bytes, dgx_pack_view* view) {
    CK(cudaMemcpyAsync(l->h_word, E.counts, 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    int rc = dgx_lane_sync(l);
    if (rc) return rc;
    const uint64_t nb = l->h_word[1], db = l->h_word[2];
    const size_t cap_nb = *nblocks, cap_db = *delta_bytes;
    *nblocks = (size_t)nb;
    *delta_bytes = (size_t)db;
    if (nb > cap_nb || nb > E.nblocks_cap || db > cap_db || db > E.delta_cap)
        return fail(DGX_ERR_CAP, "pack needs %llu blocks / %llu delta bytes (given %zu / %zu): sizes returned, call again",
                    (unsigned long long)nb, (unsigned long long)db, cap_nb, cap_db);
    if (nb) {
        CK(cudaMemcpyAsync(base, E.base, nb * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaMemcpyAsync(num_uids, E.num, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaMemcpyAsync(delta_off, E.delta_off, (nb + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
        if (db) CK(cudaMemcpyAsync(deltas, E.deltas, db, cudaMemcpyDeviceToHost, l->stream));
        CK(cudaStreamSynchronize(l->stream));
    } else if (delta_off) {
        delta_off[0] = 0;
    }
    g_stats.d2h += nb * 20 + db + 32;
    if (view) {
        view->block_size = block_size;
        view->nblocks = (size_t)nb;
        view->base = base;
        view->num_uids = num_uids;
        view->delta_off = delta_off;
        view->deltas = deltas;
    }
    return DGX_OK;
}

extern "C" int dgx_encode(const uint64_t* uids, size_t n, uint32_t block_size, uint64_t* base, uint32_t* num_uids,
                          uint64_t* delta_off, uint8_t* deltas, size_t* nblocks, size_t* delta_bytes, dgx_pack_view* view) {
    if (!nblocks || !delta_bytes) return fail(DGX_ERR_ARG, "null capacity arguments");
    if (n == 0) {  // Encoder.Done without Add: the nil pack (codec/codec.go:125-136)
        *nblocks = 0; *delta_bytes = 0;
        if (view) { view->block_size = block_size; view->nblocks = 0; view->base = base; view->num_uids = num_uids; view->delta_off = delta_off; view->deltas = deltas; }
        if (delta_off) delta_off[0] = 0;
        return DGX_OK;
    }
    if (!uids || !base || !num_uids || !delta_off || !deltas) return fail(DGX_ERR_ARG, "null argument");
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    g_stats.uids_in += n;
    uint64_t* d_u;
    int rc = upload_list(l, uids, n, &d_u);
    if (rc) return rc;
    EncOut E;
    rc = encode_impl(l, d_u, n, nullptr, block_size, *nblocks, *delta_bytes, &E);
    if (rc) return rc;
    return encode_to_host(l, E, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
}

// algo.IntersectWithLinPacked / DifferencePacked / MergeSortedPacked (algo/packed.go:35-297) by composition on
// the device: decode the operands side by side, run the plain-list kernel, encode the result -- operands and
// result cross PCIe compressed and nothing decoded leaves the device.  The reference's block-at-a-time loops
// have three behaviours its own tests never reach (oracle/packed.py, DESIGN section 5: IntersectSortedPacked
// keeps only ls[0] ∩ ls[1], DifferencePacked's handling of v running out of blocks); these entry points compute
// the set operation the function names, which is what every case of algo/packed_test.go expects.
static int packed_op_host(int kind /*0 intersect, 1 difference, 2 merge*/, const dgx_pack_ref* refs, size_t k,
                          uint32_t block_size, uint64_t* base, uint32_t* num_uids, uint64_t* delta_off, uint8_t* deltas,
                          size_t* nblocks, size_t* delta_bytes, dgx_pack_view* view) {
    if (!nblocks || !delta_bytes) return fail(DGX_ERR_ARG, "null capacity arguments");
    if (k && !refs) return fail(DGX_ERR_ARG, "null refs");
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    std::vector<PackLease> pls(k);
    std::vector<uint64_t*> d_lists(k, nullptr);
    std::vector<const dgx_pack_view*> oneshot(k, nullptr);
    int rc = DGX_OK;
    size_t got = 0;
    static const dgx_pack_view kEmpty = {0, 0, nullptr, nullptr, nullptr, nullptr};
    for (; got < k && rc == DGX_OK; ++got) {
        dgx_pack_ref r = refs[got];
        if (!r.pack || r.pack->nblocks == 0) { r.pack = &kEmpty; r.key = 0; }
        bool deferred = false;
        rc = pack_acquire(l, r, &pls[got], &deferred);
        if (deferred) oneshot[got] = r.pack;
    }
    if (rc == DGX_OK) {
        for (size_t i = 0; i < k; ++i)  // an empty view has no delta_off array: give the layout code a zero
            if (oneshot[i] == &kEmpty) oneshot[i] = nullptr;
        std::vector<dgx_dev_pack> up(k);
        rc = packs_upload_ws(l, oneshot.data(), k, up.data());
        for (size_t i = 0; i < k && rc == DGX_OK; ++i)
            if (oneshot[i]) pls[i].pk = up[i];
            else if (!pls[i].entry) { pls[i].pk = dgx_dev_pack(); pls[i].pk.pk = DPack(); pls[i].pk.pk.nblocks = 0; pls[i].pk.exact_len = 0; }
    }
    if (rc == DGX_OK) rc = decode_batch_impl(l, pls.data(), k, d_lists.data());
    size_t cap = 0;
    void *d_out = nullptr, *d_len = nullptr;
    if (rc == DGX_OK) {
        std::vector<ListDesc> ld(k);
        size_t mn = SIZE_MAX, total = 0;
        for (size_t i = 0; i < k; ++i) {
            ld[i] = {d_lists[i], pls[i].pk.exact_len, nullptr};
            mn = std::min(mn, pls[i].pk.exact_len);
            total += pls[i].pk.exact_len;
        }
        cap = kind == 0 ? (k ? mn : 0) : (kind == 1 ? (k ? pls[0].pk.exact_len : 0) : total);
        rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
        void* d_off = nullptr;
        if (rc == DGX_OK) rc = l->ws.alloc(64, &d_off);
        if (rc == DGX_OK) {
            if (kind == 2) {
                d_len = d_off;
                rc = merge_sorted_impl(l, ld.data(), k, (uint64_t*)d_out, cap, (uint64_t*)d_len);
            } else if (k == 0) {
                d_len = d_off;
                CK(cudaMemsetAsync(d_len, 0, 8, l->stream));
            } else {
                const size_t k_off[2] = {0, k};
                rc = filter_batch_impl(l, kind == 0 ? DGX_OP_INTERSECT : DGX_OP_DIFFERENCE, ld.data(), k_off, 1,
                                       (uint64_t*)d_out, cap, (uint64_t*)d_off);
                d_len = (uint64_t*)d_off + 1;
            }
        }
    }
    EncOut E;
    if (rc == DGX_OK) {
        size_t nb_cap, db_cap;
        dgx_encode_bound(cap, block_size, &nb_cap, &db_cap);
        nb_cap = std::max(nb_cap, std::min(*nblocks, cap));  // a larger capacity from the caller is honoured
        rc = encode_impl(l, (const uint64_t*)d_out, cap, (const uint64_t*)d_len, block_size, nb_cap, db_cap, &E);
    }
    if (rc == DGX_OK) rc = encode_to_host(l, E, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
    else cudaStreamSynchronize(l->stream);
    for (size_t i = 0; i < got; ++i) pack_release(pls[i]);
    return rc;
}

extern "C" int dgx_intersect_packed(const dgx_pack_ref* u, const dgx_pack_ref* v, uint32_t block_size, uint64_t* base,
                                    uint32_t* num_uids, uint64_t* delta_off, uint8_t* deltas, size_t* nblocks,
                                    size_t* delta_bytes, dgx_pack_view* view) {
    if (!u || !v) return fail(DGX_ERR_ARG, "null ref");
    const dgx_pack_ref refs[2] = {*u, *v};
    return packed_op_host(0, refs, 2, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
}
extern "C" int dgx_difference_packed(const dgx_pack_ref* u, const dgx_pack_ref* v, uint32_t block_size, uint64_t* base,
                                     uint32_t* num_uids, uint64_t* delta_off, uint8_t* deltas, size_t* nblocks,
                                     size_t* delta_bytes, dgx_pack_view* view) {
    if (!u || !v) return fail(DGX_ERR_ARG, "null ref");
    const dgx_pack_ref refs[2] = {*u, *v};
    return packed_op_host(1, refs, 2, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
}
extern "C" int dgx_merge_sorted_packed(const dgx_pack_ref* refs, size_t k, uint32_t block_size, uint64_t* base,
                                       uint32_t* num_uids, uint64_t* delta_off, uint8_t* deltas, size_t* nblocks,
                                       size_t* delta_bytes, dgx_pack_view* view) {
    return packed_op_host(2, refs, k, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
}
extern "C" int dgx_intersect_sorted_packed_out(const dgx_pack_ref* refs, size_t k, uint32_t block_size, uint64_t* base,
                                               uint32_t* num_uids, uint64_t* delta_off, uint8_t* deltas, size_t* nblocks,
                                               size_t* delta_bytes, dgx_pack_view* view) {
    return packed_op_host(0, refs, k, block_size, base, num_uids, delta_off, deltas, nblocks, delta_bytes, view);
}

// ---------------------------------------------------------------------------
// IndexOf batch, shared-list batch
// ---------------------------------------------------------------------------
extern "C" int dgx_index_of_batch(const uint64_t* u, size_t n, const uint64_t* uids, size_t m, int64_t* idx) {
    if (m == 0) return DGX_OK;
    if (!uids || !idx || (n && !u)) return fail(DGX_ERR_ARG, "null argument");
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    uint64_t *d_u, *d_q;
    void* d_idx;
    int rc = upload_list(l, u, n, &d_u);
    if (rc) return rc;
    rc = upload_list(l, uids, m, &d_q);
    if (rc) return rc;
    rc = l->ws.alloc(m * sizeof(int64_t), &d_idx);
    if (rc) return rc;
    const unsigned blocks = (unsigned)std::min<uint64_t>((m + 255) / 256, (uint64_t)g_num_sms * 16);
    index_of_kernel<<<blocks, 256, 0, l->stream>>>((const u64*)d_u, (u64)n, (const u64*)d_q, (u64)m, (long long*)d_idx);
    if (int e = launched(l)) return e;
    g_stats.uids_in += n + m;
    CK(cudaMemcpyAsync(idx, d_idx, m * sizeof(int64_t), cudaMemcpyDeviceToHost, l->stream));
    g_stats.d2h += m * sizeof(int64_t);
    return dgx_lane_sync(l);
}

static int batch_to_host(dgx_lane* l, const void* d_out, const void* d_off, size_t npairs, uint64_t* out,
                         uint64_t* out_off, size_t out_cap) {
    CK(cudaMemcpyAsync(out_off, d_off, (npairs + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
    int rc = dgx_lane_sync(l);
    if (rc) return rc;
    const uint64_t n = out_off[npairs];
    if (n > out_cap) return fail(DGX_ERR_CAP, "batch result (%llu) does not fit out_cap (%zu)", (unsigned long long)n, out_cap);
    if (n) {
        CK(cudaMemcpyAsync(out, d_out, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, l->stream));
        CK(cudaStreamSynchronize(l->stream));
    }
    g_stats.d2h += (n + npairs + 1) * sizeof(uint64_t);
    g_stats.uids_out += n;
    return DGX_OK;
}

// Intersects npairs pairs of uploaded lists and returns the results to the host.  List a of pair i is
// d_a[a_off[i] - a_off[0], a_off[i + 1] - a_off[0]), list b is the same slice of d_b through b_off[i * b_step]:
// b_step 1 gives every pair its own list b, b_step 0 gives all of them the one list [b_off[0], b_off[1]).
static int intersect_pairs(dgx_lane* l, const uint64_t* d_a, const uint64_t* a_off, const uint64_t* d_b,
                           const uint64_t* b_off, size_t b_step, size_t npairs, uint64_t* out, uint64_t* out_off,
                           size_t out_cap) {
    std::vector<ListDesc> ld(2 * npairs);
    std::vector<size_t> k_off(npairs + 1);
    size_t cap = 0;
    for (size_t i = 0; i < npairs; ++i) {
        const uint64_t* bo = b_off + i * b_step;
        const size_t la = a_off[i + 1] - a_off[i], lb = bo[1] - bo[0];
        ld[2 * i] = {d_a + (a_off[i] - a_off[0]), la, nullptr};
        ld[2 * i + 1] = {d_b + (bo[0] - b_off[0]), lb, nullptr};
        k_off[i] = 2 * i;
        cap += std::min(la, lb);
    }
    k_off[npairs] = 2 * npairs;
    void *d_out, *d_off;
    int rc = l->ws.alloc((cap + 2) * sizeof(uint64_t), &d_out);
    if (rc) return rc;
    rc = l->ws.alloc((npairs + 1) * sizeof(uint64_t), &d_off);
    if (rc) return rc;
    rc = filter_batch_impl(l, DGX_OP_INTERSECT, ld.data(), k_off.data(), npairs, (uint64_t*)d_out, cap, (uint64_t*)d_off);
    if (rc) return rc;
    return batch_to_host(l, d_out, d_off, npairs, out, out_off, out_cap);
}

extern "C" int dgx_intersect_batch(const uint64_t* a, const uint64_t* a_off, const uint64_t* b,
                                   const uint64_t* b_off, size_t npairs, uint64_t* out, uint64_t* out_off,
                                   size_t out_cap) {
    if (npairs == 0) { if (out_off) out_off[0] = 0; return DGX_OK; }
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    uint64_t *d_a, *d_b;
    int rc = upload_list(l, a + a_off[0], a_off[npairs] - a_off[0], &d_a);
    if (rc) return rc;
    rc = upload_list(l, b + b_off[0], b_off[npairs] - b_off[0], &d_b);
    if (rc) return rc;
    return intersect_pairs(l, d_a, a_off, d_b, b_off, 1, npairs, out, out_off, out_cap);
}

extern "C" int dgx_intersect_batch_shared(const uint64_t* a, const uint64_t* a_off, size_t npairs, const uint64_t* b,
                                          size_t m, uint64_t* out, uint64_t* out_off, size_t out_cap) {
    if (npairs == 0) { if (out_off) out_off[0] = 0; return DGX_OK; }
    if (!a_off || !out_off) return fail(DGX_ERR_ARG, "null argument");
    LaneLease lease;
    if (lease.rc) return lease.rc;
    dgx_lane* l = lease.l;
    g_stats.calls += 1;
    uint64_t *d_a, *d_b;
    int rc = upload_list(l, a + a_off[0], a_off[npairs] - a_off[0], &d_a);
    if (rc) return rc;
    rc = upload_list(l, b, m, &d_b);  // the shared list crosses PCIe once
    if (rc) return rc;
    const uint64_t b_off[2] = {0, m};
    return intersect_pairs(l, d_a, a_off, d_b, b_off, 0, npairs, out, out_off, out_cap);
}

// ---------------------------------------------------------------------------
// protobuf wire-format adjacency (host only; see include/dgx.h and wire.hpp)
// ---------------------------------------------------------------------------
extern "C" int dgx_wire_posting_list_pack(const uint8_t* buf, size_t len, const uint8_t** pack, size_t* pack_len) {
    if ((!buf && len) || !pack || !pack_len) return fail(DGX_ERR_ARG, "null argument");
    *pack = nullptr;
    *pack_len = 0;
    wire::Reader r{buf, buf + len};
    uint32_t f, wt;
    bool ok, seen = false;
    while (r.tag(&f, &wt, &ok)) {
        if (f == 1 && wt == 2) {
            // a sub-message split over several occurrences would have to be merged; no encoder emits that
            if (seen) return fail(DGX_ERR_ARG, "pb.PostingList.pack occurs more than once");
            if (!r.bytes(pack, pack_len)) return fail(DGX_ERR_ARG, "truncated pb.PostingList");
            seen = true;
        } else if (!r.skip(wt, f)) {
            return fail(DGX_ERR_ARG, "malformed pb.PostingList");
        }
    }
    if (!ok) return fail(DGX_ERR_ARG, "malformed pb.PostingList");
    return DGX_OK;
}

extern "C" int dgx_wire_pack_measure(const uint8_t* buf, size_t len, size_t* nblocks, size_t* delta_bytes) {
    if ((!buf && len) || !nblocks || !delta_bytes) return fail(DGX_ERR_ARG, "null argument");
    uint32_t bs;
    if (!wire::walk_pack(buf, len, &bs, nblocks, delta_bytes, nullptr)) return fail(DGX_ERR_ARG, "malformed pb.UidPack");
    return DGX_OK;
}

extern "C" int dgx_wire_pack_parse(const uint8_t* buf, size_t len, uint64_t* base, uint32_t* num_uids,
                                   uint64_t* delta_off, uint8_t* deltas, size_t nblocks_cap, size_t delta_cap,
                                   dgx_pack_view* view) {
    if ((!buf && len) || !view || !delta_off) return fail(DGX_ERR_ARG, "null argument");
    uint32_t bs;
    size_t nb, db;
    if (!wire::walk_pack(buf, len, &bs, &nb, &db, nullptr)) return fail(DGX_ERR_ARG, "malformed pb.UidPack");
    if (nb > nblocks_cap || db > delta_cap)
        return fail(DGX_ERR_CAP, "pb.UidPack has %zu blocks / %zu delta bytes, arrays hold %zu / %zu", nb, db, nblocks_cap, delta_cap);
    if ((nb && (!base || !num_uids)) || (db && !deltas)) return fail(DGX_ERR_ARG, "null array");
    const wire::PackArrays a{base, num_uids, delta_off, deltas};
    wire::walk_pack(buf, len, &bs, &nb, &db, &a);
    view->block_size = bs;
    view->nblocks = nb;
    view->base = base;
    view->num_uids = num_uids;
    view->delta_off = delta_off;
    view->deltas = deltas;
    return DGX_OK;
}

extern "C" size_t dgx_wire_list_header(size_t n, uint8_t* hdr) {
    if (n == 0 || !hdr) return 0;
    size_t w = 0;
    hdr[w++] = 0x0A;  // field 1, wire type 2
    uint64_t v = (uint64_t)n * 8u;
    while (v >= 0x80) { hdr[w++] = (uint8_t)(v | 0x80); v >>= 7; }
    hdr[w++] = (uint8_t)v;
    return w;
}

extern "C" int dgx_wire_uid_matrix(const uint64_t* out, const uint64_t* out_off, size_t nrows, uint8_t* buf, size_t buf_cap,
                                   size_t* len) {
    if (!len || (nrows && !out_off)) return fail(DGX_ERR_ARG, "null argument");
    auto varint_len = [](uint64_t v) { size_t n = 1; while (v >= 0x80) { v >>= 7; ++n; } return n; };
    auto put_varint = [](uint8_t* p, uint64_t v) { size_t n = 0; while (v >= 0x80) { p[n++] = (uint8_t)(v | 0x80); v >>= 7; } p[n++] = (uint8_t)v; return n; };
    size_t w = 0;
    for (size_t r = 0; r < nrows; ++r) {
        if (out_off[r + 1] < out_off[r]) return fail(DGX_ERR_ARG, "offsets are not ascending at row %zu", r);
        const uint64_t n = out_off[r + 1] - out_off[r];
        const uint64_t payload = n * 8;
        const uint64_t inner = n ? 1 + varint_len(payload) + payload : 0;  // the row's pb.List message
        const size_t total = 1 + varint_len(inner) + (size_t)inner;
        if (buf) {
            if (w + total > buf_cap) return fail(DGX_ERR_CAP, "uid_matrix does not fit buf_cap (%zu)", buf_cap);
            if (n && !out) return fail(DGX_ERR_ARG, "null values");
            uint8_t* p = buf + w;
            *p++ = 0x0A;
            p += put_varint(p, inner);
            if (n) {
                *p++ = 0x0A;
                p += put_varint(p, payload);
                memcpy(p, out + out_off[r], (size_t)payload);
            }
        }
        w += total;
    }
    *len = w;
    return DGX_OK;
}

extern "C" int dgx_wire_list_decode(const uint8_t* buf, size_t len, uint64_t* out, size_t out_cap, size_t* out_len) {
    if ((!buf && len) || !out_len) return fail(DGX_ERR_ARG, "null argument");
    wire::Reader r{buf, buf + len};
    uint32_t f, wt;
    bool ok;
    size_t n = 0;
    while (r.tag(&f, &wt, &ok)) {
        if (f == 1 && wt == 2) {
            const uint8_t* s;
            size_t nbytes;
            if (!r.bytes(&s, &nbytes) || (nbytes & 7)) return fail(DGX_ERR_ARG, "malformed pb.List");
            const size_t cnt = nbytes / 8;
            if (out) {
                if (n + cnt > out_cap) return fail(DGX_ERR_CAP, "pb.List does not fit out_cap (%zu)", out_cap);
                memcpy(out + n, s, nbytes);  // fixed64 is little-endian on the wire, like the hosts this runs on
            }
            n += cnt;
        } else if (f == 1 && wt == 1) {
            if (r.end - r.p < 8) return fail(DGX_ERR_ARG, "truncated pb.List");
            if (out) {
                if (n + 1 > out_cap) return fail(DGX_ERR_CAP, "pb.List does not fit out_cap (%zu)", out_cap);
                memcpy(out + n, r.p, 8);
            }
            r.p += 8;
            n += 1;
        } else if (!r.skip(wt, f)) {
            return fail(DGX_ERR_ARG, "malformed pb.List");
        }
    }
    if (!ok) return fail(DGX_ERR_ARG, "malformed pb.List");
    *out_len = n;
    return DGX_OK;
}

#ifdef DGX_PIPE_PROF
// Experimental builds only (not part of include/dgx.h): read and clear filter_pipe_kernel's wait counters.
extern "C" int dgx_debug_pprof(uint64_t* out16) {
    unsigned long long h[32];
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpyFromSymbol(h, dgx::g_pprof, sizeof(h)));
    for (int i = 0; i < 32; ++i) out16[i] = h[i];
    memset(h, 0, sizeof(h));
    CK(cudaMemcpyToSymbol(dgx::g_pprof, h, sizeof(h)));
    return DGX_OK;
}
#endif
