// gangpack_api.cu -- global kernels + the C ABI of include/gangpack.h.
// There is no CPU code path in this library: without a usable CUDA device gp_create fails.
#include "gangpack.h"
#include "gangpack_kernels.cuh"
#include "gangpack_fifo.cuh"
#include "gangpack_minfrag.cuh"
#include "gangpack_tables.cuh"
#include "gangpack_zones.cuh"
#include "gangpack_zonefifo.cuh"
#include "gangpack_resched.cuh"
#include "gangpack_sort.cuh"

#include <algorithm>
#include <chrono>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

using namespace gp;

// =============================================================================================
// kernels
// =============================================================================================

constexpr int kPrepThreads = 256;
// Thread per application: validate, derive the division magics and the driver-displacement bound (FIFO modes and
// minimal-fragmentation; independent tightly-pack / distribute-evenly prepare inside gp_pack_tables).
// Source tuple: types.SparkApplicationResources (internal/types/types.go:22-27).
__global__ void gp_prep_apps(int32_t n_apps, AppColumns cols, const uint8_t* __restrict__ skip,
                             int32_t n_groups, int64_t out_cap, const SnapMeta* __restrict__ meta,
                             GroupMin* __restrict__ gmins, PrepApp* __restrict__ prep, int* __restrict__ err,
                             volatile int* __restrict__ err_host) {
    // records are staged in shared memory and written out with fully coalesced 16-byte stores (a thread writing
    // its own 128-byte record would touch 32 different lines per warp-wide store)
    __shared__ uint4 stage[kPrepThreads * (sizeof(PrepApp) / sizeof(uint4))];
    const int32_t block0 = blockIdx.x * blockDim.x;
    int32_t i = block0 + threadIdx.x;
    const bool live = i < n_apps;
    if (!live) i = n_apps - 1;                      // keep the thread for the cooperative copy-out; its record is not stored
    int64_t d[3] = {cols.load(0, i), cols.load(1, i), cols.load(2, i)};
    int64_t e[3] = {cols.load(3, i), cols.load(4, i), cols.load(5, i)};
    int32_t k = cols.count[i];
    int32_t g = cols.group ? cols.group[i] : 0;
    int bad = 0;
    if (k < 0) bad |= kErrNegativeRequest;
    if (k > kMaxCount) bad |= kErrUnrepresentable;
    if (gmins && k > kMaxCountFifo) bad |= kErrUnrepresentable;   // FIFO modes: block-wide uint32 sums of clamped capacities stay exact
    if (g < 0 || g >= n_groups) bad |= kErrBadGroup;
    int64_t off = cols.off[i];
    if (off < 0 || cols.off[i + 1] - off != (int64_t)k || cols.off[i + 1] > out_cap) bad |= kErrBadOffsets;
    PrepApp p;
    uint64_t lmax = 0;
    bool fast = true;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        uint64_t l;
        p.drv[t] = d[t];
        p.div[t] = prep_dim(d[t], e[t], t, meta->max_avail[t], bad, l, fast);
        if (l > lmax) lmax = l;
    }
    if (bad && live) { atomicOr(err, bad); *err_host = bad; }   // err_host: mapped pinned word, no D2H copy needed
    if (bad) { k = 0; g = 0; }
    else if (gmins && live) {
        // batch-wide minima per instance group (FIFO dead-node skipping)
        GroupMin* gm = gmins + g;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            if (e[t] < gm->exe[t]) atomicMin(&gm->exe[t], (long long)e[t]);
            if (d[t] < gm->drv[t]) atomicMin(&gm->drv[t], (long long)d[t]);
        }
    }
    p.out_off = off;
    p.count = k;
    p.group = g;
    p.lmax = (int32_t)(lmax < (uint64_t)k ? lmax : (uint64_t)k);
    const bool fast32 = prep_fast32(fast, p.div[0], p.div[1], meta);
    p.flags = ((d[2] != 0 || e[2] != 0) ? kAppUsesGpu : 0u) | ((skip && skip[i]) ? kAppSkipIfNoFit : 0u) |
              (bad ? kAppInvalid : 0u) | (fast ? kAppFast : 0u) | (fast32 ? kAppFast32 : 0u);
    constexpr int kQ = sizeof(PrepApp) / sizeof(uint4);      // 8 x 16 bytes per record
    const uint4* src = reinterpret_cast<const uint4*>(&p);
#pragma unroll
    for (int w = 0; w < kQ; ++w) stage[threadIdx.x * kQ + w] = src[w];
    __syncthreads();
    const int32_t n_block = min((int32_t)blockDim.x, n_apps - block0);
    uint4* dst = reinterpret_cast<uint4*>(prep + block0);
    for (int32_t t = threadIdx.x; t < n_block * kQ; t += blockDim.x) dst[t] = stage[t];
}

// Independent minimal-fragmentation (independent tightly-pack / distribute-evenly take the tables, gangpack_tables.cuh):
// one warp per application; warps claim applications from a global counter (claim-then-broadcast, next index
// prefetched) so long scans do not leave a tail.
constexpr int kPackThreads = 256;
#ifndef GP_MF_MIN_BLOCKS
#define GP_MF_MIN_BLOCKS 4      // 64 registers (96 uncapped); measured 4.42 / 3.67 / 3.45 ms per 100 k decisions at 2 / 3 / 4 CTAs per SM
#endif
__global__ void __launch_bounds__(kPackThreads, GP_MF_MIN_BLOCKS) gp_pack_independent(Snapshot s, const PrepApp* __restrict__ prep, int32_t n_apps,
                                                                    int32_t* __restrict__ driver_node,
                                                                    int32_t* __restrict__ executor_nodes,
                                                                    int2* __restrict__ scratch,
                                                                    unsigned long long* __restrict__ stats,
                                                                    unsigned int* __restrict__ next_app) {
    const int lane = threadIdx.x & 31;
    WarpStats st{0, 0};
    const int snap_flags = s.meta->flags;          // per-kernel facts stay in registers
    // claim-then-broadcast, two applications ahead: while application i is packed, the index of i+2 is in
    // flight and the record of i+1 is being pulled into L1
    unsigned int i = 0, n1 = 0;
    if (lane == 0) { i = atomicAdd(next_app, 1u); n1 = atomicAdd(next_app, 1u); }
    i = __shfl_sync(kFull, i, 0);
    n1 = __shfl_sync(kFull, n1, 0);
    while (i < (unsigned int)n_apps) {
        unsigned int n2 = 0;
        if (lane == 0) n2 = atomicAdd(next_app, 1u);
        if (lane == 0 && n1 < (unsigned int)n_apps) asm volatile("prefetch.global.L1 [%0];" ::"l"(prep + n1));
        const PrepApp* pa = prep + i;
        int32_t d = -1;
        if (!(pa->flags & kAppInvalid)) {        // multi-pass, see gangpack_minfrag.cuh
            const bool gpu_idle = !(pa->flags & kAppUsesGpu) && !(snap_flags & kSnapGpuNegative);
            d = ((pa->flags & kAppFast32) && gpu_idle) ? pack_app_minfrag<true>(s, pa, executor_nodes, scratch, st, lane, snap_flags)
                                                       : pack_app_minfrag<false>(s, pa, executor_nodes, scratch, st, lane, snap_flags);
        }
        if (lane == 0) driver_node[i] = d;
        i = n1;
        n1 = __shfl_sync(kFull, n2, 0);
    }
    if (lane == 0) {
        atomicAdd(stats + 0, st.nodes);
        atomicAdd(stats + 1, st.drivers);
    }
}

// ---- snapshot construction -------------------------------------------------------------------
__device__ __forceinline__ int32_t find_group(const int32_t* off, int32_t n_groups, int32_t idx) {
    int32_t lo = 0, hi = n_groups - 1;
    while (lo < hi) {
        int32_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= idx) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// The slot layout is built by two kernels and nothing else (no memset, no copy node), so that a snapshot taken every
// Predicate costs two launches:
//   gp_snap_slots   executor slots, group descriptors, per-node inverse indices into both orders, and per-CTA partial
//                   maxima (every slot that gets written holds the values of a node of one of the two orders, so the
//                   snapshot-wide facts are a fold over both orders -- no need to know yet which driver takes a spare slot);
//   gp_snap_finish  SnapMeta from the partials, driver slots (spare slots included), node_slot with one writer per node,
//                   the compact view, and (gp_set_snapshot_device) the node-table copy.
// The inverse indices are never reset: inv[v] is believed only if the order holds v at that position.
// Both kernels bound the order lengths by exec_off[n_groups] / drv_off[n_groups]: gp_prepare_cluster passes upper bounds.
constexpr int kSnapThreads = 256;
constexpr int kSnapMaxParts = 256;          // grid bound of both kernels (grid-stride loops); partials gp_snap_finish folds

struct SnapPart { long long v[4]; };        // max(cpu, 0), max(mem, 0), max(gpu, 0), any gpu < 0

struct SnapLayout {
    int32_t n_exec, n_drv, n_groups, n_nodes, n_slots;     // n_exec / n_drv may be upper bounds
    const int32_t *exec_off, *drv_off, *exec_order, *drv_order;
    const int64_t *cpu, *mem, *gpu;                         // node table; gpu may be NULL (= 0)
    GroupDesc* groups;
    longlong2* pair;
    int64_t* sgpu;
    uint2* pair32;
    int32_t *slot_node, *node_slot, *drv_slot;
    int32_t *inv_exec, *inv_drv;                            // [n_nodes] each
    SnapPart* parts;                                        // [kSnapMaxParts]
    SnapMeta* meta;
    int64_t *copy_cpu, *copy_mem, *copy_gpu;                // node-table copy, or NULL
    __device__ __forceinline__ int32_t ne_all() const { return min(n_exec, exec_off[n_groups]); }
    __device__ __forceinline__ int32_t nd_all() const { return min(n_drv, drv_off[n_groups]); }
    __device__ __forceinline__ int64_t gpu_of(int32_t v) const { return gpu ? gpu[v] : 0; }
    __device__ __forceinline__ int32_t exec_slot(int32_t e) const {
        const int32_t g = find_group(exec_off, n_groups, e);
        return drv_off[g] + e;                              // exec_off[g] + drv_off[g] + (e - exec_off[g])
    }
    // position of node v in the executor order, or -1
    __device__ __forceinline__ int32_t exec_pos(int32_t v, int32_t ne) const {
        const int32_t e = inv_exec[v];
        return (e >= 0 && e < ne && exec_order[e] == v) ? e : -1;
    }
    // driver candidate j whose node has global executor slot es (-1: none): it uses that slot when it lies in the
    // driver's own group, else its spare slot ne + (j - dbase)
    struct DrvSlot { int32_t sbase, local, spare; };        // group base, group-local slot, global spare slot
    __device__ __forceinline__ DrvSlot driver_slot(int32_t j, int32_t es) const {
        const int32_t g = find_group(drv_off, n_groups, j);
        const int32_t sbase = exec_off[g] + drv_off[g], ne = exec_off[g + 1] - exec_off[g];
        const int32_t spare = ne + (j - drv_off[g]);
        return DrvSlot{sbase, (es >= sbase && es < sbase + ne) ? es - sbase : spare, sbase + spare};
    }
};

// max over the block of four non-negative values; the result is returned to every thread
__device__ __forceinline__ void block_max4(long long v[4]) {
    __shared__ long long s_red[kSnapThreads / 32][4];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) v[k] = max(v[k], __shfl_xor_sync(kFull, v[k], d));
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 4; ++k) s_red[w][k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        long long m = 0;
        for (int t = 0; t < kSnapThreads / 32; ++t) m = max(m, s_red[t][k]);
        v[k] = m;
    }
}

__device__ __forceinline__ void fold_node(long long v[4], int64_t cv, int64_t mv, int64_t gv) {
    v[0] = max(v[0], (long long)cv); v[1] = max(v[1], (long long)mv); v[2] = max(v[2], (long long)gv);
    if (gv < 0) v[3] = 1;
}

__global__ void __launch_bounds__(kSnapThreads) gp_snap_slots(SnapLayout L) {
    const int32_t ne = L.ne_all(), nd = L.nd_all();
    const int32_t n = max(max(ne, nd), L.n_groups);
    long long acc[4] = {0, 0, 0, 0};
    for (int32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        if (t < L.n_groups) {
            GroupDesc d;
            d.sbase = L.exec_off[t] + L.drv_off[t];
            d.ne = L.exec_off[t + 1] - L.exec_off[t];
            d.dbase = L.drv_off[t];
            d.nd = L.drv_off[t + 1] - L.drv_off[t];
            L.groups[t] = d;
        }
        if (t < ne) {             // executor-order entry t -> slot sbase + (t - exec_off[g])
            const int32_t slot = L.exec_slot(t);
            const int32_t v = L.exec_order[t];
            const int64_t cv = L.cpu[v], mv = L.mem[v], gv = L.gpu_of(v);
            L.pair[slot] = make_longlong2(cv, mv);
            L.sgpu[slot] = gv;
            L.slot_node[slot] = v;
            L.inv_exec[v] = t;
            fold_node(acc, cv, mv, gv);
        }
        if (t < nd) {             // driver-order entry: its slot is decided in gp_snap_finish
            const int32_t v = L.drv_order[t];
            L.inv_drv[v] = t;
            fold_node(acc, L.cpu[v], L.mem[v], L.gpu_of(v));
        }
    }
    block_max4(acc);
    if (threadIdx.x == 0) L.parts[blockIdx.x] = SnapPart{{acc[0], acc[1], acc[2], acc[3]}};
}

// compact view, 8 bytes per slot instead of 16 (negative availability -> 0: capacity 0 either way).  Its shifts are the
// smallest S with max_avail >> S < 2^32.
__device__ __forceinline__ int shift_for(long long mx) {
    if (mx <= 0) return 0;
    const int bits = 64 - __clzll(mx);
    return bits > 32 ? bits - 32 : 0;
}
__device__ __forceinline__ uint2 compact_pair(longlong2 v, int s0, int s1) {
    return make_uint2(v.x < 0 ? 0u : (uint32_t)((unsigned long long)v.x >> s0), v.y < 0 ? 0u : (uint32_t)((unsigned long long)v.y >> s1));
}

__global__ void __launch_bounds__(kSnapThreads) gp_snap_finish(SnapLayout L, int32_t n_parts) {
    long long acc[4] = {0, 0, 0, 0};
    for (int p = threadIdx.x; p < n_parts; p += blockDim.x)
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] = max(acc[k], L.parts[p].v[k]);
    block_max4(acc);
    const int s0 = shift_for(acc[0]), s1 = shift_for(acc[1]);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        SnapMeta m{};
        m.flags = acc[3] ? kSnapGpuNegative : 0;
        m.max_avail[0] = acc[0]; m.max_avail[1] = acc[1]; m.max_avail[2] = acc[2];
        m.shift32[0] = s0; m.shift32[1] = s1;
        *L.meta = m;
    }
    const int32_t ne = L.ne_all(), nd = L.nd_all();
    const int32_t used = min(L.exec_off[L.n_groups] + L.drv_off[L.n_groups], L.n_slots);
    const int32_t n = max(max(ne, nd), max(L.n_slots, L.n_nodes) + 1);
    for (int32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        if (t < nd) {             // driver candidate t: its executor slot, or its spare slot holding the node's values
            const int32_t v = L.drv_order[t];
            const int32_t e = L.exec_pos(v, ne);
            const SnapLayout::DrvSlot d = L.driver_slot(t, e >= 0 ? L.exec_slot(e) : -1);
            L.drv_slot[t] = d.local;
            if (d.sbase + d.local == d.spare) {
                const longlong2 pv = make_longlong2(L.cpu[v], L.mem[v]);
                L.pair[d.spare] = pv;
                L.sgpu[d.spare] = L.gpu_of(v);
                L.pair32[d.spare] = compact_pair(pv, s0, s1);
                L.slot_node[d.spare] = v;
            } else {
                L.slot_node[d.spare] = -1;              // unused spare slot
            }
        }
        if (t < ne) {
            const int32_t slot = L.exec_slot(t);
            L.pair32[slot] = compact_pair(L.pair[slot], s0, s1);
        }
        if (t >= used && t <= L.n_slots) L.slot_node[t] = -1;
        if (t < L.n_nodes) {      // one writer per node: its spare slot if it has one, else its executor slot, else -1
            const int32_t e = L.exec_pos(t, ne);
            int32_t slot = e >= 0 ? L.exec_slot(e) : -1;
            const int32_t j = L.inv_drv[t];
            if (j >= 0 && j < nd && L.drv_order[j] == t) {
                const SnapLayout::DrvSlot d = L.driver_slot(j, slot);
                slot = d.sbase + d.local;
            }
            L.node_slot[t] = slot;
            if (L.copy_cpu) { L.copy_cpu[t] = L.cpu[t]; L.copy_mem[t] = L.mem[t]; L.copy_gpu[t] = L.gpu_of(t); }
        } else if (t == L.n_nodes) {
            L.node_slot[t] = -1;
        }
    }
}

// Several small host->device copies in ONE launch: sources are mapped pinned host buffers read
// straight over PCIe (a chain of tiny DMA copies costs ~8-10 us each in stream order).
struct CopyJob { const void* src; void* dst; unsigned long long bytes; };
struct CopyJobs { CopyJob j[8]; int n; };
__global__ void gp_multi_copy(CopyJobs jobs) {
    for (int k = 0; k < jobs.n; ++k) {
        const unsigned long long words = jobs.j[k].bytes >> 2;     // every array here is a multiple of 4 bytes
        const unsigned int* src = static_cast<const unsigned int*>(jobs.j[k].src);
        unsigned int* dst = static_cast<unsigned int*>(jobs.j[k].dst);
        for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < words;
             i += (unsigned long long)gridDim.x * blockDim.x)
            dst[i] = src[i];
    }
}

// the compact view again after `pair` changed in place (FIFO packing, availability upkeep); thread 0 publishes the shifts
__global__ void gp_fill_pair32(int32_t n_slots, const longlong2* __restrict__ pair, SnapMeta* __restrict__ meta,
                               uint2* __restrict__ pair32) {
    const int s0 = shift_for(meta->max_avail[0]), s1 = shift_for(meta->max_avail[1]);
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { meta->shift32[0] = s0; meta->shift32[1] = s1; }
    if (i >= n_slots) return;
    pair32[i] = compact_pair(pair[i], s0, s1);
}

// slots -> node-table order (gp_get_snapshot)
__global__ void gp_scatter_slots(int32_t n_slots, const longlong2* __restrict__ pair, const int64_t* __restrict__ sgpu,
                                 const int32_t* __restrict__ slot_node,
                                 int64_t* __restrict__ cpu, int64_t* __restrict__ mem, int64_t* __restrict__ gpu) {
    int32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_slots) return;
    int32_t node = slot_node[s];
    if (node < 0) return;
    longlong2 v = pair[s];
    cpu[node] = v.x; mem[node] = v.y; gpu[node] = sgpu[s];
}

// =============================================================================================
// host side
// =============================================================================================

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// A fixed sequence of kernel launches / memsets that repeats with identical arguments (one Predicate after the other:
// same buffers, same batch shape) is captured ONCE into a CUDA graph and replayed with a single launch call -- the
// pipelined host path is bound by how fast the host thread can issue its calls, not by the GPU.  The key is the byte image
// of every argument of the sequence; it is captured when the same key is seen twice in a row.
struct GraphCache {
    cudaGraphExec_t exec = nullptr;
    std::vector<char> key, last_key;
    int launches = 0;
    void reset() { if (exec) cudaGraphExecDestroy(exec); exec = nullptr; key.clear(); last_key.clear(); }
};

static constexpr int32_t kChunkApps = 50000;       // apps per pipelined chunk of gp_pack_batch (~1.5 MB H2D, ~70 us of kernel)
static constexpr int32_t kZeroCopyOutApps = 8192;  // batches up to this size write results straight into mapped host memory

struct gp_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    static constexpr int kLanes = 3;       // H2D / kernels / D2H of consecutive chunks overlap across lanes
    static constexpr int kMaxChunks = 16;
    // what the kernels of one pack call report; pack_begin zeroes all of it with one memset
    struct DevStatus {
        int err;                              // kErr* bits
        unsigned long long stats[4];          // nodes scanned, drivers tried, scan-path applications, scan-path nodes
        unsigned int fifo_cursor;             // gp_pack_fifo_cta: next application in queue order
        unsigned int next_app[kMaxChunks];    // per pipelined chunk: next application claimed by the persistent pack kernels
    };
    // pinned host mirror: gp_last_stats copies the err / stats prefix of DevStatus into `dev`; the kernels also set
    // `err_word` through the mapping, so a pack call reads its validation errors after the stream sync without a copy
    struct HostStatus {
        DevStatus dev;
        volatile int err_word;
    };
    cudaStream_t lane[kLanes] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev[kMaxChunks][3] = {};    // per chunk: prep start, pack start, pack end
    cudaEvent_t ev_ready = nullptr, ev_done[kLanes] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_t0 = nullptr;           // GANGPACK_TRACE=2: start of the pipelined batch (timeline of the chunks on stderr)
    int ev_chunks = 0;
    std::string err;

    // snapshot
    bool have_snapshot = false;
    int32_t n_nodes = 0, n_groups = 0, n_exec = 0, n_drv = 0, n_slots = 0;
    DevBuf node_cpu, node_mem, node_gpu;        // node-table order (as given)
    DevBuf exec_off, drv_off, exec_order, drv_order;
    DevBuf pair, pair32, sgpu, slot_node, node_slot, drv_slot, groups, snap_flags;
    DevBuf snap_aux;                              // slot layout scratch (build_snapshot_device)

    // batch staging
    DevBuf a_quant, a_count, a_group, a_skip, a_off;   // a_quant: the six quantity columns, one pitched block
    DevBuf prep, r_driver, r_exec, scratch, gmin, sortbuf, usagebuf, reschedbuf;
    DevBuf status;                                // one DevStatus; never reallocated, so its address can key a graph
    HostStatus* status_host = nullptr;
    DevStatus* dev_status() const { return status.as<DevStatus>(); }
    std::vector<int64_t> host_off;
    std::vector<int32_t> v_owner;                 // gp_set_snapshot validation scratch (no per-call allocation)
    std::vector<uint8_t> v_seen_e, v_seen_d;
    std::vector<std::pair<const char*, size_t>> pinned_blocks;   // gp_alloc_pinned allocations (device-mapped under UVA)
    void* one_block = nullptr;                    // gp_pack_one staging (mapped pinned)
    size_t one_bytes = 0;
    int zero_copy = 1;                            // GANGPACK_ZERO_COPY=0 disables reading/writing mapped host buffers in kernels
    int use_tables = 1;                           // GANGPACK_TABLES=0: every independent decision takes the node-order scan
    bool async_snapshot = false;                  // gp_config.flags & GP_CFG_ASYNC_SNAPSHOT
    int chunk_apps = kChunkApps;                  // GANGPACK_CHUNK_APPS
    int trace = 0;                                // GANGPACK_TRACE=1: host-side phase timing on stderr
    int pack_ctas_per_sm = 0;                       // occupancy of gp_pack_independent on this device
    int tab_ctas_per_sm[2][2] = {{0, 0}, {0, 0}};   // occupancy of gp_pack_tables<ALGO, OUT>
    bool tab_attr_set[2] = {false, false};
    // per pipeline lane: shape hash + header, capacity tables, group totals, expansion lists, per-application shape slot
    struct TableSet { DevBuf hdr, table, total, expand, app_slot; } tabs[kLanes];
    bool record_events = true;                    // CUDA events around the kernels (gp_last_stats); the pipelined host path skips them
    int use_graphs = 1;                           // GANGPACK_GRAPHS=0: always issue the launches one by one
    GraphCache g_chunk[kMaxChunks + 1];           // per pipelined chunk (+1: an unchunked batch on the context's own stream): classify .. scan
    GraphCache g_snapshot;                        // slot layout of gp_set_snapshot
    DevBuf off_dev;                               // ExecutorNodes offsets derived on the device
    DevBuf fifo_list;                             // FIFO modes: per-instance-group application lists (queue order)
    DevBuf sched, zonebuf;                        // SchedulableResources [3][n_nodes]; staging of gp_pack_batch_zones
    bool have_sched = false;
    bool sort_attr_set = false;
    bool fifo_attr_set[2] = {false, false};       // dynamic shared-memory opt-in of gp_pack_fifo_cta<ALGO,*> done on this device

    gp_stats last{};
};

static thread_local std::string g_create_error;

static cudaError_t create_aux(gp_ctx* c) {
    cudaError_t e;
    for (auto& l : c->lane) if ((e = cudaStreamCreateWithFlags(&l, cudaStreamNonBlocking)) != cudaSuccess) return e;
    for (auto& row : c->ev) for (auto& ev : row) if ((e = cudaEventCreate(&ev)) != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&c->ev_ready, cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&c->ev_t0)) != cudaSuccess) return e;
    for (auto& ev : c->ev_done) if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    return cudaSuccess;
}

#define GP_CUDA(ctx, expr)                                                                     \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                   \
            return GP_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)

// issue(): enqueues the sequence on `st` and returns (status, launches).  See GraphCache.
template <class F>
static gp_status run_cached(gp_ctx* c, GraphCache& gc, const void* key, size_t kn, cudaStream_t st, F&& issue) {
    const char* kb = static_cast<const char*>(key);
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (!c->use_graphs || cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
        cudaGetLastError();
        int n = 0;
        gp_status s = issue(n);
        c->last.kernel_launches += n;
        return s;
    }
    if (gc.exec && gc.key.size() == kn && std::memcmp(gc.key.data(), kb, kn) == 0) {
        GP_CUDA(c, cudaGraphLaunch(gc.exec, st));
        c->last.kernel_launches += gc.launches;
        return GP_OK;
    }
    if (gc.last_key.size() == kn && std::memcmp(gc.last_key.data(), kb, kn) == 0 &&
        cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
        int n = 0;
        const gp_status s = issue(n);
        cudaGraph_t g = nullptr;
        const cudaError_t e = cudaStreamEndCapture(st, &g);
        if (s == GP_OK && e == cudaSuccess && g) {
            cudaGraphExec_t ex = nullptr;
            if (cudaGraphInstantiate(&ex, g, 0) == cudaSuccess) {
                if (gc.exec) cudaGraphExecDestroy(gc.exec);
                gc.exec = ex; gc.key.assign(kb, kb + kn); gc.launches = n;
                cudaGraphDestroy(g);
                GP_CUDA(c, cudaGraphLaunch(gc.exec, st));
                c->last.kernel_launches += n;
                return GP_OK;
            }
        }
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();                 // capture did not work out: issue directly below
        if (s != GP_OK) return s;
    } else {
        cudaGetLastError();
    }
    gc.last_key.assign(kb, kb + kn);
    int n = 0;
    gp_status s = issue(n);
    c->last.kernel_launches += n;
    return s;
}

// Device-visible alias of a host buffer, or nullptr.  Buffers from gp_alloc_pinned are known; anything
// else is asked of the driver (cudaHostRegister / cudaHostAlloc memory of the caller qualifies).
static const void* mapped_ptr(gp_ctx* c, const void* p, size_t bytes) {
    if (!p || !c->zero_copy) return nullptr;
    const char* q = static_cast<const char*>(p);
    for (const auto& b : c->pinned_blocks)
        if (q >= b.first && q + bytes <= b.first + b.second) return p;     // UVA: same address on the device
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (a.type == cudaMemoryTypeHost && a.devicePointer) return a.devicePointer;
    return nullptr;
}

static gp_status fail(gp_ctx* ctx, gp_status st, const std::string& msg) {
    ctx->err = msg;
    return st;
}

// Staging of the auxiliary entry points: stage() lays out every part(pointer, count) in one DevBuf, each sub-buffer
// 256-byte aligned, reserves the DevBuf once and points every pointer at its sub-buffer.  The same counts give the
// same addresses from one call to the next.
template <class T> struct Part { T** p; size_t n; };
template <class T> static Part<T> part(T*& p, size_t n) { return Part<T>{&p, n}; }
static size_t part_bytes(size_t bytes) { return (bytes + 255) & ~(size_t)255; }
template <class... T> static cudaError_t stage(DevBuf& buf, Part<T>... parts) {
    const cudaError_t e = buf.reserve((part_bytes(sizeof(T) * parts.n) + ... + 0));
    if (e != cudaSuccess) return e;
    char* at = buf.as<char>();
    ((*parts.p = reinterpret_cast<T*>(at), at += part_bytes(sizeof(T) * parts.n)), ...);
    return cudaSuccess;
}
// host -> device copy into a staged part; a NULL source (an optional column left out) copies nothing
static cudaError_t upload(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    return src ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
}

static Snapshot make_snapshot(const gp_ctx* c) {
    Snapshot s;
    s.pair = c->pair.as<longlong2>();
    s.pair32 = c->pair32.as<uint2>();
    s.gpu = c->sgpu.as<int64_t>();
    s.slot_node = c->slot_node.as<int32_t>();
    s.drv_slot = c->drv_slot.as<int32_t>();
    s.groups = c->groups.as<GroupDesc>();
    s.meta = c->snap_flags.as<SnapMeta>();
    s.gmins = nullptr;
    s.n_groups = c->n_groups;
    s.n_slots = c->n_slots;
    return s;
}

extern "C" {

int gp_abi_version(void) { return GP_ABI_VERSION; }

const char* gp_last_error(const gp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int gp_backend(const gp_ctx* ctx) { return ctx ? 1 : 0; }

gp_status gp_create(gp_ctx** out, const gp_config* cfg) {
    if (!out) { g_create_error = "gp_create: out is NULL"; return GP_ERR_INVALID; }
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_error = std::string("gp_create: no CUDA device (") + cudaGetErrorString(e) +
                         "); libgangpack has no CPU path";
        return GP_ERR_NO_DEVICE;
    }
    int dev = (cfg && cfg->device >= 0) ? cfg->device : -1;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= n) { g_create_error = "gp_create: device ordinal out of range"; return GP_ERR_INVALID; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, dev)) != cudaSuccess) {
        g_create_error = std::string("gp_create: cudaGetDeviceProperties: ") + cudaGetErrorString(e);
        return GP_ERR_CUDA;
    }
    if (prop.major != 10) {
        g_create_error = "gp_create: device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                         "; this library ships sm_100a code only";
        return GP_ERR_NO_DEVICE;
    }
    gp_ctx* c = new (std::nothrow) gp_ctx();
    if (!c) { g_create_error = "gp_create: out of memory"; return GP_ERR_INVALID; }
    c->device = dev;
    c->sm_count = prop.multiProcessorCount;
    c->async_snapshot = cfg && (cfg->flags & GP_CFG_ASYNC_SNAPSHOT);
    if (const char* z = std::getenv("GANGPACK_ZERO_COPY")) c->zero_copy = std::atoi(z);
    if (const char* z = std::getenv("GANGPACK_TABLES")) c->use_tables = std::atoi(z);
    if (const char* z = std::getenv("GANGPACK_GRAPHS")) c->use_graphs = std::atoi(z);
    if (const char* z = std::getenv("GANGPACK_CHUNK_APPS")) c->chunk_apps = std::max(1024, std::atoi(z));
    if (const char* z = std::getenv("GANGPACK_TRACE")) c->trace = std::atoi(z);
    void* status_host = nullptr;
    if ((e = cudaSetDevice(dev)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = create_aux(c)) != cudaSuccess ||
        (e = cudaHostAlloc(&status_host, sizeof(gp_ctx::HostStatus), cudaHostAllocDefault)) != cudaSuccess ||
        (e = c->status.reserve(sizeof(gp_ctx::DevStatus))) != cudaSuccess || (e = c->snap_flags.reserve(sizeof(SnapMeta))) != cudaSuccess) {
        g_create_error = std::string("gp_create: ") + cudaGetErrorString(e);
        delete c;
        return GP_ERR_CUDA;
    }
    c->status_host = static_cast<gp_ctx::HostStatus*>(status_host);
    *out = c;
    return GP_OK;
}

void gp_destroy(gp_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    DevBuf* bufs[] = {&c->node_cpu, &c->node_mem, &c->node_gpu, &c->exec_off, &c->drv_off, &c->exec_order, &c->drv_order,
                      &c->pair, &c->pair32, &c->sgpu, &c->slot_node, &c->node_slot, &c->drv_slot, &c->groups, &c->snap_flags, &c->snap_aux,
                      &c->a_quant, &c->a_count, &c->a_group, &c->a_skip, &c->a_off, &c->prep, &c->r_driver, &c->r_exec, &c->scratch,
                      &c->gmin, &c->sortbuf, &c->usagebuf, &c->reschedbuf, &c->status, &c->off_dev, &c->fifo_list, &c->sched, &c->zonebuf};
    for (DevBuf* b : bufs) b->release();
    for (auto& t : c->tabs) { t.hdr.release(); t.table.release(); t.total.release(); t.expand.release(); t.app_slot.release(); }
    for (auto& g : c->g_chunk) g.reset();
    c->g_snapshot.reset();
    if (c->status_host) cudaFreeHost(c->status_host);
    if (c->one_block) cudaFreeHost(c->one_block);
    for (auto& row : c->ev) for (cudaEvent_t e : row) if (e) cudaEventDestroy(e);
    if (c->ev_ready) cudaEventDestroy(c->ev_ready);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    for (cudaEvent_t e : c->ev_done) if (e) cudaEventDestroy(e);
    for (cudaStream_t l : c->lane) if (l) cudaStreamDestroy(l);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

gp_status gp_alloc_pinned(gp_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return GP_ERR_INVALID;
    GP_CUDA(ctx, cudaSetDevice(ctx->device));
    GP_CUDA(ctx, cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped));   // pinned for every device of the process (gp_multi)
    ctx->pinned_blocks.emplace_back(static_cast<const char*>(*out), bytes ? bytes : 1);
    return GP_OK;
}

gp_status gp_free_pinned(gp_ctx* ctx, void* p) {
    if (!ctx) return GP_ERR_INVALID;
    if (p) {
        for (size_t i = 0; i < ctx->pinned_blocks.size(); ++i)
            if (ctx->pinned_blocks[i].first == static_cast<const char*>(p)) { ctx->pinned_blocks.erase(ctx->pinned_blocks.begin() + (long)i); break; }
        GP_CUDA(ctx, cudaFreeHost(p));
    }
    return GP_OK;
}

gp_status gp_register_host(gp_ctx* ctx, void* p, size_t bytes) {
    if (!ctx || !p || !bytes) return GP_ERR_INVALID;
    GP_CUDA(ctx, cudaSetDevice(ctx->device));
    GP_CUDA(ctx, cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return GP_OK;
}

gp_status gp_unregister_host(gp_ctx* ctx, void* p) {
    if (!ctx || !p) return GP_ERR_INVALID;
    GP_CUDA(ctx, cudaSetDevice(ctx->device));
    GP_CUDA(ctx, cudaHostUnregister(p));
    return GP_OK;
}

void* gp_stream(gp_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

gp_status gp_synchronize(gp_ctx* ctx) {
    if (!ctx) return GP_ERR_INVALID;
    GP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return GP_OK;
}

}  // extern "C"

// ---- snapshot ---------------------------------------------------------------------------------

// Build the slot layout from DEVICE-resident gp_nodes arrays on `st` (gp_snap_slots + gp_snap_finish).  copy_nodes: the
// second kernel also copies the node table into node_cpu/mem/gpu (gp_set_snapshot_device; gp_set_snapshot has it there).
static gp_status build_snapshot_device(gp_ctx* c, const gp_nodes* dn, int32_t n_exec, int32_t n_drv, cudaStream_t st,
                                       bool copy_nodes = false) {
    const int32_t n_slots = n_exec + n_drv;
    GP_CUDA(c, c->pair.reserve(sizeof(longlong2) * (size_t)(n_slots + 1)));
    GP_CUDA(c, c->pair32.reserve(sizeof(uint2) * (size_t)(n_slots + 1)));
    GP_CUDA(c, c->sgpu.reserve(sizeof(int64_t) * (size_t)(n_slots + 1)));
    GP_CUDA(c, c->slot_node.reserve(sizeof(int32_t) * (size_t)(n_slots + 1)));
    GP_CUDA(c, c->node_slot.reserve(sizeof(int32_t) * (size_t)(dn->n_nodes + 1)));
    GP_CUDA(c, c->drv_slot.reserve(sizeof(int32_t) * (size_t)(n_drv + 1)));
    GP_CUDA(c, c->groups.reserve(sizeof(GroupDesc) * (size_t)dn->n_groups));
    // [per-CTA partials | inverse executor-order index | inverse driver-order index]
    GP_CUDA(c, c->snap_aux.reserve(sizeof(SnapPart) * (size_t)kSnapMaxParts + 2 * sizeof(int32_t) * (size_t)(dn->n_nodes + 1)));
    SnapLayout L;
    std::memset(&L, 0, sizeof(L));      // the record is also the graph key: no indeterminate padding
    L.n_exec = n_exec; L.n_drv = n_drv; L.n_groups = dn->n_groups; L.n_nodes = dn->n_nodes; L.n_slots = n_slots;
    L.exec_off = dn->exec_off; L.drv_off = dn->drv_off; L.exec_order = dn->exec_order; L.drv_order = dn->drv_order;
    L.cpu = dn->avail_cpu_milli; L.mem = dn->avail_mem_bytes; L.gpu = dn->avail_gpu;
    L.groups = c->groups.as<GroupDesc>(); L.pair = c->pair.as<longlong2>(); L.sgpu = c->sgpu.as<int64_t>();
    L.pair32 = c->pair32.as<uint2>(); L.slot_node = c->slot_node.as<int32_t>(); L.node_slot = c->node_slot.as<int32_t>();
    L.drv_slot = c->drv_slot.as<int32_t>(); L.meta = c->snap_flags.as<SnapMeta>();
    L.parts = c->snap_aux.as<SnapPart>();
    L.inv_exec = reinterpret_cast<int32_t*>(L.parts + kSnapMaxParts);
    L.inv_drv = L.inv_exec + (dn->n_nodes + 1);
    if (copy_nodes) { L.copy_cpu = c->node_cpu.as<int64_t>(); L.copy_mem = c->node_mem.as<int64_t>(); L.copy_gpu = c->node_gpu.as<int64_t>(); }
    auto grid = [](int64_t work) { return (int)std::max<int64_t>(1, std::min<int64_t>((work + kSnapThreads - 1) / kSnapThreads, kSnapMaxParts)); };
    const int g1 = grid(std::max<int64_t>(std::max(n_exec, n_drv), dn->n_groups));
    const int g2 = grid(std::max<int64_t>(std::max(n_exec, n_drv), (int64_t)std::max(n_slots, dn->n_nodes) + 1));
    // every argument of both launches: the layout record and the two grid sizes (which follow from it)
    gp_status rs = run_cached(c, c->g_snapshot, &L, sizeof(L), st, [&](int& launches) -> gp_status {
        gp_snap_slots<<<g1, kSnapThreads, 0, st>>>(L);
        gp_snap_finish<<<g2, kSnapThreads, 0, st>>>(L, g1);
        GP_CUDA(c, cudaGetLastError());
        launches = 0;       // (the snapshot layout is not part of a pack call's launch count)
        return GP_OK;
    });
    if (rs != GP_OK) return rs;
    c->n_nodes = dn->n_nodes; c->n_groups = dn->n_groups; c->n_exec = n_exec; c->n_drv = n_drv; c->n_slots = n_slots;
    c->have_snapshot = true;
    c->have_sched = false;               // SchedulableResources belong to a node table
    return GP_OK;
}

extern "C" {

gp_status gp_set_snapshot(gp_ctx* c, const gp_nodes* n) {
    if (!c) return GP_ERR_INVALID;
    if (!n || n->n_nodes < 0 || n->n_groups < 1 || !n->exec_off || !n->drv_off ||
        (n->n_nodes > 0 && (!n->avail_cpu_milli || !n->avail_mem_bytes)))
        return fail(c, GP_ERR_INVALID, "gp_set_snapshot: missing arrays or bad sizes");
    // ---- host validation (O(N)): offsets monotone, indices in range, one group per node, domain
    const int32_t G = n->n_groups;
    if (n->exec_off[0] != 0 || n->drv_off[0] != 0) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: offsets must start at 0");
    for (int32_t g = 0; g < G; ++g)
        if (n->exec_off[g + 1] < n->exec_off[g] || n->drv_off[g + 1] < n->drv_off[g])
            return fail(c, GP_ERR_INVALID, "gp_set_snapshot: offsets not monotone");
    const int32_t n_exec = n->exec_off[G], n_drv = n->drv_off[G];
    if ((n_exec > 0 && !n->exec_order) || (n_drv > 0 && !n->drv_order))
        return fail(c, GP_ERR_INVALID, "gp_set_snapshot: order arrays missing");
    {
        // owner[v] = 4 * group + (bit0: listed as executor candidate, bit1: listed as driver candidate); -1 = unseen
        std::vector<int32_t>& owner = c->v_owner;
        owner.assign((size_t)n->n_nodes, -1);
        const uint32_t N = (uint32_t)n->n_nodes;
        for (int32_t g = 0; g < G; ++g) {
            for (int32_t e = n->exec_off[g]; e < n->exec_off[g + 1]; ++e) {
                const uint32_t v = (uint32_t)n->exec_order[e];
                if (v >= N) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: exec_order index out of range");
                if (owner[v] >= 0) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: node listed twice in executor orders");
                owner[v] = 4 * g + 1;
            }
        }
        for (int32_t g = 0; g < G; ++g) {
            for (int32_t d = n->drv_off[g]; d < n->drv_off[g + 1]; ++d) {
                const uint32_t v = (uint32_t)n->drv_order[d];
                if (v >= N) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: drv_order index out of range");
                const int32_t o = owner[v];
                if (o >= 0 && (o & 2)) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: node listed twice in driver orders");
                if (o >= 0 && (o >> 2) != g) return fail(c, GP_ERR_INVALID, "gp_set_snapshot: node belongs to two instance groups");
                owner[v] = 4 * g + (o >= 0 ? (o & 3) : 0) + 2;
            }
        }
        // exact-int64 domain: branch-free so that the loop vectorises
        const int64_t* cols[3] = {n->avail_cpu_milli, n->avail_mem_bytes, n->avail_gpu};
        uint64_t out_of_domain = 0;
        for (int k = 0; k < 3; ++k) {
            const int64_t* p = cols[k];
            if (!p) continue;
            for (uint32_t i = 0; i < N; ++i) out_of_domain |= (uint64_t)(p[i] >= kMaxQuantity) | (uint64_t)(p[i] <= -kMaxQuantity);
        }
        if (out_of_domain) return fail(c, GP_ERR_UNREPRESENTABLE, "gp_set_snapshot: |quantity| >= 2^61");
    }
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t nb = sizeof(int64_t) * (size_t)(n->n_nodes + 1);
    GP_CUDA(c, c->node_cpu.reserve(nb)); GP_CUDA(c, c->node_mem.reserve(nb)); GP_CUDA(c, c->node_gpu.reserve(nb));
    GP_CUDA(c, c->exec_off.reserve(sizeof(int32_t) * (size_t)(G + 1)));
    GP_CUDA(c, c->drv_off.reserve(sizeof(int32_t) * (size_t)(G + 1)));
    GP_CUDA(c, c->exec_order.reserve(sizeof(int32_t) * (size_t)(n_exec + 1)));
    GP_CUDA(c, c->drv_order.reserve(sizeof(int32_t) * (size_t)(n_drv + 1)));
    const size_t vb = sizeof(int64_t) * (size_t)n->n_nodes;
    const size_t ob = sizeof(int32_t) * (size_t)(G + 1);
    // mapped pinned inputs: one gather-copy kernel reads them over PCIe instead of 7 chained DMA copies
    const void* m_cpu = mapped_ptr(c, n->avail_cpu_milli, vb);
    const void* m_mem = mapped_ptr(c, n->avail_mem_bytes, vb);
    const void* m_gpu = n->avail_gpu ? mapped_ptr(c, n->avail_gpu, vb) : nullptr;
    const void* m_eoff = mapped_ptr(c, n->exec_off, ob);
    const void* m_doff = mapped_ptr(c, n->drv_off, ob);
    const void* m_eord = n_exec ? mapped_ptr(c, n->exec_order, sizeof(int32_t) * (size_t)n_exec) : n->exec_order;
    const void* m_dord = n_drv ? mapped_ptr(c, n->drv_order, sizeof(int32_t) * (size_t)n_drv) : n->drv_order;
    const bool all_mapped = vb && m_cpu && m_mem && (!n->avail_gpu || m_gpu) && m_eoff && m_doff && (!n_exec || m_eord) && (!n_drv || m_dord);
    if (all_mapped) {
        CopyJobs jobs{};
        auto add = [&](const void* src, void* dst, size_t bytes) { if (bytes) jobs.j[jobs.n++] = CopyJob{src, dst, bytes}; };
        add(m_cpu, c->node_cpu.p, vb); add(m_mem, c->node_mem.p, vb);
        if (n->avail_gpu) add(m_gpu, c->node_gpu.p, vb);
        add(m_eoff, c->exec_off.p, ob); add(m_doff, c->drv_off.p, ob);
        add(m_eord, c->exec_order.p, sizeof(int32_t) * (size_t)n_exec);
        add(m_dord, c->drv_order.p, sizeof(int32_t) * (size_t)n_drv);
        if (!n->avail_gpu) GP_CUDA(c, cudaMemsetAsync(c->node_gpu.p, 0, vb, st));
        gp_multi_copy<<<c->sm_count, 512, 0, st>>>(jobs);
        GP_CUDA(c, cudaGetLastError());
    } else {
        if (vb) {
            GP_CUDA(c, cudaMemcpyAsync(c->node_cpu.p, n->avail_cpu_milli, vb, cudaMemcpyHostToDevice, st));
            GP_CUDA(c, cudaMemcpyAsync(c->node_mem.p, n->avail_mem_bytes, vb, cudaMemcpyHostToDevice, st));
            if (n->avail_gpu) GP_CUDA(c, cudaMemcpyAsync(c->node_gpu.p, n->avail_gpu, vb, cudaMemcpyHostToDevice, st));
            else GP_CUDA(c, cudaMemsetAsync(c->node_gpu.p, 0, vb, st));
        }
        GP_CUDA(c, cudaMemcpyAsync(c->exec_off.p, n->exec_off, ob, cudaMemcpyHostToDevice, st));
        GP_CUDA(c, cudaMemcpyAsync(c->drv_off.p, n->drv_off, ob, cudaMemcpyHostToDevice, st));
        if (n_exec) GP_CUDA(c, cudaMemcpyAsync(c->exec_order.p, n->exec_order, sizeof(int32_t) * (size_t)n_exec, cudaMemcpyHostToDevice, st));
        if (n_drv) GP_CUDA(c, cudaMemcpyAsync(c->drv_order.p, n->drv_order, sizeof(int32_t) * (size_t)n_drv, cudaMemcpyHostToDevice, st));
    }
    gp_nodes dn = *n;
    dn.avail_cpu_milli = c->node_cpu.as<int64_t>(); dn.avail_mem_bytes = c->node_mem.as<int64_t>();
    dn.avail_gpu = c->node_gpu.as<int64_t>();
    dn.exec_off = c->exec_off.as<int32_t>(); dn.drv_off = c->drv_off.as<int32_t>();
    dn.exec_order = c->exec_order.as<int32_t>(); dn.drv_order = c->drv_order.as<int32_t>();
    gp_status s = build_snapshot_device(c, &dn, n_exec, n_drv, st);
    if (s != GP_OK) return s;
    // GP_CFG_ASYNC_SNAPSHOT with page-locked inputs: return while the device is still reading them -- the upload and the
    // slot layout then overlap the H2D copies of the gp_pack_* call that follows
    if (!(c->async_snapshot && all_mapped)) GP_CUDA(c, cudaStreamSynchronize(st));   // the caller may reuse its host buffers
    return GP_OK;
}

gp_status gp_set_snapshot_device(gp_ctx* c, const gp_nodes* dn, int32_t n_exec, int32_t n_drv, void* stream) {
    if (!c) return GP_ERR_INVALID;
    if (!dn || dn->n_nodes < 0 || dn->n_groups < 1 || !dn->exec_off || !dn->drv_off || n_exec < 0 || n_drv < 0 ||
        (n_exec > 0 && !dn->exec_order) || (n_drv > 0 && !dn->drv_order))
        return fail(c, GP_ERR_INVALID, "gp_set_snapshot_device: missing arrays or bad sizes");
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    // keep a node-table copy so gp_get_snapshot can answer for nodes outside every group (written by gp_snap_finish)
    const size_t nb = sizeof(int64_t) * (size_t)(dn->n_nodes + 1);
    GP_CUDA(c, c->node_cpu.reserve(nb)); GP_CUDA(c, c->node_mem.reserve(nb)); GP_CUDA(c, c->node_gpu.reserve(nb));
    return build_snapshot_device(c, dn, n_exec, n_drv, st, true);
}

gp_status gp_get_snapshot(gp_ctx* c, int64_t* cpu, int64_t* mem, int64_t* gpu) {
    if (!c) return GP_ERR_INVALID;
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, "gp_get_snapshot: no snapshot");
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int T = 256;
    if (c->n_slots > 0)
        gp_scatter_slots<<<(c->n_slots + T - 1) / T, T, 0, st>>>(c->n_slots, c->pair.as<longlong2>(), c->sgpu.as<int64_t>(),
                                                                c->slot_node.as<int32_t>(), c->node_cpu.as<int64_t>(),
                                                                c->node_mem.as<int64_t>(), c->node_gpu.as<int64_t>());
    GP_CUDA(c, cudaGetLastError());
    const size_t vb = sizeof(int64_t) * (size_t)c->n_nodes;
    if (vb) {
        if (cpu) GP_CUDA(c, cudaMemcpyAsync(cpu, c->node_cpu.p, vb, cudaMemcpyDeviceToHost, st));
        if (mem) GP_CUDA(c, cudaMemcpyAsync(mem, c->node_mem.p, vb, cudaMemcpyDeviceToHost, st));
        if (gpu) GP_CUDA(c, cudaMemcpyAsync(gpu, c->node_gpu.p, vb, cudaMemcpyDeviceToHost, st));
    }
    GP_CUDA(c, cudaStreamSynchronize(st));
    return GP_OK;
}

}  // extern "C"

// ---- packing ------------------------------------------------------------------------------------

// device views of one batch
struct DevApps {
    AppColumns cols;                 // device pointers; cols.off may be NULL (derived on the device)
    const uint8_t* skip;
    int32_t n;
};
struct DevResults {
    int32_t* driver;
    void* exec;                      // int32 or uint16
    int64_t cap;
    int node_bits;
};

static AppColumns cols_at(const AppColumns& c, int32_t lo) {
    AppColumns r = c;
    const size_t es = c.bits == 64 ? 8 : 4;
    for (int k = 0; k < 6; ++k) if (c.q[k]) r.q[k] = static_cast<const char*>(c.q[k]) + es * (size_t)lo;
    r.count = c.count + lo;
    if (c.group) r.group = c.group + lo;
    if (c.off) r.off = c.off + lo;
    return r;
}

template <int ALGO>
static void launch_pack(gp_ctx* c, gp_mode mode, const Snapshot& s, const PrepApp* prep, const int32_t* app_group, int32_t n_apps,
                        int32_t* driver_node, int32_t* executor_nodes, int2* scratch, unsigned long long* stats,
                        unsigned int* next_app, cudaStream_t st) {
    if constexpr (ALGO == 2) {     // minimal-fragmentation: GP_MODE_INDEPENDENT only (check_args)
        // persistent grid: as many CTAs as fit on the device (or fewer for small batches)
        int& per_sm = c->pack_ctas_per_sm;
        if (per_sm == 0) {
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gp_pack_independent, kPackThreads, 0);
            if (per_sm < 1) per_sm = 1;
        }
        int64_t blocks = ((int64_t)n_apps * 32 + kPackThreads - 1) / kPackThreads;
        int64_t max_blocks = (int64_t)c->sm_count * per_sm;
        if (blocks > max_blocks) blocks = max_blocks;
        if (blocks < 1) blocks = 1;
        gp_pack_independent<<<(int)blocks, kPackThreads, 0, st>>>(s, prep, n_apps, driver_node, executor_nodes, scratch,
                                                                 stats, next_app);
    } else {                       // tightly-pack / distribute-evenly come here in the FIFO modes only (launch_tables)
        // FIFO: one persistent 1024-thread CTA per instance group, its slots staged in shared memory
        bool& attr_set = c->fifo_attr_set[ALGO];     // per device: function attributes live in the device's context
        if (!attr_set) {
            cudaFuncSetAttribute(gp_pack_fifo_cta<ALGO, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFifoSmemBytes);
            cudaFuncSetAttribute(gp_pack_fifo_cta<ALGO, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFifoSmemBytes);
            attr_set = true;
        }
        int32_t* app_list = c->fifo_list.as<int32_t>();
        unsigned int* cursor = &c->dev_status()->fifo_cursor;
        if (mode == GP_MODE_FIFO_REFERENCE)
            gp_pack_fifo_cta<ALGO, 1><<<s.n_groups, kFifoThreads, kFifoSmemBytes, st>>>(s, prep, app_group, n_apps, driver_node, executor_nodes, scratch, stats, s.gmins, app_list, cursor);
        else
            gp_pack_fifo_cta<ALGO, 2><<<s.n_groups, kFifoThreads, kFifoSmemBytes, st>>>(s, prep, app_group, n_apps, driver_node, executor_nodes, scratch, stats, s.gmins, app_list, cursor);
        // the FIFO kernels subtract usage from `pair` in place: refresh the compact 32-bit view so that a later
        // independent pack on this context (the driver's own pack after fitEarlierDrivers, resource.go:255 then :321)
        // sees the charged availability
        const int T = 256;
        gp_fill_pair32<<<(c->n_slots + T) / T, T, 0, st>>>(c->n_slots, c->pair.as<longlong2>(), c->snap_flags.as<SnapMeta>(), c->pair32.as<uint2>());
        c->last.kernel_launches += 1;
    }
}

// independent tightly-pack / distribute-evenly: classify -> capacity tables -> thread-per-application decisions ->
// warp-per-application scan of whatever the tables could not decide (gangpack_tables.cuh)
template <int ALGO, class OUT>
static gp_status launch_tables(gp_ctx* c, const Snapshot& s, const AppColumns& cols, const ShapeTables& tabs, const int32_t* app_slot,
                               PrepApp* prep, int32_t* listed, int32_t q, const DevResults& dr, int32_t lo, int2* scratch,
                               unsigned long long* stats, unsigned int* next_app, int* d_err, volatile int* err_host, bool use_tables,
                               cudaStream_t st, int chunk) {
    if (use_tables) {
        bool& attr = c->tab_attr_set[ALGO];
        if (!attr) {
            GP_CUDA(c, cudaFuncSetAttribute(gp_build_shape_tables<ALGO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTabSmemBytes));
            attr = true;
        }
        gp_build_shape_tables<ALGO><<<dim3(2 * kMaxShapes, (unsigned)c->n_groups), kTabThreads, kTabSmemBytes, st>>>(s, tabs);
        c->last.kernel_launches += 1;
    }
    if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][1], st));
    gp_decide_tables<ALGO, OUT><<<(q + kDecideThreads - 1) / kDecideThreads, kDecideThreads, 0, st>>>(
        s, cols, tabs, app_slot, q, dr.cap, dr.driver + lo, static_cast<OUT*>(dr.exec), prep, listed, stats, d_err, err_host, use_tables ? 0 : 1);
    int& per_sm = c->tab_ctas_per_sm[ALGO][sizeof(OUT) == 2 ? 1 : 0];
    if (per_sm == 0) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gp_pack_listed<ALGO, OUT>, kPackTabThreads, 0);
        if (per_sm < 1) per_sm = 1;
    }
    // persistent grid; with the tables on the list is normally short (or empty: the CTAs leave at once)
    int64_t blocks = ((int64_t)q * 32 + kPackTabThreads - 1) / kPackTabThreads;
    const int64_t max_blocks = (int64_t)c->sm_count * (use_tables ? 2 : per_sm);
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks < 1) blocks = 1;
    gp_pack_listed<ALGO, OUT><<<(int)blocks, kPackTabThreads, 0, st>>>(s, tabs.hdr, prep, listed, dr.driver + lo, static_cast<OUT*>(dr.exec), scratch,
                                                                      stats, next_app);
    c->last.kernel_launches += 2;
    return GP_OK;
}

// Device-resident apps [lo, hi): enqueue the kernels on `st`; chunk index selects the timing events and the table lane.
// off_base: ExecutorNodes offset of application `lo` (only used when the offsets are derived on the device).
static gp_status pack_device_range(gp_ctx* c, const DevApps& da, int32_t lo, int32_t hi, int64_t off_base, gp_algo algo, gp_mode mode,
                                   const DevResults& dr, int2* scratch, cudaStream_t st, int chunk) {
    const int32_t q = hi - lo;
    if (q <= 0) return GP_OK;
    gp_ctx::DevStatus* ds = c->dev_status();
    int* d_err = &ds->err;
    unsigned long long* d_stats = ds->stats;
    unsigned int* next_app = ds->next_app + chunk;
    volatile int* err_host = &c->status_host->err_word;
    Snapshot s = make_snapshot(c);
    AppColumns cols = cols_at(da.cols, lo);

    if (mode == GP_MODE_INDEPENDENT && algo != GP_MINIMAL_FRAGMENTATION) {
        gp_ctx::TableSet& T = c->tabs[chunk % gp_ctx::kLanes];
        const size_t hdr_bytes = 1024 + (sizeof(ShapeEntry) + sizeof(DriverEntry)) * (size_t)kShapeSlots;
        const bool use_tables = c->use_tables && q >= 32;
        GP_CUDA(c, T.hdr.reserve(hdr_bytes));
        // [executor slot | driver slot | listed | block sums of the executor counts (K0)]
        const size_t slot_words = (3 * (size_t)q + 1) & ~(size_t)1;             // keeps the block sums 8-byte aligned
        const size_t n_blocks = ((size_t)q + kClassifyThreads - 1) / kClassifyThreads;
        GP_CUDA(c, T.app_slot.reserve(sizeof(int32_t) * slot_words + sizeof(unsigned long long) * (n_blocks + 1)));
        if (use_tables) {
            GP_CUDA(c, T.table.reserve(sizeof(uint32_t) * (size_t)kMaxShapes * (size_t)((c->n_slots + 4) & ~3)));
            GP_CUDA(c, T.total.reserve(3 * sizeof(uint32_t) * (size_t)kMaxShapes * (size_t)c->n_groups));   // total | firstfit | first_host
            GP_CUDA(c, T.expand.reserve(sizeof(int32_t) * (size_t)kMaxShapes * (size_t)c->n_groups * kExpandCap));
        }
        ShapeTables tabs;
        tabs.hdr = T.hdr.as<ShapeHeader>();
        tabs.entries = reinterpret_cast<ShapeEntry*>(T.hdr.as<char>() + 1024);
        tabs.dentries = reinterpret_cast<DriverEntry*>(T.hdr.as<char>() + 1024 + sizeof(ShapeEntry) * (size_t)kShapeSlots);
        tabs.table = T.table.as<uint32_t>(); tabs.total = T.total.as<uint32_t>();
        tabs.firstfit = reinterpret_cast<int32_t*>(T.total.as<uint32_t>() + (size_t)kMaxShapes * (size_t)c->n_groups);
        tabs.first_host = tabs.firstfit + (size_t)kMaxShapes * (size_t)c->n_groups;
        tabs.expand = T.expand.as<int32_t>();
        tabs.pitch = (c->n_slots + 4) & ~3; tabs.n_groups = c->n_groups;      // rows start 16-byte aligned
        int64_t* off_out = nullptr;
        if (!da.cols.off) {                       // derive the offsets on the device
            off_out = c->off_dev.as<int64_t>() + lo;
            cols.off = off_out;
        }
        int32_t* app_slot = T.app_slot.as<int32_t>();
        int32_t* listed = app_slot + 2 * (size_t)q;
        PrepApp* prep = c->prep.as<PrepApp>() + lo;
        const bool o16 = dr.node_bits == 16;
        auto issue = [&](int& launches) -> gp_status {
            const int before = (int)c->last.kernel_launches;
            // the hash tables and the header (listed counter) start from zero: the whole block when the tables are used
            GP_CUDA(c, cudaMemsetAsync(T.hdr.p, 0, use_tables ? hdr_bytes : 1024, st));
            if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][0], st));
            if (use_tables || off_out) {
                unsigned long long* block_sums = reinterpret_cast<unsigned long long*>(app_slot + slot_words);
                if (off_out) {
                    gp_count_blocks<<<(unsigned)n_blocks, kClassifyThreads, 0, st>>>(q, cols.count, block_sums);
                    c->last.kernel_launches += 1;
                }
                gp_classify_apps<<<(unsigned)n_blocks, kClassifyThreads, 0, st>>>(
                    q, cols, tabs, c->snap_flags.as<SnapMeta>(), off_base, off_out, block_sums, app_slot, use_tables ? 1 : 0);
                c->last.kernel_launches += 1;
            }
            gp_status r;
            if (algo == GP_TIGHTLY_PACK)
                r = o16 ? launch_tables<0, uint16_t>(c, s, cols, tabs, app_slot, prep, listed, q, dr, lo, scratch, d_stats, next_app, d_err, err_host, use_tables, st, chunk)
                        : launch_tables<0, int32_t>(c, s, cols, tabs, app_slot, prep, listed, q, dr, lo, scratch, d_stats, next_app, d_err, err_host, use_tables, st, chunk);
            else
                r = o16 ? launch_tables<1, uint16_t>(c, s, cols, tabs, app_slot, prep, listed, q, dr, lo, scratch, d_stats, next_app, d_err, err_host, use_tables, st, chunk)
                        : launch_tables<1, int32_t>(c, s, cols, tabs, app_slot, prep, listed, q, dr, lo, scratch, d_stats, next_app, d_err, err_host, use_tables, st, chunk);
            if (r != GP_OK) return r;
            GP_CUDA(c, cudaGetLastError());
            if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][2], st));
            launches = (int)c->last.kernel_launches - before;
            c->last.kernel_launches = before;          // run_cached adds `launches` (also when the graph is replayed)
            return GP_OK;
        };
        if (c->record_events) {                        // timing events inside: always issued directly
            int n = 0;
            gp_status r = issue(n);
            c->last.kernel_launches += n;
            return r;
        }
        struct { int32_t algo, o16, use_tables, q, lo, chunk; int64_t off_base; AppColumns cols; ShapeTables tabs; Snapshot snap;
                 const void* p[10]; int64_t cap; } key{};
        key.algo = (int32_t)algo; key.o16 = o16; key.use_tables = use_tables; key.q = q; key.lo = lo; key.chunk = chunk; key.off_base = off_base;
        key.cols = cols; key.tabs = tabs; key.snap = s; key.cap = dr.cap;
        const void* ptrs[10] = {app_slot, prep, listed, dr.driver, dr.exec, scratch, d_stats, next_app, d_err, off_out};
        std::memcpy(key.p, ptrs, sizeof(ptrs));
        return run_cached(c, c->g_chunk[st == c->stream ? gp_ctx::kMaxChunks : chunk], &key, sizeof(key), st, issue);
    }

    // ---- FIFO modes and minimal-fragmentation: prepared records + the pack kernel ------------------------------------
    PrepApp* prep = c->prep.as<PrepApp>() + lo;
    const int T = kPrepThreads;
    if (mode != GP_MODE_INDEPENDENT) {
        GP_CUDA(c, c->fifo_list.reserve(sizeof(int32_t) * (size_t)(q + 1)));
        GP_CUDA(c, c->gmin.reserve(sizeof(GroupMin) * (size_t)c->n_groups));
        GP_CUDA(c, cudaMemsetAsync(c->gmin.p, 0x7f, sizeof(GroupMin) * (size_t)c->n_groups, st));   // +inf-ish
    }
    if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][0], st));
    gp_prep_apps<<<(q + T - 1) / T, T, 0, st>>>(
        q, cols, da.skip ? da.skip + lo : nullptr, c->n_groups, dr.cap,
        c->snap_flags.as<SnapMeta>(), mode == GP_MODE_INDEPENDENT ? nullptr : c->gmin.as<GroupMin>(), prep, d_err, err_host);
    s.gmins = c->gmin.as<GroupMin>();
    if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][1], st));
    int32_t* exec32 = static_cast<int32_t*>(dr.exec);
    if (algo == GP_TIGHTLY_PACK)
        launch_pack<0>(c, mode, s, prep, cols.group, q, dr.driver + lo, exec32, scratch, d_stats, next_app, st);
    else if (algo == GP_MINIMAL_FRAGMENTATION)
        launch_pack<2>(c, mode, s, prep, cols.group, q, dr.driver + lo, exec32, scratch, d_stats, next_app, st);
    else
        launch_pack<1>(c, mode, s, prep, cols.group, q, dr.driver + lo, exec32, scratch, d_stats, next_app, st);
    GP_CUDA(c, cudaGetLastError());
    if (c->record_events) GP_CUDA(c, cudaEventRecord(c->ev[chunk][2], st));
    c->last.kernel_launches += 2;
    return GP_OK;
}

static bool fused_path(gp_algo algo, gp_mode mode) { return mode == GP_MODE_INDEPENDENT && algo != GP_MINIMAL_FRAGMENTATION; }

// common prologue: buffers, counters
static gp_status pack_begin(gp_ctx* c, int32_t q, gp_algo algo, gp_mode mode, int64_t exec_cap, bool derive_off, int2** scratch, cudaStream_t st) {
    GP_CUDA(c, cudaMemsetAsync(c->status.p, 0, sizeof(gp_ctx::DevStatus), st));
    c->status_host->err_word = 0;
    c->last = gp_stats{};
    c->ev_chunks = 0;
    *scratch = nullptr;
    if (q == 0) return GP_OK;
    GP_CUDA(c, c->prep.reserve(sizeof(PrepApp) * (size_t)q));      // FIFO / minimal-fragmentation: every application; tables: the listed ones
    if (derive_off) GP_CUDA(c, c->off_dev.reserve(sizeof(int64_t) * (size_t)(q + 1)));
    if (algo != GP_TIGHTLY_PACK) {        // candidate list (distribute-evenly) / consumed-node list (minimal-fragmentation)
        GP_CUDA(c, c->scratch.reserve(sizeof(int2) * (size_t)(exec_cap + 1)));
        *scratch = c->scratch.as<int2>();
    }
    return GP_OK;
}

static gp_status check_args(gp_ctx* c, const gp_apps_wire* a, gp_algo algo, gp_mode mode, const gp_results_wire* out, const char* who) {
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, std::string(who) + ": gp_set_snapshot first");
    if (!a || !out || a->n_apps < 0) return fail(c, GP_ERR_INVALID, std::string(who) + ": NULL apps/results");
    if (algo != GP_TIGHTLY_PACK && algo != GP_DISTRIBUTE_EVENLY && algo != GP_MINIMAL_FRAGMENTATION)
        return fail(c, GP_ERR_INVALID, std::string(who) + ": unknown algo");
    if (algo == GP_MINIMAL_FRAGMENTATION && mode != GP_MODE_INDEPENDENT)
        return fail(c, GP_ERR_INVALID, std::string(who) + ": minimal-fragmentation is offered in GP_MODE_INDEPENDENT only "
                                                          "(its one registered caller, single-az-minimal-fragmentation, chooses a zone per application on the host)");
    if (mode != GP_MODE_INDEPENDENT && mode != GP_MODE_FIFO_REFERENCE && mode != GP_MODE_FIFO_EXACT)
        return fail(c, GP_ERR_INVALID, std::string(who) + ": unknown mode");
    if (a->quantity_bits != 64 && a->quantity_bits != 32) return fail(c, GP_ERR_INVALID, std::string(who) + ": quantity_bits must be 64 or 32");
    if (a->quantity_bits == 32 && (a->mem_shift < 0 || a->mem_shift > 40)) return fail(c, GP_ERR_INVALID, std::string(who) + ": mem_shift out of range");
    if (out->node_bits != 32 && out->node_bits != 16) return fail(c, GP_ERR_INVALID, std::string(who) + ": node_bits must be 32 or 16");
    if (out->node_bits == 16 && (!fused_path(algo, mode) || c->n_nodes > 65535))
        return fail(c, GP_ERR_INVALID, std::string(who) + ": 16-bit node indices need <= 65535 nodes and GP_MODE_INDEPENDENT tightly-pack / distribute-evenly");
    if (a->n_apps > 0 && (!a->drv_cpu || !a->drv_mem || !a->exe_cpu || !a->exe_mem || !a->exe_count || !out->driver_node))
        return fail(c, GP_ERR_INVALID, std::string(who) + ": missing app/result arrays");
    if (a->n_apps > 0 && !a->exec_out_off && !fused_path(algo, mode))
        return fail(c, GP_ERR_INVALID, std::string(who) + ": exec_out_off may only be NULL for GP_MODE_INDEPENDENT tightly-pack / distribute-evenly");
    return GP_OK;
}

// after the streams have been synchronised: event times of the last pack, summed over its chunks
static void fill_kernel_times(gp_ctx* c) {
    c->last.prep_kernel_ns = 0; c->last.pack_kernel_ns = 0;
    for (int i = 0; i < c->ev_chunks; ++i) {
        float a = 0.f, b = 0.f;
        if (cudaEventElapsedTime(&a, c->ev[i][0], c->ev[i][1]) == cudaSuccess) c->last.prep_kernel_ns += (int64_t)(a * 1.0e6);
        if (cudaEventElapsedTime(&b, c->ev[i][1], c->ev[i][2]) == cudaSuccess) c->last.pack_kernel_ns += (int64_t)(b * 1.0e6);
    }
}

static gp_status decode_device_error(gp_ctx* c, int err) {
    if (err == 0) return GP_OK;
    if (err & kErrUnrepresentable) return fail(c, GP_ERR_UNREPRESENTABLE, "pack: quantity >= 2^61 or exe_count > 2^24 (2^20 in the FIFO modes)");
    if (err & kErrNegativeRequest) return fail(c, GP_ERR_INVALID, "pack: negative resource request or executor count");
    if (err & kErrBadGroup) return fail(c, GP_ERR_INVALID, "pack: app group out of range");
    return fail(c, GP_ERR_CAPACITY, "pack: exec_out_off inconsistent with exe_count or executor_nodes_cap too small");
}

// the validation errors of the pack call just synchronised, from the host-visible error word
static gp_status pack_error(gp_ctx* c) { return decode_device_error(c, c->status_host->err_word); }

static gp_apps_wire widen(const gp_apps* a) {
    gp_apps_wire w{};
    w.n_apps = a->n_apps; w.quantity_bits = 64; w.mem_shift = 0;
    w.drv_cpu = a->drv_cpu_milli; w.drv_mem = a->drv_mem_bytes; w.drv_gpu = a->drv_gpu;
    w.exe_cpu = a->exe_cpu_milli; w.exe_mem = a->exe_mem_bytes; w.exe_gpu = a->exe_gpu;
    w.exe_count = a->exe_count; w.group = a->group; w.skip_if_no_fit = a->skip_if_no_fit; w.exec_out_off = a->exec_out_off;
    return w;
}

extern "C" {

gp_status gp_pack_batch_device(gp_ctx* c, const gp_apps* da, gp_algo algo, gp_mode mode, gp_results* dout, void* stream) {
    if (!c) return GP_ERR_INVALID;
    if (!da || !dout) return fail(c, GP_ERR_INVALID, "gp_pack_batch_device: NULL apps/results");
    const gp_apps_wire w = widen(da);
    gp_results_wire ow{dout->driver_node, dout->executor_nodes, dout->executor_nodes_cap, 32, 0};
    gp_status s = check_args(c, &w, algo, mode, &ow, "gp_pack_batch_device");
    if (s != GP_OK) return s;
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    int2* scratch = nullptr;
    s = pack_begin(c, w.n_apps, algo, mode, ow.executor_nodes_cap, !w.exec_out_off, &scratch, st);
    if (s != GP_OK || w.n_apps == 0) return s;
    DevApps dv{};
    dv.cols.q[0] = w.drv_cpu; dv.cols.q[1] = w.drv_mem; dv.cols.q[2] = w.drv_gpu;
    dv.cols.q[3] = w.exe_cpu; dv.cols.q[4] = w.exe_mem; dv.cols.q[5] = w.exe_gpu;
    dv.cols.count = w.exe_count; dv.cols.group = w.group; dv.cols.off = w.exec_out_off; dv.cols.bits = 64; dv.cols.mem_shift = 0;
    dv.skip = w.skip_if_no_fit; dv.n = w.n_apps;
    DevResults dr{ow.driver_node, ow.executor_nodes, ow.executor_nodes_cap, 32};
    s = pack_device_range(c, dv, 0, w.n_apps, 0, algo, mode, dr, scratch, st, 0);
    if (s == GP_OK) c->ev_chunks = 1;
    return s;
}

gp_status gp_last_stats(gp_ctx* c, gp_stats* out) {
    if (!c || !out) return GP_ERR_INVALID;
    GP_CUDA(c, cudaSetDevice(c->device));
    gp_ctx::DevStatus& h = c->status_host->dev;
    GP_CUDA(c, cudaMemcpyAsync(&h, c->status.p, offsetof(gp_ctx::DevStatus, stats) + sizeof(h.stats), cudaMemcpyDeviceToHost, c->stream));
    GP_CUDA(c, cudaStreamSynchronize(c->stream));
    c->last.nodes_scanned = (int64_t)h.stats[0];
    c->last.drivers_tried = (int64_t)h.stats[1];
    c->last.scan_path_apps = (int64_t)h.stats[2];
    c->last.scan_path_nodes = (int64_t)h.stats[3];
    fill_kernel_times(c);
    *out = c->last;
    return decode_device_error(c, h.err);
}

static gp_status pack_batch_impl(gp_ctx* c, const gp_apps_wire* a, gp_algo algo, gp_mode mode, gp_results_wire* out);

gp_status gp_pack_batch_wire(gp_ctx* c, const gp_apps_wire* a, gp_algo algo, gp_mode mode, gp_results_wire* out) {
    if (!c) return GP_ERR_INVALID;
    gp_status s = pack_batch_impl(c, a, algo, mode, out);
    if (s != GP_OK) {
        // Whatever was enqueued before the failure may still read the caller's buffers or write its results:
        // drain every stream of this context before handing control (and buffer ownership) back.
        const std::string keep = c->err;
        cudaSetDevice(c->device);
        for (cudaStream_t l : c->lane) if (l) cudaStreamSynchronize(l);
        if (c->stream) cudaStreamSynchronize(c->stream);
        cudaGetLastError();
        c->err = keep;
    }
    return s;
}

gp_status gp_pack_batch(gp_ctx* c, const gp_apps* a, gp_algo algo, gp_mode mode, gp_results* out) {
    if (!c) return GP_ERR_INVALID;
    if (!a || !out) return fail(c, GP_ERR_INVALID, "gp_pack_batch: NULL apps/results");
    const gp_apps_wire w = widen(a);
    gp_results_wire ow{out->driver_node, out->executor_nodes, out->executor_nodes_cap, 32, 0};
    return gp_pack_batch_wire(c, &w, algo, mode, &ow);
}

static gp_status pack_batch_impl(gp_ctx* c, const gp_apps_wire* a, gp_algo algo, gp_mode mode, gp_results_wire* out) {
    gp_status s = check_args(c, a, algo, mode, out, "gp_pack_batch");
    if (s != GP_OK) return s;
    const int32_t q = a->n_apps;
    if (q == 0) return GP_OK;
    const auto t_begin = std::chrono::steady_clock::now();
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t es = a->quantity_bits == 64 ? 8 : 4;       // bytes per quantity
    const size_t os = out->node_bits == 16 ? 2 : 4;         // bytes per ExecutorNodes entry
    const int64_t* off = a->exec_out_off;                   // may be NULL: derived on the device, chunk bases summed here
    if (off) {
        const int64_t total = off[q];
        if (total < 0 || total > out->executor_nodes_cap) return fail(c, GP_ERR_CAPACITY, "gp_pack_batch: executor_nodes_cap too small");
        if (total > 0 && !out->executor_nodes) return fail(c, GP_ERR_INVALID, "gp_pack_batch: executor_nodes is NULL");
    }
    const size_t bq = es * (size_t)q, b32 = sizeof(int32_t) * (size_t)q;
    // the quantity columns are staged in ONE pitched device block (rows: drv cpu, drv mem, exe cpu, exe mem, drv gpu,
    // exe gpu) so that equally spaced host columns can be moved by a single 2-D DMA per chunk
    const size_t dpitch = (bq + 255) & ~(size_t)255;
    GP_CUDA(c, c->a_quant.reserve(dpitch * 6));
    GP_CUDA(c, c->a_count.reserve(b32));
    if (off) GP_CUDA(c, c->a_off.reserve(sizeof(int64_t) * (size_t)(q + 1)));
    GP_CUDA(c, c->r_driver.reserve(b32));
    GP_CUDA(c, c->r_exec.reserve(os * (size_t)(out->executor_nodes_cap + 1)));
    if (a->group) GP_CUDA(c, c->a_group.reserve(b32));
    if (a->skip_if_no_fit) GP_CUDA(c, c->a_skip.reserve((size_t)q));
    // Small batches are latency-bound: inputs are gathered by ONE kernel reading the mapped host buffers (a chain of
    // tiny DMA copies costs ~8-10 us each in stream order) and results are written straight into mapped host buffers.
    // Large ones are bandwidth-bound: DMA per pipelined chunk in both directions.
    const bool small = q <= kZeroCopyOutApps;
    void* mo_driver = small ? const_cast<void*>(mapped_ptr(c, out->driver_node, b32)) : nullptr;
    void* mo_exec = (small && out->executor_nodes) ? const_cast<void*>(mapped_ptr(c, out->executor_nodes, os * (size_t)out->executor_nodes_cap)) : nullptr;
    const bool out_mapped = small && mo_driver && (out->executor_nodes_cap == 0 || !out->executor_nodes || mo_exec);
    char* blk = c->a_quant.as<char>();
    DevApps dv{};
    const void* hq[6] = {a->drv_cpu, a->drv_mem, a->exe_cpu, a->exe_mem, a->drv_gpu, a->exe_gpu};    // staging row order
    dv.cols.q[0] = blk + 0 * dpitch; dv.cols.q[1] = blk + 1 * dpitch; dv.cols.q[3] = blk + 2 * dpitch; dv.cols.q[4] = blk + 3 * dpitch;
    dv.cols.q[2] = a->drv_gpu ? blk + 4 * dpitch : nullptr;
    dv.cols.q[5] = a->exe_gpu ? blk + 5 * dpitch : nullptr;
    dv.cols.count = c->a_count.as<int32_t>();
    dv.cols.group = a->group ? c->a_group.as<int32_t>() : nullptr;
    dv.cols.off = off ? c->a_off.as<int64_t>() : nullptr;
    dv.cols.bits = a->quantity_bits; dv.cols.mem_shift = a->mem_shift;
    dv.skip = a->skip_if_no_fit ? c->a_skip.as<uint8_t>() : nullptr;
    dv.n = q;
    DevResults dr;
    dr.driver = out_mapped ? (int32_t*)mo_driver : c->r_driver.as<int32_t>();
    dr.exec = out_mapped ? mo_exec : c->r_exec.p;
    dr.cap = out->executor_nodes_cap;
    dr.node_bits = out->node_bits;

    // Independent decisions are chunked and the chunks rotate over kLanes streams, so the H2D of
    // chunk i+1, the kernels of chunk i and the D2H of chunk i-1 overlap (PCIe is full duplex).
    // FIFO modes are one sequential pass: a single chunk.
    int n_chunks = 1;
    if (mode == GP_MODE_INDEPENDENT && q >= 2 * c->chunk_apps) {
        n_chunks = (q + c->chunk_apps - 1) / c->chunk_apps;
        if (n_chunks > gp_ctx::kMaxChunks) n_chunks = gp_ctx::kMaxChunks;
    }
    int2* scratch = nullptr;
    s = pack_begin(c, q, algo, mode, out->executor_nodes_cap, !off, &scratch, st);
    if (s != GP_OK) return s;
    // per-kernel CUDA events are for gp_last_stats; the pipelined path is bound by how fast the host thread can issue
    // its ~10 calls per chunk, so it leaves them out (pack_kernel_ns / prep_kernel_ns then read 0)
    struct EvGuard { gp_ctx* c; ~EvGuard() { c->record_events = true; } } ev_guard{c};
    c->record_events = n_chunks == 1;
    GP_CUDA(c, cudaEventRecord(c->ev_ready, st));      // snapshot + zeroed counters are ready
    const bool timeline = c->trace >= 2 && !c->record_events;
    if (timeline) GP_CUDA(c, cudaEventRecord(c->ev_t0, st));
    int64_t e_run = 0;                                 // ExecutorNodes entries before the current chunk
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int32_t lo = (int32_t)((int64_t)q * ch / n_chunks), hi = (int32_t)((int64_t)q * (ch + 1) / n_chunks);
        const size_t n = (size_t)(hi - lo);
        cudaStream_t ls = n_chunks == 1 ? st : c->lane[ch % gp_ctx::kLanes];
        // ---- inputs -> HBM (the copies need not wait for the snapshot layout; the kernels below do) ----------------------------------------------------------------------------------
        bool gathered = false;
        if (small && !a->skip_if_no_fit) {
            CopyJobs jobs{};
            bool ok = true;
            auto add = [&](const void* src, void* dst, size_t bytes) {
                if (!src || !bytes) return;
                const void* m = mapped_ptr(c, src, bytes);
                if (!m || jobs.n >= 8) { ok = false; return; }
                jobs.j[jobs.n++] = CopyJob{m, dst, bytes};
            };
            // all six quantity rows when they are one equally spaced block, else row by row (<= 8 jobs in total)
            add(a->drv_cpu, blk + 0 * dpitch, bq); add(a->drv_mem, blk + 1 * dpitch, bq);
            add(a->exe_cpu, blk + 2 * dpitch, bq); add(a->exe_mem, blk + 3 * dpitch, bq);
            if (a->drv_gpu) add(a->drv_gpu, blk + 4 * dpitch, bq);
            if (a->exe_gpu) add(a->exe_gpu, blk + 5 * dpitch, bq);
            add(a->exe_count, c->a_count.p, b32);
            if (a->group) add(a->group, c->a_group.p, b32);
            if (off && ok) { if (jobs.n < 8) add(off, c->a_off.p, sizeof(int64_t) * (size_t)(q + 1)); else ok = false; }
            if (ok) {
                gp_multi_copy<<<q <= 64 ? 1 : 32, 256, 0, ls>>>(jobs);
                GP_CUDA(c, cudaGetLastError());
                c->last.kernel_launches += 1;
                gathered = true;
            }
        }
        if (!gathered) {
            // quantity columns: one 2-D DMA when the host columns are equally spaced (one pinned block laid out
            // column after column, as the shim allocates it), else one DMA per column
            int ncols = 4;
            if (a->drv_gpu && a->exe_gpu) ncols = 6;
            const ptrdiff_t spitch = (const char*)hq[1] - (const char*)hq[0];
            bool spaced = spitch >= (ptrdiff_t)bq && spitch <= ((ptrdiff_t)1 << 30);   // cudaMemcpy2D pitch limit (maxPitch ~2 GiB)
            for (int k = 2; spaced && k < ncols; ++k) spaced = ((const char*)hq[k] - (const char*)hq[k - 1]) == spitch;
            if (spaced && cudaMemcpy2DAsync(blk + es * (size_t)lo, dpitch, (const char*)hq[0] + es * (size_t)lo, (size_t)spitch,
                                            es * n, (size_t)ncols, cudaMemcpyHostToDevice, ls) != cudaSuccess) {
                cudaGetLastError();      // not accepted as a 2-D copy after all: column by column
                spaced = false;
            }
            if (!spaced) {
                for (int k = 0; k < ncols; ++k)
                    GP_CUDA(c, cudaMemcpyAsync(blk + k * dpitch + es * (size_t)lo, (const char*)hq[k] + es * (size_t)lo, es * n,
                                               cudaMemcpyHostToDevice, ls));
            }
            if (ncols == 4) {   // gpu columns given one at a time
                if (a->drv_gpu) GP_CUDA(c, cudaMemcpyAsync(blk + 4 * dpitch + es * (size_t)lo, (const char*)a->drv_gpu + es * (size_t)lo, es * n, cudaMemcpyHostToDevice, ls));
                if (a->exe_gpu) GP_CUDA(c, cudaMemcpyAsync(blk + 5 * dpitch + es * (size_t)lo, (const char*)a->exe_gpu + es * (size_t)lo, es * n, cudaMemcpyHostToDevice, ls));
            }
            GP_CUDA(c, cudaMemcpyAsync(c->a_count.as<int32_t>() + lo, a->exe_count + lo, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ls));
            if (off) GP_CUDA(c, cudaMemcpyAsync(c->a_off.as<int64_t>() + lo, off + lo, sizeof(int64_t) * (n + 1), cudaMemcpyHostToDevice, ls));
            if (a->group) GP_CUDA(c, cudaMemcpyAsync(c->a_group.as<int32_t>() + lo, a->group + lo, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ls));
            if (a->skip_if_no_fit) GP_CUDA(c, cudaMemcpyAsync(c->a_skip.as<uint8_t>() + lo, a->skip_if_no_fit + lo, n, cudaMemcpyHostToDevice, ls));
        }
        if (timeline) GP_CUDA(c, cudaEventRecord(c->ev[ch][0], ls));       // inputs of this chunk are in HBM
        if (n_chunks > 1) GP_CUDA(c, cudaStreamWaitEvent(ls, c->ev_ready, 0));
        // ---- this chunk's ExecutorNodes range ------------------------------------------------------------------
        int64_t e0, e1;
        if (off) { e0 = off[lo]; e1 = off[hi]; }
        else {
            int64_t acc = 0;
            const int32_t* cnt = a->exe_count;
            for (int32_t i = lo; i < hi; ++i) acc += cnt[i] > 0 ? cnt[i] : 0;
            e0 = e_run; e1 = e_run + acc; e_run = e1;
            if (e1 > out->executor_nodes_cap) return fail(c, GP_ERR_CAPACITY, "gp_pack_batch: executor_nodes_cap too small");
            if (e1 > 0 && !out->executor_nodes) return fail(c, GP_ERR_INVALID, "gp_pack_batch: executor_nodes is NULL");
        }
        s = pack_device_range(c, dv, lo, hi, e0, algo, mode, dr, scratch, ls, ch);
        if (s != GP_OK) return s;
        if (timeline) GP_CUDA(c, cudaEventRecord(c->ev[ch][1], ls));       // kernels of this chunk done
        if (out_mapped) continue;
        GP_CUDA(c, cudaMemcpyAsync(out->driver_node + lo, dr.driver + lo, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ls));
        if (e1 > e0)
            GP_CUDA(c, cudaMemcpyAsync((char*)out->executor_nodes + os * (size_t)e0, (char*)dr.exec + os * (size_t)e0, os * (size_t)(e1 - e0),
                                       cudaMemcpyDeviceToHost, ls));
    }
    if (timeline) for (int ch = 0; ch < n_chunks; ++ch) GP_CUDA(c, cudaEventRecord(c->ev[ch][2], n_chunks == 1 ? st : c->lane[ch % gp_ctx::kLanes]));
    c->ev_chunks = c->record_events ? n_chunks : 0;
    const auto t_issued = std::chrono::steady_clock::now();
    if (n_chunks > 1) {
        for (int l = 0; l < gp_ctx::kLanes && l < n_chunks; ++l) {
            GP_CUDA(c, cudaEventRecord(c->ev_done[l], c->lane[l]));
            GP_CUDA(c, cudaStreamWaitEvent(st, c->ev_done[l], 0));
        }
    }
    GP_CUDA(c, cudaStreamSynchronize(st));
    if (timeline) {
        for (int ch = 0; ch < n_chunks; ++ch) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, c->ev_t0, c->ev[ch][0]); cudaEventElapsedTime(&b, c->ev_t0, c->ev[ch][1]); cudaEventElapsedTime(&d, c->ev_t0, c->ev[ch][2]);
            std::fprintf(stderr, "[gangpack]   chunk %d: inputs in HBM at %.1f us, kernels done at %.1f us, results on the host at %.1f us\n", ch, a * 1e3, b * 1e3, d * 1e3);
        }
    }
    if (c->trace) {
        const auto t_done = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[gangpack] pack_batch q=%d chunks=%d bits=%d/%d out_mapped=%d issue=%.1fus wait=%.1fus\n", q, n_chunks,
                     a->quantity_bits, out->node_bits, (int)out_mapped, std::chrono::duration<double, std::micro>(t_issued - t_begin).count(),
                     std::chrono::duration<double, std::micro>(t_done - t_issued).count());
    }
    // validation errors arrive through the mapped error word; scan statistics stay on the device until
    // gp_last_stats asks for them
    return pack_error(c);
}

gp_status gp_pack_one(gp_ctx* c, gp_algo algo, int64_t drv_cpu, int64_t drv_mem, int64_t drv_gpu, int64_t exe_cpu,
                      int64_t exe_mem, int64_t exe_gpu, int32_t exe_count, int32_t* has_capacity, int32_t* driver_node,
                      int32_t* executor_nodes) {
    if (!c) return GP_ERR_INVALID;
    if (!has_capacity || !driver_node) return fail(c, GP_ERR_INVALID, "gp_pack_one: NULL outputs");
    if (exe_count > 0 && !executor_nodes) return fail(c, GP_ERR_INVALID, "gp_pack_one: executor_nodes is NULL");
    // The tuple and the result travel through a context-owned mapped pinned block: no DMA copies at all
    // on this latency-critical path (one app = one SparkBinPackFunction call).
    const size_t n_exec = exe_count > 0 ? (size_t)exe_count : 0;
    const size_t need = 128 + sizeof(int32_t) * (n_exec + 1);
    if (need > c->one_bytes) {
        GP_CUDA(c, cudaSetDevice(c->device));
        if (c->one_block) { gp_free_pinned(c, c->one_block); c->one_block = nullptr; c->one_bytes = 0; }
        void* blk = nullptr;
        gp_status st = gp_alloc_pinned(c, need * 2, &blk);
        if (st != GP_OK) return st;
        c->one_block = blk; c->one_bytes = need * 2;
    }
    int64_t* q = static_cast<int64_t*>(c->one_block);         // [0..5] tuple, [6..7] offsets
    q[0] = drv_cpu; q[1] = drv_mem; q[2] = drv_gpu; q[3] = exe_cpu; q[4] = exe_mem; q[5] = exe_gpu;
    q[6] = 0; q[7] = (int64_t)n_exec;
    int32_t* i32 = reinterpret_cast<int32_t*>(q + 8);          // [0] count, [1] driver result
    i32[0] = exe_count; i32[1] = -1;
    int32_t* exec_out = reinterpret_cast<int32_t*>(static_cast<char*>(c->one_block) + 128);
    gp_apps a{};
    a.n_apps = 1;
    a.drv_cpu_milli = q + 0; a.drv_mem_bytes = q + 1; a.drv_gpu = q + 2;
    a.exe_cpu_milli = q + 3; a.exe_mem_bytes = q + 4; a.exe_gpu = q + 5;
    a.exe_count = i32;
    a.exec_out_off = algo == GP_MINIMAL_FRAGMENTATION ? q + 6 : nullptr;   // derived on the device where the kernel can
    gp_results r{};
    r.driver_node = i32 + 1;
    r.executor_nodes = exec_out;
    r.executor_nodes_cap = (int64_t)n_exec;
    gp_status s = gp_pack_batch(c, &a, algo, GP_MODE_INDEPENDENT, &r);
    if (s != GP_OK) return s;
    const int32_t d = i32[1];
    *has_capacity = d >= 0 ? 1 : 0;
    *driver_node = d >= 0 ? d : -1;
    if (d >= 0 && n_exec) std::memcpy(executor_nodes, exec_out, sizeof(int32_t) * n_exec);
    return GP_OK;
}

// ---- single-AZ packers: pack every zone, choose by packing efficiency on the device (gangpack_zones.cuh) ----------
gp_status gp_set_schedulable(gp_ctx* c, const int64_t* cpu, const int64_t* mem, const int64_t* gpu) {
    if (!c) return GP_ERR_INVALID;
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, "gp_set_schedulable: gp_set_snapshot first");
    if (c->n_nodes > 0 && (!cpu || !mem)) return fail(c, GP_ERR_INVALID, "gp_set_schedulable: missing arrays");
    GP_CUDA(c, cudaSetDevice(c->device));
    const size_t N = (size_t)c->n_nodes;
    for (size_t i = 0; i < N; ++i) {
        const int64_t v[3] = {cpu[i], mem[i], gpu ? gpu[i] : 0};
        for (int64_t x : v) if (x >= kMaxQuantity || x <= -kMaxQuantity) return fail(c, GP_ERR_UNREPRESENTABLE, "gp_set_schedulable: |quantity| >= 2^61");
    }
    GP_CUDA(c, c->sched.reserve(24 * (N + 1)));
    char* b = c->sched.as<char>();
    if (N) {
        GP_CUDA(c, cudaMemcpyAsync(b, cpu, 8 * N, cudaMemcpyHostToDevice, c->stream));
        GP_CUDA(c, cudaMemcpyAsync(b + 8 * N, mem, 8 * N, cudaMemcpyHostToDevice, c->stream));
        if (gpu) GP_CUDA(c, cudaMemcpyAsync(b + 16 * N, gpu, 8 * N, cudaMemcpyHostToDevice, c->stream));
        else GP_CUDA(c, cudaMemsetAsync(b + 16 * N, 0, 8 * N, c->stream));
    }
    GP_CUDA(c, cudaStreamSynchronize(c->stream));
    c->have_sched = true;
    return GP_OK;
}

// the checks the two single-AZ entry points run first
static gp_status check_zone_call(gp_ctx* c, const gp_apps* a, const gp_zone_results* out, const char* who) {
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, std::string(who) + ": gp_set_snapshot first");
    if (!c->have_sched) return fail(c, GP_ERR_INVALID, std::string(who) + ": gp_set_schedulable first (the efficiencies need SchedulableResources)");
    if (!a || !out || a->n_apps < 0) return fail(c, GP_ERR_INVALID, std::string(who) + ": NULL apps/results");
    return GP_OK;
}

static bool has_requests(const gp_apps* a) {
    return a->drv_cpu_milli && a->drv_mem_bytes && a->exe_cpu_milli && a->exe_mem_bytes && a->exe_count;
}

// c->host_off = exclusive prefix sum of the executor counts (negative counts as 0); returns the largest count, at least 1
static int64_t count_offsets(gp_ctx* c, const gp_apps* a) {
    std::vector<int64_t>& off = c->host_off;
    off.resize((size_t)a->n_apps + 1);
    int64_t acc = 0, widest = 1;
    for (int32_t i = 0; i < a->n_apps; ++i) {
        const int64_t k = a->exe_count[i] > 0 ? a->exe_count[i] : 0;
        off[(size_t)i] = acc; acc += k;
        if (k > widest) widest = k;
    }
    off[(size_t)a->n_apps] = acc;
    return widest;
}

// the six int64 request columns into req[6][q] (a gpu column not given stays NULL in `cols`), the executor counts and
// the [q + 1] ExecutorNodes offsets `off`
static gp_status upload_apps(gp_ctx* c, const gp_apps* a, const int64_t* off, size_t q, cudaStream_t st, int64_t* req, int32_t* cnt,
                             int64_t* d_off, SixCols& cols) {
    const int64_t* hc[6] = {a->drv_cpu_milli, a->drv_mem_bytes, a->drv_gpu, a->exe_cpu_milli, a->exe_mem_bytes, a->exe_gpu};
    for (int k = 0; k < 6; ++k) {
        GP_CUDA(c, upload(req + q * (size_t)k, hc[k], 8 * q, st));
        cols.p[k] = hc[k] ? req + q * (size_t)k : nullptr;
    }
    GP_CUDA(c, upload(cnt, a->exe_count, 4 * q, st));
    GP_CUDA(c, upload(d_off, off, 8 * (q + 1), st));
    return GP_OK;
}

// results of a single-AZ call to the host; after the stream sync, the validation errors of its pack
static gp_status zone_results_back(gp_ctx* c, gp_zone_results* out, const int32_t* zone, const int32_t* driver, const int32_t* exec,
                                   const double* avg, size_t q, size_t total, cudaStream_t st) {
    GP_CUDA(c, cudaMemcpyAsync(out->zone, zone, 4 * q, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaMemcpyAsync(out->driver_node, driver, 4 * q, cudaMemcpyDeviceToHost, st));
    if (total) GP_CUDA(c, cudaMemcpyAsync(out->executor_nodes, exec, 4 * total, cudaMemcpyDeviceToHost, st));
    if (out->avg_efficiency) GP_CUDA(c, cudaMemcpyAsync(out->avg_efficiency, avg, 32 * q, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    return pack_error(c);
}

gp_status gp_pack_batch_zones(gp_ctx* c, const gp_apps* a, gp_algo algo, gp_zone_results* out) {
    if (!c) return GP_ERR_INVALID;
    gp_status s = check_zone_call(c, a, out, "gp_pack_batch_zones");
    if (s != GP_OK) return s;
    if (algo != GP_TIGHTLY_PACK && algo != GP_MINIMAL_FRAGMENTATION)
        return fail(c, GP_ERR_INVALID, "gp_pack_batch_zones: the single-AZ packers are tightly-pack and minimal-fragmentation (single_az_pack_tightly.go, single_az_minimal_fragmentation.go)");
    const int32_t Q = a->n_apps, Z = c->n_groups;
    if (Q == 0) return GP_OK;
    if (!has_requests(a) || !out->zone || !out->driver_node) return fail(c, GP_ERR_INVALID, "gp_pack_batch_zones: missing app/result arrays");
    if ((int64_t)Q * Z > 0x7fffffffLL) return fail(c, GP_ERR_INVALID, "gp_pack_batch_zones: n_apps x zones too large");
    const int64_t* off = a->exec_out_off;
    if (!off) {
        count_offsets(c, a);
        off = c->host_off.data();
    }
    const int64_t total = off[Q];
    if (total < 0 || total > out->executor_nodes_cap) return fail(c, GP_ERR_CAPACITY, "gp_pack_batch_zones: executor_nodes_cap too small");
    if (total > 0 && !out->executor_nodes) return fail(c, GP_ERR_INVALID, "gp_pack_batch_zones: executor_nodes is NULL");
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t q = (size_t)Q, R = q * (size_t)Z, T = (size_t)total;
    int64_t *in, *d_off, *rows, *roff;
    int32_t *cnt, *rcnt, *rgrp, *rdrv, *rexe, *zone, *drv, *exe;
    double* avg;
    GP_CUDA(c, stage(c->zonebuf, part(in, 6 * q), part(cnt, q), part(d_off, q + 1), part(rows, 6 * R), part(rcnt, R), part(rgrp, R),
                     part(roff, R + 1), part(rdrv, R), part(rexe, (size_t)Z * T + 1), part(zone, q), part(drv, q), part(exe, T + 1),
                     part(avg, 4 * q)));
    SixCols six{};
    s = upload_apps(c, a, off, q, st, in, cnt, d_off, six);
    if (s != GP_OK) return s;
    const int TH = 256;
    // the efficiencies read the availability in node-table order: refresh that copy from the slots (a FIFO batch may
    // have charged them since gp_set_snapshot)
    if (c->n_slots > 0)
        gp_scatter_slots<<<(c->n_slots + TH - 1) / TH, TH, 0, st>>>(c->n_slots, c->pair.as<longlong2>(), c->sgpu.as<int64_t>(), c->slot_node.as<int32_t>(),
                                                                   c->node_cpu.as<int64_t>(), c->node_mem.as<int64_t>(), c->node_gpu.as<int64_t>());
    gp_zone_expand<<<(unsigned)((R + 1 + TH - 1) / TH), TH, 0, st>>>(Q, Z, six, cnt, d_off, rows, rcnt, rgrp, roff);
    int2* scratch = nullptr;
    s = pack_begin(c, (int32_t)R, algo, GP_MODE_INDEPENDENT, (int64_t)Z * total, false, &scratch, st);
    if (s != GP_OK) return s;
    DevApps dv{};
    for (int k = 0; k < 6; ++k) dv.cols.q[k] = rows + R * (size_t)k;
    dv.cols.count = rcnt; dv.cols.group = rgrp; dv.cols.off = roff;
    dv.cols.bits = 64; dv.cols.mem_shift = 0; dv.skip = nullptr; dv.n = (int32_t)R;
    DevResults dr{rdrv, rexe, (int64_t)Z * total, 32};
    s = pack_device_range(c, dv, 0, (int32_t)R, 0, algo, GP_MODE_INDEPENDENT, dr, scratch, st, 0);
    if (s != GP_OK) return s;
    c->ev_chunks = 1;
    ZoneChooseIn zi{};
    const size_t N = (size_t)c->n_nodes;
    zi.avail[0] = c->node_cpu.as<long long>(); zi.avail[1] = c->node_mem.as<long long>(); zi.avail[2] = c->node_gpu.as<long long>();
    zi.sched[0] = c->sched.as<long long>(); zi.sched[1] = c->sched.as<long long>() + N; zi.sched[2] = c->sched.as<long long>() + 2 * N;
    for (int k = 0; k < 3; ++k) { zi.drv[k] = six.p[k]; zi.exe[k] = six.p[3 + k]; }
    zi.count = cnt; zi.out_off = d_off;
    zi.row_driver = rdrv; zi.row_exec = rexe;
    zi.n_apps = Q; zi.n_zones = Z; zi.executors_reserved = algo == GP_TIGHTLY_PACK ? 1 : 0;
    gp_zone_choose<<<(unsigned)((q * 32 + TH - 1) / TH), TH, 0, st>>>(zi, zone, drv, exe, out->avg_efficiency ? avg : nullptr);
    GP_CUDA(c, cudaGetLastError());
    c->last.kernel_launches += 2;
    return zone_results_back(c, out, zone, drv, exe, avg, q, T, st);
}

// ---- reservation table + device-resident snapshot upkeep (gangpack_zones.cuh) -------------------------------------------
// the snapshot-wide facts and the compact view after availabilities changed in place
static gp_status refresh_views(gp_ctx* c, cudaStream_t st) {
    const int T = 256;
    if (c->n_slots <= 0) return GP_OK;
    SnapMeta* meta = c->snap_flags.as<SnapMeta>();
    gp_refresh_meta<<<(c->n_slots + T - 1) / T, T, 0, st>>>(c->n_slots, c->pair.as<longlong2>(), c->sgpu.as<long long>(), c->slot_node.as<int32_t>(),
                                                           &meta->flags, meta->max_avail);
    gp_fill_pair32<<<(c->n_slots + T) / T, T, 0, st>>>(c->n_slots, c->pair.as<longlong2>(), meta, c->pair32.as<uint2>());
    GP_CUDA(c, cudaGetLastError());
    return GP_OK;
}

// the FIFO loop with a single-AZ packer in one launch (gangpack_zonefifo.cuh)
gp_status gp_pack_fifo_zones(gp_ctx* c, const gp_apps* a, gp_algo algo, gp_mode mode, gp_zone_results* out) {
    if (!c) return GP_ERR_INVALID;
    gp_status s = check_zone_call(c, a, out, "gp_pack_fifo_zones");
    if (s != GP_OK) return s;
    if (algo != GP_TIGHTLY_PACK && algo != GP_MINIMAL_FRAGMENTATION)
        return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: the single-AZ packers are tightly-pack and minimal-fragmentation");
    if (mode != GP_MODE_FIFO_REFERENCE && mode != GP_MODE_FIFO_EXACT)
        return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: mode must be one of the FIFO modes (independent decisions: gp_pack_batch_zones)");
    const int32_t Q = a->n_apps, Z = c->n_groups;
    if (Z > kZoneFifoMaxZones) return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: more than 64 zones");
    if (Q == 0) return GP_OK;
    if (!has_requests(a) || !out->zone || !out->driver_node) return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: missing app/result arrays");
    int64_t pitch = count_offsets(c, a);
    const std::vector<int64_t>& hoff = c->host_off;
    if (a->exec_out_off)
        for (int32_t i = 0; i <= Q; ++i)
            if (a->exec_out_off[i] != hoff[(size_t)i]) return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: exec_out_off must be the prefix sum of exe_count (or NULL)");
    const int64_t total = hoff[(size_t)Q];
    if (total > out->executor_nodes_cap) return fail(c, GP_ERR_CAPACITY, "gp_pack_fifo_zones: executor_nodes_cap too small");
    if (total > 0 && !out->executor_nodes) return fail(c, GP_ERR_INVALID, "gp_pack_fifo_zones: executor_nodes is NULL");
    pitch = (pitch + 3) & ~(int64_t)3;
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const bool mf = algo == GP_MINIMAL_FRAGMENTATION;
    const size_t q = (size_t)Q, T = (size_t)total, RP = (size_t)Z * (size_t)pitch;
    int64_t *in, *d_off;
    int32_t *cnt, *rexe, *zone, *drv, *exe;
    uint8_t* skip;
    int2* rlist;
    double* avg;
    GP_CUDA(c, stage(c->zonebuf, part(in, 6 * q), part(cnt, q), part(d_off, q + 1), part(skip, q), part(rexe, RP), part(rlist, mf ? RP : 0),
                     part(zone, q), part(drv, q), part(exe, T + 1), part(avg, 4 * q)));
    int2* unused = nullptr;
    s = pack_begin(c, Q, GP_TIGHTLY_PACK, mode, total, false, &unused, st);
    if (s != GP_OK) return s;
    SixCols six{};
    s = upload_apps(c, a, hoff.data(), q, st, in, cnt, d_off, six);
    if (s != GP_OK) return s;
    GP_CUDA(c, upload(skip, a->skip_if_no_fit, q, st));
    AppColumns cols{};
    for (int k = 0; k < 6; ++k) cols.q[k] = six.p[k];
    cols.count = cnt; cols.group = nullptr; cols.off = d_off; cols.bits = 64; cols.mem_shift = 0;
    gp_ctx::DevStatus* ds = c->dev_status();
    PrepApp* prep = c->prep.as<PrepApp>();
    gp_prep_apps<<<(Q + kPrepThreads - 1) / kPrepThreads, kPrepThreads, 0, st>>>(
        Q, cols, a->skip_if_no_fit ? skip : nullptr, c->n_groups, total, c->snap_flags.as<SnapMeta>(), nullptr, prep, &ds->err, &c->status_host->err_word);
    Snapshot snap = make_snapshot(c);
    ZoneFifoIn zi{};
    const size_t N = (size_t)c->n_nodes;
    zi.sched[0] = c->sched.as<long long>(); zi.sched[1] = c->sched.as<long long>() + N; zi.sched[2] = c->sched.as<long long>() + 2 * N;
    zi.node_slot = c->node_slot.as<int32_t>();
    zi.row_exec = rexe;
    zi.row_list = mf ? rlist : nullptr;
    zi.row_pitch = pitch; zi.n_apps = Q; zi.n_zones = Z;
    double* avg_out = out->avg_efficiency ? avg : nullptr;
    if (algo == GP_TIGHTLY_PACK) {
        if (mode == GP_MODE_FIFO_REFERENCE) gp_pack_fifo_zones_cta<0, 1><<<1, kZoneFifoThreads, 0, st>>>(snap, prep, zi, zone, drv, exe, avg_out, ds->stats);
        else gp_pack_fifo_zones_cta<0, 2><<<1, kZoneFifoThreads, 0, st>>>(snap, prep, zi, zone, drv, exe, avg_out, ds->stats);
    } else {
        if (mode == GP_MODE_FIFO_REFERENCE) gp_pack_fifo_zones_cta<2, 1><<<1, kZoneFifoThreads, 0, st>>>(snap, prep, zi, zone, drv, exe, avg_out, ds->stats);
        else gp_pack_fifo_zones_cta<2, 2><<<1, kZoneFifoThreads, 0, st>>>(snap, prep, zi, zone, drv, exe, avg_out, ds->stats);
    }
    GP_CUDA(c, cudaGetLastError());
    c->last.kernel_launches += 2;
    s = refresh_views(c, st);                          // the compact view follows the charged slots
    if (s != GP_OK) return s;
    return zone_results_back(c, out, zone, drv, exe, avg, q, T, st);
}

gp_status gp_reserve_placements(gp_ctx* c, const gp_apps* a, const gp_results* placed, int32_t subtract, gp_reservation_table* out) {
    if (!c) return GP_ERR_INVALID;
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, "gp_reserve_placements: gp_set_snapshot first");
    if (!a || !placed || a->n_apps < 0 || (!out && !subtract)) return fail(c, GP_ERR_INVALID, "gp_reserve_placements: NULL arguments");
    const int32_t Q = a->n_apps;
    if (out) out->n_rows = 0;
    if (Q == 0) return GP_OK;
    if (!has_requests(a) || !placed->driver_node) return fail(c, GP_ERR_INVALID, "gp_reserve_placements: missing app/result arrays");
    // host pass: offsets, rows per placed application, index validation
    std::vector<int64_t>& off = c->host_off;
    off.resize(2 * ((size_t)Q + 1));
    int64_t* roff = off.data() + Q + 1;
    int64_t acc = 0, rows = 0;
    for (int32_t i = 0; i < Q; ++i) {
        const int64_t k = a->exe_count[i] > 0 ? a->exe_count[i] : 0;
        off[(size_t)i] = a->exec_out_off ? a->exec_out_off[i] : acc;
        acc += k;
        roff[i] = rows;
        const int32_t d = placed->driver_node[i];
        if (d >= c->n_nodes) return fail(c, GP_ERR_INVALID, "gp_reserve_placements: driver_node out of range");
        if (d >= 0) {
            if (k > 0 && !placed->executor_nodes) return fail(c, GP_ERR_INVALID, "gp_reserve_placements: executor_nodes is NULL");
            if (off[(size_t)i] < 0 || off[(size_t)i] + k > placed->executor_nodes_cap) return fail(c, GP_ERR_CAPACITY, "gp_reserve_placements: offsets exceed executor_nodes_cap");
            for (int64_t t = 0; t < k; ++t) {
                const int32_t n = placed->executor_nodes[off[(size_t)i] + t];
                if (n < 0 || n >= c->n_nodes) return fail(c, GP_ERR_INVALID, "gp_reserve_placements: executor node out of range");
            }
            rows += 1 + k;
        }
    }
    off[(size_t)Q] = a->exec_out_off ? a->exec_out_off[Q] : acc;
    roff[Q] = rows;
    const int64_t total = placed->executor_nodes_cap < off[(size_t)Q] ? placed->executor_nodes_cap : off[(size_t)Q];
    if (out && rows > out->rows_cap) return fail(c, GP_ERR_CAPACITY, "gp_reserve_placements: rows_cap too small");
    if (out && rows > 0 && (!out->app || !out->slot || !out->node || !out->cpu_milli || !out->mem_bytes))
        return fail(c, GP_ERR_INVALID, "gp_reserve_placements: missing table arrays");
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t q = (size_t)Q, T = (size_t)(total > 0 ? total : 0), R = (size_t)rows;
    int64_t *in, *d_off, *d_roff;
    int32_t *cnt, *drv, *exe;
    ReserveOut ro;
    GP_CUDA(c, stage(c->zonebuf, part(in, 6 * q), part(cnt, q), part(d_off, q + 1), part(d_roff, q + 1), part(drv, q), part(exe, T + 1),
                     part(ro.app, R + 1), part(ro.slot, R + 1), part(ro.node, R + 1), part(ro.cpu, R + 1), part(ro.mem, R + 1), part(ro.gpu, R + 1)));
    ReserveIn ri{};
    gp_status s = upload_apps(c, a, off.data(), q, st, in, cnt, d_off, ri.cols);
    if (s != GP_OK) return s;
    GP_CUDA(c, upload(d_roff, roff, 8 * (q + 1), st));
    GP_CUDA(c, upload(drv, placed->driver_node, 4 * q, st));
    if (T) GP_CUDA(c, upload(exe, placed->executor_nodes, 4 * T, st));
    ri.count = cnt; ri.off = d_off; ri.row_off = d_roff;
    ri.driver = drv; ri.exec = exe; ri.n_apps = Q; ri.subtract = subtract ? 1 : 0;
    const int TH = 256;
    gp_reserve_rows<<<(unsigned)((q * 32 + TH - 1) / TH), TH, 0, st>>>(ri, ro, c->node_slot.as<int32_t>(), c->pair.as<longlong2>(), c->sgpu.as<long long>(),
                                                                        c->node_cpu.as<long long>(), c->node_mem.as<long long>(), c->node_gpu.as<long long>());
    GP_CUDA(c, cudaGetLastError());
    if (subtract) { s = refresh_views(c, st); if (s != GP_OK) return s; }
    if (out && R) {
        GP_CUDA(c, cudaMemcpyAsync(out->app, ro.app, 4 * R, cudaMemcpyDeviceToHost, st));
        GP_CUDA(c, cudaMemcpyAsync(out->slot, ro.slot, 4 * R, cudaMemcpyDeviceToHost, st));
        GP_CUDA(c, cudaMemcpyAsync(out->node, ro.node, 4 * R, cudaMemcpyDeviceToHost, st));
        GP_CUDA(c, cudaMemcpyAsync(out->cpu_milli, ro.cpu, 8 * R, cudaMemcpyDeviceToHost, st));
        GP_CUDA(c, cudaMemcpyAsync(out->mem_bytes, ro.mem, 8 * R, cudaMemcpyDeviceToHost, st));
        if (out->gpu) GP_CUDA(c, cudaMemcpyAsync(out->gpu, ro.gpu, 8 * R, cudaMemcpyDeviceToHost, st));
    }
    GP_CUDA(c, cudaStreamSynchronize(st));
    if (out) out->n_rows = rows;
    return GP_OK;
}

gp_status gp_apply_usage_delta(gp_ctx* c, int64_t n_rows, const int32_t* node, const int64_t* cpu, const int64_t* mem, const int64_t* gpu, int32_t sign) {
    if (!c) return GP_ERR_INVALID;
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, "gp_apply_usage_delta: gp_set_snapshot first");
    if (n_rows < 0 || (sign != 1 && sign != -1) || (n_rows > 0 && (!node || !cpu || !mem))) return fail(c, GP_ERR_INVALID, "gp_apply_usage_delta: bad arguments");
    if (n_rows == 0) return GP_OK;
    for (int64_t r = 0; r < n_rows; ++r) {
        const int64_t v[3] = {cpu[r], mem[r], gpu ? gpu[r] : 0};
        for (int64_t x : v) if (x >= kMaxQuantity || x <= -kMaxQuantity) return fail(c, GP_ERR_UNREPRESENTABLE, "gp_apply_usage_delta: |quantity| >= 2^61");
    }
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t R = (size_t)n_rows;
    long long *d_cpu, *d_mem, *d_gpu;
    int32_t* d_node;
    GP_CUDA(c, stage(c->zonebuf, part(d_cpu, R), part(d_mem, R), part(d_gpu, R), part(d_node, R)));
    GP_CUDA(c, upload(d_cpu, cpu, 8 * R, st));
    GP_CUDA(c, upload(d_mem, mem, 8 * R, st));
    GP_CUDA(c, upload(d_gpu, gpu, 8 * R, st));
    GP_CUDA(c, upload(d_node, node, 4 * R, st));
    const int TH = 256;
    gp_usage_delta<<<(unsigned)((R + TH - 1) / TH), TH, 0, st>>>(n_rows, d_node, d_cpu, d_mem, gpu ? d_gpu : nullptr, sign, c->n_nodes, c->node_slot.as<int32_t>(),
                                                                  c->pair.as<longlong2>(), c->sgpu.as<long long>(), c->node_cpu.as<long long>(),
                                                                  c->node_mem.as<long long>(), c->node_gpu.as<long long>());
    GP_CUDA(c, cudaGetLastError());
    gp_status s = refresh_views(c, st);
    if (s != GP_OK) return s;
    GP_CUDA(c, cudaStreamSynchronize(st));
    return GP_OK;
}

// ---- node priority order (f1) and availability snapshot (f2): device stages + the entries built on them ----
}  // extern "C"

// f2 stage: uploads the inputs, leaves avail[3][N] / sched[3][N] on the device (usagebuf).
static gp_status stage_availability(gp_ctx* c, const gp_usage_input* in, cudaStream_t st, long long** d_avail, long long** d_sched,
                                    long long** d_resched = nullptr) {
    const int32_t n = in->n_nodes;
    const size_t N = (size_t)n, R = (size_t)in->n_reservations;
    long long *al, *ov, *avail, *sched, *resched, *rc, *rm, *rg;
    char* usage_has;                            // usage sums [3][N] u64, then the has-reservation flags [N] u32: one memset
    int32_t* rn;
    GP_CUDA(c, stage(c->usagebuf, part(al, 3 * N), part(ov, 3 * N), part(usage_has, 28 * N), part(avail, 3 * N), part(sched, 3 * N),
                     part(resched, 3 * N), part(rn, R), part(rc, R), part(rm, R), part(rg, R)));
    unsigned long long* usage = reinterpret_cast<unsigned long long*>(usage_has);
    unsigned int* has = reinterpret_cast<unsigned int*>(usage_has + 24 * N);
    GP_CUDA(c, upload(al, in->alloc_cpu_milli, 8 * N, st));
    GP_CUDA(c, upload(al + N, in->alloc_mem_bytes, 8 * N, st));
    GP_CUDA(c, upload(al + 2 * N, in->alloc_gpu, 8 * N, st));
    GP_CUDA(c, upload(ov, in->overhead_cpu_milli, 8 * N, st));
    GP_CUDA(c, upload(ov + N, in->overhead_mem_bytes, 8 * N, st));
    GP_CUDA(c, upload(ov + 2 * N, in->overhead_gpu, 8 * N, st));
    GP_CUDA(c, cudaMemsetAsync(usage_has, 0, 28 * N, st));
    const int T = 256;
    if (R) {
        GP_CUDA(c, upload(rn, in->res_node, 4 * R, st));
        GP_CUDA(c, upload(rc, in->res_cpu_milli, 8 * R, st));
        GP_CUDA(c, upload(rm, in->res_mem_bytes, 8 * R, st));
        GP_CUDA(c, upload(rg, in->res_gpu, 8 * R, st));
        gp_usage_scatter<<<(unsigned)((R + T - 1) / T), T, 0, st>>>((long long)R, rn, rc, rm, in->res_gpu ? rg : nullptr, n, usage,
                                                                   d_resched ? has : nullptr);
    }
    gp_availability<<<(n + T - 1) / T, T, 0, st>>>(n, al, al + N, in->alloc_gpu ? al + 2 * N : nullptr, in->overhead_cpu_milli ? ov : nullptr,
                                                   in->overhead_mem_bytes ? ov + N : nullptr, in->overhead_gpu ? ov + 2 * N : nullptr,
                                                   usage, avail, sched, has, d_resched ? resched : nullptr);
    if (d_resched) *d_resched = resched;
    GP_CUDA(c, cudaGetLastError());
    *d_avail = avail;
    *d_sched = sched;
    return GP_OK;
}

struct SortStage { const int32_t* drv; const int32_t* exe; const int32_t* counts; };

// f1 stage: d_cpu / d_mem / d_gpu are device arrays (NULL: uploaded from `in`; gpu optional); leaves the two orders and
// counts[3] = {#driver candidates, #executor candidates, #undefined ties} on the device.
static gp_status stage_sort(gp_ctx* c, const gp_sort_input* in, const long long* d_cpu, const long long* d_mem, const long long* d_gpu,
                            cudaStream_t st, SortStage* out) {
    const int32_t n = in->n_nodes;
    // cheap host validation of the two id arrays the kernels index with
    if (in->zone_id) for (int32_t i = 0; i < n; ++i)
        if (in->zone_id[i] < 0 || in->zone_id[i] >= in->n_zones) return fail(c, GP_ERR_INVALID, "gp_potential_nodes: zone_id out of range");
    if (in->name_rank) for (int32_t i = 0; i < n; ++i)
        if (in->name_rank[i] < 0 || in->name_rank[i] >= n) return fail(c, GP_ERR_INVALID, "gp_potential_nodes: name_rank out of range");
    const size_t N = (size_t)n, Z = (size_t)in->n_zones;
    long long *cpu, *mem, *gpu;
    SortKey *keys, *sorted;
    LabelKey *lk, *lks;
    unsigned long long* tot;
    int32_t *zone, *nr, *prio, *pos, *order, *drv, *exe, *drv2, *exe2, *lrd, *lre, *cnt;
    uint8_t *fc, *fu, *fr;
    GP_CUDA(c, stage(c->sortbuf, part(cpu, N), part(mem, N), part(gpu, N), part(keys, N), part(sorted, N), part(tot, 2 * Z), part(zone, N),
                     part(nr, N), part(prio, Z), part(pos, N), part(order, N), part(drv, N), part(exe, N), part(drv2, N), part(exe2, N),
                     part(lrd, N), part(lre, N), part(lk, N), part(lks, N), part(cnt, 4), part(fc, N), part(fu, N), part(fr, N)));
    if (!d_cpu) { GP_CUDA(c, upload(cpu, in->avail_cpu_milli, 8 * N, st)); d_cpu = cpu; }
    if (!d_mem) { GP_CUDA(c, upload(mem, in->avail_mem_bytes, 8 * N, st)); d_mem = mem; }
    if (!d_gpu && in->avail_gpu) { GP_CUDA(c, upload(gpu, in->avail_gpu, 8 * N, st)); d_gpu = gpu; }
    const bool zoned = in->zone_id != nullptr && in->n_zones > 1;       // one zone: priority 0 for every node, nothing to total
    if (zoned) GP_CUDA(c, upload(zone, in->zone_id, 4 * N, st));
    GP_CUDA(c, upload(nr, in->name_rank, 4 * N, st));
    GP_CUDA(c, upload(fc, in->is_driver_candidate, N, st));
    GP_CUDA(c, upload(fu, in->unschedulable, N, st));
    GP_CUDA(c, upload(fr, in->ready, N, st));
    GP_CUDA(c, upload(lrd, in->driver_label_rank, 4 * N, st));
    GP_CUDA(c, upload(lre, in->executor_label_rank, 4 * N, st));
    if (zoned) GP_CUDA(c, cudaMemsetAsync(tot, 0, 16 * Z, st));
    if (!c->sort_attr_set) {
        GP_CUDA(c, cudaFuncSetAttribute(gp_sort_tiles<SortKey>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSortTile * sizeof(SortKey))));
        c->sort_attr_set = true;
    }
    const int T = 256;
    const int nb = (n + T - 1) / T;
    const int ntile = (n + kSortTile - 1) / kSortTile;
    if (zoned) {
        gp_zone_totals<<<nb, T, 0, st>>>(n, d_cpu, d_mem, zone, tot);
        gp_zone_priority<<<(in->n_zones + T - 1) / T, T, 0, st>>>(in->n_zones, tot, prio);
    }
    gp_make_keys<<<nb, T, 0, st>>>(n, d_cpu, d_mem, zoned ? zone : nullptr, prio, in->name_rank ? nr : nullptr, keys);
    gp_sort_tiles<SortKey><<<ntile, kSortThreads, kSortTile * sizeof(SortKey), st>>>(n, nullptr, keys, sorted);
    gp_rank_by_search<SortKey><<<nb, T, 0, st>>>(n, nullptr, keys, sorted, pos);
    gp_scatter_order<<<nb, T, 0, st>>>(n, pos, order);
    gp_split_candidates<<<1, 1024, 0, st>>>(n, order, in->is_driver_candidate ? fc : nullptr, in->unschedulable ? fu : nullptr,
                                           in->ready ? fr : nullptr, keys, d_gpu, drv, exe, cnt);
    out->drv = drv;
    out->exe = exe;
    out->counts = cnt;
    auto label_sort = [&](const int32_t* count, const int32_t* list, const int32_t* rank, int32_t* sorted_list) {
        gp_label_keys<<<nb, T, 0, st>>>(count, list, rank, lk);
        gp_sort_tiles<LabelKey><<<ntile, kSortThreads, kSortTile * sizeof(LabelKey), st>>>(n, count, lk, lks);
        gp_rank_by_search<LabelKey><<<nb, T, 0, st>>>(n, count, lk, lks, pos);
        gp_label_scatter<<<nb, T, 0, st>>>(count, list, pos, sorted_list);
        return sorted_list;
    };
    if (in->driver_label_rank) out->drv = label_sort(out->counts, out->drv, lrd, drv2);
    if (in->executor_label_rank) out->exe = label_sort(out->counts + 1, out->exe, lre, exe2);
    GP_CUDA(c, cudaGetLastError());
    return GP_OK;
}

// offsets of the single instance group from the device-resident candidate counts
__global__ void gp_offsets_from_counts(const int32_t* __restrict__ counts, int32_t* __restrict__ exec_off, int32_t* __restrict__ drv_off) {
    if (threadIdx.x == 0) { drv_off[0] = 0; drv_off[1] = counts[0]; exec_off[0] = 0; exec_off[1] = counts[1]; }
}

extern "C" {

gp_status gp_potential_nodes(gp_ctx* c, const gp_sort_input* in, int32_t* driver_order, int32_t* n_driver,
                             int32_t* executor_order, int32_t* n_executor) {
    if (!c) return GP_ERR_INVALID;
    if (!in || in->n_nodes < 0 || in->n_zones < 1 || !n_driver || !n_executor ||
        (in->n_nodes > 0 && (!in->avail_cpu_milli || !in->avail_mem_bytes || !driver_order || !executor_order)))
        return fail(c, GP_ERR_INVALID, "gp_potential_nodes: missing arrays or bad sizes");
    const int32_t n = in->n_nodes;
    *n_driver = 0; *n_executor = 0;
    if (n == 0) return GP_OK;
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    SortStage so{};
    gp_status s = stage_sort(c, in, nullptr, nullptr, nullptr, st, &so);
    if (s != GP_OK) return s;
    int32_t counts[3] = {0, 0, 0};
    GP_CUDA(c, cudaMemcpyAsync(counts, so.counts, 12, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaMemcpyAsync(driver_order, so.drv, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaMemcpyAsync(executor_order, so.exe, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    *n_driver = counts[0];
    *n_executor = counts[1];
    if (in->undefined_ties) *in->undefined_ties = counts[2];
    return GP_OK;
}

gp_status gp_build_availability(gp_ctx* c, const gp_usage_input* in, int64_t* avail_cpu, int64_t* avail_mem, int64_t* avail_gpu,
                                int64_t* sched_cpu, int64_t* sched_mem, int64_t* sched_gpu) {
    if (!c) return GP_ERR_INVALID;
    if (!in || in->n_nodes < 0 || in->n_reservations < 0 || (in->n_nodes > 0 && (!in->alloc_cpu_milli || !in->alloc_mem_bytes)) ||
        (in->n_reservations > 0 && (!in->res_node || !in->res_cpu_milli || !in->res_mem_bytes)))
        return fail(c, GP_ERR_INVALID, "gp_build_availability: missing arrays or bad sizes");
    const int32_t n = in->n_nodes;
    if (n == 0) return GP_OK;
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    long long *d_avail = nullptr, *d_sched = nullptr;
    gp_status s = stage_availability(c, in, st, &d_avail, &d_sched);
    if (s != GP_OK) return s;
    const size_t N = (size_t)n;
    int64_t* outs[6] = {avail_cpu, avail_mem, avail_gpu, sched_cpu, sched_mem, sched_gpu};
    for (int k = 0; k < 6; ++k)
        if (outs[k]) GP_CUDA(c, cudaMemcpyAsync(outs[k], (k < 3 ? d_avail : d_sched) + N * (size_t)(k % 3), 8 * N, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    return GP_OK;
}

// availableResources of rescheduleExecutor's first-fit branch: the availability to upload before gp_reschedule_executors(min_frag = 0)
gp_status gp_build_reschedule_availability(gp_ctx* c, const gp_usage_input* in, int64_t* avail_cpu, int64_t* avail_mem, int64_t* avail_gpu) {
    if (!c) return GP_ERR_INVALID;
    if (!in || in->n_nodes < 0 || in->n_reservations < 0 || (in->n_nodes > 0 && (!in->alloc_cpu_milli || !in->alloc_mem_bytes)) ||
        (in->n_reservations > 0 && (!in->res_node || !in->res_cpu_milli || !in->res_mem_bytes)))
        return fail(c, GP_ERR_INVALID, "gp_build_reschedule_availability: missing arrays or bad sizes");
    const int32_t n = in->n_nodes;
    if (n == 0) return GP_OK;
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    long long *d_avail = nullptr, *d_sched = nullptr, *d_re = nullptr;
    gp_status s = stage_availability(c, in, st, &d_avail, &d_sched, &d_re);
    if (s != GP_OK) return s;
    const size_t N = (size_t)n;
    int64_t* outs[3] = {avail_cpu, avail_mem, avail_gpu};
    for (int k = 0; k < 3; ++k)
        if (outs[k]) GP_CUDA(c, cudaMemcpyAsync(outs[k], d_re + N * (size_t)k, 8 * N, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    return GP_OK;
}

// reservations -> availability -> priority orders -> slot layout, without leaving the device
gp_status gp_prepare_cluster(gp_ctx* c, const gp_usage_input* usage, const gp_sort_input* sort, int32_t* n_driver, int32_t* n_executor) {
    if (!c) return GP_ERR_INVALID;
    if (!usage || !sort || usage->n_nodes != sort->n_nodes || usage->n_nodes < 0 || sort->n_zones < 1 || usage->n_reservations < 0 ||
        (usage->n_nodes > 0 && (!usage->alloc_cpu_milli || !usage->alloc_mem_bytes)) ||
        (usage->n_reservations > 0 && (!usage->res_node || !usage->res_cpu_milli || !usage->res_mem_bytes)))
        return fail(c, GP_ERR_INVALID, "gp_prepare_cluster: missing arrays or mismatched sizes");
    const int32_t n = usage->n_nodes;
    if (n_driver) *n_driver = 0;
    if (n_executor) *n_executor = 0;
    if (n == 0) return fail(c, GP_ERR_INVALID, "gp_prepare_cluster: empty node table");
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    long long *d_avail = nullptr, *d_sched = nullptr;
    gp_status s = stage_availability(c, usage, st, &d_avail, &d_sched);
    if (s != GP_OK) return s;
    const size_t N = (size_t)n;
    SortStage so{};
    s = stage_sort(c, sort, d_avail, d_avail + N, d_avail + 2 * N, st, &so);
    if (s != GP_OK) return s;
    // node-table copy (gp_get_snapshot) and the one-group offsets, then the usual slot layout with N as the upper bound
    const size_t nb = sizeof(int64_t) * (N + 1);
    GP_CUDA(c, c->node_cpu.reserve(nb)); GP_CUDA(c, c->node_mem.reserve(nb)); GP_CUDA(c, c->node_gpu.reserve(nb));
    GP_CUDA(c, cudaMemcpyAsync(c->node_cpu.p, d_avail, 8 * N, cudaMemcpyDeviceToDevice, st));
    GP_CUDA(c, cudaMemcpyAsync(c->node_mem.p, d_avail + N, 8 * N, cudaMemcpyDeviceToDevice, st));
    GP_CUDA(c, cudaMemcpyAsync(c->node_gpu.p, d_avail + 2 * N, 8 * N, cudaMemcpyDeviceToDevice, st));
    GP_CUDA(c, c->exec_off.reserve(8)); GP_CUDA(c, c->drv_off.reserve(8));
    gp_offsets_from_counts<<<1, 32, 0, st>>>(so.counts, c->exec_off.as<int32_t>(), c->drv_off.as<int32_t>());
    gp_nodes dn{};
    dn.n_nodes = n;
    dn.avail_cpu_milli = c->node_cpu.as<int64_t>(); dn.avail_mem_bytes = c->node_mem.as<int64_t>(); dn.avail_gpu = c->node_gpu.as<int64_t>();
    dn.n_groups = 1;
    dn.exec_off = c->exec_off.as<int32_t>(); dn.exec_order = so.exe;
    dn.drv_off = c->drv_off.as<int32_t>(); dn.drv_order = so.drv;
    s = build_snapshot_device(c, &dn, n, n, st);      // n is the upper bound of both order lengths
    if (s != GP_OK) return s;
    int32_t counts[3] = {0, 0, 0};
    GP_CUDA(c, cudaMemcpyAsync(counts, so.counts, 12, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    c->n_drv = counts[0]; c->n_exec = counts[1];
    if (sort->undefined_ties) *sort->undefined_ties = counts[2];
    if (n_driver) *n_driver = counts[0];
    if (n_executor) *n_executor = counts[1];
    return GP_OK;
}

// rescheduleExecutor's node choice for a batch of executors (SURVEY 8f row f4); see gangpack_resched.cuh
gp_status gp_reschedule_executors(gp_ctx* c, const gp_reschedule* in, int32_t* node_out) {
    if (!c) return GP_ERR_INVALID;
    if (!c->have_snapshot) return fail(c, GP_ERR_NO_SNAPSHOT, "gp_reschedule_executors: gp_set_snapshot first");
    if (!in || in->n_execs < 0 || (in->n_execs > 0 && (!in->exe_cpu_milli || !in->exe_mem_bytes || !node_out)))
        return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: missing arrays or bad sizes");
    const int32_t q = in->n_execs;
    if (q == 0) return GP_OK;
    const bool mf = in->min_frag != 0;
    const bool has_res = mf && in->reserved_cpu_milli;
    const bool has_host = mf && in->host_off;
    if (has_res && !in->reserved_mem_bytes) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: reserved_mem_bytes missing");
    // host validation (O(q + n_nodes + hosted)): the exact-int64 domain, non-negative requests, CSR shape
    for (int32_t i = 0; i < q; ++i) {
        const int64_t v[3] = {in->exe_cpu_milli[i], in->exe_mem_bytes[i], in->exe_gpu ? in->exe_gpu[i] : 0};
        for (int64_t x : v) {
            if (x < 0) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: negative resource request");
            if (x >= kMaxQuantity) return fail(c, GP_ERR_UNREPRESENTABLE, "gp_reschedule_executors: quantity >= 2^61");
        }
        if (in->group && (in->group[i] < 0 || in->group[i] >= c->n_groups))
            return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: instance group out of range");
    }
    if (has_res)
        for (int32_t n = 0; n < c->n_nodes; ++n) {
            const int64_t v[3] = {in->reserved_cpu_milli[n], in->reserved_mem_bytes[n], in->reserved_gpu ? in->reserved_gpu[n] : 0};
            for (int64_t x : v)
                if (x >= kMaxQuantity || x <= -kMaxQuantity) return fail(c, GP_ERR_UNREPRESENTABLE, "gp_reschedule_executors: |reserved| >= 2^61");
        }
    int64_t hosted = 0;
    if (has_host) {
        if (in->host_off[0] != 0) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: host_off must start at 0");
        for (int32_t i = 0; i < q; ++i)
            if (in->host_off[i + 1] < in->host_off[i]) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: host_off not monotone");
        hosted = in->host_off[q];
        if (hosted > 0 && !in->host_nodes) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: host_nodes missing");
        for (int64_t t = 0; t < hosted; ++t)
            if (in->host_nodes[t] < 0 || in->host_nodes[t] >= c->n_nodes)
                return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: host_nodes index out of range");
    }
    GP_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const size_t Q = (size_t)q, N = (size_t)c->n_nodes, H = (size_t)hosted;
    int64_t *d_exe, *d_res, *d_hoff;
    int32_t *d_grp, *d_hn, *d_out;
    int* d_err;
    GP_CUDA(c, stage(c->reschedbuf, part(d_exe, 3 * Q), part(d_res, 3 * N), part(d_hoff, Q + 1), part(d_grp, Q), part(d_hn, H + 1),
                     part(d_out, Q), part(d_err, 1)));
    GP_CUDA(c, cudaMemsetAsync(d_err, 0, sizeof(int), st));
    GP_CUDA(c, upload(d_exe, in->exe_cpu_milli, 8 * Q, st));
    GP_CUDA(c, upload(d_exe + Q, in->exe_mem_bytes, 8 * Q, st));
    GP_CUDA(c, upload(d_exe + 2 * Q, in->exe_gpu, 8 * Q, st));
    GP_CUDA(c, upload(d_grp, in->group, 4 * Q, st));
    if (has_res && N) {
        GP_CUDA(c, upload(d_res, in->reserved_cpu_milli, 8 * N, st));
        GP_CUDA(c, upload(d_res + N, in->reserved_mem_bytes, 8 * N, st));
        GP_CUDA(c, upload(d_res + 2 * N, in->reserved_gpu, 8 * N, st));
    }
    if (has_host) {
        GP_CUDA(c, upload(d_hoff, in->host_off, 8 * (Q + 1), st));
        if (H) GP_CUDA(c, upload(d_hn, in->host_nodes, 4 * H, st));
    }
    ReschedIn ri{};
    ri.exe_cpu = d_exe; ri.exe_mem = d_exe + Q; ri.exe_gpu = in->exe_gpu ? d_exe + 2 * Q : nullptr;
    ri.group = in->group ? d_grp : nullptr;
    ri.res_cpu = has_res ? d_res : nullptr; ri.res_mem = has_res ? d_res + N : nullptr;
    ri.res_gpu = (has_res && in->reserved_gpu) ? d_res + 2 * N : nullptr;
    ri.host_off = has_host ? d_hoff : nullptr; ri.host_nodes = d_hn;
    ri.node_slot = c->node_slot.as<int32_t>();
    ri.n_execs = q;
    const Snapshot s = make_snapshot(c);
    const int T = 256;
    int64_t blocks = ((int64_t)q * 32 + T - 1) / T;
    const int64_t max_blocks = (int64_t)c->sm_count * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    if (mf) gp_reschedule_kernel<true><<<(int)blocks, T, 0, st>>>(s, ri, d_out, d_err);
    else gp_reschedule_kernel<false><<<(int)blocks, T, 0, st>>>(s, ri, d_out, d_err);
    GP_CUDA(c, cudaGetLastError());
    int err = 0;
    GP_CUDA(c, cudaMemcpyAsync(node_out, d_out, 4 * Q, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, st));
    GP_CUDA(c, cudaStreamSynchronize(st));
    if (err) return fail(c, GP_ERR_INVALID, "gp_reschedule_executors: instance group out of range");
    return GP_OK;
}


}  // extern "C"
