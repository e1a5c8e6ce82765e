// gangpack_tables.cuh -- independent mode (GP_MODE_INDEPENDENT) for tightly-pack / distribute-evenly:
// per-executor-shape capacity tables + the fused (prep + pack) warp-per-application kernel.
//
// Reference semantics (all under /root/reference; LIB = vendor/github.com/palantir/k8s-spark-scheduler-lib/pkg):
//   SparkBinPack driver loop        LIB/binpack/binpack.go:60-87
//   tightlyPackExecutors            LIB/binpack/pack_tightly.go:34-63
//   distributeExecutorsEvenly       LIB/binpack/distribute_evenly.go:34-73
//   node capacity                   LIB/capacity/capacity.go:36-75
//
// Why tables.  Every application of an independent batch is packed against the SAME snapshot
// (internal/extender/unschedulablepods.go:132-166; each Predicate's own pack, resource.go:321), and a node's executor
// capacity depends only on the executor request -- the "shape" (cpu, mem, gpu).  Real queues hold few shapes (the
// synthetic one: 12).  So instead of every application re-scanning the node order, each distinct shape is scanned ONCE:
//   K1 gp_classify_apps   thread per application: intern its shape in a small hash table (atomicCAS on a 64-bit
//                         fingerprint; the full tuple is verified again by the consumer, so a fingerprint collision costs
//                         a fallback, never a wrong answer) and derive the ExecutorNodes offsets when the caller gave none;
//   K2 gp_build_shape_tables  one CTA per (shape, instance group): the group's (cpu, mem) slots are staged tile by tile
//                         into shared memory by TMA bulk copies (cp.async.bulk + mbarrier, double-buffered), every
//                         thread evaluates 4 consecutive nodes, a block-wide exclusive scan turns capacities into the
//                         prefix table  S[i] = sum_{n<i} min(cap(n|0), CLAMP)   (tightly-pack) or
//                                       M[i] = #{n<i : cap(n|0) >= 1}            (distribute-evenly);
//                         and, from the same tile, the expansion list E (node n repeated c(n) times, cut at kExpandCap);
//       (same launch, second half of the grid: one CTA per (driver shape, instance group) finds the first driver candidate
//       the shape fits on);
//   K3 gp_decide_tables   ONE THREAD per application (with the tables a decision is O(log N + k) scalar work -- a warp per
//                         application, right for an O(N) scan, would idle 31 lanes): feasibility is
//                         S[ne] - delta(d) >= k  per driver candidate d starting at the shape's first fit (delta = what the
//                         driver displaces on its own node: O(1) per candidate, the reference's loop binpack.go:67-85
//                         verbatim); ExecutorNodes is a prefix of E with the driver's node spliced in, copied by the whole
//                         warp (32 entries per step); placements longer than E walk the table from the shape's first
//                         hosting node (one word per (shape, group), written by K2) with the next word always in flight
//                         (zero-capacity runs are jumped by a galloping search).
// What the tables cannot answer exactly -- more than kMaxShapes distinct shapes in a batch, executor counts above the table
// clamp, distribute-evenly placements that need more than one round -- is appended, already prepared (PrepApp), to a list
// that the warp-per-application scan kernel gp_pack_listed (the node-order scan of gangpack_kernels.cuh) works off.
// GANGPACK_TABLES=0 sends every application down that path.
#pragma once

#include "gangpack_kernels.cuh"
#include "gangpack_fifo.cuh"     // TMA / mbarrier helpers

namespace gp {

constexpr int kShapeSlots = 1024;     // hash slots (power of two)
constexpr int kShapeProbes = 16;      // linear probes before giving up (-> scan path)
constexpr int kMaxShapes = 64;        // dense tables per batch
constexpr int kTabThreads = 1024;
constexpr int kTabPerThread = 4;
constexpr int kTabTile = kTabThreads * kTabPerThread;     // 4096 nodes per tile: 64 KB of (cpu, mem)
// Entries of the expansion list of one (shape, instance group): the node-major expansion E of the shape's capacities
// (node n repeated c(n) times, E[S[n] .. S[n+1]) = n), cut at kExpandCap.  The placement of every application of the
// shape that needs at most kExpandCap entries (k executors plus what its driver displaces) is copied from it; longer
// ones walk the prefix table.  The bench.py workloads place at most 128 executors per application.
constexpr int kExpandCap = 1024;

struct __align__(16) ShapeEntry {     // 96 bytes
    unsigned long long key;           // fingerprint, never 0; 0 = empty (claimed with atomicCAS)
    int32_t id;                       // dense table id in claim order; -1: more than kMaxShapes shapes in this batch
    uint32_t flags;                   // bit0: gpu request != 0
    DimDiv div[3];                    // executor cpu, mem, gpu: the request itself (div[t].e) and how to divide by it
};
static_assert(sizeof(ShapeEntry) == 96, "ShapeEntry layout");

struct __align__(16) DriverEntry {    // 48 bytes: interned driver request
    unsigned long long key;
    int32_t id;
    uint32_t pad;
    int64_t d[3];
    int64_t pad2;
};
static_assert(sizeof(DriverEntry) == 48, "DriverEntry layout");

// device-side header of one table set
struct ShapeHeader {
    int32_t n_shapes;                 // executor shapes claimed so far (may exceed kMaxShapes)
    int32_t n_dshapes;                // driver shapes claimed so far
    int32_t n_listed;                 // applications handed to the scan kernel
    int32_t pad;
    int32_t id_slot[kMaxShapes];      // dense executor-shape id -> hash slot
    int32_t did_slot[kMaxShapes];     // dense driver-shape id -> hash slot
};
static_assert(sizeof(ShapeHeader) <= 1024, "ShapeHeader");

struct ShapeTables {
    ShapeEntry* entries;              // [kShapeSlots]
    DriverEntry* dentries;            // [kShapeSlots]
    ShapeHeader* hdr;
    uint32_t* table;                  // [kMaxShapes][pitch] exclusive prefix per instance group, indexed by slot
    uint32_t* total;                  // [kMaxShapes][n_groups]
    int32_t* firstfit;                // [kMaxShapes][n_groups] first driver-order position the driver shape fits on (nd: none)
    int32_t* first_host;              // [kMaxShapes][n_groups] first executor-order position with capacity > 0 for the shape (ne: none)
    int32_t* expand;                  // [kMaxShapes][n_groups][kExpandCap] expansion list: entry t is the node that hosts executor t
    int32_t pitch;                    // row length (>= n_slots, multiple of 4)
    int32_t n_groups;
};

// largest executor count / per-node capacity the uint32 prefix of a group can carry without wrapping
__device__ __forceinline__ uint32_t table_clamp(int32_t ne) {
    const uint32_t by_len = 0xFFFFFFFFu / (uint32_t)(ne > 0 ? ne : 1);
    return by_len < (uint32_t)kMaxCount ? by_len : (uint32_t)kMaxCount;
}

__device__ __forceinline__ unsigned long long shape_fingerprint(int64_t a, int64_t b, int64_t c) {
    unsigned long long z = (unsigned long long)a * 0x9E3779B97F4A7C15ull;
    z ^= ((unsigned long long)b + 0xBF58476D1CE4E5B9ull) * 0x94D049BB133111EBull;
    z ^= ((unsigned long long)c + 0x2545F4914F6CDD1Dull) * 0xD6E8FEB86659FD93ull;
    z ^= z >> 29; z *= 0xBF58476D1CE4E5B9ull; z ^= z >> 32;
    return z ? z : 1ull;
}

// ---- raw application columns in either wire width --------------------------------------------------------------
// 64-bit layout: exact int64 quantities (gp_apps).  32-bit layout (gp_apps_wire.quantity_bits == 32): int32 millicores /
// int32 (bytes >> mem_shift) / int32 gpu units -- 28 bytes per application instead of 60.
struct AppColumns {
    const void* q[6];                 // drv cpu, drv mem, drv gpu, exe cpu, exe mem, exe gpu (gpu columns may be NULL = 0)
    const int32_t* count;
    const int32_t* group;             // or NULL (= 0)
    const int64_t* off;               // [n+1] ExecutorNodes offsets (the caller's, or the ones K1 derived)
    int32_t bits;                     // 64 or 32
    int32_t mem_shift;                // 32-bit layout only
    __device__ __forceinline__ int64_t load(int c, int32_t i) const {
        const void* p = q[c];
        if (!p) return 0;
        if (bits == 64) return static_cast<const int64_t*>(p)[i];
        const int64_t v = static_cast<const int32_t*>(p)[i];
        return (c == 1 || c == 4) ? (v < 0 ? v : (v << mem_shift)) : v;     // negative stays negative -> validation error
    }
};

// ---------------------------------------------------------------------------------------------------------------
// K1: intern executor shapes, derive offsets
// ---------------------------------------------------------------------------------------------------------------
constexpr int kClassifyThreads = 256;

// K0: executor counts per block of kClassifyThreads applications (the offsets K1 derives are an exclusive prefix sum: every
// CTA of K1 adds up the <= n/256 block sums before its own block instead of re-reading every count before it -- the
// redundant form moved q^2/512 words through L2)
__global__ void __launch_bounds__(kClassifyThreads) gp_count_blocks(int32_t n_apps, const int32_t* __restrict__ count,
                                                                    unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned long long s_part[kClassifyThreads / 32];
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int32_t c = i < n_apps ? count[i] : 0;
    unsigned long long v = c > 0 ? (unsigned long long)c : 0ull;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(kFull, v, d);
    if (lane == 0) s_part[w] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int k = 0; k < kClassifyThreads / 32; ++k) t += s_part[k];
        block_sums[blockIdx.x] = t;
    }
}

// intern one request tuple (fingerprint fp) into the open-addressing table of ENTRY records; returns the slot or -1.
// `init(entry, slot)` fills a freshly claimed entry.  Called by ONE lane per distinct fingerprint of a warp.
template <class ENTRY, class INIT>
__device__ __forceinline__ int32_t intern_shape(ENTRY* table, unsigned long long fp, INIT init) {
    int32_t slot = (int32_t)(fp & (kShapeSlots - 1));
    for (int p = 0; p < kShapeProbes; ++p) {
        ENTRY* en = table + slot;
        // plain (L1-cacheable) load: a key never changes once set, and a stale 0 is resolved by the CAS below
        unsigned long long cur = en->key;
        if (cur == 0) {
            cur = atomicCAS(&en->key, 0ull, fp);
            if (cur == 0) { init(en, slot); cur = fp; }
        }
        if (cur == fp) return slot;
        slot = (slot + 1) & (kShapeSlots - 1);
    }
    return -1;
}

__global__ void __launch_bounds__(kClassifyThreads) gp_classify_apps(int32_t n_apps, AppColumns cols, ShapeTables tabs,
                                                                     const SnapMeta* __restrict__ meta,
                                                                     int64_t off_base, int64_t* __restrict__ off_out /* or NULL */,
                                                                     const unsigned long long* __restrict__ block_sums /* with off_out */,
                                                                     int32_t* __restrict__ app_slot, int use_tables) {
    __shared__ unsigned long long s_part[kClassifyThreads / 32];
    const int32_t block0 = blockIdx.x * blockDim.x;
    const int32_t i = block0 + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;

    // ---- ExecutorNodes offsets = exclusive prefix sum of max(count, 0), when the caller passed none: the block sums of
    // K0 before this block + a block-wide scan of this block's counts (no inter-CTA dependency inside this launch)
    if (off_out) {
        unsigned long long before = 0;
        for (int32_t t = threadIdx.x; t < (int32_t)blockIdx.x; t += blockDim.x) before += block_sums[t];
        const int32_t mine = (i < n_apps) ? max(cols.count[i], 0) : 0;
        unsigned long long wb = before;
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) wb += __shfl_xor_sync(kFull, wb, d);
        uint32_t incl = warp_incl_scan((uint32_t)mine, lane);
        __shared__ unsigned long long s_before[kClassifyThreads / 32];
        if (lane == 31) s_part[w] = incl;
        if (lane == 0) s_before[w] = wb;
        __syncthreads();
        unsigned long long base = (unsigned long long)off_base, prev = 0;
        for (int t = 0; t < kClassifyThreads / 32; ++t) { base += s_before[t]; if (t < w) prev += s_part[t]; }
        if (i < n_apps) off_out[i] = (int64_t)(base + prev + incl - (uint32_t)mine);
        if (i == n_apps - 1) off_out[n_apps] = (int64_t)(base + prev + incl);
        __syncthreads();
    }
    const unsigned act = __ballot_sync(kFull, i < n_apps);     // the lanes that intern (the whole warp except in the last block)
    if (i >= n_apps) return;
    if (!use_tables) { app_slot[i] = -1; return; }

    // A queue has few distinct requests: the lanes of a warp that carry the same fingerprint elect ONE of them to probe /
    // claim the entry (100 000 threads doing their own CAS on a dozen lines serialise on those lines); the consumer
    // verifies the full tuple, so a fingerprint collision inside a warp only sends an application to the scan.
    const int64_t e0 = cols.load(3, i), e1 = cols.load(4, i), e2 = cols.load(5, i);
    const bool e_ok = e0 >= 0 && e1 >= 0 && e2 >= 0 && e0 < kMaxQuantity && e1 < kMaxQuantity && e2 < kMaxQuantity;
    const unsigned long long efp = e_ok ? shape_fingerprint(e0, e1, e2) : 0ull;
    {
        const unsigned same = __match_any_sync(act, efp);
        const int leader = __ffs(same) - 1;
        int32_t found = -1;
        if (lane == leader && e_ok)
            found = intern_shape(tabs.entries, efp, [&](ShapeEntry* en, int32_t slot) {
                // this lane owns the entry: dense id, division recipes (verified by every consumer against its own tuple)
                int32_t id = atomicAdd(&tabs.hdr->n_shapes, 1);
                if (id >= kMaxShapes) id = -1;
                int bad = 0; uint64_t l; bool fast = true;
                en->div[0] = prep_dim(0, e0, 0, meta->max_avail[0], bad, l, fast);
                en->div[1] = prep_dim(0, e1, 1, meta->max_avail[1], bad, l, fast);
                en->div[2] = prep_dim(0, e2, 2, meta->max_avail[2], bad, l, fast);
                en->flags = e2 != 0 ? 1u : 0u;
                en->id = id;
                if (id >= 0) tabs.hdr->id_slot[id] = slot;
            });
        app_slot[i] = __shfl_sync(act, found, leader);
    }

    // ---- the driver request, interned the same way: its first fitting candidate is searched once per shape (K2d) ----
    const int64_t d0 = cols.load(0, i), d1 = cols.load(1, i), d2 = cols.load(2, i);
    const bool d_ok = d0 >= 0 && d1 >= 0 && d2 >= 0 && d0 < kMaxQuantity && d1 < kMaxQuantity && d2 < kMaxQuantity;
    const unsigned long long dfp = d_ok ? shape_fingerprint(d0 ^ 0x5bd1e995, d1, d2) : 0ull;
    {
        const unsigned same = __match_any_sync(act, dfp);
        const int leader = __ffs(same) - 1;
        int32_t dfound = -1;
        if (lane == leader && d_ok)
            dfound = intern_shape(tabs.dentries, dfp, [&](DriverEntry* en, int32_t slot) {
                int32_t id = atomicAdd(&tabs.hdr->n_dshapes, 1);
                if (id >= kMaxShapes) id = -1;
                en->d[0] = d0; en->d[1] = d1; en->d[2] = d2;
                en->id = id;
                if (id >= 0) tabs.hdr->did_slot[id] = slot;
            });
        app_slot[n_apps + i] = __shfl_sync(act, dfound, leader);         // second half of the array: driver-shape slots
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K2: capacity prefix tables, one CTA per (shape, instance group)
// ---------------------------------------------------------------------------------------------------------------
struct TabScratch {
    unsigned long long bar[2];
    uint32_t part[2][kTabThreads / 32];
    int32_t first_host;
};
constexpr size_t kTabSmemBytes = 1024 + 2 * (size_t)kTabTile * sizeof(longlong2);      // 1 KB scratch + 2 x 64 KB tiles

__device__ __forceinline__ void driver_firstfit_block(const Snapshot& s, const ShapeTables& tabs, int id, int grp);

// grid (2 * kMaxShapes, n_groups): blocks [0, kMaxShapes) build the capacity table of executor shape blockIdx.x, blocks
// [kMaxShapes, 2 kMaxShapes) find the first fitting candidate of driver shape blockIdx.x - kMaxShapes (one launch for both)
template <int ALGO>
__global__ void __launch_bounds__(kTabThreads, 1) gp_build_shape_tables(Snapshot s, ShapeTables tabs) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    if (blockIdx.x >= kMaxShapes) { driver_firstfit_block(s, tabs, (int)blockIdx.x - kMaxShapes, (int)blockIdx.y); return; }
    TabScratch& sh = *reinterpret_cast<TabScratch*>(smem_raw);
    longlong2* tile[2] = {reinterpret_cast<longlong2*>(smem_raw + 1024), reinterpret_cast<longlong2*>(smem_raw + 1024) + kTabTile};
    const int id = blockIdx.x, grp = blockIdx.y;
    const int n_shapes = min(tabs.hdr->n_shapes, kMaxShapes);
    if (id >= n_shapes) return;
    const ShapeEntry& en = tabs.entries[tabs.hdr->id_slot[id]];
    const DimDiv dc = en.div[0], dm = en.div[1], dg = en.div[2];
    const bool ug = (en.flags & 1u) || (s.meta->flags & kSnapGpuNegative);
    const GroupDesc g = s.groups[grp];
    const int32_t ne = g.ne;
    const uint32_t clamp = table_clamp(ne);
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const longlong2* gpair = s.pair + g.sbase;
    const int64_t* ggpu = s.gpu + g.sbase;
    uint32_t* out = tabs.table + (size_t)id * tabs.pitch + g.sbase;
    int32_t* ex = tabs.expand + ((size_t)id * tabs.n_groups + grp) * kExpandCap;

    if (tid == 0) { mbar_init(&sh.bar[0], 1); mbar_init(&sh.bar[1], 1); sh.first_host = ne; }
    __syncthreads();
    const int n_tiles = (ne + kTabTile - 1) / kTabTile;
    auto issue = [&](int t) {          // thread 0: TMA bulk copies of tile t into buffer t & 1 (<= 32 KB per copy)
        const int32_t lo = t * kTabTile;
        const uint32_t bytes = (uint32_t)min(kTabTile, ne - lo) * (uint32_t)sizeof(longlong2);
        mbar_expect_tx(&sh.bar[t & 1], bytes);
        for (uint32_t off = 0; off < bytes; off += 32768u) {
            const uint32_t n = bytes - off < 32768u ? bytes - off : 32768u;
            tma_load_1d(reinterpret_cast<unsigned char*>(tile[t & 1]) + off, reinterpret_cast<const unsigned char*>(gpair + lo) + off, n,
                        &sh.bar[t & 1]);
        }
    };
    if (tid == 0 && n_tiles > 0) issue(0);
    uint32_t carry = 0;
    for (int t = 0; t < n_tiles; ++t) {
        if (tid == 0 && t + 1 < n_tiles) issue(t + 1);           // buffer (t+1)&1 was released by the barrier that ended tile t-1
        mbar_wait(&sh.bar[t & 1], (uint32_t)((t >> 1) & 1));
        const longlong2* tp = tile[t & 1];
        const int32_t lo = t * kTabTile;
        const int32_t i0 = lo + tid * kTabPerThread;
        uint32_t v[kTabPerThread];
        uint32_t sum = 0;
        int32_t my_first = 0x7fffffff;
#pragma unroll
        for (int j = 0; j < kTabPerThread; ++j) {
            const int32_t i = i0 + j;
            uint32_t c = 0;
            if (i < ne) {
                const longlong2 a = tp[i - lo];
                c = min(cap_dim(a.x, dc, clamp), cap_dim(a.y, dm, clamp));
                if (ug) c = min(c, cap_dim(__ldg(ggpu + i), dg, clamp));
                if (ALGO == 1) c = c != 0 ? 1u : 0u;
            }
            if (c != 0 && i < my_first) my_first = i;
            v[j] = sum;             // exclusive within the thread
            sum += c;
        }
        // the first hosting node of the shape: every decision of the shape starts its walk there (no search per application)
        {
            const uint32_t wmin = __reduce_min_sync(kFull, (uint32_t)my_first);
            if (lane == 0 && wmin != 0x7fffffffu) atomicMin(&sh.first_host, (int32_t)wmin);
        }
        // block-wide exclusive scan of the per-thread sums
        const uint32_t incl = warp_incl_scan(sum, lane);
        if (lane == 31) sh.part[t & 1][w] = incl;
        __syncthreads();            // also: every thread is done reading tile[t & 1]... of the PREVIOUS use (see issue())
        const uint32_t pt = sh.part[t & 1][lane];
        const uint32_t pti = warp_incl_scan(pt, lane);
        const uint32_t before = __shfl_sync(kFull, pti - pt, w);
        const uint32_t tile_total = __shfl_sync(kFull, pti, 31);
        const uint32_t base = carry + before + incl - sum;
        if (i0 + kTabPerThread <= ne && ((g.sbase + i0) & 3) == 0) {
            *reinterpret_cast<uint4*>(out + i0) = make_uint4(base + v[0], base + v[1], base + v[2], base + v[3]);
        } else {
#pragma unroll
            for (int j = 0; j < kTabPerThread; ++j) if (i0 + j < ne) out[i0 + j] = base + v[j];
        }
        // the expansion list: node i0 + j fills entries [S, S + c) of it, as far as they are below kExpandCap
        if (base < (uint32_t)kExpandCap) {
#pragma unroll
            for (int j = 0; j < kTabPerThread; ++j) {
                const uint32_t lo = base + v[j];
                const uint32_t hi = min(base + (j + 1 < kTabPerThread ? v[j + 1] : sum), (uint32_t)kExpandCap);
                if (lo < hi) {
                    const int32_t node = __ldg(s.slot_node + g.sbase + i0 + j);
                    for (uint32_t t = lo; t < hi; ++t) ex[t] = node;
                }
            }
        }
        carry += tile_total;
        __syncthreads();            // tile[t & 1] and part[t & 1] may be overwritten from here on
    }
    if (tid == 0) {
        tabs.total[(size_t)id * tabs.n_groups + grp] = carry;
        tabs.first_host[(size_t)id * tabs.n_groups + grp] = sh.first_host;     // ordered by the barrier that ended the last tile
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K2d: first fitting driver candidate per (driver shape, instance group)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void driver_firstfit_block(const Snapshot& s, const ShapeTables& tabs, int id, int grp) {
    __shared__ int32_t s_first;
    const int n = min(tabs.hdr->n_dshapes, kMaxShapes);
    if (id >= n) return;
    const DriverEntry& en = tabs.dentries[tabs.hdr->did_slot[id]];
    const int64_t d0 = en.d[0], d1 = en.d[1], d2 = en.d[2];
    const GroupDesc g = s.groups[grp];
    const bool ug = d2 != 0 || (s.meta->flags & kSnapGpuNegative);
    const longlong2* gpair = s.pair + g.sbase;
    const int64_t* ggpu = s.gpu + g.sbase;
    if (threadIdx.x == 0) s_first = g.nd;
    __syncthreads();
    for (int32_t j0 = 0; j0 < g.nd; j0 += blockDim.x) {
        const int32_t j = j0 + threadIdx.x;
        bool fits = false;
        if (j < g.nd) {
            const int32_t ls = s.drv_slot[g.dbase + j];
            const longlong2 v = __ldg(gpair + ls);
            fits = !(d0 > v.x) && !(d1 > v.y) && !(ug && d2 > __ldg(ggpu + ls));     // driverResources.GreaterThan(available) == false
        }
        if (fits) atomicMin(&s_first, j);
        __syncthreads();
        if (s_first < g.nd) break;               // block-uniform
    }
    if (threadIdx.x == 0) tabs.firstfit[(size_t)id * tabs.n_groups + grp] = s_first;
}

// ---------------------------------------------------------------------------------------------------------------
// K3: one thread per application
// ---------------------------------------------------------------------------------------------------------------
// prefix value S(i), i in [0, ne]
__device__ __forceinline__ uint32_t tab_at(const uint32_t* __restrict__ tab, int32_t i, int32_t ne, uint32_t total) {
    return i < ne ? __ldg(tab + i) : total;
}
// smallest p in (lo, ne] with S(p) > val; requires S(ne) = total > val
__device__ __forceinline__ int32_t tab_next_above(const uint32_t* __restrict__ tab, int32_t lo, int32_t ne, uint32_t total, uint32_t val,
                                                  unsigned long long& probes) {
    int32_t a = lo + 1, b = ne;                     // answer in [a, b], S(b) > val
    // gallop first: the zero-capacity runs inside a walk are short (1-2 probes instead of log2(ne))
    int32_t step = 1;
    while (a < b) {
        const int32_t t = a + step - 1 < b - 1 ? a + step - 1 : b - 1;      // t in [a, b-1]
        ++probes;
        if (tab_at(tab, t, ne, total) > val) { b = t; break; }             // answer in [a, t]
        a = t + 1;                                                          // answer in [t+1, b]
        step <<= 1;
    }
    while (a < b) {
        const int32_t mid = (a + b) >> 1;
        if (tab_at(tab, mid, ne, total) > val) b = mid; else a = mid + 1;
        ++probes;
    }
    return a;
}

constexpr int kDecideThreads = 128;
// cols: raw application columns; app_slot: [2][n_apps] executor / driver shape slots from K1.  Applications the tables
// cannot decide are prepared (PrepApp) and appended to `listed`; force_scan appends every application.
template <int ALGO, class OUT>
__global__ void __launch_bounds__(kDecideThreads) gp_decide_tables(Snapshot s, AppColumns cols, ShapeTables tabs,
                                                                   const int32_t* __restrict__ app_slot, int32_t n_apps, int64_t out_cap,
                                                                   int32_t* __restrict__ driver_node, OUT* __restrict__ executor_nodes,
                                                                   PrepApp* __restrict__ prep, int32_t* __restrict__ listed,
                                                                   unsigned long long* __restrict__ stats, int* __restrict__ err,
                                                                   volatile int* __restrict__ err_host, int force_scan) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long probes = 0, drivers = 0;
    // placement to copy from an expansion list (see below): out[t] = list[t] for t < a, node for a <= t < a + b,
    // list[t + skip] after that
    bool copy = false;
    const int32_t* list = nullptr;
    int64_t copy_off = 0;
    uint32_t copy_k = 0, copy_a = 0, copy_b = 0, copy_skip = 0;
    int32_t copy_node = 0;
    if (i < n_apps) {
        const int64_t d_cpu = cols.load(0, i), d_mem = cols.load(1, i), d_gpu = cols.load(2, i);
        const int64_t e_cpu = cols.load(3, i), e_mem = cols.load(4, i), e_gpu = cols.load(5, i);
        const int32_t kk = cols.count[i];
        const int32_t grp = cols.group ? cols.group[i] : 0;
        const int64_t off = cols.off[i], off1 = cols.off[i + 1];
        // ---- validation (types.SparkApplicationResources must be non-negative and inside the exact-int64 domain) ----
        int bad = 0;
        if (d_cpu < 0 || d_mem < 0 || d_gpu < 0 || e_cpu < 0 || e_mem < 0 || e_gpu < 0 || kk < 0) bad |= kErrNegativeRequest;
        if (d_cpu >= kMaxQuantity || d_mem >= kMaxQuantity || d_gpu >= kMaxQuantity || e_cpu >= kMaxQuantity || e_mem >= kMaxQuantity ||
            e_gpu >= kMaxQuantity || kk > kMaxCount) bad |= kErrUnrepresentable;
        if (grp < 0 || grp >= s.n_groups) bad |= kErrBadGroup;
        if (off < 0 || off1 - off != (int64_t)(kk > 0 ? kk : 0) || off1 > out_cap) bad |= kErrBadOffsets;
        if (bad) {
            atomicOr(err, bad); *err_host = bad;
            driver_node[i] = -1;
        } else {
            const GroupDesc g = s.groups[grp];
            const int32_t ne = g.ne, nd = g.nd;
            const uint32_t k = (uint32_t)kk;
            const int snap_flags = s.meta->flags;
            bool need_scan = force_scan != 0;
            int32_t result = -1;
            const ShapeEntry* en = nullptr;
            const uint32_t* tab = nullptr;
            uint32_t total = 0;
            const uint32_t clamp = table_clamp(ne);
            if (!need_scan) {
                const int32_t slot = app_slot[i];
                if (slot < 0) need_scan = true;
                else {
                    en = tabs.entries + slot;       // the full tuple decides, not the fingerprint
                    if (en->id < 0 || en->div[0].e != e_cpu || en->div[1].e != e_mem || en->div[2].e != e_gpu || k > clamp) need_scan = true;
                    else {
                        tab = tabs.table + (size_t)en->id * tabs.pitch + g.sbase;
                        total = tabs.total[(size_t)en->id * tabs.n_groups + grp];
                        // distribute-evenly: no hosting node at all -> no executor can be placed (distribute_evenly.go:72);
                        // 1..k hosting nodes: several rounds or an exact per-candidate test -> the scan decides
                        if (ALGO == 1 && k != 0 && total != 0 && total < k + 1) need_scan = true;
                    }
                }
            }
            if (!need_scan && !(k != 0 && (ALGO == 0 ? total < k : total == 0))) {   // not even without a driver (pack_tightly.go:62, distribute_evenly.go:72)
                const bool drv_gpu = d_gpu != 0 || (snap_flags & kSnapGpuNegative);
                const bool cap_gpu = drv_gpu || (en->flags & 1u);
                const longlong2* gpair = s.pair + g.sbase;
                const int64_t* ggpu = s.gpu + g.sbase;
                // ---- driver loop (binpack.go:67-85) from the shape's first fitting candidate ---------------------------
                int32_t j = 0;
                {
                    const int32_t ds = app_slot[n_apps + i];
                    if (ds >= 0) {
                        const DriverEntry& de = tabs.dentries[ds];
                        if (de.id >= 0 && de.d[0] == d_cpu && de.d[1] == d_mem && de.d[2] == d_gpu) j = tabs.firstfit[(size_t)de.id * tabs.n_groups + grp];
                    }
                }
                int32_t dslot = -1;
                uint32_t cd = 0, c0d = 0, spd = 0;
                for (; j < nd; ++j) {
                    ++drivers;
                    const int32_t ls = s.drv_slot[g.dbase + j];
                    const longlong2 v = __ldg(gpair + ls);
                    const int64_t gv = (drv_gpu || cap_gpu) ? __ldg(ggpu + ls) : 0;
                    if ((d_cpu > v.x) || (d_mem > v.y) || (drv_gpu && d_gpu > gv)) continue;
                    uint32_t my_c0 = 0, my_cd = 0, sp = 0;
                    if (ls < ne && k != 0) {
                        sp = __ldg(tab + ls);
                        my_c0 = tab_at(tab, ls + 1, ne, total) - sp;
                        probes += 2;
                        if (my_c0 != 0) {        // what the node can still take once the driver sits on it
                            uint32_t c = min(cap_dim(v.x - d_cpu, en->div[0], clamp), cap_dim(v.y - d_mem, en->div[1], clamp));
                            if (cap_gpu) c = min(c, cap_dim(gv - d_gpu, en->div[2], clamp));
                            if (ALGO == 1) c = c != 0 ? 1u : 0u;
                            my_cd = c;
                        }
                        if (ALGO == 0 && total - (my_c0 - my_cd) < k) continue;       // the executors do not fit with this driver
                        // distribute-evenly: >= k+1 hosting nodes, the driver removes at most its own
                    }
                    dslot = ls; cd = my_cd; c0d = my_c0; spd = sp;
                    break;
                }
                if (dslot >= 0) {
                    result = s.slot_node[g.sbase + dslot];
                    if (k != 0 && k + (c0d - cd) <= (uint32_t)kExpandCap) {
                        // ---- emission from the expansion list E: the driver's node p takes cd executors instead of
                        // c0d, so the placement is  E[0, S[p]) ++ p x min(cd, k - S[p]) ++ E[S[p+1], ...)  when S[p] < k,
                        // else E[0, k) (also for a driver in a spare slot).  Copied by the whole warp below.
                        copy = true;
                        list = tabs.expand + ((size_t)en->id * tabs.n_groups + grp) * kExpandCap;
                        copy_off = off; copy_k = k; copy_node = result;
                        copy_a = (dslot < ne && spd < k) ? spd : k;
                        copy_b = min(cd, k - copy_a);
                        copy_skip = c0d - copy_b;
                        probes += k - copy_b;
                    } else if (k != 0) {
                        // ---- emission: walk the prefix table from the first hosting node ---------------------------------
                        OUT* out = executor_nodes + off;
                        const int32_t* slot_node = s.slot_node + g.sbase;
                        const int32_t dpos = (dslot < ne) ? dslot : 0x7fffffff;
                        int32_t pos = __ldg(tabs.first_host + (size_t)en->id * tabs.n_groups + grp);    // first node with room for the shape
                        ++probes;
                        uint32_t prev = 0, placed = 0;
                        uint32_t nxt = tab_at(tab, pos + 1, ne, total);
                        ++probes;
                        while (placed < k && pos < ne) {
                            // S(pos + 2) is requested before S(pos + 1) is consumed: the walk's dependent-load chain is
                            // what bounds this kernel (one thread per application), so the next word is always in flight
                            const uint32_t nxt2 = tab_at(tab, pos + 2, ne, total);
                            ++probes;
                            uint32_t c = nxt - prev;
                            if (pos == dpos) c = cd;
                            if (c == 0) {                               // zero-capacity run (or the driver ate its node): jump
                                if (nxt >= total) break;                // cannot happen for a feasible placement
                                pos = tab_next_above(tab, pos + 1, ne, total, nxt, probes) - 1;
                                prev = nxt;
                                nxt = tab_at(tab, pos + 1, ne, total);
                                ++probes;
                                continue;
                            }
                            const uint32_t take = c < k - placed ? c : k - placed;
                            const OUT node = (OUT)__ldg(slot_node + pos);
                            for (uint32_t t = 0; t < take; ++t) out[placed + t] = node;
                            placed += take;
                            prev = nxt;
                            nxt = nxt2;
                            ++pos;
                        }
                    }
                }
            }
            if (need_scan) {
                // ---- prepared record for the scan kernel ------------------------------------------------------------------
                const int32_t at = atomicAdd(&tabs.hdr->n_listed, 1);
                PrepApp p;
                int b2 = 0; uint64_t lmax = 0; bool fast = true;
                const int64_t dd[3] = {d_cpu, d_mem, d_gpu}, ee[3] = {e_cpu, e_mem, e_gpu};
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    uint64_t l;
                    p.drv[t] = dd[t];
                    p.div[t] = prep_dim(dd[t], ee[t], t, s.meta->max_avail[t], b2, l, fast);
                    if (l > lmax) lmax = l;
                }
                p.out_off = off; p.count = kk; p.group = grp;
                p.lmax = (int32_t)(lmax < (uint64_t)k ? lmax : (uint64_t)k);
                const bool f32 = prep_fast32(fast, p.div[0], p.div[1], s.meta);
                p.flags = ((d_gpu != 0 || e_gpu != 0) ? kAppUsesGpu : 0u) | (fast ? kAppFast : 0u) | (f32 ? kAppFast32 : 0u);
                const uint4* src = reinterpret_cast<const uint4*>(&p);
                uint4* dst = reinterpret_cast<uint4*>(prep + at);
#pragma unroll
                for (int t = 0; t < (int)(sizeof(PrepApp) / sizeof(uint4)); ++t) dst[t] = src[t];
                listed[at] = i;
            } else {
                driver_node[i] = result;
            }
        }
    }
    // ---- the copies, one application of the warp after the other: coalesced loads from E, coalesced stores ----------
    const int lane = threadIdx.x & 31;
    for (unsigned todo = __ballot_sync(kFull, copy); todo; todo &= todo - 1) {
        const int src = __ffs(todo) - 1;
        const int32_t* l = reinterpret_cast<const int32_t*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(list), src));
        OUT* out = executor_nodes + __shfl_sync(kFull, copy_off, src);
        const uint32_t k = __shfl_sync(kFull, copy_k, src), a = __shfl_sync(kFull, copy_a, src);
        const uint32_t ab = a + __shfl_sync(kFull, copy_b, src), skip = __shfl_sync(kFull, copy_skip, src);
        const int32_t node = __shfl_sync(kFull, copy_node, src);
        for (uint32_t t = lane; t < k; t += 32) out[t] = (OUT)(t < a ? __ldg(l + t) : (t < ab ? node : __ldg(l + t + skip)));
    }
    // statistics: one atomic per warp
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) { probes += __shfl_xor_sync(kFull, probes, d); drivers += __shfl_xor_sync(kFull, drivers, d); }
    if ((threadIdx.x & 31) == 0 && (probes | drivers)) { atomicAdd(stats + 0, probes); atomicAdd(stats + 1, drivers); }
}

// ---------------------------------------------------------------------------------------------------------------
// the node-order scan for the listed applications: one warp per application (gangpack_kernels.cuh)
// ---------------------------------------------------------------------------------------------------------------
constexpr int kPackTabThreads = 256;
#ifndef GP_TAB_MIN_BLOCKS
#define GP_TAB_MIN_BLOCKS 4
#endif
template <int ALGO, class OUT>
__global__ void __launch_bounds__(kPackTabThreads, GP_TAB_MIN_BLOCKS) gp_pack_listed(Snapshot s, const ShapeHeader* __restrict__ hdr,
                                                                                     const PrepApp* __restrict__ prep,
                                                                                     const int32_t* __restrict__ listed,
                                                                                     int32_t* __restrict__ driver_node,
                                                                                     OUT* __restrict__ executor_nodes,
                                                                                     int2* __restrict__ scratch,
                                                                                     unsigned long long* __restrict__ stats,
                                                                                     unsigned int* __restrict__ next_app) {
    __shared__ uint16_t cap_cache[kPackTabThreads / 32][kCapCache];
    const int n = hdr->n_listed;
    if (n == 0) return;
    const int lane = threadIdx.x & 31;
    uint16_t* wcache = cap_cache[threadIdx.x >> 5];
    WarpStats st{0, 0};
    const int snap_flags = s.meta->flags;
    const GroupDesc g0 = s.groups[0];
    unsigned int i = 0, n1 = 0;
    if (lane == 0) { i = atomicAdd(next_app, 1u); n1 = atomicAdd(next_app, 1u); }
    i = __shfl_sync(kFull, i, 0);
    n1 = __shfl_sync(kFull, n1, 0);
    unsigned long long apps_done = 0;
    while (i < (unsigned int)n) {
        unsigned int n2 = 0;
        if (lane == 0) n2 = atomicAdd(next_app, 1u);
        if (lane == 0 && n1 < (unsigned int)n) asm volatile("prefetch.global.L1 [%0];" ::"l"(prep + n1));
        const PrepApp* pa = prep + i;
        const int32_t d = pack_app<ALGO, OUT>(s, pa, executor_nodes, scratch, wcache, st, lane, snap_flags, g0);
        if (lane == 0) driver_node[listed[i]] = d;
        ++apps_done;
        i = n1;
        n1 = __shfl_sync(kFull, n2, 0);
    }
    if (lane == 0) {
        atomicAdd(stats + 0, st.nodes);
        atomicAdd(stats + 1, st.drivers);
        atomicAdd(stats + 2, apps_done);
        atomicAdd(stats + 3, st.nodes);
    }
}

}  // namespace gp
