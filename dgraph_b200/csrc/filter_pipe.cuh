// filter_pipe.cuh -- persistent, TMA-fed version of the batched sorted-set filter.
//
// Same contract as filter_kernel.cuh (IntersectWith / IntersectSorted chain /
// Difference over a batch of queries, bit-exact incl. duplicate semantics), built
// as a Blackwell pipeline:
//
//   filter_tiles_kernel  one thread per tile: owning task, driving offset, plan index,
//                        predecessor value -> a tile table in HBM.
//   filter_plan_kernel   one thread per (tile, filter list): both slice bounds
//                        [lower_bound(L_j, tile first), upper_bound(L_j, tile last))
//                        as two interleaved binary searches -> a small plan in HBM.
//   filter_pipe_kernel   persistent CTAs (grid = resident capacity, 2 per SM).  Warp roles:
//     M  (1 warp)  metadata: claims the next tile(s) (atomic ticket = look-back order),
//                  reads the tile table, list descriptors and plan entries and pushes a
//                  tile descriptor into a small ring in shared memory;
//     T  (1 warp)  waits for a free stage, lays the tile's slices out and issues ONE
//                  TMA bulk copy (cp.async.bulk, mbarrier complete_tx) per list plus
//                  one for the 512 driving values: global -> shared with no
//                  register staging and no consumer instruction spent on loads;
//     C  (8 warps) consume a stage, each warp on its own 64 candidates (2 rows in
//                  registers) and with NO block barrier: binary-lifting searches over
//                  the staged 64-bit keys, interleaved across rows / lists for ILP,
//                  warp-level re-packs between lists, survivors dropped into the
//                  warp's fixed segment of an output slot; the last warp to deliver a
//                  tile publishes the tile's aggregate for the look-back;
//     O  (1 warp)  drains output slots: decoupled look-back -> ordered stores.  Only
//                  this warp ever waits on other CTAs.
//   Two stages and six output slots are in flight per CTA, so the TMA traffic of
//   tile i+1 and the look-back of tiles i-1.. overlap the searches of tile i.
//
// Lists that are not pre-staged (slice larger than the stage, or more than 8
// filter lists) are binary-searched in HBM by the surviving candidates.
#pragma once

#include "decode_kernel.cuh"   // mbarrier / TMA helpers
#include "filter_kernel.cuh"

namespace dgx {

// Tile geometry is a template parameter of the kernel: VA candidate rows per consumer warp, 32 VA candidates per
// warp, 8 consumer warps, 256 VA candidates per tile.  Wide queries (k >= 3) run VA = 2 (512-value tiles: more
// tiles in flight per byte of shared memory, measured best on C2); 2-list batches run VA = 4 (1024-value tiles:
// their per-tile costs -- metadata, TMA issue, look-back, delivery -- are spread over twice the values).
constexpr int P_CW = 8;                  // consumer warps
constexpr int P_CT = P_CW * 32;          // consumer threads
constexpr int P_NT = P_CT + 96;          // + metadata warp + TMA warp + output warp
#define DGX_GEOM(VA)                                                                     \
    constexpr int P_VA = (VA);           /* candidate rows per consumer warp */           \
    constexpr int P_WC = 32 * (VA);      /* candidates per consumer warp */               \
    constexpr int P_TA = P_CW * 32 * (VA); /* candidates per tile */                      \
    static_assert(P_VA == 2 || P_VA == 4, "rows per consumer warp")
constexpr int p_tile_size(int va) { return P_CW * 32 * va; }
#ifndef DGX_P_OS
#define DGX_P_OS 6
#endif
constexpr int P_OS = DGX_P_OS;           // output slots in flight (6 vs 4: 2-list batches +4.5 %, C2 unchanged)
#ifndef DGX_P_ST
#define DGX_P_ST 2
#endif
#ifndef DGX_P_PAIR2
#define DGX_P_PAIR2 1   // two-row warps search two lists per iteration (four chains) once past the first list
#endif
#ifndef DGX_P_FAST
#define DGX_P_FAST 1   // 0: build without the 32-bit fast path (A/B measurements, fallback-path tests)
#endif
constexpr int P_ST = DGX_P_ST;           // data stages in flight
constexpr int P_MAXL = 8;                // filter lists a stage can hold
constexpr int P_RING = 8;                // tile descriptors in flight between M and T
constexpr int P_GRP = 4;                 // most tiles the metadata warp can resolve per iteration (8 lanes each)
constexpr u32 P_END = 0xffffffffu;
// Back-off between polls of a waiting helper warp (ns): TMA warp / metadata + output warps / look-back.
// The helpers share schedulers with consumer warps and every poll is an issue slot taken from them
// (polling was 14 % of the issued instructions at 128 ns); measured -0.8 % (C2) / -2 % (C1 batch).
#ifndef DGX_P_SLEEP_T
#define DGX_P_SLEEP_T 600
#endif
#ifndef DGX_P_SLEEP_MO
#define DGX_P_SLEEP_MO 2000
#endif
#ifndef DGX_P_SLEEP_LB
#define DGX_P_SLEEP_LB 1000
#endif

struct PPlanEntry { u64 r0, r1; };
struct PTileEntry {            // everything the metadata warp needs about a tile, resolved by filter_tiles_kernel
    u32 task, list_first, k, na;
    u64 a0, plan_idx, prev;
    u32 has_prev, pad;
};

struct PParams {
    FParams f;                 // tasks, lists, op, outputs, look-back state (ticket unused)
    const u64* plan_base;      // per task: index of its first plan entry
    const PPlanEntry* plan;    // per (tile, filter list)
    const struct PTileEntry* tiles;  // per tile
    u32 slice_cap;             // stage capacity for slices, in u64 values
    u32 nctas;
    u32 grp;                   // tiles the metadata warp claims per ticket (1 .. P_GRP)
};

// ---- plan ---------------------------------------------------------------------------
// One THREAD per (tile, filter list): r0 = first i with L[i] >= tile first, r1 = first i
// with L[i] > tile last, as two interleaved binary searches.  A binary search touches one
// new 32-byte sector per level only near its end (~8 sectors), where the 32-ary warp
// search of filter_kernel.cuh touches ~70: the plan must not cost a second pass over HBM.
__global__ void __launch_bounds__(256) filter_plan_kernel(const FTask* __restrict__ tasks, const FList* __restrict__ lists,
                                                          const u64* __restrict__ plan_base, u32 ntasks, u64 npairs,
                                                          PPlanEntry* __restrict__ plan, u32 tile_sz) {
    const u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npairs) return;
    u32 lo = 0, hi = ntasks;  // last task with plan_base <= p (the one that owns pair p)
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (plan_base[mid] <= p) lo = mid; else hi = mid;
    }
    const FTask T = tasks[lo];
    const u64 local = p - plan_base[lo];
    const u32 km1 = T.k - 1;
    const u64 tl = local / km1;
    const u32 j = (u32)(local - tl * km1) + 1;
    const FList LA = lists[T.list_first];
    const u64 lenA = flist_len(LA);
    const u64 a0 = tl * (u64)tile_sz;
    u64 r0 = 0, r1 = 0;
    if (a0 < lenA) {
        const u64 na = lenA - a0 < (u64)tile_sz ? lenA - a0 : (u64)tile_sz;
        const u64 tlo = ld_probe(LA.ptr + a0), thi = ld_probe(LA.ptr + a0 + na - 1);
        const FList Lj = lists[T.list_first + j];
        const u64* __restrict__ B = Lj.ptr;
        u64 l0 = 0, h0 = flist_len(Lj), l1 = 0, h1 = h0;
        while (l0 < h0 || l1 < h1) {
            const u64 m0 = l0 + ((h0 - l0) >> 1), m1 = l1 + ((h1 - l1) >> 1);
            const bool a = l0 < h0, c = l1 < h1;
            const u64 v0 = a ? ld_probe(B + m0) : 0, v1 = c ? ld_probe(B + m1) : 0;
            if (a) { if (v0 < tlo) l0 = m0 + 1; else h0 = m0; }
            if (c) { if (v1 <= thi) l1 = m1 + 1; else h1 = m1; }
        }
        r0 = l0; r1 = l1;
    }
    plan[p].r0 = r0;
    plan[p].r1 = r1;
}

// One thread per tile: which task it belongs to and where its driving values start.
__global__ void __launch_bounds__(256) filter_tiles_kernel(const FTask* __restrict__ tasks, const FList* __restrict__ lists,
                                                           const u64* __restrict__ plan_base, u32 ntasks, u32 ntiles,
                                                           PTileEntry* __restrict__ tiles, u32 tile_sz) {
    const u32 tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= ntiles) return;
    u32 lo = 0, hi = ntasks;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (tasks[mid].tile_base <= (u64)tile) lo = mid; else hi = mid;
    }
    const FTask T = tasks[lo];
    const FList LA = lists[T.list_first];
    const u64 lenA = flist_len(LA);
    PTileEntry e;
    e.task = lo; e.list_first = T.list_first; e.k = T.k;
    e.a0 = ((u64)tile - T.tile_base) * (u64)tile_sz;
    e.na = e.a0 < lenA ? (u32)((lenA - e.a0 < (u64)tile_sz) ? (lenA - e.a0) : (u64)tile_sz) : 0u;
    e.plan_idx = plan_base[lo] + ((u64)tile - T.tile_base) * (u64)(T.k - 1);
    e.has_prev = (e.a0 > 0 && e.na > 0) ? 1u : 0u;
    e.prev = e.has_prev ? ld_probe(LA.ptr + e.a0 - 1) : 0;
    e.pad = 0;
    tiles[tile] = e;
}

// ---- pipeline state in shared memory -------------------------------------------------
struct PDesc {                 // one tile, produced by M, consumed by T
    u32 tile, task, na, k, list_first, has_prev;
    u64 a0, prev, plan_idx;
    const u64* A;
    const u64* ptr[P_MAXL];
    u64 len[P_MAXL], r0[P_MAXL], r1[P_MAXL];
};
struct PStageInfo {            // one stage, produced by T, consumed by C
    u32 tile, task, na, k, list_first, has_prev, nstaged, headA;
    u64 a0, prev, plan_idx;
    const u64* A;
    const u64* ptr[P_MAXL];
    u64 len[P_MAXL], r0[P_MAXL];
    u32 off[P_MAXL], n[P_MAXL];
};
struct POutSlot {              // survivors of one tile: warp w owns data[P_WC*w ..) and cnt[w]
    u32 tile, task;
    u32 first;                 // the tile opens its task's output range (driving offset 0)
    u32 total, arrived;        // running sum of cnt / number of warps that delivered (reset by O)
    u32 cnt[P_CW];
};
struct PShared {
    u64 full[P_ST], empty[P_ST], ofull[P_OS], oempty[P_OS], ready[P_RING], freed[P_RING];
    PDesc ring[P_RING];
    PStageInfo st[P_ST];
    POutSlot os[P_OS];
};

__device__ __forceinline__ void mbar_arrive(u32 bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// Re-pack a consumer warp's survivors into rows 0..ceil(live/32)-1 (order preserved).
template <int P_VA>
__device__ __forceinline__ void pwarp_repack(u64 (&c)[P_VA], unsigned& alive, int& rows, u64* s_w, int lane) {
    unsigned b[P_VA];
    int tot = 0;
#pragma unroll
    for (int i = 0; i < P_VA; ++i) {
        b[i] = __ballot_sync(0xffffffffu, (i < rows) && ((alive >> i) & 1u));
        tot += __popc(b[i]);
    }
    const int nrows = (tot + 31) >> 5;
    if (nrows >= rows) return;
    if (nrows == 0) { rows = 0; alive = 0; return; }
    const unsigned lt = (1u << lane) - 1u;
    int before = 0;
#pragma unroll
    for (int i = 0; i < P_VA; ++i) {
        if ((b[i] >> lane) & 1u) s_w[before + __popc(b[i] & lt)] = c[i];
        before += __popc(b[i]);
    }
    __syncwarp();
    alive = 0;
#pragma unroll
    for (int i = 0; i < P_VA; ++i) {
        if (i < nrows && 32 * i + lane < tot) { c[i] = s_w[32 * i + lane]; alive |= 1u << i; }
    }
    __syncwarp();
    rows = nrows;
}

struct PTile {          // per-thread constants of the tile being consumed
    const u64* cand;    // staged driving values (tile order)
    const u64* A;
    u64 a0, prev;
    bool has_prev;
    int cidx0;
    int op;
};

// NJ independent lower-bound searches advanced in lock step (binary lifting): job j
// looks for x[j] in sb[j][0..n[j]).  The ladder starts at the largest power of two
// <= max n, every step is guarded by t <= n[j], so the NJ dependent chains overlap.
template <int NJ>
__device__ __forceinline__ void lift_multi(const u64* const (&sb)[NJ], const int (&n)[NJ], const u64 (&x)[NJ],
                                           int (&pos)[NJ]) {
    int nmax = 1;
#pragma unroll
    for (int j = 0; j < NJ; ++j) { pos[j] = 0; nmax = n[j] > nmax ? n[j] : nmax; }
#define DGX_LIFTM(H)                                                              \
    {                                                                             \
        _Pragma("unroll") for (int j = 0; j < NJ; ++j) {                          \
            const int t_ = pos[j] + (H);                                          \
            if (t_ <= n[j] && sb[j][t_ - 1] < x[j]) pos[j] = t_;                  \
        }                                                                         \
    }
    switch (31 - __clz(nmax)) {
        case 14: DGX_LIFTM(16384)
        case 13: DGX_LIFTM(8192)
        case 12: DGX_LIFTM(4096)
        case 11: DGX_LIFTM(2048)
        case 10: DGX_LIFTM(1024)
        case 9: DGX_LIFTM(512)
        case 8: DGX_LIFTM(256)
        case 7: DGX_LIFTM(128)
        case 6: DGX_LIFTM(64)
        case 5: DGX_LIFTM(32)
        case 4: DGX_LIFTM(16)
        case 3: DGX_LIFTM(8)
        case 2: DGX_LIFTM(4)
        case 1: DGX_LIFTM(2)
        default: DGX_LIFTM(1)
    }
#undef DGX_LIFTM
}

// hit test of candidate value x (row i of this lane) at staged position p of list (sb, n, g0, B, lenB)
__device__ __forceinline__ bool phit(const PTile& X, u64 x, int i, unsigned dup, const u64* sb, int n, int p, u64 g0,
                                     const u64* __restrict__ B, u64 lenB) {
    if (!((dup >> i) & 1u)) return (p < n) && (sb[p] == x);
    const u64 g = g0 + (u64)p + cand_rank(X.cand, X.cidx0 + 32 * i, x, X.has_prev, X.prev, X.A, X.a0);
    return (g < lenB) && (ld_probe(B + g) == x);
}

// ---- 32-bit fast path ---------------------------------------------------------------------
// When every value of a tile shares its upper 32 bits (the rule for real UID ranges: a tile of 512
// driving values rarely straddles a multiple of 2^32) the staged slices, which lie inside
// [tile first, tile last], share them too, and membership is decided on the LOW words alone, read in
// place (ld.shared.u32 at an 8-byte stride) with 32-bit compares.  A search is: one probe of element
// p2-1 (p2 = largest power of two <= n) choosing the window [0, p2) or [n-p2, n), then log2(p2)
// lifting steps with compile-time strides -- load with an immediate offset, compare, predicated add:
// three instructions a step, against seven for the guarded 64-bit ladder (lift_multi).
template <int OFF>
__device__ __forceinline__ u32 lds32(u32 addr) {
    u32 v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}
__device__ __forceinline__ u32 lds32r(u32 addr) {
    u32 v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
// R rows of one lane against NL staged slices at once (slice j: shared byte address sb[j], n[j] >= P values at an
// 8-byte stride), every (row, list) pair an independent dependency chain.  All chains run the SAME ladder: a window
// of P = 2^l2P values per slice, P <= n[j] <= 3P.  The window is chosen by three pivots -- the last elements of
// windows starting at 0, s1, s2 (s1 = ceil((n-P)/3), s2 = 2 s1, both clamped to n-P); a fourth window ends the
// slice.  Neighbouring windows touch or overlap (s1 <= P), so the lower bound of x lies in the first window whose
// last element is >= x, or nowhere.  hit[j] bit i = x[i] is present in slice j.
template <int R, int NL>
__device__ __forceinline__ void lift32m(const u32 (&sb)[NL], const u32 (&n)[NL], int l2P, const u32 (&x)[R],
                                        unsigned (&hit)[NL]) {
    const u32 Pw = 1u << l2P;
    u32 a[NL][R];
#pragma unroll
    for (int j = 0; j < NL; ++j) {
        const u32 y = n[j] - Pw;
        const u32 d = (y + 2u) / 3u;
        const u32 s1 = d < y ? d : y, s2 = 2u * d < y ? 2u * d : y;
        const u32 e0 = sb[j] + (Pw - 1u) * 8u;
        const u32 p0 = lds32r(e0), p1 = lds32r(e0 + s1 * 8u), p2 = lds32r(e0 + s2 * 8u);
#pragma unroll
        for (int i = 0; i < R; ++i) {
            u32 st = sb[j];
            if (p0 < x[i]) st = sb[j] + s1 * 8u;
            if (p1 < x[i]) st = sb[j] + s2 * 8u;
            if (p2 < x[i]) st = sb[j] + y * 8u;
            a[j][i] = st;
        }
    }
#define DGX_L32(H)                                                          \
    {                                                                       \
        _Pragma("unroll") for (int j = 0; j < NL; ++j)                      \
        _Pragma("unroll") for (int i = 0; i < R; ++i) {                     \
            const u32 v_ = lds32<((H) - 1) * 8>(a[j][i]);                   \
            if (v_ < x[i]) a[j][i] += (H) * 8;                              \
        }                                                                   \
    }
    switch (l2P) {
        case 15: DGX_L32(16384)
        case 14: DGX_L32(8192)
        case 13: DGX_L32(4096)
        case 12: DGX_L32(2048)
        case 11: DGX_L32(1024)
        case 10: DGX_L32(512)
        case 9: DGX_L32(256)
        case 8: DGX_L32(128)
        case 7: DGX_L32(64)
        case 6: DGX_L32(32)
        case 5: DGX_L32(16)
        case 4: DGX_L32(8)
        case 3: DGX_L32(4)
        case 2: DGX_L32(2)
        case 1: DGX_L32(1)
        default: break;
    }
#undef DGX_L32
#pragma unroll
    for (int j = 0; j < NL; ++j) {
        hit[j] = 0;
#pragma unroll
        for (int i = 0; i < R; ++i) hit[j] |= (lds32r(a[j][i]) == x[i]) ? (1u << i) : 0u;
    }
}

#ifdef DGX_PIPE_PROF
// Wait-time breakdown per warp role (cycles, summed over warps / CTAs); experimental builds only.
__device__ unsigned long long g_pprof[32];
#define PPROF_VARS unsigned long long pp_t = 0, pp_w0 = 0, pp_w1 = 0, pp_w2 = 0; const long long pp_start = clock64();
#define PPROF_T() pp_t = clock64();
#define PPROF_ACC(v) v += clock64() - pp_t;
#define PPROF_PHASE_VARS unsigned long long pp_ph[4] = {0, 0, 0, 0}; long long pp_pt = 0;
#define PPROF_PHASE_T() pp_pt = clock64();
#define PPROF_PHASE(k) { const long long n_ = clock64(); pp_ph[k] += n_ - pp_pt; pp_pt = n_; }
#define PPROF_PHASE_FLUSH() if (lane == 0) { for (int k_ = 0; k_ < 4; ++k_) atomicAdd(&g_pprof[16 + k_], pp_ph[k_]); }
#define PPROF_FLUSH(i) if (lane == 0) { atomicAdd(&g_pprof[i], (unsigned long long)(clock64() - pp_start)); atomicAdd(&g_pprof[i + 1], pp_w0); atomicAdd(&g_pprof[i + 2], pp_w1); atomicAdd(&g_pprof[i + 3], pp_w2); }
#else
#define PPROF_VARS
#define PPROF_T()
#define PPROF_ACC(v)
#define PPROF_FLUSH(i)
#define PPROF_PHASE_VARS
#define PPROF_PHASE_T()
#define PPROF_PHASE(k)
#define PPROF_PHASE_FLUSH()
#endif

template <int VA>
__global__ void __launch_bounds__(P_NT, 2) filter_pipe_kernel(const PParams PP) {
    DGX_GEOM(VA);
    extern __shared__ __align__(128) unsigned char p_smem[];
    const FParams& P = PP.f;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const u32 scap = PP.slice_cap;
    // layout: [PShared | s_work P_TA | out slots P_OS x P_TA | stage0: A (P_TA+2) | slices scap | stage1: ...]
    PShared& S = *reinterpret_cast<PShared*>(p_smem);
    u64* s_work = reinterpret_cast<u64*>(p_smem + ((sizeof(PShared) + 127) & ~size_t(127)));
    u64* s_out = s_work + P_TA;  // P_OS slots of P_TA values
    u64* stage_mem = s_work + (1 + P_OS) * P_TA;
    const size_t stage_words = (size_t)(P_TA + 2) + scap;
    auto s_A = [&](u32 st_) { return stage_mem + (size_t)st_ * stage_words; };
    auto s_SL = [&](u32 st_) { return stage_mem + (size_t)st_ * stage_words + (P_TA + 2); };

    if (tid == 0) {
        for (int s = 0; s < P_ST; ++s) { mbar_init(smem_u32(&S.full[s]), 1); mbar_init(smem_u32(&S.empty[s]), P_CW); }
        for (int s = 0; s < P_OS; ++s) { mbar_init(smem_u32(&S.ofull[s]), P_CW); mbar_init(smem_u32(&S.oempty[s]), 1); }
        for (int r = 0; r < P_RING; ++r) { mbar_init(smem_u32(&S.ready[r]), 1); mbar_init(smem_u32(&S.freed[r]), 1); }
        for (int s = 0; s < P_OS; ++s) { S.os[s].total = 0; S.os[s].arrived = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();


    if (wid == P_CW) {
        // =========================== M: metadata warp ===============================
        // PP.grp (1 .. P_GRP) tiles per iteration, eight lanes each, claimed with ONE atomic so a
        // CTA's tiles stay in look-back order; the ticket for the next iteration is fetched before
        // this iteration's loads, so the chain per group is two global latencies: tile table ->
        // {list descriptors, plan entries}.  Sub-lane u < 8 resolves filter list u of its tile.
        const int h = lane >> 3, u = lane & 7;
        u32 next_base = 0;
        const u32 grp = PP.grp;
        if (lane == 0) next_base = atomicAdd(P.ticket, grp);
        PPROF_VARS
        for (u32 itn = 0;; ++itn) {
            const u32 seq = grp * itn + h;
            const u32 slot = seq % P_RING, use = seq / P_RING;
            const u32 base_ticket = __shfl_sync(0xffffffffu, next_base, 0);
            if (lane == 0) next_base = atomicAdd(P.ticket, grp);  // prefetch (harmless past the end)
            const bool act = (u32)h < grp;  // lane groups beyond grp idle
            PPROF_T()
            if (act && u == 0) mbar_wait_relaxed<DGX_P_SLEEP_MO>(smem_u32(&S.freed[slot]), (use & 1u) ^ 1u);
            __syncwarp();
            PPROF_ACC(pp_w0)
            const u64 tile64 = (u64)base_ticket + h;
            const bool valid = act && tile64 < (u64)P.ntiles;
            const u32 tile = valid ? (u32)tile64 : P_END;
            PTileEntry e;
            e.task = 0; e.list_first = 0; e.k = 0; e.na = 0; e.a0 = 0; e.plan_idx = 0; e.prev = 0; e.has_prev = 0;
            if (valid) e = PP.tiles[tile];
            u64 r0 = 0, r1 = 0, lenj = 0;
            const u64* ptrj = nullptr;
            const u64* A = nullptr;
            if (valid) {
                if (u < P_MAXL && (u32)u + 1 < e.k) {
                    const FList Lj = P.lists[e.list_first + 1 + u];
                    ptrj = Lj.ptr;
                    lenj = flist_len(Lj);
                    const PPlanEntry pe = PP.plan[e.plan_idx + u];
                    r0 = pe.r0; r1 = pe.r1;
                }
                if (u == 0) A = P.lists[e.list_first].ptr;
            }
            PDesc& D = S.ring[slot];
            if (act && u == 0) {
                D.tile = tile; D.task = e.task; D.na = e.na; D.k = e.k; D.list_first = e.list_first;
                D.has_prev = e.has_prev; D.a0 = e.a0; D.prev = e.prev; D.plan_idx = e.plan_idx; D.A = A;
            }
            if (act && u < P_MAXL) { D.ptr[u] = ptrj; D.len[u] = lenj; D.r0[u] = r0; D.r1[u] = r1; }
            __syncwarp();
            if (act && u == 0) mbar_arrive(smem_u32(&S.ready[slot]));
            if (__ballot_sync(0xffffffffu, act && !valid)) break;  // an END descriptor was published
        }
        PPROF_FLUSH(8)
    } else if (wid == P_CW + 1) {
        // =========================== T: TMA warp ====================================
        PPROF_VARS
        for (u32 seq = 0;; ++seq) {
            const u32 slot = seq % P_RING, use = seq / P_RING;
            PPROF_T()
            mbar_wait_relaxed<DGX_P_SLEEP_T>(smem_u32(&S.ready[slot]), use & 1u);
            PPROF_ACC(pp_w0)
            const PDesc& D = S.ring[slot];
            const u32 st = seq % P_ST, suse = seq / P_ST;
            PPROF_T()
            mbar_wait_relaxed<DGX_P_SLEEP_T>(smem_u32(&S.empty[st]), (suse & 1u) ^ 1u);
            PPROF_ACC(pp_w1)
            PStageInfo& G = S.st[st];
            const u32 tile = D.tile;
            if (tile == P_END) {
                if (lane == 0) { G.tile = P_END; mbar_arrive(smem_u32(&S.full[st])); }
                break;
            }
            // layout of the staged slices: lane t owns filter list t
            const u32 km1 = D.k - 1;
            const bool mine = (u32)lane < km1 && lane < P_MAXL;
            u64 n64 = 0;
            const u64* src = nullptr;
            u32 head = 0;
            if (mine) {
                n64 = D.r1[lane] - D.r0[lane];
                src = D.ptr[lane] + D.r0[lane];
                head = (u32)((reinterpret_cast<uintptr_t>(src) >> 3) & 1);
            }
            const u32 words = (mine && n64 <= (u64)scap) ? (u32)((n64 + head + 1) & ~1ull) : 0u;  // 16-byte granules
            u32 incl = words;
#pragma unroll
            for (int dlt = 1; dlt < 8; dlt <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, incl, dlt);
                if (lane >= dlt) incl += v;
            }
            const bool fits = mine && n64 <= (u64)scap && incl <= scap;
            const unsigned fm = __ballot_sync(0xffffffffu, fits);
            u32 nstaged = (u32)(__ffs(~fm) - 1);  // leading run of lists that fit
            if (nstaged > km1) nstaged = km1;
            if (nstaged > P_MAXL) nstaged = P_MAXL;
            const u32 na = D.na;
            const u32 headA = na ? (u32)((reinterpret_cast<uintptr_t>(D.A + D.a0) >> 3) & 1) : 0u;
            const u32 bytesA = na ? (u32)(((na + headA + 1) & ~1u) * 8u) : 0u;
            const u32 my_bytes = ((u32)lane < nstaged) ? words * 8u : 0u;
            u32 tot = my_bytes;
#pragma unroll
            for (int dlt = 16; dlt > 0; dlt >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, dlt);
            tot += bytesA;
            if (lane < P_MAXL) {
                G.ptr[lane] = D.ptr[lane]; G.len[lane] = D.len[lane]; G.r0[lane] = D.r0[lane];
                G.off[lane] = incl - words + head; G.n[lane] = (u32)(n64 < 0xffffffffull ? n64 : 0xffffffffull);
            }
            if (lane == 0) {
                G.tile = tile; G.task = D.task; G.na = na; G.k = D.k; G.list_first = D.list_first;
                G.has_prev = D.has_prev; G.nstaged = nstaged; G.headA = headA;
                G.a0 = D.a0; G.prev = D.prev; G.plan_idx = D.plan_idx; G.A = D.A;
            }
            __syncwarp();
            const u32 bar = smem_u32(&S.full[st]);
            if (lane == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                if (tot) mbar_expect_tx(bar, tot); else mbar_arrive(bar);
                if (bytesA) tma_bulk_g2s(smem_u32(s_A(st)), D.A + D.a0 - headA, bytesA, bar);
            }
            __syncwarp();
            if (my_bytes) tma_bulk_g2s(smem_u32(s_SL(st) + (incl - words)), src - head, my_bytes, bar);
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&S.freed[slot]));  // descriptor consumed
        }
        PPROF_FLUSH(4)
    } else if (wid == P_CW + 2) {
        // =========================== O: output warp =================================
        PPROF_VARS
        for (u32 it = 0;; ++it) {
            const u32 sl = it % P_OS, use = it / P_OS;
            PPROF_T()
            mbar_wait_relaxed<DGX_P_SLEEP_MO>(smem_u32(&S.ofull[sl]), use & 1u);
            PPROF_ACC(pp_w0)
            const POutSlot& O = S.os[sl];
            const u32 tile = O.tile;
            if (tile == P_END) break;
            const u32 q = O.task;
            u32 cw = lane < P_CW ? O.cnt[lane] : 0u;
            u32 incl = cw;
#pragma unroll
            for (int dlt = 1; dlt < 32; dlt <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, incl, dlt);
                if (lane >= dlt) incl += v;
            }
            const u32 total = __shfl_sync(0xffffffffu, incl, 31);
            PPROF_T()
            const u64 base = lookback_exclusive<true, DGX_P_SLEEP_LB>(P.status, tile, (u64)total, lane);
            PPROF_ACC(pp_w1)
            if (lane == 0) {
                if (O.first) P.out_off[q] = base;
                if (tile == P.ntiles - 1) P.out_off[P.ntasks] = base + (u64)total;
            }
            if (base + (u64)total > P.out_cap) {
                if (lane == 0) atomicExch(P.err, 1);
            } else if (total != 0) {
                // a warp's segment holds at most P_WC survivors: P_VA predicated stores per segment,
                // the shuffles of all segments independent of each other
                const u64* data = s_out + (size_t)sl * P_TA;
                u64* dst = P.out + base;
#pragma unroll
                for (int w = 0; w < P_CW; ++w) {
                    const u32 nw = __shfl_sync(0xffffffffu, cw, w);
                    const u32 ow = __shfl_sync(0xffffffffu, incl, w) - nw;
#pragma unroll
                    for (int r = 0; r < P_VA; ++r)
                        if ((u32)(lane + 32 * r) < nw) st_stream(dst + ow + lane + 32 * r, data[P_WC * w + lane + 32 * r]);
                }
            }
            __syncwarp();
            if (lane == 0) {
                S.os[sl].total = 0;
                S.os[sl].arrived = 0;
                mbar_arrive(smem_u32(&S.oempty[sl]));
            }
        }
        PPROF_FLUSH(12)
    } else {
        // =========================== C: consumer warps ==============================
        u64* s_w = s_work + P_WC * wid;
        PPROF_VARS
        PPROF_PHASE_VARS
        for (u32 it = 0;; ++it) {
            const u32 st = it % P_ST, suse = it / P_ST;
            PPROF_T()
            mbar_wait(smem_u32(&S.full[st]), suse & 1u);
            PPROF_ACC(pp_w0)
            PPROF_PHASE_T()
            const PStageInfo& G = S.st[st];
            const u32 tile = G.tile;
            const u32 osl = it % P_OS, ouse = it / P_OS;
            POutSlot& O = S.os[osl];
            if (tile == P_END) {
                mbar_wait(smem_u32(&S.oempty[osl]), (ouse & 1u) ^ 1u);
                if (wid == 0 && lane == 0) O.tile = P_END;
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(&S.ofull[osl]));
                break;
            }
            const u32 na = G.na, k = G.k, q = G.task;
            const u32 tile_first = G.a0 == 0 ? 1u : 0u;
            const u64* cand = s_A(st) + G.headA;
            const u64* sl = s_SL(st);
            PTile X;
            X.cand = cand; X.A = G.A; X.a0 = G.a0; X.prev = G.prev; X.has_prev = G.has_prev != 0;
            X.cidx0 = P_WC * wid + lane; X.op = P.op;

            u64 c[P_VA] = {};
            unsigned alive = 0, dup = 0;
            int rows;
            {
                const int wn = (int)na - P_WC * wid;
                rows = wn <= 0 ? 0 : (wn >= P_WC ? P_VA : (wn + 31) >> 5);
#pragma unroll
                for (int i = 0; i < P_VA; ++i) {
                    const int idx = X.cidx0 + 32 * i;
                    if (idx < (int)na) {
                        c[i] = cand[idx];
                        alive |= 1u << i;
                        const u64 before = idx > 0 ? cand[idx - 1] : X.prev;
                        if ((idx > 0 || X.has_prev) && before == c[i]) dup |= 1u << i;
                    }
                }
            }
            const bool warp_dup = __any_sync(0xffffffffu, dup != 0);  // repeated values: candidates stay in place
            const u32 km1 = (k > 1) ? k - 1 : 0u;
            const u32 nstaged = G.nstaged < km1 ? G.nstaged : km1;

            u32 t = 0;
            PPROF_PHASE(0)
            // ---- fast path: one upper word for the whole tile, no repeated values in this warp's rows,
            //      every filter list staged -> 32-bit searches on the low words (see lift32) ----------
            bool fast = DGX_P_FAST && !warp_dup && nstaged == km1 && na > 0;
            u32 hiword = 0;
            if (fast) {
                const u32 cb = smem_u32(cand);
                hiword = lds32r(cb + 4u);
                fast = hiword == lds32r(cb + (na - 1u) * 8u + 4u);
            }
            if (fast) {
                u32 x[P_VA];
#pragma unroll
                for (int i = 0; i < P_VA; ++i) x[i] = (u32)c[i];
                const u32 slb = smem_u32(sl);
                const bool keep_hits = P.op == 0;
                while (t < km1 && rows > 0) {
#if DGX_P_PAIR2
                    // (only after the first list: a warp that still fills two rows then has lost less than half of its
                    //  candidates, so the second search is rarely wasted; sparse workloads drop to one row and take
                    //  the three-list path below -- measured: always pairing costs C2 6 %, never pairing costs the
                    //  dense variant 24 %)
                    if (rows == 2 && t >= 1 && t + 1 < km1 && G.n[t] != 0 && G.n[t + 1] != 0 &&
                        (G.n[t] > G.n[t + 1] ? G.n[t] : G.n[t + 1]) <= 3u << (31 - __clz(G.n[t] < G.n[t + 1] ? G.n[t] : G.n[t + 1]))) {
                        // ---- two rows against TWO lists at once (four chains; the second list is searched for
                        //      candidates the first may reject -- cheap while most candidates survive) -------------
                        const u32 n2[2] = {G.n[t], G.n[t + 1]};
                        const u32 s2[2] = {slb + G.off[t] * 8u, slb + G.off[t + 1] * 8u};
                        const int l2 = 31 - __clz(n2[0] < n2[1] ? n2[0] : n2[1]);
                        const u32 x2[2] = {x[0], x[1]};
                        unsigned h2[2] = {0, 0};
                        lift32m<2, 2>(s2, n2, l2, x2, h2);
                        alive &= h2[0] & h2[1];   // intersect only: a difference has a single filter list
                        t += 2;
                    } else
#endif
                    if (rows >= 2) {
                        // ---- every row of the warp against ONE list (rows chains) ----------------------
                        const u32 nn[1] = {G.n[t]};
                        unsigned hit[1] = {0};
                        if (nn[0] != 0) {
                            const u32 sbs[1] = {slb + G.off[t] * 8u};
                            const int l2 = 31 - __clz(nn[0]);
                            if (P_VA == 2 || rows == 2) {
                                const u32 x2[2] = {x[0], x[1]};
                                lift32m<2, 1>(sbs, nn, l2, x2, hit);
                            } else {
                                lift32m<P_VA, 1>(sbs, nn, l2, x, hit);
                            }
                        }
                        alive &= keep_hits ? hit[0] : ~hit[0];
                        t += 1;
                    } else {
                        // ---- one row against up to three lists at once (speculative: a candidate that fails the
                        //      first is searched in the others anyway -- the lanes are there, the chains overlap) ----
                        u32 g = km1 - t < 3u ? km1 - t : 3u;
                        u32 nn[3], sbs[3];
                        u32 nmin = 0xffffffffu, nmax = 0;
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            const u32 tj = (u32)j < g ? t + j : t;
                            nn[j] = G.n[tj];
                            sbs[j] = slb + G.off[tj] * 8u;
                            nmin = nn[j] < nmin ? nn[j] : nmin;
                            nmax = nn[j] > nmax ? nn[j] : nmax;
                        }
                        const u32 x1[1] = {x[0]};
                        unsigned ok = 1u;
                        if (nmin == 0) {
                            // an empty slice: nothing survives an intersection; a difference (one list) keeps everything
                            ok = keep_hits ? 0u : 1u;
                            g = keep_hits ? g : 1u;
                        } else {
                            int l2 = 31 - __clz(nmin);
                            if (nmax > 3u << l2) { g = 1; l2 = 31 - __clz(nn[0]); }  // lengths too far apart for one ladder
                            unsigned h3[3] = {0, 0, 0};
                            if (g == 3) {
                                lift32m<1, 3>(sbs, nn, l2, x1, h3);
                                ok = h3[0] & h3[1] & h3[2] & 1u;
                            } else if (g == 2) {
                                const u32 s2[2] = {sbs[0], sbs[1]}, n2[2] = {nn[0], nn[1]};
                                unsigned h2[2] = {0, 0};
                                lift32m<1, 2>(s2, n2, l2, x1, h2);
                                ok = h2[0] & h2[1] & 1u;
                            } else {
                                const u32 s1[1] = {sbs[0]}, n1[1] = {nn[0]};
                                unsigned h1[1] = {0};
                                lift32m<1, 1>(s1, n1, l2, x1, h1);
                                ok = keep_hits ? (h1[0] & 1u) : (~h1[0] & 1u);
                            }
                        }
                        alive &= ok;
                        t += g;
                    }
                    if (t < km1 && rows == 1) {
                        if (!__any_sync(0xffffffffu, alive & 1u)) { rows = 0; alive = 0; }  // nobody left: done with the tile
                    } else if (t < km1) {
                        // re-pack into fewer rows (order preserved)
                        unsigned b[P_VA];
                        int tot = 0;
#pragma unroll
                        for (int i = 0; i < P_VA; ++i) {
                            b[i] = __ballot_sync(0xffffffffu, (i < rows) && ((alive >> i) & 1u));
                            tot += __popc(b[i]);
                        }
                        const int nrows = (tot + 31) >> 5;
                        if (nrows == 0) { rows = 0; alive = 0; }
                        else if (nrows < rows) {
                            u32* s32 = reinterpret_cast<u32*>(s_w);
                            const unsigned lt = (1u << lane) - 1u;
                            int before = 0;
#pragma unroll
                            for (int i = 0; i < P_VA; ++i) {
                                if ((b[i] >> lane) & 1u) s32[before + __popc(b[i] & lt)] = x[i];
                                before += __popc(b[i]);
                            }
                            __syncwarp();
                            alive = 0;
#pragma unroll
                            for (int i = 0; i < P_VA; ++i)
                                if (i < nrows && 32 * i + lane < tot) { x[i] = s32[32 * i + lane]; alive |= 1u << i; }
                            __syncwarp();
                            rows = nrows;
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < P_VA; ++i) c[i] = ((u64)hiword << 32) | (u64)x[i];
                t = km1;
            }
            while (t < km1 && rows > 0) {
                if (t < nstaged) {
                    if (rows >= 2 || t + 1 >= nstaged) {
                        // ---- one staged list, the warp's rows interleaved in pairs ------------
                        const int n = (int)G.n[t];
                        if (n == 0) {
                            if (P.op == 0) { alive = 0; rows = 0; }
                        } else {
                            const u64* sb = sl + G.off[t];
                            const u64* const sbs[2] = {sb, sb};
                            const int ns[2] = {n, n};
#pragma unroll
                            for (int r0 = 0; r0 < P_VA; r0 += 2) {
                                if (r0 < rows) {
                                    const u64 xs[2] = {c[r0], c[r0 + 1]};
                                    int pos[2];
                                    lift_multi<2>(sbs, ns, xs, pos);
#pragma unroll
                                    for (int i = r0; i < r0 + 2; ++i)
                                        if ((alive >> i) & 1u) {
                                            const bool h = phit(X, c[i], i, dup, sb, n, pos[i - r0], G.r0[t], G.ptr[t], G.len[t]);
                                            if ((P.op == 0) != h) alive &= ~(1u << i);
                                        }
                                }
                            }
                        }
                        t += 1;
                    } else {
                        // ---- single row: up to three staged lists interleaved ---------------
                        const u32 nl = (nstaged - t >= 3) ? 3u : 2u;
                        const u64* sbs[3];
                        int ns[3];
                        u64 xs[3];
                        int pos[3];
                        bool empty_list = false;
#pragma unroll
                        for (int j = 0; j < 3; ++j) {
                            const u32 tj = (u32)j < nl ? t + j : t;
                            sbs[j] = sl + G.off[tj];
                            ns[j] = (int)G.n[tj];
                            xs[j] = c[0];
                            if ((u32)j < nl && ns[j] == 0) empty_list = true;
                            if (ns[j] == 0) { ns[j] = 1; sbs[j] = cand; }  // harmless dummy search
                        }
                        const u64* const (&sbr)[3] = sbs;
                        lift_multi<3>(sbr, ns, xs, pos);
                        if (empty_list && P.op == 0) {
                            alive = 0; rows = 0;
                        } else if (alive & 1u) {
#pragma unroll
                            for (int j = 0; j < 3; ++j)
                                if ((u32)j < nl && (alive & 1u) && (int)G.n[t + j] > 0) {
                                    const bool h = phit(X, c[0], 0, dup, sbs[j], (int)G.n[t + j], pos[j], G.r0[t + j],
                                                        G.ptr[t + j], G.len[t + j]);
                                    if ((P.op == 0) != h) alive &= ~1u;
                                }
                        }
                        t += nl;
                    }
                } else {
                    // ---- list not staged: live candidates binary-search it in HBM -----------
                    const FList Lj = P.lists[G.list_first + 1 + t];
                    const u64* __restrict__ B = Lj.ptr;
                    const u64 lenB = flist_len(Lj);
                    const PPlanEntry e = PP.plan[G.plan_idx + t];
                    const u64 sz = e.r1 - e.r0;
#pragma unroll
                    for (int i = 0; i < P_VA; ++i) {
                        if ((alive >> i) & 1u) {
                            const u64 x = c[i];
                            u64 gpos = e.r0 + (sz ? lower_bound_g(B + e.r0, sz, x) : 0);
                            if ((dup >> i) & 1u) gpos += cand_rank(cand, X.cidx0 + 32 * i, x, X.has_prev, X.prev, X.A, X.a0);
                            const bool h = (gpos < lenB) && (ld_probe(B + gpos) == x);
                            if ((P.op == 0) != h) alive &= ~(1u << i);
                        }
                    }
                    t += 1;
                }
                if (t < km1) {
                    if (!warp_dup) pwarp_repack<P_VA>(c, alive, rows, s_w, lane);
                    else if (!__any_sync(0xffffffffu, alive != 0)) rows = 0;
                }
            }
            if (rows == 0) alive = 0;
            PPROF_PHASE(1)

            // ---- this warp is done with the stage: hand it back to T ---------------------------
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&S.empty[st]));

            // ---- survivors -> this warp's segment of the output slot -----------------------------
            PPROF_T()
            mbar_wait_relaxed(smem_u32(&S.oempty[osl]), (ouse & 1u) ^ 1u);
            PPROF_ACC(pp_w1)
            PPROF_PHASE_T()
            {
                u64* od = s_out + (size_t)osl * P_TA + P_WC * wid;
                const unsigned lt = (1u << lane) - 1u;
                int before = 0;
#pragma unroll
                for (int i = 0; i < P_VA; ++i) {
                    const unsigned bo = __ballot_sync(0xffffffffu, (alive >> i) & 1u);
                    if ((bo >> lane) & 1u) od[before + __popc(bo & lt)] = c[i];
                    before += __popc(bo);
                }
                if (lane == 0) {
                    O.cnt[wid] = (u32)before;
                    if (wid == 0) { O.tile = tile; O.task = q; O.first = tile_first; }
                    // The last warp to deliver publishes the tile's aggregate for the look-back
                    // right away: successors never wait for this CTA's output warp to get here.
                    atomicAdd(&O.total, (u32)before);
                    __threadfence_block();
                    if (atomicAdd(&O.arrived, 1u) == P_CW - 1) {
                        const u32 tot = atomicAdd(&O.total, 0u);
                        st_relaxed(P.status + tile, (tile == 0 ? kFlagPrefix : kFlagAgg) | (u64)tot);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&S.ofull[osl]));
            PPROF_PHASE(2)
        }
        PPROF_FLUSH(0)
        PPROF_PHASE_FLUSH()
    }
}

}  // namespace dgx
