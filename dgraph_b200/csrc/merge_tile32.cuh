// merge_tile32.cuh -- the bounds and tile kernels of the single-pass multiway MergeSorted.
//
// The pipeline (samples -> distinct splitters -> per-(boundary, run) bounds -> one CTA per tile -> scan of the tile
// counts -> compaction) is described in merge_multi.cuh.  The two kernels here:
//   mplan2_kernel   bounds, run-major (threads of a warp search neighbouring splitters in the SAME run, so their
//                   probes share sectors), each search confined to the gap between two samples of the run (the
//                   samples are already in HBM/L2: 9 steps instead of 24 over the whole run).
//   mmerge3_kernel  all values of a tile lie in [lo, hi]; when hi - lo fits 32 bits (any realistic uid distribution)
//                   the k slices are loaded as 32-bit offsets from lo and the six levels of pairwise merge-path merges
//                   run on u32 keys: one-instruction compares and selects, half the shared-memory bytes (so a
//                   round holds 7680 slots instead of 4096), T_VT = 15 consecutive slots per thread -- an odd stride,
//                   so the threads of a warp hit different banks without index padding.  About a third of the
//                   instructions of the 64-bit levels per slot.  Tiles whose span does not fit 32 bits use the 64-bit
//                   engine of merge_multi.cuh (mm_levels_tile) in the same kernel.
// An LSD radix sort of the tile (8-bit digits, match.any ranking) and a decoupled look-back straight to the final
// position were built and measured first (profiles/README.md): ~3 warp-instructions per value and pass for the sort,
// and in-order retirement behind the slowest tile for the look-back; both slower than this.
// algo.MergeSorted: algo/uidlist.go:448-542.
#pragma once

#include "merge_multi.cuh"

namespace dgx {

constexpr int T_NT = MM_NT;                 // 512 threads
constexpr int T_VT = 15;                    // slots per thread (odd: conflict-free strided stores)
constexpr int T_C = T_NT * T_VT;            // 7680 slots per round
constexpr u32 T_INF = 0xFFFFFFFFu;          // padding key; real keys are < T_INF
constexpr size_t T_SMEM_32 = (size_t)2 * T_C * sizeof(u32);
constexpr size_t T_SMEM_64 = (size_t)2 * MM_CP * sizeof(u64);
constexpr size_t T_SMEM = T_SMEM_32 > T_SMEM_64 ? T_SMEM_32 : T_SMEM_64;
#ifndef DGX_T_PIECE
#define DGX_T_PIECE 128  // 256 measured slower (1.677 vs 1.642 ms on C5)
#endif
constexpr int T_PIECE = DGX_T_PIECE;         // slots per load piece (T_PIECE / 32 independent loads per lane)
constexpr int T_NCH = T_VT * (T_NT / 32);   // 32-position chunks of a round (de-duplication scan)
static_assert(T_NCH <= 256, "chunk scan handles 8 chunks per lane");
static_assert(MM_K == 64, "six merge levels");

// ---- bounds, run-major: bounds[j * nbs + b] = position of boundary b in run j ---------------------------------
__global__ void __launch_bounds__(256) mplan2_kernel(const MMParams P) {
    const u32 ns = (u32)(*P.nsplit / P.stride);
    const u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 j = (u32)(idx / P.nbs), b = (u32)(idx % P.nbs);
    if (j >= P.k || b > ns + 1) return;
    const u64* p; u64 n;
    mref_resolve(P.runs[j], p, n);
    u64 pos;
    if (b == 0 || n == 0) pos = 0;
    else if (b == ns + 1) pos = n;
    else {
        const u64 S = P.splitters[(u64)b * P.stride - 1];
        // the samples of run j sit at positions q(r) = (r + 1) * n / (s + 1) (msample_kernel): the samples below S
        // and the first one not below S fence the answer in
        const u64* sm = P.samples + P.samp_off[j];
        const u32 s = P.samp_off[j + 1] - P.samp_off[j];
        u32 l = 0, h = s;
        while (l < h) {
            const u32 m = (l + h) >> 1;
            if (ld_probe(sm + m) < S) l = m + 1; else h = m;
        }
        const u64 wlo = l > 0 ? (u64)(((unsigned __int128)l * n) / (s + 1)) + 1 : 0;
        const u64 whi = l < s ? (u64)(((unsigned __int128)(l + 1) * n) / (s + 1)) : n;
        pos = wlo + lower_bound_g(p + wlo, whi - wlo, S);
    }
    P.bounds[(u64)j * P.nbs + b] = pos;
}

__device__ __forceinline__ void t32_st_stream(u32* p, u32 v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ u32 t32_saddr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u32 t32_lds(u32 a) {
    u32 v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}

// One level of pairwise merges on u32 keys.  The 64 run slots of the round (run r = [off0[r], off0[r+1]), every slot a
// multiple of T_VT long, padded with T_INF, unused slots empty) are merged as a complete binary tree: at level L the
// groups of 2^L slots (2i, 2i+1) of src are merged into dst at the same positions, so a thread finds its pair from the
// slot r0 that holds its first position -- no per-level offset table.  A thread produces T_VT consecutive outputs:
// merge-path search, then T_VT serial steps.
__device__ __forceinline__ void t32_merge_level(const u32* __restrict__ src, u32* __restrict__ dst, const int* off0,
                                                int level, int r0, int np, int tid) {
    const int pos = tid * T_VT;
    if (pos >= np) return;
    const int g = 1 << level;
    const int first = (r0 >> (level + 1)) << (level + 1);
    const int a0 = off0[first], a1 = off0[first + g], b1 = off0[first + 2 * g];
    const int na = a1 - a0, nb = b1 - a1;
    const int d = pos - a0;  // diagonal inside the pair
    // 32-bit shared-memory addresses from here on: one register per cursor, ld.shared with no address arithmetic
    const u32 sA = t32_saddr(src + a0), sB = t32_saddr(src + a1), sE = t32_saddr(src + b1);
    int l = d > nb ? d - nb : 0, h = d < na ? d : na;
    const u32 sBd = sB + 4u * (u32)(d - 1);
    while (l < h) {
        const int m = (l + h) >> 1;
        if (t32_lds(sA + 4u * (u32)m) <= t32_lds(sBd - 4u * (u32)m)) l = m + 1; else h = m;
    }
    // Serial steps without divergence: an exhausted side reads as T_INF, which also is the padding value, so "take A"
    // is a plain av <= bv (when both are T_INF everything left is padding and either side will do); the cursors are
    // read only below their run's end (A ends where B starts).
    u32 pa = sA + 4u * (u32)l, pb = sB + 4u * (u32)(d - l);
    u32 av = pa < sB ? t32_lds(pa) : T_INF, bv = pb < sE ? t32_lds(pb) : T_INF;
    u32* o = dst + pos;
#pragma unroll
    for (int s_ = 0; s_ < T_VT; ++s_) {
        const bool takeA = av <= bv;
        o[s_] = takeA ? av : bv;
        const u32 p = (takeA ? pa : pb) + 4u;
        const u32 lim = takeA ? sB : sE;
        u32 nv = T_INF;
        if (p < lim) nv = t32_lds(p);
        pa = takeA ? p : pa;
        pb = takeA ? pb : p;
        av = takeA ? nv : av;
        bv = takeA ? bv : nv;
    }
}

// The 32-bit engine for one tile (same contract as mm_levels_tile): the slices [s_cur[r], s_end[r]) of the k runs are
// merged in rounds of at most T_C slots as offsets from lo, repeats are dropped, the distinct KEYS (v - lo, 4 bytes each)
// are appended to dst -- the compaction adds lo back, so the scratch pass moves half the bytes.
// Every value of the tile must satisfy 0 <= v - lo < T_INF.  Called by all T_NT threads; returns the number written.
__device__ __noinline__ u32 t32_tile(u32* s_k, const u64* const* s_ptr, u64* s_cur, const u64* s_end, int k, u32* dst,
                                     u64 lo) {
    u32* s_x = s_k;
    u32* s_y = s_k + T_C;
    __shared__ int s_off[2][MM_K + 2];
    __shared__ u64 s_tot[2], s_mn[2];
    __shared__ u32 s_inc[2], s_tk[2];
    __shared__ int s_len[MM_K];
    __shared__ int s_coff[MM_K + 1];  // first load piece of every run
    __shared__ u32 s_cinc[2];
    __shared__ unsigned char s_prun[T_C / T_PIECE + MM_K + 4];  // run of every load piece
    __shared__ u64 s_bound;
    __shared__ u32 s_cc[256];
    __shared__ u32 s_rtot;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    u32 produced = 0;
    // A value equal to a round's bound can have more copies waiting in runs that had loaded only part of them, so the
    // last value written is remembered across rounds.
    bool have_last = false;
    u32 lastkey = 0;

    for (;;) {
        // ---- how much of every run enters this round -------------------------------------------
        u64 rem = 0;
        if (tid < k) rem = s_end[tid] - s_cur[tid];
        u64 tot = rem;
        // every run gets a slot padded to a multiple of T_VT; the tile fits when the slots do
        u64 padded = ((rem + T_VT - 1) / T_VT) * T_VT;
        if (wid < 2) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                tot += __shfl_xor_sync(0xffffffffu, tot, d);
                padded += __shfl_xor_sync(0xffffffffu, padded, d);
            }
            if (lane == 0) { s_tot[wid] = tot; s_mn[wid] = padded; }
        }
        __syncthreads();
        const u64 total_rem = s_tot[0] + s_tot[1];
        const bool fits = (s_mn[0] + s_mn[1]) <= (u64)T_C;
        if (total_rem == 0) break;
        __syncthreads();  // s_mn is written again below
        // A tile that does not fit is merged in rounds: every run contributes a share of the chunk proportional to
        // what it has left (at least one value), so the runs' loaded prefixes end at about the same value and most of
        // the chunk is final in this round.
        u64 take = 0, bnd = kU64Max;
        if (tid < k) {
            if (fits) {
                take = rem;
            } else if (rem > 0) {
                const u64 share = (u64)(((unsigned __int128)rem * (u64)(T_C - T_VT * MM_K)) / total_rem);
                take = share < 1 ? 1 : share;
                if (take > rem) take = rem;
                if (take < rem) bnd = ld_probe(s_ptr[tid] + s_cur[tid] + take - 1);
            }
        }
        const u32 slot = (u32)(((take + T_VT - 1) / T_VT) * T_VT);
        // exclusive scan of the slots over the 64 run positions + min of the bounds + sum of takes
        if (wid < 2) {
            const u32 pieces = (slot + (u32)T_PIECE - 1u) / (u32)T_PIECE;
            u32 inc = slot, inc2 = pieces, tsum = (u32)take;
            u64 mn = bnd;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, inc, d);
                const u32 v2 = __shfl_up_sync(0xffffffffu, inc2, d);
                if (lane >= d) { inc += v; inc2 += v2; }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const u64 o = __shfl_xor_sync(0xffffffffu, mn, d);
                mn = o < mn ? o : mn;
                tsum += __shfl_xor_sync(0xffffffffu, tsum, d);
            }
            if (lane == 31) { s_inc[wid] = inc; s_cinc[wid] = inc2; }
            if (lane == 0) { s_mn[wid] = mn; s_tk[wid] = tsum; }
            s_coff[tid] = (int)(inc2 - pieces);
            // exclusive offset inside the warp; the second warp adds the first warp's total below
            s_len[tid] = (int)take;
            s_off[1][tid] = (int)(inc - slot);
        }
        __syncthreads();
        if (tid < MM_K) {
            s_off[0][tid] = s_off[1][tid] + (wid == 1 ? (int)s_inc[0] : 0);
            if (wid == 1) s_coff[tid] += (int)s_cinc[0];
        }
        if (tid == 0) {
            s_coff[MM_K] = (int)(s_cinc[0] + s_cinc[1]);
            s_off[0][MM_K] = (int)(s_inc[0] + s_inc[1]);
            s_off[0][MM_K + 1] = s_off[0][MM_K];
            s_bound = s_mn[0] < s_mn[1] ? s_mn[0] : s_mn[1];
        }
        __syncthreads();
        const int np = s_off[0][MM_K];                 // padded size of the chunk
        const int n = (int)(s_tk[0] + s_tk[1]);        // real values in the chunk
        const u64 bound = s_bound;
        // ---- load the runs' contributions as offsets from lo, pad every slot.  The runs are cut into pieces of T_PIECE
        // slots and the pieces dealt to the warps round-robin: a run that holds a fifth of the tile does not make one
        // warp the straggler of the barrier below.
        const int nitems = s_coff[MM_K];  // <= T_C / T_PIECE + MM_K
        if (tid < nitems) {
            int l = 0, h = MM_K;  // last r with s_coff[r] <= tid (runs without pieces share their successor's offset)
            while (h - l > 1) {
                const int mid = (l + h) >> 1;
                if (s_coff[mid] <= tid) l = mid; else h = mid;
            }
            s_prun[tid] = (unsigned char)l;
        }
        __syncthreads();
        {
            for (int it = wid; it < nitems; it += T_NT / 32) {
                const int l = s_prun[it];
                const int r = l;
                const int o = s_off[0][r], cnt = s_len[r], slot_n = s_off[0][r + 1] - o;
                const u64* src = s_ptr[r] + s_cur[r];
                const int base = (it - s_coff[r]) * T_PIECE + lane;
#pragma unroll
                for (int q = 0; q < T_PIECE / 32; ++q) {
                    const int i = base + q * 32;
                    if (i < slot_n) s_x[o + i] = i < cnt ? (u32)(ld_stream(src + i) - lo) : T_INF;
                }
            }
        }
        __syncthreads();
        // ---- log2(64) levels of pairwise merges, ping-pong between s_x and s_y -------------------
        int r0 = 0;  // slot holding this thread's first position: last r with off0[r] <= pos
        {
            const int pos = tid * T_VT;
            int l = 0, h = MM_K;
            while (h - l > 1) {
                const int mid = (l + h) >> 1;
                if (s_off[0][mid] <= pos) l = mid; else h = mid;
            }
            r0 = l;
        }
        u32* src = s_x;
        u32* out = s_y;
#pragma unroll 1
        for (int level = 0; level < 6; ++level) {
            t32_merge_level(src, out, s_off[0], level, r0, np, tid);
            __syncthreads();
            u32* t = src; src = out; out = t;
        }
        const u32* Z = src;  // n real sorted keys followed by the padding
        // ---- values <= bound are final this round ---------------------------------------------
        int nsafe = n;
        if (!fits) {
            const u32 bd = (u32)(bound - lo);
            int l = 0, h = n;
            while (l < h) {
                const int m = (l + h) >> 1;
                if (Z[m] <= bd) l = m + 1; else h = m;
            }
            nsafe = l;
        }
        // ---- drop repeats; position order is (j, thread): chunk (j, warp) holds 32 consecutive positions -------
        unsigned keepbits = 0;  // bit j: position j * T_NT + tid is a first occurrence
#pragma unroll
        for (int j = 0; j < T_VT; ++j) {
            if (j * T_NT < nsafe) {  // the same for the whole CTA
                const int pos = j * T_NT + tid;
                bool keep = false;
                if (pos < nsafe) {
                    const u32 v = Z[pos];
                    keep = pos == 0 ? (!have_last || v != lastkey) : (Z[pos - 1] != v);
                }
                const unsigned bal = __ballot_sync(0xffffffffu, keep);
                if (keep) keepbits |= 1u << j;
                if (lane == 0) s_cc[j * (T_NT / 32) + wid] = __popc(bal);
            } else if (lane == 0) {
                s_cc[j * (T_NT / 32) + wid] = 0;
            }
        }
        if (nsafe > 0) { lastkey = Z[nsafe - 1]; have_last = true; }
        if (tid >= T_NCH && tid < 256) s_cc[tid] = 0;
        __syncthreads();
        if (wid == 0) {  // exclusive scan of the chunk counts: eight per lane
            u32 c[8], mine = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { c[q] = s_cc[lane * 8 + q]; mine += c[q]; }
            u32 inc = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u32 v = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += v;
            }
            u32 run = inc - mine;
#pragma unroll
            for (int q = 0; q < 8; ++q) { s_cc[lane * 8 + q] = run; run += c[q]; }
            if (lane == 31) s_rtot = inc;
        }
        __syncthreads();
        {
            u32* dstp = dst + produced;
#pragma unroll
            for (int j = 0; j < T_VT; ++j) {
                if (j * T_NT < nsafe) {
                    const bool keep = (keepbits >> j) & 1u;
                    const unsigned bal = __ballot_sync(0xffffffffu, keep);
                    if (keep) t32_st_stream(dstp + s_cc[j * (T_NT / 32) + wid] + __popc(bal & lt), Z[j * T_NT + tid]);
                }
            }
            produced += s_rtot;
        }
        // ---- advance the runs past everything that was final --------------------------------------
        if (tid < k) {
            u64 adv = take;  // this run's contribution
            if (!fits) {
                const u64* srcp = s_ptr[tid] + s_cur[tid];
                u64 l = 0, h = take;  // first loaded value of the run that is > bound
                while (l < h) {
                    const u64 m = l + ((h - l) >> 1);
                    if (ld_probe(srcp + m) <= bound) l = m + 1; else h = m;
                }
                adv = l;
            }
            s_cur[tid] += adv;
        }
        __syncthreads();
        if (fits) break;
    }
    return produced;
}

constexpr u32 kTileWide = 0x80000000u;  // tile_cnt flag: the tile's scratch holds u64 values, not u32 offsets from tile_lo

__global__ void __launch_bounds__(T_NT, 3) mmerge3_kernel(const MMParams P) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ u64 s_cur[MM_K], s_end[MM_K];
    __shared__ const u64* s_ptr[MM_K];
    __shared__ u64 s_r[2][4];

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const u32 b = blockIdx.x;
    const u32 ns = (u32)(*P.nsplit / P.stride);
    if (b > ns) return;
    const int k = (int)P.k;

    // ---- the tile's slice of every run; input offset, size, smallest and largest value ---------------------
    // An interior tile holds the values in [S(b), S(b+1)) (S(b) = splitter of boundary b), which bounds its span without
    // touching the runs; the first and the last tile read their runs' end values.
    const bool interior = b >= 1 && b < ns;
    u64 lo = 0, hi = 0;
    bool exact = !interior;  // read the runs' end values (also when the splitters are too far apart for 32-bit keys
    if (interior) {          // although the values between them may not be)
        lo = P.splitters[(u64)b * P.stride - 1];
        hi = P.splitters[(u64)(b + 1) * P.stride - 1] - 1;  // splitters are distinct and ascending: hi >= lo
        exact = hi - lo >= (u64)T_INF;
    }
    {
        u64 c = 0, len = 0, vmin = kU64Max, vmax = 0;
        if (tid < k) {
            const u64* p; u64 n;
            mref_resolve(P.runs[tid], p, n);
            c = P.bounds[(u64)tid * P.nbs + b];
            const u64 e = P.bounds[(u64)tid * P.nbs + b + 1];
            s_ptr[tid] = p; s_cur[tid] = c; s_end[tid] = e;
            len = e - c;
            if (len && exact) { vmin = ld_probe(p + c); vmax = ld_probe(p + e - 1); }
        }
        if (wid < 2) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                c += __shfl_xor_sync(0xffffffffu, c, d);
                len += __shfl_xor_sync(0xffffffffu, len, d);
                const u64 a = __shfl_xor_sync(0xffffffffu, vmin, d);
                const u64 z = __shfl_xor_sync(0xffffffffu, vmax, d);
                vmin = a < vmin ? a : vmin;
                vmax = z > vmax ? z : vmax;
            }
            if (lane == 0) { s_r[wid][0] = c; s_r[wid][1] = len; s_r[wid][2] = vmin; s_r[wid][3] = vmax; }
        }
    }
    __syncthreads();
    const u64 inbase = s_r[0][0] + s_r[1][0];
    const u64 total = s_r[0][1] + s_r[1][1];
    if (exact) {
        lo = s_r[0][2] < s_r[1][2] ? s_r[0][2] : s_r[1][2];
        hi = s_r[0][3] > s_r[1][3] ? s_r[0][3] : s_r[1][3];
    }

    // Pull the slices of the tile this SM slot will most likely run next (P.ahead tiles on) into L2 while this one is
    // merged: its loads then pay an L2 hit instead of a DRAM round trip.
    if (P.ahead && tid < k && b + P.ahead <= ns) {
        const u64 c2 = P.bounds[(u64)tid * P.nbs + b + P.ahead], e2 = P.bounds[(u64)tid * P.nbs + b + P.ahead + 1];
        const u64* q = s_ptr[tid];
        for (u64 i = c2 & ~(u64)15; i < e2; i += 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(q + i));
    }

    // Equal values always fall into the same tile (every run is cut at lower_bound of the same splitter), so a tile
    // never has to look at its predecessor's last value.
    u32 produced = 0;
    const bool wide = hi - lo >= (u64)T_INF;
    if (total != 0) {
        if (!wide) produced = t32_tile((u32*)s_raw, s_ptr, s_cur, s_end, k, (u32*)(P.scratch + inbase), lo);
        else produced = mm_levels_tile((u64*)s_raw, s_ptr, s_cur, s_end, k, P.scratch + inbase);
    }
    if (tid == 0) {
        P.tile_in[b] = inbase;
        P.tile_lo[b] = lo;
        P.tile_cnt[b] = produced | (wide ? kTileWide : 0u);
    }
}

}  // namespace dgx
