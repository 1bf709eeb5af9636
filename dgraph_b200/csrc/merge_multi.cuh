// merge_multi.cuh -- single-pass multiway MergeSorted (k <= 64 runs) for sm_100a: shared pieces.
//
// algo.MergeSorted (algo/uidlist.go:448-542) pops a k-way heap and drops values equal
// to the last one written: a sorted union with global de-duplication.  A pairwise
// merge tree moves the data ceil(log2 k) times through HBM; here every input value is
// read once:
//   msample_kernel   evenly spaced samples of every run (count proportional to its length)
//   (merge tree)     the k sample runs are themselves sorted, so the existing pairwise
//                    merge tree (merge_kernel, with de-duplication) turns them into the
//                    sorted distinct splitters; splitters b-1 .. b bound tile b.
//   mplan2_kernel    position of every splitter in every run (merge_tile32.cuh)
//   mmerge3_kernel   one CTA per tile merges the tile's slices of the k runs, drops repeats
//                    and writes the result to a scratch buffer at the tile's INPUT offset
//                    (output <= input, so regions never overlap) (merge_tile32.cuh)
//   mscan_kernel     exclusive scan of the tile counts (one CTA)
//   mcompact_kernel  moves every tile's output to its final, compact position.
// This file holds the 64-bit tile engine (mm_levels_tile), which mmerge3_kernel runs for
// tiles whose value span does not fit 32 bits.  A tile larger than the shared-memory chunk
// is processed in rounds: every run contributes a quota, only values <= the smallest "last
// loaded value of a run that has more" are final in that round (classic block-wise k-way
// merge), so no distribution of the input can overflow shared memory.
#pragma once

#include "common.cuh"
#include "merge_kernel.cuh"

namespace dgx {

constexpr int MM_K = 64;          // maximum fan-in
constexpr int MM_NT = 512;        // threads per merge CTA
constexpr int MM_C = 4096;        // values merged in shared memory at once
constexpr int MM_VT = MM_C / MM_NT;
// Tile buffers are indexed through mm_pad(): one spare slot per 16 values.  A thread owns MM_VT = 8
// consecutive outputs, so unpadded 8-byte accesses of a warp sit 16 banks apart (a 16-way conflict on
// the stores, ~8-way on the data-dependent reads); the padding brings both to the 2-way minimum of
// 64-bit accesses.
__device__ __forceinline__ int mm_pad(int i) { return i + (i >> 4); }
constexpr int MM_CP = MM_C + MM_C / 16 + 2;  // padded buffer length

struct MMParams {
    const MRef* runs;       // k run references (plain arrays or CSR slices of a previous level)
    u32 k;
    const u32* samp_off;    // k + 1: first sample index of every run
    u32 nsamp;
    u64* samples;           // nsamp
    u64* splitters;         // <= nsamp
    const u64* nsplit;      // device word: number of distinct sample values
    u32 stride;             // every stride-th distinct sample is a splitter (evens out tile sizes)
    u64* bounds;            // k * nbs, run-major: bounds[j * nbs + b] = position of boundary b in run j
    u64* tile_in;           // nsamp + 1: input offset of every tile (= scratch offset)
    u32* tile_cnt;          // nsamp + 1: values the tile produced
    u64* tile_out;          // nsamp + 2: exclusive scan of tile_cnt
    u64* scratch;           // sum of run lengths
    u64* out;
    u64 out_cap;
    u64* out_len;
    int* err;
    u32 nbs;                // boundaries per run in the bounds table
    u32 ahead;              // prefetch the tile this many tiles on into L2 (0 = off)
    u64* tile_lo;           // nsamp + 2: base of a tile's 32-bit scratch keys
};

// ---- samples ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) msample_kernel(const MMParams P) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.nsamp) return;
    u32 lo = 0, hi = P.k;  // run whose sample range holds i
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (P.samp_off[mid] <= i) lo = mid; else hi = mid;
    }
    const u64* p; u64 n;
    mref_resolve(P.runs[lo], p, n);
    const u32 s = P.samp_off[lo + 1] - P.samp_off[lo];
    const u32 r = i - P.samp_off[lo];
    u64 v = kU64Max;  // an empty (fully de-duplicated) run contributes "+inf" samples
    if (n > 0) v = ld_probe(p + (u64)(((unsigned __int128)(r + 1) * n) / (s + 1)));
    P.samples[i] = v;
}

// ---- the merge -----------------------------------------------------------------------------
// One level of pairwise merges over `nruns` sorted runs laid out back to back in `src`
// (run r = [off[r], off[r+1])): runs (2i, 2i+1) are merged into dst at the same positions.
// Every run occupies a slot whose size is a multiple of MM_VT (padded with +inf, which sorts
// to the end of every merged run), so a thread's MM_VT outputs never straddle two pairs and
// every thread runs the same instruction sequence: pair lookup, merge-path search, MM_VT steps.
__device__ __forceinline__ void mm_merge_level(const u64* src, u64* dst, const int* off, int nruns, int n, int tid) {
    const int pos = tid * MM_VT;
    if (pos >= n) return;
    int lo = 0, hi = (nruns + 1) >> 1;  // pair that holds `pos`: last pair pi with off[2*pi] <= pos
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[2 * mid] <= pos) lo = mid; else hi = mid;
    }
    const int a0 = off[2 * lo];
    const int a1 = (2 * lo + 1 <= nruns) ? off[2 * lo + 1] : a0;
    const int b1 = (2 * lo + 2 <= nruns) ? off[2 * lo + 2] : a1;
    const int na = a1 - a0, nb = b1 - a1;
    const int d = pos - a0;  // diagonal inside the pair
#define MM_A(i) src[mm_pad(a0 + (i))]
#define MM_B(i) src[mm_pad(a1 + (i))]
    int l = d > nb ? d - nb : 0, h = d < na ? d : na;
    while (l < h) {
        const int m = (l + h) >> 1;
        if (MM_A(m) <= MM_B(d - 1 - m)) l = m + 1; else h = m;
    }
    int ai = l, bi = d - l;
    u64 av = ai < na ? MM_A(ai) : kU64Max, bv = bi < nb ? MM_B(bi) : kU64Max;
#pragma unroll
    for (int s_ = 0; s_ < MM_VT; ++s_) {
        const bool takeA = (bi >= nb) || (ai < na && av <= bv);
        dst[mm_pad(pos + s_)] = takeA ? av : bv;
        if (takeA) { ++ai; av = ai < na ? MM_A(ai) : kU64Max; }
        else { ++bi; bv = bi < nb ? MM_B(bi) : kU64Max; }
    }
#undef MM_A
#undef MM_B
}

// The levels engine for ONE tile: the slices [s_cur[r], s_end[r]) of the k runs s_ptr[r] are merged in rounds of at
// most MM_C values (two ping-pong buffers of MM_CP values in s_mm), values equal to their predecessor are dropped and
// the rest is appended to dst.  Called by all MM_NT threads of the CTA; returns the number of values written.
__device__ __noinline__ u32 mm_levels_tile(u64* s_mm, const u64* const* s_ptr, u64* s_cur, const u64* s_end, int k,
                                           u64* dst) {
    u64* s_x = s_mm;
    u64* s_y = s_mm + MM_CP;
    __shared__ int s_off[2][MM_K + 2];
    __shared__ u64 s_tot[2], s_inc[2], s_mn[2], s_pad[2], s_tk[2];
    __shared__ int s_len[MM_K];
    __shared__ u64 s_bound;
    __shared__ u32 s_scan[MM_NT / 32 + 1];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    u32 produced = 0;
    // A value equal to a round's bound can have more copies waiting in runs that had loaded only part of them, so the
    // last value written is remembered across rounds.
    bool have_last = false;
    u64 last = 0;

    for (;;) {
        // ---- how much of every run enters this round -------------------------------------------
        u64 rem = 0;
        if (tid < k) rem = s_end[tid] - s_cur[tid];
        u64 tot = rem;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, d);
        if (lane == 0 && wid < 2) s_tot[wid] = tot;
        __syncthreads();
        const u64 total_rem = s_tot[0] + s_tot[1];
        if (total_rem == 0) break;
        // every run gets a slot padded to a multiple of MM_VT; the tile fits when the slots do
        u64 padded = tid < k ? ((rem + MM_VT - 1) & ~(u64)(MM_VT - 1)) : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) padded += __shfl_xor_sync(0xffffffffu, padded, d);
        if (lane == 0 && wid < 2) s_pad[wid] = padded;
        __syncthreads();
        const bool fits = (s_pad[0] + s_pad[1]) <= (u64)MM_C;
        // A tile that does not fit is merged in rounds: every run contributes a share of the
        // chunk proportional to what it has left (at least one value), so the runs' loaded
        // prefixes end at about the same value and most of the chunk is final in this round.
        u64 take = 0, bnd = kU64Max;
        if (tid < k) {
            if (fits) {
                take = rem;
            } else if (rem > 0) {
                const u64 share = (u64)(((unsigned __int128)rem * (u64)(MM_C - MM_VT * MM_K)) / total_rem);
                take = share < 1 ? 1 : share;
                if (take > rem) take = rem;
                if (take < rem) bnd = ld_probe(s_ptr[tid] + s_cur[tid] + take - 1);
            }
        }
        const u64 slot = (take + MM_VT - 1) & ~(u64)(MM_VT - 1);
        // exclusive scan of the slots over the 64 run positions + min of the bounds + sum of takes
        {
            u64 inc = slot, mn = bnd, tsum = take;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const u64 v = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += v;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const u64 o = __shfl_xor_sync(0xffffffffu, mn, d);
                mn = o < mn ? o : mn;
                tsum += __shfl_xor_sync(0xffffffffu, tsum, d);
            }
            if (wid < 2) {
                if (lane == 31) s_inc[wid] = inc;
                if (lane == 0) { s_mn[wid] = mn; s_tk[wid] = tsum; }
            }
            __syncthreads();
            if (tid < MM_K) {
                const u64 basew = wid == 1 ? s_inc[0] : 0;
                s_off[0][tid] = (int)(basew + inc - slot);
                s_len[tid] = (int)take;
            }
            if (tid == 0) {
                s_off[0][MM_K] = (int)(s_inc[0] + s_inc[1]);
                s_off[0][MM_K + 1] = s_off[0][MM_K];
                s_bound = s_mn[0] < s_mn[1] ? s_mn[0] : s_mn[1];
            }
            __syncthreads();
        }
        const int np = s_off[0][MM_K];                 // padded size of the chunk
        const int n = (int)(s_tk[0] + s_tk[1]);        // real values in the chunk
        const u64 bound = s_bound;
        // ---- load the runs' contributions, pad every slot with +inf (warp w: runs w, w+8, ...) ------
        for (int r = wid; r < k; r += MM_NT / 32) {
            const int o = s_off[0][r], cnt = s_len[r], slot_n = s_off[0][r + 1] - o;
            const u64* src = s_ptr[r] + s_cur[r];
            for (int i = lane; i < slot_n; i += 32) s_x[mm_pad(o + i)] = i < cnt ? ld_stream(src + i) : kU64Max;
        }
        for (int r = k + tid; r <= MM_K; r += MM_NT) s_off[0][r] = np;  // unused slots are empty runs
        __syncthreads();
        // ---- log2(64) levels of pairwise merges, ping-pong between s_x and s_y -------------------
        u64* src = s_x;
        u64* out = s_y;
        int cur = 0;
        for (int nruns = MM_K; nruns > 1; nruns = (nruns + 1) >> 1) {
            mm_merge_level(src, out, s_off[cur], nruns, np, tid);
            const int nn = (nruns + 1) >> 1;
            for (int r = tid; r <= nn; r += MM_NT) {
                const int q = 2 * r;
                s_off[cur ^ 1][r] = q <= nruns ? s_off[cur][q] : np;
            }
            if (tid == 0) s_off[cur ^ 1][nn + 1] = np;
            __syncthreads();
            u64* t = src; src = out; out = t;
            cur ^= 1;
        }
        const u64* Z = src;  // n real sorted values followed by the +inf padding
        // ---- values <= bound are final this round ---------------------------------------------
        int nsafe = n;
        if (!fits) {
            int l = 0, h = n;
            while (l < h) {
                const int m = (l + h) >> 1;
                if (Z[mm_pad(m)] <= bound) l = m + 1; else h = m;
            }
            nsafe = l;
        }
        // ---- drop repeats, append to the tile's scratch region -----------------------------------
        {
            const int i0 = tid * MM_VT;
            u64 vals[MM_VT];
            unsigned keep = 0;
            u64 prevv = last;
            bool havep = have_last;
            if (i0 > 0 && i0 <= nsafe) { prevv = Z[mm_pad(i0 - 1)]; havep = true; }
#pragma unroll
            for (int j = 0; j < MM_VT; ++j) {
                if (i0 + j < nsafe) {
                    const u64 v = Z[mm_pad(i0 + j)];
                    vals[j] = v;
                    if (!havep || v != prevv) keep |= 1u << j;
                    prevv = v;
                    havep = true;
                }
            }
            u32 tot_keep;
            u32 off = block_exclusive_scan<MM_NT>(__popc(keep), s_scan, &tot_keep);
#pragma unroll
            for (int j = 0; j < MM_VT; ++j)
                if ((keep >> j) & 1u) st_stream(dst + produced + off++, vals[j]);
            produced += tot_keep;
        }
        if (nsafe > 0) { last = Z[mm_pad(nsafe - 1)]; have_last = true; }
        // ---- advance the runs past everything that was final --------------------------------------
        if (tid < k) {
            const u64 tk = take;  // this run's contribution
            u64 adv = tk;
            if (!fits) {
                const u64* srcp = s_ptr[tid] + s_cur[tid];
                u64 l = 0, h = tk;  // first loaded value of the run that is > bound
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

// ---- scan of the tile counts (one CTA) --------------------------------------------------------
__global__ void __launch_bounds__(1024) mscan_kernel(const MMParams P) {
    __shared__ u32 s_warp[1024 / 32 + 1];
    const u32 ntiles = (u32)(*P.nsplit / P.stride) + 1;
    u64 base = 0;
    for (u32 start = 0; start < ntiles; start += 1024) {
        const u32 i = start + threadIdx.x;
        const u32 v = i < ntiles ? (P.tile_cnt[i] & 0x7fffffffu) : 0u;
        u32 total;
        const u32 off = block_exclusive_scan<1024>(v, s_warp, &total);
        if (i < ntiles) P.tile_out[i] = base + off;
        base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        P.tile_out[ntiles] = base;
        *P.out_len = base;
        if (base > P.out_cap) atomicExch(P.err, 1);
    }
}

// ---- compaction: scratch (tile-local offsets) -> out (final offsets) ------------------------------
__global__ void __launch_bounds__(256) mcompact_kernel(const MMParams P) {
    const u32 ntiles = (u32)(*P.nsplit / P.stride) + 1;
    const u32 b = blockIdx.x;
    if (b >= ntiles) return;
    const u64 o = P.tile_out[b];
    const u32 cnt = P.tile_cnt[b] & 0x7fffffffu;
    if (o + cnt > P.out_cap) return;  // error already flagged by mscan_kernel
    u64* dst = P.out + o;
    if (P.tile_cnt[b] & 0x80000000u) {  // u64 values
        const u64* src = P.scratch + P.tile_in[b];
        for (u32 i = threadIdx.x; i < cnt; i += 256) st_stream(dst + i, ld_stream(src + i));
    } else {                            // 32-bit offsets from tile_lo (merge_tile32.cuh)
        const u32* src = (const u32*)(P.scratch + P.tile_in[b]);
        const u64 lo = P.tile_lo[b];
        for (u32 i = threadIdx.x; i < cnt; i += 256) st_stream(dst + i, lo + __ldg(src + i));
    }
}

}  // namespace dgx
