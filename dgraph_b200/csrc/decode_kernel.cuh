// decode_kernel.cuh -- group-varint UidPack decode for sm_100a.
//
// codec.Decode / Decoder.UnpackBlock (codec/codec.go:154-200, 444-452): block b
// yields Base, then running sums of its group-varint u32 deltas, truncated to
// NumUids.  A group is 1 tag byte + 4 little-endian values of 1..4 bytes
// (go-groupvarint; value j's length-1 in tag bits [2j+1:2j]).
//
// Mapping: a warp owns a run of consecutive blocks and streams it in batches of
// up to 32 blocks.  Per batch: (1) ONE TMA bulk copy (cp.async.bulk + mbarrier)
// brings the batch's contiguous delta bytes into the warp's shared-memory
// window; (2) lane i walks block i's tag bytes (the only serial dependence:
// group g+1 starts BytesUsed[tag_g] after group g) and records group offsets;
// (3) all lanes decode a block's groups in parallel -- unaligned 16-byte read,
// four extractions, warp prefix sum of deltas (64-bit, `last + uint64(delta)` as in
// codec.go:191-196) -- into a staging row that is written out as coalesced 16-byte stores.
#pragma once

#include "common.cuh"

namespace dgx {

constexpr int D_WARPS = 4;                  // warps per CTA
constexpr int D_NT = D_WARPS * 32;
constexpr int D_BPW = 64;                   // blocks owned by one warp
constexpr int D_WB = 4096;                  // payload window per warp (bytes)
constexpr int D_MAXG = 64;                  // groups per block at BlockSize 256
constexpr int D_TSTRIDE = 33;               // group-offset table row stride (u16)
constexpr int D_STAGE = 260;                // staging row (u64)

struct DPack {
    u64 nblocks;
    const u64* base;       // nblocks
    const u32* num;        // nblocks
    const u64* delta_off;  // nblocks + 1
    const unsigned char* deltas;  // 16-byte aligned, >= 32 bytes of slack after the end
    const u64* uid_off;    // nblocks + 1: exclusive prefix of num
    u32 max_num;           // largest NumUids of any block
};
struct DSeek {            // written by decode_seek_kernel
    u64 first_block;
    u64 skip;             // uids (in pack order) before the first emitted one
    u64 out_len;
};

__device__ __forceinline__ u32 gv_bytes_used(u32 t) {
    return 5u + (t & 3u) + ((t >> 2) & 3u) + ((t >> 4) & 3u) + (t >> 6);
}

// Decoder.Seek(seek, SeekStart), codec/codec.go:279-337, restated for one thread.
__global__ void decode_seek_kernel(const DPack pk, u64 seek, DSeek* out, u64* out_len_word, u64 out_cap, int* err) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    u64 first = 0, trim = 0;
    const u64 nb = pk.nblocks;
    if (nb > 0 && seek != 0) {
        u64 idx = lower_bound_g(pk.base, nb, seek);  // first block with Base >= seek
        if (idx == 0) {
            first = 0;
        } else if (idx < nb && pk.base[idx] == seek) {
            first = idx;
        } else {
            const u64 b = idx - 1;  // unpack the previous block, count uids < seek
            const u32 num = pk.num[b];
            const unsigned char* p = pk.deltas + pk.delta_off[b];
            u64 last = pk.base[b];
            u32 produced = 1, below = last < seek ? 1u : 0u;
            while (produced < num) {
                const u32 tag = p[0];
                const unsigned char* d = p + 1;
                for (int j = 0; j < 4 && produced < num; ++j) {
                    const u32 l = ((tag >> (2 * j)) & 3u) + 1u;
                    u32 v = 0;
                    for (u32 k = 0; k < l; ++k) v |= (u32)d[k] << (8 * k);
                    d += l;
                    last += v;
                    ++produced;
                    if (last < seek) ++below;
                }
                p += gv_bytes_used(tag);
            }
            if (below < num) { first = b; trim = below; }
            else { first = idx; }  // Next(): nothing >= seek in that block
        }
    }
    DSeek s;
    s.first_block = first;
    const u64 total = nb ? pk.uid_off[nb] : 0;
    s.skip = (first < nb ? pk.uid_off[first] : total) + trim;
    s.out_len = total - s.skip;
    *out = s;
    *out_len_word = s.out_len;
    if (s.out_len > out_cap) atomicExch(err, 1);
}

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u32 bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(u32 dst, const void* src, u32 bytes, u32 bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(u32 bar, u32 parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}

// Same wait for the pipeline's helper warps: the try_wait carries a suspend-time hint and a miss
// backs off with nanosleep, so a waiting warp does not compete with working warps for issue slots.
template <unsigned kSleepNs = 128>
__device__ __forceinline__ void mbar_wait_relaxed(u32 bar, u32 parity) {
    u32 done = 0;
    while (true) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(bar), "r"(parity), "r"(2000u) : "memory");
        if (done) break;
        __nanosleep(kSleepNs);
    }
}

struct __align__(128) DWarpSmem {
    unsigned char payload[D_WB + 64];
    unsigned short goff[D_MAXG * D_TSTRIDE + 2];
    u64 stage[D_STAGE];
    u64 mbar;
};

// One warp decodes blocks [first_block + gw*D_BPW, +D_BPW) of `pk` into out[uid_off - skip ...].
__device__ __forceinline__ void decode_warp_run(const DPack& pk, u64 first_block, u64 skip, u64* __restrict__ out,
                                                u64 gw, DWarpSmem& S, int lane) {
    u64 b = first_block + gw * D_BPW;
    const u64 bend = (b + D_BPW < pk.nblocks) ? b + D_BPW : pk.nblocks;
    if (b >= bend) return;  // whole warp

    const u32 bar = smem_u32(&S.mbar);
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    u32 parity = 0;

    while (b < bend) {
        // ---- batch geometry ----------------------------------------------------
        const u64 bi = b + lane;
        const bool in = bi < bend;
        const u64 doff = in ? pk.delta_off[bi] : 0;
        const u64 dnext = in ? pk.delta_off[bi + 1] : 0;
        const u64 win0 = __shfl_sync(0xffffffffu, doff, 0) & ~15ull;  // 16-byte aligned window start
        const bool fits = in && (dnext - win0 <= (u64)D_WB);
        const unsigned fm = __ballot_sync(0xffffffffu, fits);
        // leading run of blocks that fit (at least one: a block is <= 1088 B at BlockSize 256)
        int nb = __ffs(~fm) - 1;
        if (fm == 0xffffffffu) nb = 32;
        if (nb == 0) nb = 1;  // oversize block (BlockSize > 256*7): handled by the slow path below
        const u64 wend = __shfl_sync(0xffffffffu, dnext, nb - 1);
        const u32 num = in ? pk.num[bi] : 0;
        const u64 base = in ? pk.base[bi] : 0;
        const u64 uoff = in ? pk.uid_off[bi] : 0;
        const u32 ngroups = num > 1 ? (num + 2) / 4 : 0;  // ceil((num-1)/4) groups carry data

        const bool oversize = (wend - win0 > (u64)D_WB) || (num > 256u && lane < nb);
        if (__any_sync(0xffffffffu, oversize)) {
            // Generic slow path (BlockSize > 256 packs): lane-serial decode straight from
            // global memory, one block per lane.  Never taken at the reference's BlockSize 256.
            if (lane < nb && in) {
                const unsigned char* p = pk.deltas + doff;
                u64 last = base;
                u64 gi = uoff;
                if (gi >= skip) st_stream(out + (gi - skip), last);
                u32 produced = 1;
                while (produced < num) {
                    const u32 tag = p[0];
                    const unsigned char* d = p + 1;
                    for (int j = 0; j < 4 && produced < num; ++j) {
                        const u32 l = ((tag >> (2 * j)) & 3u) + 1u;
                        u32 v = 0;
                        for (u32 k = 0; k < l; ++k) v |= (u32)d[k] << (8 * k);
                        d += l;
                        last += v;
                        gi = uoff + produced;
                        if (gi >= skip) st_stream(out + (gi - skip), last);
                        ++produced;
                    }
                    p += gv_bytes_used(tag);
                }
            }
            b += nb;
            continue;
        }

        // ---- (1) TMA bulk copy of the batch's delta bytes ------------------------
        const u32 bytes = (u32)(((wend - win0) + 15ull) & ~15ull);
        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar, bytes);
            tma_bulk_g2s(smem_u32(S.payload), pk.deltas + win0, bytes, bar);
        }
        mbar_wait(bar, parity);
        parity ^= 1u;

        // ---- (2) tag walk: lane i records the byte offset of every group of block i
        if (lane < nb) {
            // a corrupt tag may claim more bytes than the block holds: the walk stops at the block's
            // end (the reference zero-pads a short tail, codec.go:176-188; here the next block's
            // bytes are read instead -- garbage in, garbage out, but never outside the window)
            u32 off = (u32)(doff - win0);
            const u32 off_end = (u32)(dnext - win0);
            for (u32 g = 0; g < ngroups; ++g) {
                S.goff[g * D_TSTRIDE + lane] = (unsigned short)off;
                off += gv_bytes_used(S.payload[off]);
                off = off < off_end ? off : off_end;
            }
        }
        __syncwarp();

        // ---- (3) cooperative decode, block by block --------------------------------
        const u32* pl32 = reinterpret_cast<const u32*>(S.payload);
        for (int i = 0; i < nb; ++i) {
            const u32 n_i = __shfl_sync(0xffffffffu, num, i);
            const u64 base_i = __shfl_sync(0xffffffffu, base, i);
            const u64 uoff_i = __shfl_sync(0xffffffffu, uoff, i);
            const u32 ng_i = __shfl_sync(0xffffffffu, ngroups, i);
            if (lane == 0) S.stage[0] = base_i;
            u64 carry = 0;
            for (u32 g0 = 0; g0 < ng_i; g0 += 32) {
                const u32 g = g0 + lane;
                u32 d0 = 0, d1 = 0, d2 = 0, d3 = 0;
                if (g < ng_i) {
                    const u32 off = S.goff[g * D_TSTRIDE + i];
                    const u32 tag = S.payload[off];
                    const u32 a = off + 1;
                    const u32 wb = a >> 2, sh = (a & 3u) * 8u;
                    const u32 w0 = pl32[wb], w1 = pl32[wb + 1], w2 = pl32[wb + 2], w3 = pl32[wb + 3], w4 = pl32[wb + 4];
                    const u32 D0 = __funnelshift_r(w0, w1, sh), D1 = __funnelshift_r(w1, w2, sh);
                    const u32 D2 = __funnelshift_r(w2, w3, sh), D3 = __funnelshift_r(w3, w4, sh);
                    const u32 l0 = (tag & 3u) + 1u, l1 = ((tag >> 2) & 3u) + 1u;
                    const u32 l2 = ((tag >> 4) & 3u) + 1u, l3 = (tag >> 6) + 1u;
                    auto extract = [&](u32 s, u32 l) -> u32 {
                        const u32 wi = s >> 2, sh2 = (s & 3u) * 8u;
                        const u32 lo = wi == 0 ? D0 : (wi == 1 ? D1 : (wi == 2 ? D2 : D3));
                        const u32 hi = wi == 0 ? D1 : (wi == 1 ? D2 : (wi == 2 ? D3 : 0u));
                        return __funnelshift_r(lo, hi, sh2) & (0xffffffffu >> (32u - 8u * l));
                    };
                    d0 = extract(0, l0);
                    d1 = extract(l0, l1);
                    d2 = extract(l0 + l1, l2);
                    d3 = extract(l0 + l1 + l2, l3);
                }
                // running sums are 64-bit like the reference's `last + uint64(delta)` (codec.go:191-196):
                // packs produced by the Encoder never carry more than 2^32 per block, hand-built ones may
                const u64 p1 = d0, p2 = p1 + d1, p3 = p2 + d2, p4 = p3 + d3;
                u64 inc = p4;
#pragma unroll
                for (int dlt = 1; dlt < 32; dlt <<= 1) {
                    u64 t = __shfl_up_sync(0xffffffffu, inc, dlt);
                    if (lane >= dlt) inc += t;
                }
                const u64 ex = base_i + carry + inc - p4;
                if (g < ng_i) {
                    const u32 idx = 1u + 4u * g;  // uid index of this group's first value
                    S.stage[idx] = ex + p1;
                    S.stage[idx + 1] = ex + p2;
                    S.stage[idx + 2] = ex + p3;
                    S.stage[idx + 3] = ex + p4;
                }
                carry += __shfl_sync(0xffffffffu, inc, 31);
            }
            __syncwarp();
            // coalesced write-out of uids [e0, n_i) of the block
            const u64 e0 = skip > uoff_i ? skip - uoff_i : 0;  // trimmed head (first block only)
            if (e0 < (u64)n_i) {
                u64* dst = out + (uoff_i + e0 - skip);
                const u64* src = S.stage + e0;
                const int cnt = (int)((u64)n_i - e0);
                const int head = (int)((reinterpret_cast<uintptr_t>(dst) >> 3) & 1);
                if (lane == 0 && head) st_stream(dst, src[0]);
                const int npairs = (cnt - head) >> 1;
                for (int p = lane; p < npairs; p += 32)
                    st_stream2(dst + head + 2 * p, src[head + 2 * p], src[head + 2 * p + 1]);
                if (lane == 31 && ((cnt - head) & 1)) st_stream(dst + cnt - 1, src[cnt - 1]);
            }
            __syncwarp();
        }
        b += nb;
    }
}

__global__ void __launch_bounds__(D_NT) decode_kernel(const DPack pk, const DSeek* __restrict__ seekp,
                                                      u64* __restrict__ out, u64 out_cap) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    DWarpSmem& S = reinterpret_cast<DWarpSmem*>(smem_raw)[wid];
    if (seekp->out_len > out_cap) return;  // error already flagged by decode_seek_kernel
    decode_warp_run(pk, seekp->first_block, seekp->skip, out, (u64)blockIdx.x * D_WARPS + wid, S, lane);
}

// Several packs decoded in full (seek 0) by ONE launch: the k posting lists of a query arrive as
// UidPacks (1.3-1.6 B/UID over PCIe) and are expanded side by side.  Job j owns warps
// [warp_base[j], warp_base[j+1]) of the grid.
struct DJob {
    DPack pk;
    u64* out;
    u64 warp_base;
};
__global__ void __launch_bounds__(D_NT) decode_batch_kernel(const DJob* __restrict__ jobs, u32 njobs, u64 nwarps) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    DWarpSmem& S = reinterpret_cast<DWarpSmem*>(smem_raw)[wid];
    const u64 gw = (u64)blockIdx.x * D_WARPS + wid;
    if (gw >= nwarps) return;
    u32 lo = 0, hi = njobs;  // last job with warp_base <= gw
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (jobs[mid].warp_base <= gw) lo = mid; else hi = mid;
    }
    const DPack pk = jobs[lo].pk;
    decode_warp_run(pk, 0, 0, jobs[lo].out, gw - jobs[lo].warp_base, S, lane);
}

}  // namespace dgx
