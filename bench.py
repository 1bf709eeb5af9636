#!/usr/bin/env python
"""bench.py -- headline benchmark of the posting-list set-op hot path on B200.

Workload (BASELINE.json configs[1]): k-way algo.IntersectSorted, k = 8 Zipf-gap lists of ~1e6 UIDs each
(independent thinnings, p = 0.25, of a shared 4e6 master), as a batch of Q independent queries per GPU per
step so that one step's inputs (Q x 64 MB) exceed the 126 MB L2.  Metric: input UIDs intersected per
second, bit-exact vs the CPU oracle (every query of the step is checked).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2dense]
                  [--dump-outputs DIR]

value   device-resident: lists already in HBM, one batched launch per step, CUDA events on the launching stream.
e2e     the same step through the host-pointer C ABI, HOST buffers, copies inside the timed region.  The
        headline contract is what production holds: every posting list is a pb.UidPack in (pinned) host
        memory (posting/list.go:1795-1800); dgx_intersect_sorted_packed copies the packs (~1.5 B/UID), decodes
        and intersects on the device and returns the result -- every step, no caching.  Beside it:
        e2e_raw_u64 (decoded uint64 lists cross PCIe, 8 B/UID: the PCIe wall) and e2e_cached (packs named with
        (key, version) stay resident in HBM, steady state: only descriptors and results cross PCIe).

N > 1 is launched by torchrun (one rank per GPU).  Queries are independent, so they shard across ranks with
no data-path collective (weak scaling: Q per rank); the only exchange is the NCCL all-gatherv that
concatenates the per-rank results; it is inside the timed region, on a side stream, so the gather of step i
overlaps the filter of step i+1.

`--impl reference` times the reference's CPU algorithm (the C oracle restating algo/uidlist.go; the Go
toolchain is absent) on the same workload -- N x Q queries at N GPUs -- one query per host thread, the only
parallelism the reference has for this path (IntersectSorted itself is single-threaded).

`--dump-outputs DIR` writes the result of the last timed step of the device-resident loop, as a caller of
dgx_dev_filter_batch receives it, to DIR/offsets.npy (Q + 1 per-query offsets) and DIR/uids.npy (the
concatenated result UIDs), both float64.  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.  At N > 1 every rank writes its own queries' result, named
offsets_rank<r>.npy and uids_rank<r>.npy.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

K_LISTS = 8
LIST_LEN = 1_000_000
METRIC = "UIDs/sec intersected (bit-exact)"
UNIT = "UIDs/s"
WORKLOADS = {
    # name: (keep probability, master size, description)
    "c2": (0.25, 4_000_000, "thinnings p=0.25 of a 4e6 master"),
    "c2dense": (0.9, 1_111_111, "thinnings p=0.9 of a 1.11e6 master (dense variant: ~43 % of the driving list survives)"),
}


def make_query(seed: int, keep: float = 0.25, master_n: int = 4_000_000):
    """One config[1] query: 8 thinnings of a Zipf-gap master (a=1.5, clip 2^20)."""
    rng = np.random.default_rng(seed)
    gaps = np.minimum(rng.zipf(1.5, master_n), 1 << 20).astype(np.uint64)
    master = np.cumsum(gaps, dtype=np.uint64)
    return [master[rng.random(master_n) < keep] for _ in range(K_LISTS)]


def make_queries(q: int, rank: int, workload: str = "c2"):
    keep, master_n, _ = WORKLOADS[workload]
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda s: make_query(s, keep, master_n), [201 + 1000 * rank + i for i in range(q)]))


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons through NVML during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.active = False   # only samples taken while the timed region runs are kept
        self.ok = False

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            self.ok = True
            while not self._halt.is_set():
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_intersect_batch(orc, queries, threads: int) -> float:
    """Seconds for the oracle (algo.IntersectSorted restatement) over all queries on `threads` threads."""
    t0 = time.perf_counter()
    if threads <= 1:
        for q in queries:
            orc.intersect_sorted(q)
    else:
        with ThreadPoolExecutor(max_workers=threads) as ex:  # ctypes releases the GIL
            list(ex.map(orc.intersect_sorted, queries))
    return time.perf_counter() - t0


DUMP_MAX_BYTES = 64 << 20  # --dump-outputs budget over all ranks' files


def dump_outputs(out_dir: str, offsets: np.ndarray, uids: np.ndarray, rank: int, world: int):
    """Writes one step's result as float64 .npy files.  float64 holds every UID below 2^53 exactly, which
    covers these workloads (masters of <= 4e6 gaps of <= 2^20).  A result larger than this rank's share of
    DUMP_MAX_BYTES is replaced by a fixed, seeded sample of its positions, written as uids_index.npy."""
    if uids.size and int(uids.max()) >= 1 << 53:
        raise SystemExit("--dump-outputs: a result UID does not fit float64 exactly")
    arrays = {"offsets": offsets, "uids": uids}
    room = DUMP_MAX_BYTES // world - 8 * offsets.size
    if 8 * uids.size > room:
        idx = np.sort(np.random.default_rng(0).choice(uids.size, room // 16, replace=False))
        arrays["uids"], arrays["uids_index"] = uids[idx], idx
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a.astype(np.float64))


def workload_config(q: int, world: int, workload: str = "c2"):
    _, _, desc = WORKLOADS[workload]
    return {
        "workload": f"configs[1]: k-way IntersectSorted, k=8 Zipf-gap lists of ~1e6 UIDs ({desc}), "
                    f"batch of {q} independent queries per GPU per step",
        "k": K_LISTS, "list_len": LIST_LEN, "queries_per_gpu": q, "parallelism": f"queries sharded over {world} GPU(s)",
        "l2": f"inputs {q * K_LISTS * LIST_LEN * 8 / 1e9:.2f} GB per GPU per step > 126 MB L2 (no flush needed)",
        "lists": "resident in HBM and declared so to the lane (dgx_lane_set_resident_inputs): the plan pre-pass of a step overlaps the previous step's kernel",
    }


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference CPU algorithm on the host cores (rank 0 only), the whole job's queries."""
    if rank != 0:
        return
    from oracle import pyoracle as orc

    orc.lib()
    q = args.queries
    queries = []
    for r in range(world):  # the same N x Q queries the GPU arm shards over its ranks
        queries += make_queries(q, r, args.workload)
    uids = sum(l.size for qq in queries for l in qq)
    host_threads = os.cpu_count() or 1
    busy = min(host_threads, len(queries))  # IntersectSorted is single-threaded: one query per thread
    for _ in range(args.warmup):
        cpu_intersect_batch(orc, queries, busy)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_intersect_batch(orc, queries, busy)
    dt = time.perf_counter() - t0
    val = uids * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(q, world, args.workload),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": busy, "kind": "port",
                         "sample": f"{len(queries)} queries ({world} x {q}) x {K_LISTS} lists x ~{LIST_LEN} UIDs per step, C restatement of "
                                   f"algo.IntersectSorted, one query per thread: {busy} busy threads of {host_threads} logical CPUs "
                                   "(the reference has no parallelism inside one IntersectSorted)",
                         "host_threads": host_threads},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def kernel_source_sha() -> str:
    """Hash of the sources the dominant kernel is built from; stamps profiles/filter_kernel_traffic.json."""
    h = hashlib.sha256()
    for f in ("filter_pipe.cuh", "filter_kernel.cuh", "common.cuh"):
        h.update(open(os.path.join(ROOT, "dgraph_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def run_e2e_legs(args, lib, queries, want, uids_all, uids_per_step, rank, world, dev):
    """The three end-to-end legs (packs / named packs / decoded lists) through the host-pointer C ABI."""
    import torch
    import torch.distributed as dist

    import gen
    from dgraph_b200 import _lib

    Q = len(queries)

    T = max(1, args.e2e_threads)
    res_cap = max(min(l.size for l in qq) for qq in queries)
    pool = ThreadPoolExecutor(max_workers=T)
    outs = [(lib.dgx_host_alloc(res_cap * 8), C.c_size_t(0)) for _ in range(T)]
    pinned = []

    def pin(a: np.ndarray):
        p = lib.dgx_host_alloc(max(a.nbytes, 16))
        assert p
        C.memmove(p, a.ctypes.data, a.nbytes)
        pinned.append(p)
        return p

    def run_e2e(call, nsteps):
        """`call(slot, qi)` = one query through the C ABI on thread `slot`; returns (seconds per step, out values per step).
        The reference is called from many goroutines at once (x.DivideAndRule, worker/task.go:816); here T host
        threads issue the queries, each call borrowing its own lane, so one query's sync gap is another's copy."""
        def worker(slot, steps):
            # thread `slot` issues queries slot, slot+T, ... of every step, back to back: the timed region is a
            # continuous stream of nsteps x Q calls (no barrier between steps -- a server does not have one)
            tot = 0
            for _ in range(steps):
                for qi in range(slot, Q, T):
                    tot += call(slot, qi)
            return tot

        sum(pool.map(lambda s_: worker(s_, 1), range(T)))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        outn = sum(pool.map(lambda s_: worker(s_, nsteps), range(T))) // nsteps
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt / nsteps, outn

    def check_e2e(call):
        ok = True
        for qi in range(Q):
            n = call(0, qi)
            got = np.ctypeslib.as_array(C.cast(outs[0][0], C.POINTER(C.c_uint64)), shape=(max(n, 1),))[:n]
            ok = ok and np.array_equal(got, want[qi])
        return bool(ok)

    # (a) packs: what production holds.  numpy generator (tests/gen.encode_pack_np, checked against the oracle's
    #     Encode byte for byte in tests/test_gen_encoder.py); arrays live in dgx_host_alloc (pinned) memory.
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        enc = list(ex.map(lambda l: gen.encode_pack_np(l, 256), [l for qq in queries for l in qq]))
    # every query's 8 packs are flattened back to back into ONE pinned buffer in the library's flat-image layout
    # (dgx_pack_image_view) -- what a cgo shim's flatten() writes from pb.UidPack.Blocks -- so a query's packs
    # cross PCIe as one transfer
    views, pack_bytes = [], 0
    for qi in range(Q):
        group = enc[qi * K_LISTS:(qi + 1) * K_LISTS]
        sizes = [lib.dgx_pack_image_size(base.size, deltas.size) for (_, base, _, _, deltas) in group]
        blob = lib.dgx_host_alloc(sum(sizes) + 64)
        assert blob
        pinned.append(blob)
        o = 0
        for (bs, base, num, doff_, deltas), sz in zip(group, sizes):
            v = _lib.PackView()
            _lib.check(lib.dgx_pack_image_view(C.c_void_p(blob + o), bs, base.size, deltas.size, C.byref(v)))
            C.memmove(v.base, base.ctypes.data, base.nbytes)
            C.memmove(v.delta_off, doff_.ctypes.data, doff_.nbytes)
            C.memmove(v.num_uids, num.ctypes.data, num.nbytes)
            C.memmove(v.deltas, deltas.ctypes.data, deltas.nbytes)
            pack_bytes += base.nbytes + num.nbytes + doff_.nbytes + deltas.nbytes
            views.append(v)
            o += sz
    del enc

    def make_refs(named: bool):
        tabs = []
        for qi in range(Q):
            refs = (_lib.PackRef * K_LISTS)()
            for j in range(K_LISTS):
                refs[j].pack = C.pointer(views[qi * K_LISTS + j])
                refs[j].key = (1 + rank * 1_000_000 + qi * K_LISTS + j) if named else 0
                refs[j].version = 1
            tabs.append(refs)
        return tabs

    def packed_call(tabs):
        def call(slot, qi):
            buf, cnt = outs[slot]
            _lib.check(lib.dgx_intersect_sorted_packed(tabs[qi], K_LISTS, buf, res_cap, C.byref(cnt)))
            return cnt.value
        return call

    anon, named = make_refs(False), make_refs(True)
    ok_packed = check_e2e(packed_call(anon))
    hb0 = _lib.stats()["h2d_bytes"]
    s_packed, outn = run_e2e(packed_call(anon), args.e2e_steps)
    pack_bytes_moved = (_lib.stats()["h2d_bytes"] - hb0) / (args.e2e_steps + 1)   # counted by the library per copy it issues
    e2e = {"value": uids_all / s_packed, "unit": UNIT, "h2d_bytes_per_step": int(pack_bytes_moved),
           "d2h_bytes_per_step": int(outn * 8 + 8 * Q), "ms_per_step": 1e3 * s_packed, "bit_exact": ok_packed,
           "api": f"dgx_intersect_sorted_packed: every list a pb.UidPack (BlockSize 256, {pack_bytes / uids_per_step:.2f} B/UID) in pinned host "
                  f"memory (a query's 8 packs flattened back to back, as the cgo shim's flatten writes them), copied, decoded and "
                  f"intersected on the device every step (no caching), one call per query, {T} host threads",
           "pack_bytes_per_step": int(pack_bytes), "pcie_GBps": pack_bytes_moved / s_packed / 1e9}
    lib.dgx_cache_clear()
    ok_cached = check_e2e(packed_call(named))               # first pass fills the cache
    st = _lib.CacheStats()
    lib.dgx_cache_get_stats(C.byref(st))
    h0 = _lib.stats()["h2d_bytes"]
    s_cached, outn_c = run_e2e(packed_call(named), args.e2e_steps)
    h2d_cached = (_lib.stats()["h2d_bytes"] - h0) / (args.e2e_steps + 1)
    e2e_cached = {"value": uids_all / s_cached, "unit": UNIT, "h2d_bytes_per_step": int(h2d_cached),
                  "d2h_bytes_per_step": int(outn_c * 8 + 8 * Q), "ms_per_step": 1e3 * s_cached, "bit_exact": ok_cached,
                  "api": "dgx_intersect_sorted_packed with (key, version) on every pack: packs resident in HBM (compressed) after "
                         "their first use, steady state; only descriptors and results cross PCIe",
                  "cache_bytes": int(st.bytes), "cache_entries": int(st.entries)}
    lib.dgx_cache_clear()
    for p in pinned:
        lib.dgx_host_free(p)
    pinned.clear()

    # (b) decoded uint64 lists over PCIe (8 B/UID): the round-1 contract, kept for comparison
    tables = []
    for qq in queries:
        tables.append(((C.c_void_p * K_LISTS)(*[pin(l) for l in qq]), (C.c_size_t * K_LISTS)(*[l.size for l in qq])))

    def raw_call(slot, qi):
        buf, cnt = outs[slot]
        tp, tl = tables[qi]
        _lib.check(lib.dgx_intersect_sorted(tp, tl, K_LISTS, buf, res_cap, C.byref(cnt)))
        return cnt.value

    ok_raw = check_e2e(raw_call)
    s_raw, outn_r = run_e2e(raw_call, max(2, args.e2e_steps // 2))
    e2e_raw = {"value": uids_all / s_raw, "unit": UNIT, "h2d_bytes_per_step": int(uids_per_step * 8),
               "d2h_bytes_per_step": int(outn_r * 8 + 8 * Q), "ms_per_step": 1e3 * s_raw, "bit_exact": ok_raw,
               "api": f"dgx_intersect_sorted (decoded uint64 lists in pinned host memory, 8 B/UID over PCIe), one call per query, {T} host threads",
               "pcie_GBps": uids_per_step * 8 / s_raw / 1e9}
    for p in pinned:
        lib.dgx_host_free(p)
    for buf, _ in outs:
        lib.dgx_host_free(buf)
    pool.shutdown()
    return e2e, e2e_cached, e2e_raw, bool(ok_packed and ok_cached and ok_raw)



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--queries", type=int, default=16, help="independent queries per GPU per step")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--e2e-threads", type=int, default=4)
    ap.add_argument("--no-ops", action="store_true", help="skip the per-config (C1/C3/C4/C5) one-liners under `ops`")
    ap.add_argument("--no-dense", action="store_true", help="skip the p=0.9 variant of the headline step")
    ap.add_argument("--no-resident", action="store_true", help="do not declare the lists resident (no pre-pass / pipeline overlap across steps)")
    ap.add_argument("--no-e2e", action="store_true", help="kernel iteration runs only: skip the end-to-end legs (the line then has no e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from dgraph_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's log (NCCL_DEBUG=INFO/VERSION) goes to stderr, never to stdout: stdout carries ONE JSON line
        if os.environ.get("NCCL_DEBUG"):
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.dgx_init(local_rank))

    Q = args.queries
    queries = make_queries(Q, rank, args.workload)
    uids_per_step = sum(l.size for qq in queries for l in qq)

    # ---- device-resident inputs (torch owns the HBM; libdgx gets raw pointers) -------
    # a real (non-default) torch stream: libdgx launches on it and torch.cuda.Event times it
    stream = torch.cuda.Stream(device=dev)
    comm_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    lane = lib.dgx_lane_create(local_rank, C.c_void_p(stream.cuda_stream))
    assert lane, lib.dgx_last_error()
    # the lists of the device-resident loop are complete in HBM before the first call and never written: declared to
    # the lane, the plan pre-pass of step i+1 may then overlap the pipeline kernel of step i (include/dgx.h)
    if not args.no_resident:
        _lib.check(lib.dgx_lane_set_resident_inputs(lane, 1))

    def to_device(qs):
        keep, ptrs, lens, k_off = [], [], [], [0]
        for qq in qs:
            for l in qq:
                t = torch.from_numpy(l.view(np.int64)).to(dev)
                keep.append(t)
                ptrs.append(t.data_ptr())
                lens.append(l.size)
            k_off.append(len(ptrs))
        nl = len(ptrs)
        return keep, (C.c_void_p * nl)(*ptrs), (C.c_size_t * nl)(*lens), (C.c_size_t * (len(qs) + 1))(*k_off)

    d_lists, c_ptrs, c_lens, c_koff = to_device(queries)
    out_cap = sum(min(l.size for l in qq) for qq in queries)
    # Result buffers, double-buffered so the gather of step i (side stream) overlaps the filter of step i+1.
    # Layout of one buffer: [out_off (Q+1 words) | values]: words Q .. Q+pad are [total count | first pad values],
    # one contiguous slice that the all-gatherv sends as is.
    NBUF = 2
    bufs = [torch.zeros(Q + 1 + out_cap + 2, dtype=torch.int64, device=dev) for _ in range(NBUF)]

    def launch(b):
        buf = bufs[b]
        _lib.check(lib.dgx_dev_filter_batch(lane, _lib.OP_INTERSECT, c_ptrs, c_lens, c_koff, Q,
                                            C.c_void_p(buf.data_ptr() + 8 * (Q + 1)), out_cap, C.c_void_p(buf.data_ptr())))

    # ---- parity check (outside the timed region): EVERY query of the step against the oracle ----------
    from oracle import pyoracle as orc

    launch(0)
    torch.cuda.synchronize()
    host = bufs[0].cpu().numpy().view(np.uint64)
    off, res = host[: Q + 1], host[Q + 1:]
    want = [orc.intersect_sorted(qq) for qq in queries]
    bit_exact = all(np.array_equal(res[int(off[i]):int(off[i + 1])], want[i]) for i in range(Q))
    out_uids = int(off[Q])

    # all-gatherv sized by the real result: every rank sends [count | values padded to `pad`], pad = twice the
    # largest per-rank result of this workload (power of two, agreed across ranks); a step whose result
    # outgrows it fails the run loudly (checked after the timed loop), nothing is truncated silently.
    pad = 1024
    while pad < 2 * out_uids:
        pad *= 2
    if world > 1:
        t = torch.tensor([pad], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pad = int(t.item())
    pad = min(pad, out_cap + 1)
    gathered = [torch.empty(world * (1 + pad), dtype=torch.int64, device=dev) for _ in range(NBUF)]
    ev_done = [torch.cuda.Event() for _ in range(NBUF)]      # filter of buffer b finished
    ev_free = [torch.cuda.Event() for _ in range(NBUF)]      # gather of buffer b finished (buffer reusable)

    def step(i):
        b = i % NBUF
        if world > 1:
            stream.wait_event(ev_free[b])                    # the gather that last read this buffer is done
        launch(b)
        if world > 1:
            ev_done[b].record(stream)
            with torch.cuda.stream(comm_stream):
                comm_stream.wait_event(ev_done[b])
                dist.all_gather_into_tensor(gathered[b], bufs[b][Q: Q + 1 + pad])
                ev_free[b].record(comm_stream)

    if world > 1:  # the gathered block of this rank must be its own [count | results]
        for b in range(NBUF):
            ev_free[b].record(comm_stream)
        step(0)
        torch.cuda.synchronize()
        mine = gathered[0][rank * (1 + pad):(rank + 1) * (1 + pad)].cpu().numpy().view(np.uint64)
        bit_exact = bit_exact and out_uids <= pad and int(mine[0]) == out_uids and bool(np.array_equal(mine[1:1 + out_uids], res[:out_uids]))
        counts = gathered[0].view(world, 1 + pad)[:, 0].cpu().numpy()
        bit_exact = bit_exact and bool(np.all(counts <= pad))

    # ---- device-resident timing --------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    for _ in range(200):  # NVML init can take a while when 8 ranks start at once
        if sampler.ok or hasattr(sampler, "err"):
            break
        time.sleep(0.01)
    sampler.active = True
    launches0 = lib.dgx_lane_launches(lane)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev_end = torch.cuda.Event(enable_timing=True)
    # barrier + synchronize immediately before the first timed launch: a rank that enters the loop late
    # would make its peers' first gather wait inside their timed region
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    evs[0].record()
    host_t0 = time.perf_counter()
    for i in range(args.steps):
        step(i)
        evs[i + 1].record()
    if world > 1:
        stream.wait_stream(comm_stream)                      # the last gathers belong to the timed region
    ev_end.record()
    host_submit_ms = (time.perf_counter() - host_t0) * 1e3 / args.steps  # host time to enqueue one step
    torch.cuda.synchronize()
    sampler.active = False
    rc_sync = lib.dgx_lane_sync(lane)                        # DGX_ERR_CAP here = some step overflowed out_cap
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    launches = int(lib.dgx_lane_launches(lane) - launches0)
    if args.dump_outputs:
        last = bufs[(args.steps - 1) % NBUF].cpu().numpy().view(np.uint64)
        dump_outputs(args.dump_outputs, last[: Q + 1], last[Q + 1: Q + 1 + int(last[Q])], rank, world)
    total_ms = evs[0].elapsed_time(ev_end)
    step_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    bit_exact = bit_exact and rc_sync == 0
    if world > 1:
        cnt = torch.stack([g.view(world, 1 + pad)[:, 0].max() for g in gathered]).max()
        bit_exact = bit_exact and int(cnt.item()) <= pad     # no step's result outgrew the gather slot
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        tot = torch.tensor([uids_per_step, launches, int(bit_exact)], dtype=torch.int64, device=dev)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        uids_all, launches_all = int(tot[0].item()), int(tot[1].item())
        bit_exact = int(tot[2].item()) == world
    else:
        uids_all, launches_all = uids_per_step, launches
    ms_per_step = total_ms / args.steps
    value = uids_all / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel (filter_pipe_kernel: one launch per step, ~90 % of it) -----------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    algo_bytes = 8.0 * (uids_per_step + out_uids)  # 8*(sum|L_i| + |Out|), SURVEY 8(d)
    kern_ms = float(np.median(step_ms)) if world == 1 else ms_per_step
    achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
    # DRAM bytes per launch come from an `ncu --set full` capture (tools/collect_round.sh); the file is stamped
    # with the hash of the kernel sources it was measured on and a stale stamp prints null, never an old number
    traffic, traffic_note = None, "no capture"
    tpath = os.path.join(ROOT, "profiles", "filter_kernel_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("kernel_src_sha") == kernel_source_sha() and tj.get("workload", "c2") == args.workload:
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), f"ncu capture {tj.get('capture', '?')}"
            else:
                traffic_note = "capture is older than the kernel sources (or another workload): not reported"
        except Exception:  # noqa: BLE001
            pass
    roofline = {"bound": "hbm", "kernel": "dgx::filter_pipe_kernel (timed with its plan pre-pass: filter_tiles_kernel + filter_plan_kernel)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": kern_ms}

    # ---- the dense variant of the same step (p = 0.9: ~43 % of the driving list survives all 8 lists) -----
    dense = None
    if world == 1 and args.workload == "c2" and not args.no_dense:
        dq = make_queries(Q, rank, "c2dense")
        dk, dp, dl, dko = to_device(dq)
        dcap = sum(min(l.size for l in qq) for qq in dq)
        dbuf = torch.zeros(Q + 1 + dcap + 2, dtype=torch.int64, device=dev)

        def dstep():
            _lib.check(lib.dgx_dev_filter_batch(lane, _lib.OP_INTERSECT, dp, dl, dko, Q,
                                                C.c_void_p(dbuf.data_ptr() + 8 * (Q + 1)), dcap, C.c_void_p(dbuf.data_ptr())))
        for _ in range(3):
            dstep()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            dstep()
        e1.record()
        torch.cuda.synchronize()
        dms = e0.elapsed_time(e1) / 20
        dh = dbuf.cpu().numpy().view(np.uint64)
        doff, dres = dh[: Q + 1], dh[Q + 1:]
        dok = all(np.array_equal(dres[int(doff[i]):int(doff[i + 1])], orc.intersect_sorted(dq[i])) for i in range(Q))
        duids = sum(l.size for qq in dq for l in qq)
        dbytes = 8.0 * (duids + int(doff[Q]))
        dense = {"workload": WORKLOADS["c2dense"][2], "ms_per_step": dms, "value": duids / (dms * 1e-3), "unit": UNIT,
                 "out_uids_per_step": int(doff[Q]), "bit_exact": bool(dok),
                 "roofline_frac": dbytes / (dms * 1e-3) / 1e9 / peak}
        del dk, dbuf

    # ---- end to end through the host-pointer C ABI (pinned host buffers, copies timed) ------
    e2e = e2e_cached = e2e_raw = None
    if not args.no_e2e:
        e2e, e2e_cached, e2e_raw, ok_e2e = run_e2e_legs(args, lib, queries, want, uids_all, uids_per_step, rank, world, dev)
        bit_exact = bit_exact and ok_e2e

    ops = None
    if world == 1 and not args.no_ops:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_ops

            # the per-op rows chain producers and consumers on one stream (Decode -> IntersectSorted): measured, like
            # tools/bench_ops.py alone, on a lane WITHOUT the resident-inputs declaration of the headline loop
            _lib.check(lib.dgx_lane_set_resident_inputs(lane, 0))
            ops = bench_ops.quick_rows(lib, lane, dev, peak)
        except Exception as e:  # noqa: BLE001
            ops = {"error": repr(e)}

    if rank == 0:
        # CPU baseline: the oracle (port of algo.IntersectSorted), 1 thread like the Go code
        sample = queries[: min(Q, 8)]
        cpu_intersect_batch(orc, sample[:1], 1)
        reps, t_cpu = 0, 0.0
        while t_cpu < 2.0 and reps < 8:
            t_cpu += cpu_intersect_batch(orc, sample, 1)
            reps += 1
        s_uids = sum(l.size for qq in sample for l in qq)
        cpu_baseline = {"value": s_uids * reps / t_cpu, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": f"{len(sample)} of the step's {Q} queries x {reps} repetitions, single thread "
                                  "(algo.IntersectSorted is single-threaded in the reference)",
                        "host": f"{os.cpu_count()} logical CPUs"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(Q, world, args.workload),
            "bit_exact": bool(bit_exact), "queries_checked": Q, "out_uids_per_step": out_uids,
            "host_submit_ms_per_step": round(host_submit_ms, 4),
            "step_ms_rank0": {"median": round(float(np.median(step_ms)), 4), "p10": round(float(np.percentile(step_ms, 10)), 4),
                              "p90": round(float(np.percentile(step_ms, 90)), 4), "max": round(float(np.max(step_ms)), 4)},
            "roofline": roofline, "dense_variant": dense, "cpu_baseline": cpu_baseline,
            "e2e": e2e, "e2e_cached": e2e_cached, "e2e_raw_u64": e2e_raw,
            "gather": None if world == 1 else {"collective": "all_gather_into_tensor on a side stream, overlapped with the next step",
                                               "slot_values": pad, "bytes_per_rank_per_step": 8 * (1 + pad)},
            "ops": ops, "gpu_launches": launches_all, "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
