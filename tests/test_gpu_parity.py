"""GPU parity: libdgx (through the C ABI) vs the CPU oracle, bit-exact.

Runs on a B200 only (`pytest -m gpu`).  Known-answer cases transcribe the
reference's own tests; randomized cases compare with oracle/ on the same seeded
inputs; large cases use size-independent properties plus the oracle.
"""
import os
import sys
import threading

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(__file__))
import gen  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dgx():
    import dgraph_b200
    from dgraph_b200 import _lib

    lib = _lib.load()
    _lib.check(lib.dgx_init(-1))
    print(_lib.describe())
    return dgraph_b200


def L(dgx, xs):
    return dgx.pb.List(np.asarray(xs, dtype=np.uint64))


def eq(got, want, what=""):
    got = np.asarray(got, dtype=np.uint64)
    want = np.asarray(want, dtype=np.uint64)
    if got.size != want.size or not np.array_equal(got, want):
        n = min(got.size, want.size)
        bad = np.nonzero(got[:n] != want[:n])[0]
        first = int(bad[0]) if bad.size else n
        raise AssertionError(
            f"{what}: len got {got.size} want {want.size}; first diff at {first}: "
            f"got {got[max(0, first - 2): first + 3].tolist()} want {want[max(0, first - 2): first + 3].tolist()}"
        )


def to_pack(dgx, op):
    """oracle Pack -> dgraph_b200.pb.UidPack (same bytes)"""
    if op.is_nil:
        return None
    return dgx.pb.UidPack(op.block_size, op.base, op.num_uids, op.delta_off, op.deltas)


# ---- known answers from algo/uidlist_test.go ------------------------------------

def test_merge_sorted_kat(dgx):
    from test_oracle_algo import MERGE_CASES
    for lists, want in MERGE_CASES:
        got = dgx.algo.MergeSorted([L(dgx, l) for l in lists])
        eq(got.Uids, want, f"MergeSorted{lists}")


def test_intersect_sorted_kat(dgx):
    from test_oracle_algo import ISECT_SORTED_CASES
    for lists, want in ISECT_SORTED_CASES:
        got = dgx.algo.IntersectSorted([L(dgx, l) for l in lists])
        if not lists:
            assert got.Uids is None  # &pb.List{}: nil Uids (algo/uidlist.go:298-300)
        else:
            eq(got.Uids, want, f"IntersectSorted{lists}")


def test_difference_kat(dgx):
    from test_oracle_algo import DIFF_CASES
    for u, v, want in DIFF_CASES:
        got = dgx.algo.Difference(L(dgx, u), L(dgx, v))
        assert got.Uids is not None  # non-nil empty (uidlist_test.go:246)
        eq(got.Uids, want, f"Difference({u},{v})")
    assert dgx.algo.Difference(None, L(dgx, [1])).tolist() == []


def test_intersect_with_kat(dgx):
    cases = [([1, 2, 3], [], []), ([1, 2, 3], [1, 2, 3, 4, 5], [1, 2, 3]), ([1, 2, 3], [2], [2]),
             ([1, 2, 3], [0, 5], []), ([1, 2, 3], [3, 5], [3]),
             # duplicates: multiset-min (uidlist_test.go:329-348)
             ([1, 1, 2, 3], [1, 2], [1, 2]), ([1, 1, 2, 3, 5], [1, 1, 2, 4], [1, 1, 2]), ([1, 2, 3, 5], [1, 1, 2, 4], [1, 2])]
    for u, v, want in cases:
        ul, vl = L(dgx, u), L(dgx, v)
        dgx.algo.IntersectWith(ul, vl, ul)  # in place, like every caller
        eq(ul.Uids, want, f"IntersectWith({u},{v})")
        eq(vl.Uids, v, "v must be untouched")
        o = dgx.pb.List(None)
        dgx.algo.IntersectWith(L(dgx, u), vl, o)
        eq(o.Uids, want, "o nil")


@pytest.mark.parametrize("n2", [500, 2500, 20000])
def test_intersect_with_ratio_branches(dgx, orc, n2):
    rng = np.random.default_rng(n2)
    common, _, other = gen.fill_nums(rng, 10, n2)
    for a, b in ((common, other), (other, common)):
        o = dgx.pb.List(None)
        dgx.algo.IntersectWith(L(dgx, a), L(dgx, b), o)
        eq(o.Uids, orc.intersect_with(a, b), f"ratio case {n2}")
        eq(o.Uids, common)


# ---- randomized parity vs the oracle ----------------------------------------------

SIZES = [0, 1, 2, 3, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4097, 10000, 65537]


def test_intersect_with_sizes(dgx, orc):
    rng = np.random.default_rng(1)
    for n in SIZES:
        for m in (0, 1, 7, 1024, 5000, 300000):
            hi = max(4 * max(n, m), 16)
            u = gen.uniform_unique(rng, n, hi)
            v = gen.uniform_unique(rng, m, hi)
            o = dgx.pb.List(None)
            dgx.algo.IntersectWith(L(dgx, u), L(dgx, v), o)
            eq(o.Uids, orc.intersect_with(u, v), f"n={n} m={m}")
            eq(dgx.algo.Difference(L(dgx, u), L(dgx, v)).Uids, orc.difference(u, v), f"diff n={n} m={m}")


def test_intersect_regimes_large(dgx, orc):
    rng = np.random.default_rng(2)
    # dense overlap, sparse overlap, disjoint ranges, identical lists, skewed ratios
    master = gen.zipf_gaps(rng, 600000)
    cases = [
        (gen.thin(rng, master, 0.5), gen.thin(rng, master, 0.5)),
        (gen.thin(rng, master, 0.9), gen.thin(rng, master, 0.9)),
        (gen.thin(rng, master, 0.01), gen.thin(rng, master, 0.9)),
        (gen.thin(rng, master, 0.9), gen.thin(rng, master, 0.001)),
        (master[:1000], master[-1000:]),
        (master, master),
        (gen.uniform_unique(rng, 100000, 10**7), gen.uniform_unique(rng, 100000, 10**7)),
        (gen.uniform_unique(rng, 50, 10**12), gen.zipf_gaps(rng, 500000)),
    ]
    for i, (u, v) in enumerate(cases):
        o = dgx.pb.List(None)
        dgx.algo.IntersectWith(L(dgx, u), L(dgx, v), o)
        want = orc.intersect_with(u, v)
        eq(o.Uids, want, f"case {i}")
        eq(o.Uids, np.intersect1d(u, v), f"case {i} numpy")
        eq(dgx.algo.Difference(L(dgx, u), L(dgx, v)).Uids, orc.difference(u, v), f"diff case {i}")
        eq(dgx.algo.Difference(L(dgx, v), L(dgx, u)).Uids, np.setdiff1d(v, u), f"diff rev case {i}")


def test_duplicates_multiset(dgx, orc):
    rng = np.random.default_rng(3)
    for trial in range(60):
        n, m = (int(x) for x in rng.integers(0, 6000, 2))
        hi = int(rng.choice([5, 50, 2000]))
        u = gen.with_dups(rng, n, hi)
        v = gen.with_dups(rng, m, hi)
        if orc.intersect_with_branch(n, m) == 2:
            continue  # Bin regime: duplicates undefined in the reference (uidlist_test.go:394)
        o = dgx.pb.List(None)
        dgx.algo.IntersectWith(L(dgx, u), L(dgx, v), o)
        eq(o.Uids, orc.intersect_with(u, v), f"dups trial {trial} n={n} m={m} hi={hi}")
        eq(dgx.algo.Difference(L(dgx, u), L(dgx, v)).Uids, orc.difference(u, v), f"dups diff trial {trial}")
    # long runs crossing tile boundaries
    u = np.sort(np.concatenate([np.full(3000, 7), np.full(2500, 9), np.arange(10, 3000)]).astype(np.uint64))
    v = np.sort(np.concatenate([np.full(1500, 7), np.full(2600, 9), np.arange(5, 2000, 3)]).astype(np.uint64))
    o = dgx.pb.List(None)
    dgx.algo.IntersectWith(L(dgx, u), L(dgx, v), o)
    eq(o.Uids, orc.intersect_with(u, v), "long runs")
    eq(dgx.algo.Difference(L(dgx, u), L(dgx, v)).Uids, orc.difference(u, v), "long runs diff")
    eq(dgx.algo.Difference(L(dgx, v), L(dgx, u)).Uids, orc.difference(v, u), "long runs diff rev")


def test_intersect_sorted_random(dgx, orc):
    rng = np.random.default_rng(4)
    for k in (1, 2, 3, 5, 8, 9, 17, 40):
        master = gen.zipf_gaps(rng, 200000)
        lists = [gen.thin(rng, master, float(p)) for p in rng.uniform(0.05, 0.95, k)]
        got = dgx.algo.IntersectSorted([L(dgx, l) for l in lists])
        eq(got.Uids, orc.intersect_sorted(lists), f"k={k}")
    # empty list in the mix, and wildly different lengths
    lists = [master, master[:10], np.zeros(0, np.uint64)]
    eq(dgx.algo.IntersectSorted([L(dgx, l) for l in lists]).Uids, [], "with empty")
    lists = [master, master[::1000], master[::7], master[3::5]]
    eq(dgx.algo.IntersectSorted([L(dgx, l) for l in lists]).Uids, orc.intersect_sorted(lists), "skewed")


def test_config2_shape(dgx, orc):
    """BASELINE config[1]: k=8 Zipf lists of ~1e6 (thinnings of a shared master)."""
    rng = np.random.default_rng(201)
    for p, msize in ((0.25, 4_000_000), (0.9, 1_110_000)):
        master = gen.zipf_gaps(rng, msize)
        lists = [gen.thin(rng, master, p) for _ in range(8)]
        got = dgx.algo.IntersectSorted([L(dgx, l) for l in lists])
        eq(got.Uids, orc.intersect_sorted(lists), f"config2 p={p}")


def test_merge_sorted_random(dgx, orc):
    rng = np.random.default_rng(5)
    for k in (1, 2, 3, 4, 7, 16, 33, 64, 100, 257):
        lists = [np.sort(rng.integers(0, 50000, int(rng.integers(0, 3000)), dtype=np.uint64)) for _ in range(k)]
        got = dgx.algo.MergeSorted([L(dgx, l) for l in lists])
        eq(got.Uids, orc.merge_sorted(lists), f"merge k={k}")
    # TestMergeSortedRandom (uidlist_test.go:109-127) shape
    lists = [np.sort(rng.integers(0, 2**63, 1000, dtype=np.uint64)) for _ in range(1000)]
    got = dgx.algo.MergeSorted([L(dgx, l) for l in lists])
    eq(got.Uids, orc.merge_sorted(lists), "1000x1000")
    # large skewed lengths with heavy cross-list duplication (config 5 shape, scaled)
    master = gen.zipf_gaps(rng, 2_000_000)
    lens = (1_000_000 / np.arange(1, 17)).astype(int)
    lists = [gen.thin(rng, master, min(1.0, l / master.size)) for l in lens]
    got = dgx.algo.MergeSorted([L(dgx, l) for l in lists])
    eq(got.Uids, np.unique(np.concatenate(lists)), "skewed merge")


def test_intersect_batch(dgx, orc):
    rng = np.random.default_rng(6)
    npairs = 300
    As, Bs = [], []
    for i in range(npairs):
        n = int(rng.choice([0, 1, 50, 1024, 3000, 20000]))
        m = int(rng.choice([0, 3, 700, 1025, 9000, 60000]))
        master = gen.zipf_gaps(rng, max(n, m) * 2 + 10)
        As.append(gen.thin(rng, master, n / master.size))
        Bs.append(gen.thin(rng, master, m / master.size))
    a = np.concatenate(As); b = np.concatenate(Bs)
    a_off = np.concatenate([[0], np.cumsum([x.size for x in As])]).astype(np.uint64)
    b_off = np.concatenate([[0], np.cumsum([x.size for x in Bs])]).astype(np.uint64)
    out, out_off = dgx.algo.IntersectBatch(a, a_off, b, b_off)
    for i in range(npairs):
        eq(out[int(out_off[i]): int(out_off[i + 1])], orc.intersect_with(As[i], Bs[i]), f"pair {i}")


# ---- codec ---------------------------------------------------------------------------

def test_decode_roundtrip(dgx, orc):
    rng = np.random.default_rng(7)
    for size in (1, 2, 5, 255, 256, 257, 1000, 16384, 16385, 100000, 1234567):
        uids = gen.get_uids(rng, size)  # duplicates allowed (gap 0), like the reference's getUids
        for bs in (256,):
            pack = orc.encode(uids, bs)
            got = dgx.codec.Decode(to_pack(dgx, pack), 0)
            eq(got, uids, f"decode size={size} bs={bs}")
            assert dgx.codec.ExactLen(to_pack(dgx, pack)) == uids.size
    assert dgx.codec.Decode(None, 0).size == 0


def test_decode_block_sizes_and_msb(dgx, orc):
    rng = np.random.default_rng(8)
    big = [0xF000000000000000, 0xF00F000000000000, 0x00F00F0000000000, 0x000F0F0000000000, 0x0F0F0F0F00000000]
    ints = np.sort(np.concatenate([rng.integers(0, 2**32, 3000, dtype=np.uint64)] +
                                  [rng.integers(0, 2**32, 700, dtype=np.uint64) + np.uint64(b) for b in big]))
    for bs in (0, 1, 2, 5, 10, 100, 256, 257, 1000, 5000):
        pack = orc.encode(ints, bs)
        eq(dgx.codec.Decode(to_pack(dgx, pack), 0), ints, f"msb bs={bs}")
    wide = gen.zipf_gaps(rng, 300000, a=1.2, clip=1 << 31)  # 1..4-byte deltas, MSB splits
    pack = orc.encode(wide, 256)
    eq(dgx.codec.Decode(to_pack(dgx, pack), 0), wide, "wide gaps")


def test_decode_seek(dgx, orc):
    # TestDecoder (codec_test.go:190-217) + TestSeek table semantics via Decode(pack, seek)
    expected = np.arange(3, 10001, 3, dtype=np.uint64)
    pack = orc.encode(expected, 10)
    p = to_pack(dgx, pack)
    for seek in [0, 1, 2, 3, 4, 29, 30, 31, 33, 34, 5000, 9998, 9999, 10000, 10001, 2**64 - 1]:
        eq(dgx.codec.Decode(p, seek), orc.decode(pack, seek), f"seek={seek}")
    rng = np.random.default_rng(9)
    uids = gen.get_uids(rng, 200000)  # with duplicates across block boundaries
    pack = orc.encode(uids, 256)
    p = to_pack(dgx, pack)
    for seek in rng.integers(0, int(uids[-1]) + 10, 40):
        eq(dgx.codec.Decode(p, int(seek)), orc.decode(pack, int(seek)), f"seek={seek}")
    for seek in uids[[0, 255, 256, 257, 511, 512, 1000, -1]]:
        eq(dgx.codec.Decode(p, int(seek)), orc.decode(pack, int(seek)), f"seek=uid {seek}")


def test_golden_fixture_decode(dgx):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "clustered_head.npz"))
    p = dgx.pb.UidPack(256, g["base"], g["num_uids"], g["delta_off"], g["deltas"])
    eq(dgx.codec.Decode(p, 0), g["uids"], "golden clustered fixture")


def test_decode_intersect_pipeline(dgx, orc):
    rng = np.random.default_rng(10)
    master = gen.zipf_gaps(rng, 1_000_000)
    pack = orc.encode(master, 256)
    l1 = gen.thin(rng, master, 0.1)
    l2 = gen.thin(rng, master, 0.01)
    for seek in (0, int(master[500000])):
        got = dgx.codec.DecodeIntersectSorted(to_pack(dgx, pack), seek, [L(dgx, l1), L(dgx, l2)])
        want = orc.intersect_sorted([orc.decode(pack, seek), l1, l2])
        eq(got.Uids, want, f"pipeline seek={seek}")


def test_intersect_compressed_with(dgx, orc):
    """algo.IntersectCompressedWith vs the oracle's restatement (LinJump and Bin branches,
    afterUID seeks), on duplicate-free inputs like the reference's own tests
    (algo/uidlist_test.go:607-681)."""
    rng = np.random.default_rng(21)
    # the reference's fillNums cases at BlockSize 10
    for n1 in (0, 1, 3, 11, 100):
        for n2 in (0, 1, 3, 11, 100):
            common, block, other = gen.fill_nums(rng, n1, n2)
            pack = orc.encode(block, 10)
            o = dgx.pb.List(None)
            dgx.algo.IntersectCompressedWith(to_pack(dgx, pack), 0, L(dgx, other), o)
            if pack.is_nil:
                assert o.Uids is None
            else:
                eq(o.Uids, common, f"fillNums {n1},{n2}")
    for n, m in ((1000, 1000), (1000, 50), (50, 20000), (5000, 30), (300000, 2000), (2000, 300000)):
        u = gen.uniform_unique(rng, n, 10 * max(n, m))
        v = gen.uniform_unique(rng, m, 10 * max(n, m))
        pack = orc.encode(u, 256)
        for after in (0, 1, int(u[n // 2]), int(u[n // 2]) + 1, int(u[-1]), int(u[-1]) + 5):
            o = dgx.pb.List(None)
            dgx.algo.IntersectCompressedWith(to_pack(dgx, pack), after, L(dgx, v), o)
            eq(o.Uids, orc.intersect_compressed_with(pack, after, v), f"n={n} m={m} after={after}")


# ---- error behaviour, concurrency, properties at size --------------------------------

def test_out_cap_error(dgx):
    import ctypes as C
    from dgraph_b200 import _lib
    lib = _lib.load()
    u = np.arange(5000, dtype=np.uint64)
    out = np.zeros(10, dtype=np.uint64)
    n = C.c_size_t(0)
    rc = lib.dgx_intersect2(u.ctypes.data, u.size, u.ctypes.data, u.size, out.ctypes.data, 10, C.byref(n))
    assert rc == -4, (rc, lib.dgx_last_error())
    # the library stays usable afterwards
    o = dgx.pb.List(None)
    dgx.algo.IntersectWith(L(dgx, u), L(dgx, u), o)
    eq(o.Uids, u)


def test_concurrent_callers(dgx, orc):
    rng = np.random.default_rng(11)
    master = gen.zipf_gaps(rng, 300000)
    jobs = [(gen.thin(rng, master, 0.5), gen.thin(rng, master, 0.3)) for _ in range(16)]
    want = [orc.intersect_with(u, v) for u, v in jobs]
    errs = []

    def work(i):
        try:
            for _ in range(5):
                o = dgx.pb.List(None)
                dgx.algo.IntersectWith(L(dgx, jobs[i][0]), L(dgx, jobs[i][1]), o)
                eq(o.Uids, want[i], f"thread {i}")
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(16)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs[0]


def test_properties_at_scale(dgx):
    """Size-independent properties at 1e7: idempotence, A∩B ⊎ A\\B = A, sortedness, merge == unique."""
    rng = np.random.default_rng(12)
    master = gen.zipf_gaps(rng, 12_000_000)
    a = gen.thin(rng, master, 0.8)
    b = gen.thin(rng, master, 0.5)
    la, lb = L(dgx, a), L(dgx, b)
    i = dgx.pb.List(None)
    dgx.algo.IntersectWith(la, lb, i)
    d = dgx.algo.Difference(la, lb)
    assert i.Uids.size + d.Uids.size == a.size
    assert np.all(np.diff(i.Uids.astype(np.int64)) > 0) and np.all(np.diff(d.Uids.astype(np.int64)) > 0)
    eq(i.Uids, np.intersect1d(a, b, assume_unique=True), "1e7 intersect")
    eq(d.Uids, np.setdiff1d(a, b, assume_unique=True), "1e7 difference")
    ii = dgx.pb.List(None)
    dgx.algo.IntersectWith(i, lb, ii)
    eq(ii.Uids, i.Uids, "idempotence")
    m = dgx.algo.MergeSorted([i, d])
    eq(m.Uids, a, "merge(A∩B, A\\B) == A")
    m2 = dgx.algo.MergeSorted([la, lb, la])
    eq(m2.Uids, np.union1d(a, b), "union")


@pytest.mark.parametrize("knobs", [{}, {"DGX_MERGE_STRIDE": "16"}, {"DGX_MERGE": "tree"}],
                         ids=["default", "stride16", "tree"])
def test_merge_multiway_forced(orc, knobs):
    """The multiway MergeSorted path with its size threshold removed (DGX_MERGE_MULTI_MIN=0), in a
    subprocess because libdgx reads its knobs once: known answers, random k, adversarial shapes that
    force the block-wise rounds (identical lists, one dense cluster, long duplicate runs).  Variants: tiles so large
    that most need several rounds (stride 16), and the pairwise tree forced for every k.  The launch count of a small
    k = 9 merge shows which path ran: the tree takes ceil(log2 9) = 4 launches, the multiway path more."""
    import subprocess
    code = r'''
import os, sys
import numpy as np
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import gen
from dgraph_b200 import _lib, algo, pb
from oracle import pyoracle as orc
from test_oracle_algo import MERGE_CASES
def L(x): return pb.List(np.asarray(x, dtype=np.uint64))
def chk(lists, what):
    got = algo.MergeSorted([L(l) for l in lists]).Uids
    want = orc.merge_sorted(lists)
    assert got.size == want.size and np.array_equal(got, want), (what, got.size, want.size)
before = _lib.stats()["kernel_launches"]
chk([np.arange(j, 9000, 9, dtype=np.uint64) for j in range(9)], "k=9, 9000 values")
launches = _lib.stats()["kernel_launches"] - before
if os.environ.get("DGX_MERGE") == "tree":
    assert launches == 4, ("forced tree", launches)
else:
    assert launches > 4, ("multiway threshold not lifted", launches)
for lists, want in MERGE_CASES:
    got = algo.MergeSorted([L(l) for l in lists])
    assert got.tolist() == want, (lists, got.tolist())
rng = np.random.default_rng(77)
for k in (3, 4, 5, 17, 33, 63, 64):
    chk([np.sort(rng.integers(0, 50000, int(rng.integers(0, 3000)), dtype=np.uint64)) for _ in range(k)], f"small k={k}")
# more than 64 lists: groups of <= 64 merged multiway into intermediate runs (device-side lengths), then merged again
for k in (65, 130, 257):
    chk([np.sort(rng.integers(0, 200000, int(rng.integers(0, 4000)), dtype=np.uint64)) for _ in range(k)], f"grouped k={k}")
wide = gen.zipf_gaps(rng, 1500000)
chk([gen.thin(rng, wide, float(rng.uniform(0.002, 0.03))) for _ in range(200)], "grouped k=200, 3e6 values")
chk([np.zeros(0, np.uint64)] * 70 + [wide[::5], wide[1::7]] + [np.zeros(0, np.uint64)] * 70, "mostly empty, k=142")
master = gen.zipf_gaps(rng, 400000)
chk([master] * 64, "64 identical lists")
chk([master[::3], master[1::3], master[2::3]] * 8, "interleaved x8")
dense = np.arange(10**6, 10**6 + 300000, dtype=np.uint64)
chk([dense] + [gen.thin(rng, master, 0.01) for _ in range(40)], "one dense cluster")
runs = np.sort(np.concatenate([np.full(50000, 7), np.full(70000, 9), rng.integers(0, 100, 5000)]).astype(np.uint64))
chk([runs, runs[::2], np.arange(0, 200, dtype=np.uint64)] * 5, "long duplicate runs")
lens = (2_000_000 / np.arange(1, 65)).astype(int)
big = gen.zipf_gaps(rng, 4_000_000)
chk([gen.thin(rng, big, min(1.0, l / big.size)) for l in lens], "config-5 shape")
chk([np.array([2**64 - 1, 2**64 - 1], dtype=np.uint64), np.array([0, 2**64 - 1], dtype=np.uint64), np.array([5], dtype=np.uint64)], "max values")
# key widths: tiles whose value span fits 32 bits merge on u32 keys, wide ones on u64 -- cover both and the mix
chk([np.sort(rng.integers(0, 2**64 - 1, 20000, dtype=np.uint64)) for _ in range(9)], "full-range 64-bit values")
far = (np.arange(30000, dtype=np.uint64) << np.uint64(33)) + np.uint64(12345)
chk([far[::2], far[1::3], np.arange(5 * 10**9, 5 * 10**9 + 40000, dtype=np.uint64), far[::7]], "wide gaps around a dense cluster")
edge = np.uint64(2**32 - 2) * np.arange(1, 20001, dtype=np.uint64)
chk([edge, edge + np.uint64(1), edge[::2] + np.uint64(2**32 - 3)], "spans at the 32-bit boundary")
print("MULTIWAY_OK")
'''
    env = dict(os.environ, DGX_MERGE_MULTI_MIN="0", **knobs)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert "MULTIWAY_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
