"""Keyframe database: knnMatch k=2 -> Lowe ratio test -> database-wide mutual check (ShardedKeyframeDatabase.match*).

The contract is row P of the frame-to-frame pipeline applied to the concatenated database: keep query q iff its global
top-2 passes the ratio test (when asked) and q is the lowest-index nearest query of its best row t1 among the batch
(when asked).  cv2 has nothing to compare with here (``BFMatcher(crossCheck=True)`` on a collection of more than one
image fails ``batch_distance.cpp:303``), so the references are ``hamming_oracle.pipeline`` over the concatenation and
``BFMatcher.match_tensors`` on the concatenated array.

CPU part: gloo worlds of 2 and 3 with an oracle-backed stand-in for the device ops -- shard ownership of t1, the MAX
all-reduce of the per-shard flags, empty ranks, decoding.  GPU part (``gpu``): every variant, edge sizes, growth and
full C4, bit-exact.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from slam_experiments_b200 import _native as nat
from slam_experiments_b200.keyframe_db import ShardedKeyframeDatabase, shard_ranges
from oracle import hamming_oracle as ho

COMBOS = ((None, False), (0.75, False), (None, True), (0.75, True))


def expected(q, kfs, ratio, cross):
    """(queryIdx, imgIdx, trainIdx, distance) from hamming_oracle.pipeline over the concatenation."""
    sizes = np.array([np.asarray(k).shape[0] for k in kfs], np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    cat = np.concatenate([np.asarray(k).reshape(-1, 32) for k in kfs]) if len(kfs) else np.empty((0, 32), np.uint8)
    eq, et, ed = ho.pipeline(q, cat, ratio, cross)
    img = (np.searchsorted(starts, et, side="right") - 1).astype(np.int32)
    return eq, img, (et - starts[img]).astype(np.int32), ed


def same(got, exp):
    return all(np.array_equal(np.asarray(g), np.asarray(e)) for g, e in zip(got, exp)) and len(got) == len(exp)


# =====================================================================================================================
# CPU: oracle-backed stand-in for the device ops, gloo worlds
# =====================================================================================================================
class PipelineOracleOps:
    """CPU stand-in for NativeOps with the pipeline hooks (tests only).  Records, per call, which queries this rank's
    shard flagged, so the test can check that only the owner of t1 ever answers for it."""

    def __init__(self):
        self.flag_log = []

    def upload(self, a):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint8).reshape(-1, 32))

    def make_shard(self, train):
        return {"bits": train, "prepared": None, "nt": train.shape[0]}

    def append_rows(self, shard, rows):
        cat = np.concatenate([shard["bits"].numpy(), rows]) if shard["nt"] else rows
        return self.make_shard(torch.from_numpy(np.ascontiguousarray(cat)))

    def local_knn2(self, query, shard, train_base):
        return torch.from_numpy(ho.knn2_keys(query.numpy(), shard["bits"].numpy(), train_base=train_base).view(np.int64))

    def all_gather(self, keys, group):
        out = [torch.empty_like(keys) for _ in range(dist.get_world_size(group))]
        dist.all_gather(out, keys.contiguous(), group=group)
        return torch.stack(out)

    def merge(self, gathered):
        return torch.from_numpy(ho.merge_top2_keys(gathered.numpy().view(np.uint64)).view(np.int64))

    def to_host(self, t):
        return t.numpy()

    def mutual_flags(self, keys, query, shard, row_lo, ratio):
        k = keys.numpy().view(np.uint64).reshape(-1, 2)
        q = query.numpy()
        bits = shard["bits"].numpy()
        flags = np.zeros(k.shape[0], np.uint8)
        lut = ho.ratio_lut(ratio) if ratio is not None else None
        for i in range(k.shape[0]):
            if k[i, 0] == ho.NO_MATCH_KEY:
                continue
            t1 = int(k[i, 0] & np.uint64(0xFFFFFFFF))
            if not (row_lo <= t1 < row_lo + bits.shape[0]):
                continue
            if lut is not None and (k[i, 1] == ho.NO_MATCH_KEY or int(k[i, 0] >> np.uint64(32)) >= lut[min(int(k[i, 1] >> np.uint64(32)), 256)]):
                continue
            col = ho.hamming_matrix(bits[t1 - row_lo:t1 - row_lo + 1], q)[0]
            flags[i] = int(np.argmin(col)) == i
        self.flag_log.append((row_lo, row_lo + bits.shape[0], np.nonzero(flags)[0].tolist()))
        return torch.from_numpy(flags)

    def all_reduce_max(self, flags, group):
        buf = flags.clone() if flags.numel() else torch.zeros(1, dtype=torch.uint8)
        dist.all_reduce(buf, op=dist.ReduceOp.MAX, group=group)
        return buf

    def filter_matches(self, keys, flags, ratio):
        k = keys.numpy().view(np.uint64).reshape(-1, 2)
        nq = k.shape[0]
        keep = k[:, 0] != ho.NO_MATCH_KEY
        d1 = (k[:, 0] >> np.uint64(32)).astype(np.int64)
        if ratio is not None:
            has2 = k[:, 1] != ho.NO_MATCH_KEY
            d2 = np.where(has2, (k[:, 1] >> np.uint64(32)).astype(np.int64), 0)
            keep &= has2 & (d1 < ho.ratio_lut(ratio)[np.clip(d2, 0, 256)])
        if flags is not None:
            keep &= flags.numpy()[:nq] != 0
        qi = np.nonzero(keep)[0]
        out = np.zeros((3, nq), np.int32)
        out[0, :qi.size] = qi
        out[1, :qi.size] = (k[qi, 0] & np.uint64(0xFFFFFFFF)).astype(np.int64)
        out[2, :qi.size] = d1[qi]
        t = torch.from_numpy(out)
        return t[0], t[1], t[2], torch.tensor([qi.size], dtype=torch.int32)


def gloo_db(seed=21):
    """Tie-heavy keyframes with empty ones, cross-shard duplicates, and query rows planted on shard boundaries."""
    rng = np.random.default_rng(seed)
    sizes = [5, 0, 0, 60, 3, 0, 40]           # world 3: the last rank owns no keyframe at all
    kfs = [rng.integers(0, 4, (s, 32), dtype=np.uint8) for s in sizes]
    kfs[6][:4] = kfs[0][:4]                   # duplicates across shards: the lower global row must win
    kfs[4][1] = kfs[3][59]
    cat = np.concatenate(kfs)
    q = rng.integers(0, 4, (40, 32), dtype=np.uint8)
    plant = []
    for world in (2, 3):
        for _, _, lo, hi in shard_ranges(sizes, world):
            if hi > lo:
                plant += [lo, hi - 1]
    plant = sorted(set(plant)) + [0, 1, 65, 106]
    q[:len(plant)] = cat[plant]
    q[len(plant)] = q[0]                      # duplicate query rows: only the lower index may be mutual
    q_rank0 = cat[:12].copy()                 # every best row on the first rank: the others own no candidate
    return sizes, kfs, q, q_rank0


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sizes, kfs, q, q_rank0 = gloo_db()
        lo, hi, rlo, rhi = shard_ranges(sizes, world)[rank]
        ops = PipelineOracleOps()
        db = ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, ops=ops)
        out = {}
        for name, qq in (("q", q), ("rank0", q_rank0), ("empty", np.empty((0, 32), np.uint8))):
            for ratio, cross in COMBOS:
                out[(name, ratio, cross)] = db.match_tensors(qq, ratio=ratio, cross_check=cross)
        rows = db.match(q, ratio=0.75, cross_check=True)
        out["dmatch"] = [(m.queryIdx, m.imgIdx, m.trainIdx, int(m.distance)) for m in rows]
        # growth: a database built from the first four keyframes and grown by appends
        db2 = ShardedKeyframeDatabase(sizes[:4], [kfs[i] for i in range(*shard_ranges(sizes[:4], world)[rank][:2])],
                                      rank=rank, world_size=world, ops=PipelineOracleOps())
        for k in kfs[4:]:
            db2.append_keyframe(k)
        out["grown"] = db2.match_tensors(q, ratio=0.8, cross_check=True)
        ret[rank] = (out, ops.flag_log, (rlo, rhi))
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_pipeline_matches_oracle(world):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    sizes, kfs, q, q_rank0 = gloo_db()
    cat = np.concatenate(kfs)
    ranges = [ret[r][2] for r in range(world)]
    if world == 3:
        assert ranges[2][0] == ranges[2][1], "the test wants an empty rank"
    for name, qq in (("q", q), ("rank0", q_rank0), ("empty", np.empty((0, 32), np.uint8))):
        for ratio, cross in COMBOS:
            exp = expected(qq, kfs, ratio, cross)
            for r in range(world):
                assert same(ret[r][0][(name, ratio, cross)], exp), (world, r, name, ratio, cross)
    exp = expected(q, kfs, 0.75, True)
    assert ret[0][0]["dmatch"] == list(zip(*[a.tolist() for a in exp]))
    for r in range(world):
        assert same(ret[r][0]["grown"], expected(q, kfs, 0.8, True)), r
    # ownership: every rank is asked about its own row range, flags only queries whose best row it holds, and the
    # flags of the ranks never overlap.  Mutual calls in order: ("q", None), ("q", 0.75), ("rank0", None),
    # ("rank0", 0.75), ("empty", None), ("empty", 0.75), match(q, 0.75).
    t1_of = {"q": ho.knn2_keys(q, cat)[:, 0], "rank0": ho.knn2_keys(q_rank0, cat)[:, 0]}
    t1_of = {k: (v & np.uint64(0xFFFFFFFF)).astype(np.int64) for k, v in t1_of.items()}
    calls = ["q", "q", "rank0", "rank0", None, None, "q"]
    for r in range(world):
        assert len(ret[r][1]) == len(calls)
        for lo, hi, _ in ret[r][1]:
            assert (lo, hi) == ranges[r]
    for c, name in enumerate(calls):
        per_rank = [set(ret[r][1][c][2]) for r in range(world)]
        assert sum(len(s) for s in per_rank) == len(set().union(*per_rank))
        for r in range(world):
            lo, hi = ranges[r]
            assert all(lo <= t1_of[name][i] < hi for i in per_rank[r]), (c, r)
    assert len(ret[0][1][0][2]) > 0 and len(ret[1][1][0][2]) > 0        # both sides of the first boundary answer
    # the planted rows really are best rows on both sides of every boundary
    assert {lo for lo, hi in ranges if hi > lo} <= set(t1_of["q"].tolist())
    assert {hi - 1 for lo, hi in ranges if hi > lo} <= set(t1_of["q"].tolist())
    # "rank0" queries: every best row on rank 0; the other ranks own no candidate yet join the all-reduce
    assert (t1_of["rank0"] < ranges[0][1]).all()
    assert all(not ret[r][1][c][2] for r in range(1, world) for c in (2, 3))


def test_single_rank_pipeline_and_one_row_database():
    sizes, kfs, q, _ = gloo_db(5)
    db = ShardedKeyframeDatabase(sizes, kfs, ops=PipelineOracleOps())
    for ratio, cross in COMBOS:
        assert same(db.match_tensors(q, ratio=ratio, cross_check=cross), expected(q, kfs, ratio, cross)), (ratio, cross)
    one = [np.zeros((0, 32), np.uint8), q[3:4].copy()]
    db = ShardedKeyframeDatabase([0, 1], one, ops=PipelineOracleOps())
    assert db.match_tensors(q, ratio=0.75)[0].size == 0                       # the ratio test needs two rows
    qi, img, loc, d = db.match_tensors(q, cross_check=True)
    assert qi.tolist() == [3] and img.tolist() == [1] and loc.tolist() == [0] and d.tolist() == [0]


def test_db_oracle_equals_pipeline_oracle():
    from oracle import db_oracle
    rng = np.random.default_rng(3)
    for nq, nt, hi in ((1, 1, 256), (30, 1, 256), (50, 2, 4), (300, 700, 3), (257, 1200, 256), (40, 90, 2)):
        q = rng.integers(0, hi, (nq, 32), dtype=np.uint8)
        t = rng.integers(0, hi, (nt, 32), dtype=np.uint8)
        q[: nq // 3] = t[rng.integers(0, nt, nq // 3)]
        for ratio, cross in COMBOS + ((0.9, True),):
            got = db_oracle.pipeline(q, t, ratio, cross)
            assert same(got, ho.pipeline(q, t, ratio, cross)), (nq, nt, ratio, cross)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_db_entry_points_fail_loudly_without_gpu():
    from slam_experiments_b200 import build as hm_build
    hm_build.build()
    L = nat.lib()
    buf = np.zeros((4, 32), np.uint8)
    keys = np.zeros((4, 2), np.uint64)
    out = np.zeros(16, np.int32)
    assert L.hm_db_mutual_flags(keys.ctypes.data, 4, buf.ctypes.data, 32, buf.ctypes.data, 4, 32, 0, nat.FLAG_MUTUAL,
                                None, out.ctypes.data, 0, None, 0, None) == -5
    assert L.hm_db_filter(keys.ctypes.data, 4, None, 0, None, out.ctypes.data, out.ctypes.data, out.ctypes.data,
                          out.ctypes.data, None) == -5
    # sizing is host arithmetic and depends on the query batch only
    assert L.hm_db_mutual_workspace_bytes(2000, nat.VARIANT_F4) > 0
    assert L.hm_db_mutual_workspace_bytes(0, 0) == 256 and L.hm_db_mutual_workspace_bytes(-1, 0) == 0


# =====================================================================================================================
# GPU
# =====================================================================================================================
VARIANTS = ("popc", "i8", "f4", "auto")
gpu = pytest.mark.gpu


def collection(seed, sizes, hi=256):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, hi, (s, 32), dtype=np.uint8) for s in sizes], rng


def check_db(db, q, kfs, bf_variant="popc"):
    """every option combination: database result == oracle == BFMatcher.match_tensors on the concatenation"""
    import slam_experiments_b200 as sx
    cat = np.concatenate([k.reshape(-1, 32) for k in kfs]) if kfs else np.empty((0, 32), np.uint8)
    starts = np.concatenate([[0], np.cumsum([k.shape[0] for k in kfs])])
    bf = sx.BFMatcher(sx.NORM_HAMMING, variant=bf_variant)
    for ratio, cross in COMBOS:
        got = db.match_tensors(q, ratio=ratio, cross_check=cross)
        exp = expected(q, kfs, ratio, cross)
        assert same(got, exp), (ratio, cross, q.shape[0])
        if q.shape[0] and cat.shape[0]:
            bq, bt, bd = bf.match_tensors(q, cat, ratio=ratio, cross_check=cross)
            assert np.array_equal(bq, got[0]) and np.array_equal(bt, starts[got[1]] + got[2]) and np.array_equal(bd, got[3])
    return got


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_small_and_tie_heavy_collections(variant):
    kfs, rng = collection(1, [300, 90, 1, 515, 0, 128, 127, 700])
    q = rng.integers(0, 256, (400, 32), dtype=np.uint8)
    cat = np.concatenate(kfs)
    q[:150] = cat[rng.choice(cat.shape[0], 150, replace=False)] ^ rng.integers(0, 2, (150, 32), dtype=np.uint8)
    db = ShardedKeyframeDatabase([k.shape[0] for k in kfs], kfs, variant=variant)
    check_db(db, q, kfs)
    tie, rng = collection(2, [200, 0, 333, 64, 1000], hi=3)                     # a handful of distinct distances
    tie[4][:50] = tie[0][:50]                                                   # duplicates across keyframes
    qt = rng.integers(0, 3, (513, 32), dtype=np.uint8)
    qt[:20] = tie[0][:20]
    qt[20:40] = qt[:20]                                                         # duplicate query rows
    db = ShardedKeyframeDatabase([k.shape[0] for k in tie], tie, variant=variant)
    check_db(db, qt, tie)


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_edge_sizes(variant):
    rng = np.random.default_rng(17)
    # a one-row database: the ratio test drops everything, the mutual check alone keeps the row's nearest query
    row = rng.integers(0, 256, (1, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (50, 32), dtype=np.uint8)
    q[7] = row[0]
    q[9] = row[0]
    kfs = [np.empty((0, 32), np.uint8), row, np.empty((0, 32), np.uint8)]
    db = ShardedKeyframeDatabase([0, 1, 0], kfs, variant=variant)
    got = check_db(db, q, kfs)
    assert db.match_tensors(q, ratio=0.75)[0].size == 0
    qi, img, loc, d = db.match_tensors(q, cross_check=True)
    assert qi.tolist() == [7] and img.tolist() == [1] and loc.tolist() == [0] and d.tolist() == [0]
    # batch sizes 0, 1, 2, 129, 2000 and 4097 against one database (duplicated rows across keyframes, duplicated queries)
    kfs, rng = collection(18, [1000, 0, 2500, 1, 3000])
    kfs[4][100:200] = kfs[0][:100]
    cat = np.concatenate(kfs)
    db = ShardedKeyframeDatabase([k.shape[0] for k in kfs], kfs, variant=variant)
    for nq in (0, 1, 2, 129, 2000, 4097):
        q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
        m = nq // 2
        q[:m] = cat[rng.integers(0, cat.shape[0], m)] ^ (rng.integers(0, 8, (m, 32), dtype=np.uint8) == 0).astype(np.uint8)
        if nq >= 4:
            q[nq - 1] = q[0]
        check_db(db, q, kfs)
    # an empty database: nothing to match, every option
    db = ShardedKeyframeDatabase([0, 0], [np.empty((0, 32), np.uint8)] * 2, variant=variant)
    for ratio, cross in COMBOS:
        assert db.match_tensors(q[:10], ratio=ratio, cross_check=cross)[0].size == 0


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_growth_through_append_keyframe(variant):
    sizes = [300, 90, 1, 515, 0, 128, 127, 700, 70000]
    kfs, rng = collection(8, sizes, hi=3)
    q = rng.integers(0, 3, (600, 32), dtype=np.uint8)
    q[:100] = np.concatenate(kfs)[rng.integers(0, sum(sizes), 100)]
    db = ShardedKeyframeDatabase(sizes[:1], kfs[:1], variant=variant)
    for i in range(1, len(sizes)):
        db.append_keyframe(kfs[i])
        if i in (1, 4, len(sizes) - 1):
            for ratio, cross in COMBOS:
                assert same(db.match_tensors(q, ratio=ratio, cross_check=cross), expected(q, kfs[:i + 1], ratio, cross)), (i, ratio, cross)
    at_once = ShardedKeyframeDatabase(sizes, kfs, variant=variant)
    for ratio, cross in COMBOS:
        assert same(db.match_tensors(q, ratio=ratio, cross_check=cross), at_once.match_tensors(q, ratio=ratio, cross_check=cross))


@gpu
def test_match_device_and_dmatch_list():
    import slam_experiments_b200 as sx
    kfs, rng = collection(4, [400, 0, 900, 333])
    q = rng.integers(0, 256, (700, 32), dtype=np.uint8)
    q[:300] = np.concatenate(kfs)[rng.integers(0, 1633, 300)]
    db = ShardedKeyframeDatabase([k.shape[0] for k in kfs], kfs, variant="f4")
    oq, ot, od, cnt = db.match_device(torch.from_numpy(q).cuda(), ratio=0.8, cross_check=True)
    assert oq.is_cuda and oq.dtype == torch.int32 and cnt.shape == (1,)
    eq, img, loc, ed = expected(q, kfs, 0.8, True)
    n = int(cnt[0])
    assert n == len(eq) and np.array_equal(oq[:n].cpu().numpy(), eq) and np.array_equal(od[:n].cpu().numpy(), ed)
    assert np.array_equal(ot[:n].cpu().numpy(), db.starts[img] + loc)
    rows = db.match(q, ratio=0.8, cross_check=True)
    assert isinstance(rows, tuple) and all(isinstance(m, type(sx.DMatch())) for m in rows[:1])
    assert [(m.queryIdx, m.imgIdx, m.trainIdx, m.distance) for m in rows] == \
        list(zip(eq.tolist(), img.tolist(), loc.tolist(), [float(x) for x in ed]))


@gpu
def test_bad_arguments_are_rejected_before_any_work():
    L = nat.lib()
    d = torch.zeros((8, 32), dtype=torch.uint8, device="cuda")
    keys = torch.zeros((8, 2), dtype=torch.int64, device="cuda")
    out = torch.zeros(64, dtype=torch.int32, device="cuda")
    ws = torch.empty(nat.db_mutual_workspace_bytes(8, "popc"), dtype=torch.uint8, device="cuda")
    args = lambda **kw: dict(dict(keys=keys.data_ptr(), nq=8, q=d.data_ptr(), qs=32, t=d.data_ptr(), nt=8, ts=32, lo=0,
                                  flags=nat.FLAG_MUTUAL, lut=None, out=out.data_ptr(), v=nat.VARIANT_POPC,
                                  ws=ws.data_ptr(), wsb=ws.numel(), st=None), **kw)
    call = lambda a: L.hm_db_mutual_flags(*a.values())
    assert call(args()) == 0
    assert call(args(flags=nat.FLAG_MUTUAL | nat.FLAG_DIST_THRESHOLD)) == -1
    assert call(args(flags=nat.FLAG_MUTUAL | nat.FLAG_RATIO)) == -1                    # ratio without its table
    assert call(args(nq=-1)) == -1 and call(args(v=7)) == -1 and call(args(lo=0xFFFFFFFF)) == -1
    assert call(args(ts=24)) == -1 and call(args(out=None)) == -1
    assert call(args(wsb=16)) == -3
    f = lambda **kw: L.hm_db_filter(*dict(dict(k=keys.data_ptr(), nq=8, m=None, fl=0, lut=None, q=out.data_ptr(),
                                               t=out.data_ptr(), d=out.data_ptr(), c=out.data_ptr(), st=None), **kw).values())
    assert f() == 0 and f(fl=nat.FLAG_MUTUAL) == -1 and f(fl=nat.FLAG_DIST_THRESHOLD) == -1 and f(c=None) == -1
    torch.cuda.synchronize()


@gpu
def test_per_call_memory_does_not_grow_with_the_database():
    """The mutual step has no buffer proportional to the database: its workspace is a function of the batch alone and a
    pipeline call allocates the same on a 20k-row and a 600k-row database."""
    rng = np.random.default_rng(6)
    q = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    peaks = []
    for nt in (20000, 600000):
        t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
        db = ShardedKeyframeDatabase([nt], [t], variant="f4")
        qd = torch.from_numpy(q).cuda()
        db.match_device(qd, ratio=0.75, cross_check=True)                   # warm: cached workspaces reach their size
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = db.match_device(qd, ratio=0.75, cross_check=True)
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del out, db
    assert peaks[0] == peaks[1], peaks
    for v in VARIANTS:
        assert nat.db_mutual_workspace_bytes(2000, v) < 64 << 20


# ---- full C4 (2000 queries x 4096 keyframes x 2000 rows): the three databases of the full-size k-NN parity tests ----
def _c4_database(kind):
    from slam_experiments_b200 import synth
    if kind == "uniform":                      # the bench's own input
        return synth.keyframe_database(4096, 2000, 2000, seed=4096)
    rng = np.random.default_rng(4097)
    nt, nq = 4096 * 2000, 2000
    if kind == "dups":
        t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
        pool = rng.integers(0, 256, (64, 32), dtype=np.uint8)
        where = rng.choice(nt, 64 * 1280, replace=False)
        t[where] = pool[rng.integers(0, 64, where.size)]
        q = pool[rng.integers(0, 64, nq)].copy()
        flips = rng.integers(0, 4, nq)
        for i in range(nq):
            for b in rng.choice(256, flips[i], replace=False):
                q[i, b >> 3] ^= 1 << (b & 7)
        return q, t
    return rng.integers(0, 3, (nq, 32), dtype=np.uint8), rng.integers(0, 3, (nt, 32), dtype=np.uint8)


@pytest.fixture(scope="module", params=("uniform", "dups", "lowentropy"))
def c4_pipeline_case(request):
    from oracle import c_oracle as co, db_oracle
    q, t = _c4_database(request.param)
    keys = co.knn2_keys(q, t)
    return request.param, q, t, {(r, c): db_oracle.pipeline_from_keys(q, t, keys, r, c) for r, c in COMBOS}


def _c4_db(t, variant):
    return ShardedKeyframeDatabase([2000] * 4096, [t[i * 2000:(i + 1) * 2000] for i in range(4096)], variant=variant)


@gpu
@pytest.mark.parametrize("variant", ("f4", "i8"))
def test_full_c4_pipeline_all_rows(c4_pipeline_case, variant):
    kind, q, t, exp = c4_pipeline_case
    if variant == "i8" and kind != "uniform":
        pytest.skip("i8 on one database keeps the suite short")
    db = _c4_db(t, variant)
    for (ratio, cross), (eq, et, ed) in exp.items():
        qi, img, loc, d = db.match_tensors(q, ratio=ratio, cross_check=cross)
        assert np.array_equal(qi, eq) and np.array_equal(img * 2000 + loc, et) and np.array_equal(d, ed), (kind, ratio, cross)
    if kind == "dups":
        assert len(exp[(None, True)][0]) < 2000 // 2          # many queries share a best row: the mutual check bites


@gpu
def test_full_c4_pipeline_repeated_is_stable(c4_pipeline_case):
    kind, q, t, exp = c4_pipeline_case
    if kind != "uniform":
        pytest.skip("one database is enough")
    db = _c4_db(t, "f4")
    eq, et, ed = exp[(0.75, True)]
    qd = torch.from_numpy(q).cuda()
    for it in range(30):
        oq, ot, od, cnt = db.match_device(qd, ratio=0.75, cross_check=True)
        n = int(cnt[0])
        assert n == len(eq) and np.array_equal(oq[:n].cpu().numpy(), eq) and np.array_equal(ot[:n].cpu().numpy(), et) and \
            np.array_equal(od[:n].cpu().numpy(), ed), it
