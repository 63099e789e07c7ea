"""Keyframe database: search only a chosen subset of keyframes (``keyframes=`` on every query entry point).

The contract: the result over a selection S equals cv2's collection ``knnMatch`` over the collection made of the
keyframes of S (in imgIdx order), and ``hamming_oracle.pipeline`` over the concatenation of S, with imgIdx mapped back
to the whole database.  "Select everything" equals ``keyframes=None`` bit for bit.

CPU part: validation and run building on every rank of ``shard_ranges``, the library's run planning (no device needed),
and gloo worlds of 2 and 3 with an oracle-backed stand-in for the device ops.  GPU part (``gpu``): POPC, i8 and f4,
bit-exact, from single keyframes to full C4.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from slam_experiments_b200 import _native as nat
from slam_experiments_b200.feature_matchers import MatcherError
from slam_experiments_b200.keyframe_db import ShardedKeyframeDatabase, selection_mask, shard_ranges, shard_runs
from oracle import hamming_oracle as ho

from test_keyframe_db_pipeline import COMBOS, PipelineOracleOps, _free_port, expected, same

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sel_list(sel, n):
    return np.flatnonzero(selection_mask(sel, n))


def expected_sub(q, kfs, sel, ratio, cross):
    """the pipeline over the concatenation of the selected keyframes, imgIdx mapped back"""
    idx = sel_list(sel, len(kfs))
    eq, img, loc, ed = expected(q, [kfs[i] for i in idx], ratio, cross)
    return eq, idx[img].astype(np.int32) if idx.size else img, loc, ed


def knn_sub(q, kfs, sel, k=2):
    """(imgIdx, trainIdx, distance) [Nq, k'] over the selected keyframes: the global stable top-k of their concatenation"""
    idx = sel_list(sel, len(kfs))
    sub = [np.asarray(kfs[i]).reshape(-1, 32) for i in idx]
    cat = np.concatenate(sub) if sub else np.empty((0, 32), np.uint8)
    starts = np.concatenate([[0], np.cumsum([s.shape[0] for s in sub])]).astype(np.int64)
    keys = ho.knn2_keys(q, cat)
    kk = min(k, cat.shape[0])
    g = (keys[:, :kk] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    d = (keys[:, :kk] >> np.uint64(32)).astype(np.int32)
    img = np.searchsorted(starts, g, side="right") - 1
    return idx[img].astype(np.int32) if kk else img.astype(np.int32), (g - starts[img]).astype(np.int32), d


def same_knn(got, exp):
    return all(np.array_equal(np.asarray(g).reshape(np.asarray(e).shape), e) for g, e in zip(got, exp)) and \
        all(np.asarray(g).shape == np.asarray(e).shape for g, e in zip(got, exp))


# =====================================================================================================================
# CPU: validation, run building, run planning
# =====================================================================================================================
def brute_runs(mask, sizes, lo_kf, hi_kf):
    """shard-local runs from the row set itself: maximal ranges of consecutive selected rows"""
    starts = np.concatenate([[0], np.cumsum(sizes)])
    rows = [r - starts[lo_kf] for k in range(lo_kf, hi_kf) if mask[k] for r in range(starts[k], starts[k + 1])]
    out = []
    for r in rows:
        if out and out[-1][1] == r:
            out[-1][1] = r + 1
        else:
            out.append([r, r + 1])
    return np.array(out, np.int64).reshape(-1, 2)


def test_run_building_on_every_rank():
    rng = np.random.default_rng(0)
    sizes = np.array([5, 0, 0, 60, 3, 0, 40, 1, 0, 1, 128, 0, 7, 300, 0], np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    masks = [np.ones(len(sizes), bool), np.zeros(len(sizes), bool)]
    masks += [rng.random(len(sizes)) < p for p in (0.2, 0.5, 0.8) for _ in range(20)]
    m = np.zeros(len(sizes), bool)
    m[[0, 3, 6, 9]] = True                                   # zero-row keyframes inside runs, 1-row keyframe gaps
    masks.append(m)
    for world in (1, 2, 3, 4, 7):
        ranges = shard_ranges(sizes, world)
        for mask in masks:
            total = 0
            for lo, hi, rlo, rhi in ranges:
                runs = shard_runs(mask, starts, lo, hi, rlo)
                assert runs.dtype == np.int64 and runs.shape[1] == 2
                assert np.array_equal(runs, brute_runs(mask, sizes, lo, hi)), (world, mask, lo, hi)
                if runs.size:
                    assert (runs[:, 1] > runs[:, 0]).all() and (runs[1:, 0] > runs[:-1, 1]).all()
                    assert runs[0, 0] >= 0 and runs[-1, 1] <= rhi - rlo
                total += int((runs[:, 1] - runs[:, 0]).sum())
            assert total == int(sizes[mask].sum())


def test_selection_forms_and_rejections():
    n = 6
    assert np.array_equal(selection_mask([4, 1, 1, 4], n), [0, 1, 0, 0, 1, 0])            # a set
    assert np.array_equal(selection_mask(np.array([5, 0], np.uint16), n), [1, 0, 0, 0, 0, 1])
    assert np.array_equal(selection_mask(np.array([1, 0, 0, 0, 0, 1], bool), n), [1, 0, 0, 0, 0, 1])
    assert not selection_mask([], n).any() and not selection_mask(np.array([], np.int64), n).any()
    bad = [np.ones(5, bool), np.ones(7, bool), [6], [-1], [0, 9], np.array([0.0, 1.0]), np.array([1.5]),
           np.zeros((2, 3), np.int64), np.ones((1, 6), bool), 3, "abc", ["a"], [None], np.array([], np.float64)]
    sizes = [3, 0, 5, 1, 2, 4]
    db = ShardedKeyframeDatabase(sizes, [np.zeros((s, 32), np.uint8) for s in sizes], ops=PipelineOracleOps())
    q = np.zeros((3, 32), np.uint8)
    for b in bad:
        with pytest.raises(MatcherError):
            selection_mask(b, n)
        for call in (lambda: db.knn_tensors(q, 2, keyframes=b), lambda: db.knnMatch(q, 2, keyframes=b),
                     lambda: db.match_tensors(q, ratio=0.75, keyframes=b), lambda: db.match(q, keyframes=b),
                     lambda: db.match_device(torch.from_numpy(q), cross_check=True, keyframes=b),
                     lambda: db.knn2_keys_device(torch.from_numpy(q), keyframes=b)):
            with pytest.raises(MatcherError):
                call()


@pytest.fixture(scope="module")
def built():
    from slam_experiments_b200 import build as hm_build
    hm_build.build()
    return nat.lib()


def test_run_planning_covers_the_selected_tiles(built):
    """hm_describe_runs_launch: host arithmetic, no device -- the planned pieces are the selected tiles, in order"""
    rng = np.random.default_rng(1)
    cases = [np.array([[0, 1]]), np.array([[5, 9]]), np.array([[0, 300], [301, 391]]),
             np.array([[100, 200], [250, 260], [383, 385], [1000, 70000]])]
    for _ in range(30):
        nt = int(rng.integers(1, 400000))
        cuts = np.unique(rng.integers(0, nt + 1, int(rng.integers(2, 200))))
        runs = np.stack([cuts[:-1], cuts[1:]], 1)[::2]
        if runs.shape[0]:
            cases.append(runs)
    cases.append(np.stack([np.arange(0, 200000, 2), np.arange(1, 200001, 2)], 1))   # more pieces than SMs
    for runs in cases:
        runs = runs.astype(np.int64)
        nt = int(runs[-1, 1]) + 3
        for variant in ("i8", "f4"):
            for nq in (1, 2000, 4097):
                text, pieces = nat.describe_runs_launch(nq, nt, runs, variant, pieces=True)
                assert f"hm_{variant}_knn2_runs" in text
                tiles = -(-runs[:, 1] // 128) - runs[:, 0] // 128
                assert pieces.shape == (tiles.sum(), 4), text
                assert (np.diff(pieces[:, 0]) >= 0).all()                         # splits take consecutive tiles
                # every run's tiles in order; rows clipped to the run; together exactly the selected rows, ascending
                want = np.concatenate([np.arange(lo // 128, -(-hi // 128)) for lo, hi in runs])
                assert np.array_equal(pieces[:, 1], want)
                assert (pieces[:, 2] < pieces[:, 3]).all() and (pieces[:, 2] >= pieces[:, 1] * 128).all()
                assert (pieces[:, 3] <= pieces[:, 1] * 128 + 128).all()
                rows = np.concatenate([np.arange(a, b) for a, b in pieces[:, 2:]])
                assert np.array_equal(rows, np.concatenate([np.arange(a, b) for a, b in runs]))
                splits = int(text.split("grid=(")[1].split(",")[1])
                assert pieces[-1, 0] == splits - 1 and ("_floor" in text) == (splits > 1)
    # the workspace follows the selection, not the database
    few = np.array([[0, 1000]], np.int64)
    far = np.array([[8_000_000, 8_001_000]], np.int64)
    for prepared in (0, 1):
        assert nat.runs_workspace_bytes(2000, few, prepared, "f4") == nat.runs_workspace_bytes(2000, far, prepared, "f4") > 0
    assert nat.runs_workspace_bytes(2000, np.array([[0, 4000]]), 0, "popc") < 64 << 20


def test_run_lists_are_rejected_on_the_host(built):
    L = built
    for bad in ([[5, 5]], [[0, 10], [9, 20]], [[10, 20], [0, 5]], [[-1, 4]], [[0, 101]], [[3, 2]]):
        r = np.ascontiguousarray(bad, dtype=np.int64)
        assert L.hm_describe_runs_launch(10, 100, r.ctypes.data, r.shape[0], nat.VARIANT_F4, None, 0, None) == -1, bad
        if bad != [[0, 101]]:                                                   # (the workspace query has no nt)
            assert L.hm_runs_workspace_bytes(10, r.ctypes.data, r.shape[0], 0, 0) == 0, bad
        with pytest.raises(nat.NativeError):
            nat.describe_runs_launch(10, 100, r, "f4")
    r = np.array([[0, 10]], np.int64)
    assert L.hm_describe_runs_launch(10, 1 << 32, r.ctypes.data, 1, nat.VARIANT_F4, None, 0, None) == -1
    assert L.hm_describe_runs_launch(10, 100, None, 1, nat.VARIANT_F4, None, 0, None) == -1
    assert L.hm_describe_runs_launch(10, 100, None, 0, nat.VARIANT_F4, None, 0, None) == 0
    assert L.hm_describe_runs_launch(10, 100, r.ctypes.data, 1, nat.VARIANT_POPC, None, 0, None) == -1
    if not torch.cuda.is_available():                                           # no device: compute entry points fail
        q = np.zeros((4, 32), np.uint8)
        keys = np.zeros((4, 2), np.uint64)
        assert L.hm_knn2_runs(q.ctypes.data, 4, 32, q.ctypes.data, 4, 32, r.ctypes.data, r.ctypes.data, 1, 0,
                              keys.ctypes.data, 0, None, 0, None) == -5


# ---- gloo worlds with an oracle-backed stand-in --------------------------------------------------------------------
class SubsetOracleOps(PipelineOracleOps):
    """PipelineOracleOps plus the run hook: the oracle's top-2 over the gathered rows of the runs, mapped back."""

    def __init__(self):
        super().__init__()
        self.runs_log = []

    def local_knn2_runs(self, query, shard, train_base, runs):
        self.runs_log.append(runs.copy())
        bits = shard["bits"].numpy()
        rows = np.concatenate([np.arange(lo, hi) for lo, hi in runs])
        keys = ho.knn2_keys(query.numpy(), bits[rows])
        ok = keys != ho.NO_MATCH_KEY
        mapped = (keys & np.uint64(0xFFFF_FFFF_0000_0000)) + np.uint64(train_base) + rows[(keys & np.uint64(0xFFFFFFFF)).astype(np.int64) * ok].astype(np.uint64)
        return torch.from_numpy(np.where(ok, mapped, keys).view(np.int64))


def gloo_selections(n):
    return {"all": np.ones(n, bool), "none": [], "first": [0], "last": [n - 1], "first_last": [n - 1, 0, 0],
            "odd": np.arange(1, n, 2), "even": np.arange(0, n, 2), "kf4": [4], "no_rank2": [0, 3, 4],
            "tail": np.arange(n // 2, n)}


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from test_keyframe_db_pipeline import gloo_db
        sizes, kfs, q, _ = gloo_db()
        lo, hi, rlo, rhi = shard_ranges(sizes, world)[rank]
        ops = SubsetOracleOps()
        db = ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, ops=ops)
        out = {}
        for name, sel in gloo_selections(len(sizes)).items():
            for k in (1, 2):
                out[("knn", name, k)] = db.knn_tensors(q, k, keyframes=sel)
                rows = db.knnMatch(q, k, keyframes=sel)
                out[("dm", name, k)] = [[(m.queryIdx, m.imgIdx, m.trainIdx, int(m.distance)) for m in r] for r in rows]
            for ratio, cross in COMBOS:
                out[(name, ratio, cross)] = db.match_tensors(q, ratio=ratio, cross_check=cross, keyframes=sel)
        out["none_knn"] = db.knn_tensors(q, 2)
        out["grown"] = None
        db.append_keyframe(kfs[0][:3])
        out["grown"] = db.knn_tensors(q, 2, keyframes=[len(sizes)])
        ret[rank] = (out, (rlo, rhi), len(ops.runs_log))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_subset_matches_oracle(world):
    from test_keyframe_db_pipeline import gloo_db
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    sizes, kfs, q, _ = gloo_db()
    n = len(sizes)
    for name, sel in gloo_selections(n).items():
        for k in (1, 2):
            exp = knn_sub(q, kfs, sel, k)
            for r in range(world):
                assert same_knn(ret[r][0][("knn", name, k)], exp), (world, r, name, k)
                dm = ret[r][0][("dm", name, k)]
                assert len(dm) == q.shape[0]
                assert dm == [[(i, int(exp[0][i, j]), int(exp[1][i, j]), int(exp[2][i, j])) for j in range(exp[0].shape[1])]
                              for i in range(q.shape[0])], (world, r, name, k)
        for ratio, cross in COMBOS:
            exp = expected_sub(q, kfs, sel, ratio, cross)
            for r in range(world):
                assert same(ret[r][0][(name, ratio, cross)], exp), (world, r, name, ratio, cross)
    assert all(len(ret[r][0][("dm", "none", 2)][0]) == 0 for r in range(world))      # Nq empty tuples
    kfs2 = kfs + [kfs[0][:3]]
    for r in range(world):
        assert same_knn(ret[r][0]["grown"], knn_sub(q, kfs2, [n], 2)), r
    # the selection "no_rank2" holds rows on rank 0 only; world 3's last rank owns no keyframe: both join every exchange
    ranges = [ret[r][1] for r in range(world)]
    if world == 3:
        assert ranges[2][0] == ranges[2][1]


def test_single_rank_all_selected_equals_unselected():
    from test_keyframe_db_pipeline import gloo_db
    sizes, kfs, q, _ = gloo_db(5)
    db = ShardedKeyframeDatabase(sizes, kfs, ops=SubsetOracleOps())
    assert same_knn(db.knn_tensors(q, 2, keyframes=np.ones(len(sizes), bool)), db.knn_tensors(q, 2))
    for ratio, cross in COMBOS:
        assert same(db.match_tensors(q, ratio=ratio, cross_check=cross, keyframes=list(range(len(sizes)))),
                    db.match_tensors(q, ratio=ratio, cross_check=cross))
    one = db.match_tensors(q, ratio=0.75, keyframes=[0, 4])                    # 8 rows: the ratio test can pass
    assert same(one, expected_sub(q, kfs, [0, 4], 0.75, False))
    assert db.match_tensors(q, ratio=0.75, keyframes=[1, 2, 5])[0].size == 0  # no rows: nothing passes


# =====================================================================================================================
# GPU
# =====================================================================================================================
gpu = pytest.mark.gpu
VARIANTS = ("popc", "i8", "f4")


def collection(seed, sizes, hi=256):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, hi, (s, 32), dtype=np.uint8) for s in sizes], rng


# keyframe sizes chosen so that runs start and end inside tiles, two runs share a tile across a one-row keyframe
# (keyframes 0 and 2 around keyframe 1), keyframes have 1 row, a run is shorter than 8 columns (keyframe 9)
SHAPE_SIZES = [300, 1, 90, 1, 515, 0, 128, 127, 700, 5, 1, 2000, 3, 64]
SHAPE_SELECTIONS = {
    "single": [4], "first": [0], "last": [13], "first_last": [0, 13], "every_other": np.arange(0, 14, 2),
    "every_other_odd": np.arange(1, 14, 2), "shared_tile": [0, 2], "short_run": [9], "one_row": [1, 3, 10],
    "inside_tiles": [2, 7, 12], "all": np.ones(14, bool), "none": [], "all_but_last": np.arange(13),
}


def check_selection(db, q, kfs, sel, what, combos=True):
    for k in (1, 2):
        got = db.knn_tensors(q, k, keyframes=sel)
        assert same_knn(got, knn_sub(q, kfs, sel, k)), (what, k)
    if combos:
        for ratio, cross in COMBOS:
            assert same(db.match_tensors(q, ratio=ratio, cross_check=cross, keyframes=sel),
                        expected_sub(q, kfs, sel, ratio, cross)), (what, ratio, cross)


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_selection_shapes(variant):
    kfs, rng = collection(31, SHAPE_SIZES)
    cat = np.concatenate(kfs)
    q = rng.integers(0, 256, (600, 32), dtype=np.uint8)
    q[:300] = cat[rng.choice(cat.shape[0], 300, replace=False)] ^ (rng.integers(0, 16, (300, 32), dtype=np.uint8) == 0)
    db = ShardedKeyframeDatabase(SHAPE_SIZES, kfs, variant=variant)
    for name, sel in SHAPE_SELECTIONS.items():
        check_selection(db, q, kfs, sel, (variant, name))
    # "all selected" equals keyframes=None bit for bit
    qd = torch.from_numpy(q).cuda()
    a = db.knn2_keys_device(qd, keyframes=np.ones(len(kfs), bool)).cpu().numpy()
    assert np.array_equal(a, db.knn2_keys_device(qd).cpu().numpy())
    # tie-heavy low-entropy rows: the lowest global row inside the selection wins
    tie, rng = collection(32, SHAPE_SIZES, hi=3)
    tie[11][:300] = tie[0]
    qt = rng.integers(0, 3, (513, 32), dtype=np.uint8)
    dbt = ShardedKeyframeDatabase(SHAPE_SIZES, tie, variant=variant)
    for name in ("every_other", "shared_tile", "all_but_last", "inside_tiles", "one_row"):
        check_selection(dbt, qt, tie, SHAPE_SELECTIONS[name], (variant, "tie", name), combos=name == "every_other")


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_against_cv2_subcollection(variant):
    cv2 = pytest.importorskip("cv2")
    kfs, rng = collection(33, SHAPE_SIZES)
    q = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    q[:100] = np.concatenate(kfs)[rng.integers(0, sum(SHAPE_SIZES), 100)]
    db = ShardedKeyframeDatabase(SHAPE_SIZES, kfs, variant=variant)
    sizes = np.array(SHAPE_SIZES)
    for name in ("every_other", "shared_tile", "first_last", "inside_tiles", "all"):
        # cv2's collection is made of the selected keyframes that have rows (an empty image adds nothing)
        idx = np.array([i for i in sel_list(SHAPE_SELECTIONS[name], len(kfs)) if sizes[i] > 0])
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)
        bf.add([kfs[i] for i in idx])
        for k in (1, 2):
            got = db.knnMatch(q, k, keyframes=SHAPE_SELECTIONS[name])
            got = [[(m.queryIdx, m.imgIdx, m.trainIdx, m.distance) for m in r] for r in got]
            if sizes[idx].min() < k:
                # cv2's collection knnMatch returns uninitialised entries when an image has fewer than k rows
                # (DESIGN.md §1): the oracle over the concatenation is the reference there
                img, loc, d = knn_sub(q, kfs, SHAPE_SELECTIONS[name], k)
                exp = [[(i, int(img[i, j]), int(loc[i, j]), float(d[i, j])) for j in range(img.shape[1])]
                       for i in range(q.shape[0])]
            else:
                exp = [[(m.queryIdx, int(idx[m.imgIdx]), m.trainIdx, m.distance) for m in r] for r in bf.knnMatch(q, k=k)]
            assert exp == got, (variant, name, k)
    # cv2 masks= on the whole collection (every image has >= 2 rows, where whole-image masks are exact)
    big = [k for k in kfs if k.shape[0] >= 2]
    db2 = ShardedKeyframeDatabase([k.shape[0] for k in big], big, variant=variant)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    bf.add(big)
    sel = np.arange(len(big)) % 3 != 1
    masks = [np.full((q.shape[0], k.shape[0]), 255 if s else 0, np.uint8) for k, s in zip(big, sel)]
    ref = bf.knnMatch(q, k=2, masks=masks)
    got = db2.knnMatch(q, 2, keyframes=sel)
    assert [[(m.queryIdx, m.imgIdx, m.trainIdx, m.distance) for m in r] for r in ref] == \
        [[(m.queryIdx, m.imgIdx, m.trainIdx, m.distance) for m in r] for r in got], variant


@gpu
@pytest.mark.parametrize("variant", ("i8", "f4"))
def test_runs_across_splits(variant):
    """a big shard: the planner splits the walk over many CTAs, runs are cut at split boundaries, and the walk of
    every-other 64-row keyframes has more pieces than SMs"""
    sizes = [64] * 4000 + [1, 77, 129, 3]
    kfs, rng = collection(34, sizes)
    cat = np.concatenate(kfs)
    q = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    q[:1000] = cat[rng.integers(0, cat.shape[0], 1000)] ^ (rng.integers(0, 8, (1000, 32), dtype=np.uint8) == 0)
    db = ShardedKeyframeDatabase(sizes, kfs, variant=variant)
    for name, sel in (("every_other", np.arange(0, len(sizes), 2)), ("every_third", np.arange(0, len(sizes), 3)),
                      ("odd_tail", np.arange(1, len(sizes), 2)), ("all_but_64", np.arange(len(sizes) - 64))):
        runs = shard_runs(selection_mask(sel, len(sizes)), db.starts, 0, len(sizes), 0)
        text, pieces = nat.describe_runs_launch(2000, cat.shape[0], runs, variant, pieces=True)
        assert int(text.split("grid=(")[1].split(",")[1]) > 1, text
        check_selection(db, q, kfs, sel, (variant, name), combos=name == "every_other")
    assert pieces.shape[0] > 148


_CLUSTER_CHILD = r'''
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from test_keyframe_db_subset import collection, check_selection, SHAPE_SIZES, SHAPE_SELECTIONS
from slam_experiments_b200.keyframe_db import ShardedKeyframeDatabase
sizes = SHAPE_SIZES * 40
kfs, rng = collection(35, sizes)
q = rng.integers(0, 256, (700, 32), dtype=np.uint8)
q[:300] = np.concatenate(kfs)[rng.integers(0, sum(sizes), 300)]
for variant in ("i8", "f4"):
    db = ShardedKeyframeDatabase(sizes, kfs, variant=variant)
    for sel in (np.arange(0, len(sizes), 2), np.arange(len(sizes)) % 14 == 2, [0, 2, 555]):
        check_selection(db, q, kfs, sel, (variant, "cluster"), combos=False)
print("CLUSTER OK")
'''


@gpu
def test_cluster_pairs_share_run_tiles():
    env = dict(os.environ, HM_I8_CLUSTER="2")
    r = subprocess.run([sys.executable, "-c", _CLUSTER_CHILD, ROOT], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "CLUSTER OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


@gpu
@pytest.mark.parametrize("variant", VARIANTS)
def test_growth_then_select_the_new_keyframe(variant):
    sizes = [300, 90, 1, 515]
    kfs, rng = collection(36, sizes + [200, 1, 70000])
    q = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    q[:200] = np.concatenate(kfs)[rng.integers(0, sum(k.shape[0] for k in kfs), 200)]
    db = ShardedKeyframeDatabase(sizes, kfs[:4], variant=variant)
    for i in range(4, len(kfs)):
        assert db.append_keyframe(kfs[i]) == i
        check_selection(db, q, kfs[:i + 1], [i], (variant, "new", i), combos=False)
        check_selection(db, q, kfs[:i + 1], [0, i], (variant, "first+new", i), combos=i == len(kfs) - 1)


@gpu
def test_per_call_memory_does_not_grow_with_unselected_rows():
    rng = np.random.default_rng(37)
    q = torch.from_numpy(rng.integers(0, 256, (2000, 32), dtype=np.uint8)).cuda()
    for variant in ("f4", "popc"):
        peaks = []
        for n_kf in (20, 600):
            kfs = [rng.integers(0, 256, (1000, 32), dtype=np.uint8) for _ in range(n_kf)]
            db = ShardedKeyframeDatabase([1000] * n_kf, kfs, variant=variant)
            sel = [0, 3, 7, n_kf - 1]
            db.match_device(q, ratio=0.75, cross_check=True, keyframes=sel)       # warm the cached workspaces
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            out = db.match_device(q, ratio=0.75, cross_check=True, keyframes=sel)
            torch.cuda.synchronize()
            peaks.append(torch.cuda.max_memory_allocated() - base)
            del out, db
        assert peaks[0] == peaks[1], (variant, peaks)


# ---- full C4: the three databases of the full-size pipeline tests ----------------------------------------------------
C4_SELECTIONS = {"all_but_last_64": np.arange(4096 - 64), "every_third": np.arange(0, 4096, 3)}


@pytest.fixture(scope="module", params=("uniform", "dups", "lowentropy"))
def c4_subset_case(request):
    from oracle import c_oracle as co
    from test_keyframe_db_pipeline import _c4_database
    q, t = _c4_database(request.param)
    exp = {}
    for name, sel in C4_SELECTIONS.items():
        rows = np.concatenate([np.arange(k * 2000, (k + 1) * 2000) for k in sel])
        keys = co.knn2_keys(q, t[rows])
        ok = keys != ho.NO_MATCH_KEY
        exp[name] = np.where(ok, (keys & np.uint64(0xFFFF_FFFF_0000_0000)) + rows[(keys & np.uint64(0xFFFFFFFF)).astype(np.int64)].astype(np.uint64), keys)
    return request.param, q, t, exp


@gpu
def test_full_c4_subsets_all_rows(c4_subset_case):
    from test_keyframe_db_pipeline import _c4_db
    kind, q, t, exp = c4_subset_case
    qd = torch.from_numpy(q).cuda()
    for variant in ("f4", "i8") if kind == "uniform" else ("f4",):
        db = _c4_db(t, variant)
        for name, sel in C4_SELECTIONS.items():
            got = db.knn2_keys_device(qd, keyframes=sel).cpu().numpy().view(np.uint64)
            assert np.array_equal(got, exp[name]), (kind, variant, name, int((got != exp[name]).any(1).sum()))
        a = db.knn2_keys_device(qd, keyframes=np.ones(4096, bool)).cpu().numpy()
        assert np.array_equal(a, db.knn2_keys_device(qd).cpu().numpy()), (kind, variant)
        if kind == "uniform" and variant == "f4":
            for it in range(30):
                got = db.knn2_keys_device(qd, keyframes=C4_SELECTIONS["all_but_last_64"]).cpu().numpy().view(np.uint64)
                assert np.array_equal(got, exp["all_but_last_64"]), it
        del db
