"""The matching pipeline (knnMatch k=2 -> Lowe's ratio test -> mutual check, and cv2's k=1 ``match()``) at the edges
where its device pieces go wrong, bit-exact against the oracle.

The pieces under test, beyond the k-NN keys that tests/test_gpu_parity.py covers:
  - the top-1 kernels (scan mode 2) of the forward ``match()`` pass and of every swapped pass, which have no shared
    row thresholds, so ties across groups, tiles and splits are resolved by the scan and the merge alone;
  - the ratio test + candidate selection in the k-NN tail (``select_candidate``: slot table, count, list);
  - the candidate pass of the kind::mxf4 mutual check (rows gathered through the candidate list, row count read from
    device memory, clusters past the count return early) and the filter that reads it through ``slot_of``;
  - the single-launch small-problem kernel (hm_small.cu) at its size limits, and the graph path one step past them.

Every case compares q, t, d and the count of every problem with oracle/c_oracle.py (or the goldens the reference
wrote).  The candidate-count recipe itself is checked on the CPU with the numpy oracle.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden, pair_goldens
from oracle import c_oracle as co
from oracle import hamming_oracle as ho

VARIANTS = ("popc", "i8", "f4")
NO_MATCH = np.uint64(0xFFFFFFFFFFFFFFFF)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def expected(q, t, ratio=None, cross=False, thr=None):
    """(q, t, d) of the fused pipeline: ratio test, mutual check, then the reference's distance filter
    ``d < max(2 * min_d, thr)`` where min_d is the smallest forward distance over ALL query rows."""
    eq, et, ed = co.pipeline(q, t, ratio=ratio, cross_check=cross)
    if thr and q.shape[0] and t.shape[0]:
        d1 = (co.knn2_keys(q, t)[:, 0] >> np.uint64(32)).astype(np.int64)
        keep = ed.astype(np.float64) < max(2 * float(d1.min()), float(thr))
        eq, et, ed = eq[keep], et[keep], ed[keep]
    return eq, et, ed


def device_match(qs, ts, variant, ratio=None, cross=False, thr=None, want_keys=False):
    """``nat.match_fused`` on ``[B, n, 32]`` host arrays; returns one (q, t, d) per problem (and the keys)."""
    import torch
    from slam_experiments_b200 import _native as nat
    qd = torch.from_numpy(np.ascontiguousarray(qs)).cuda()
    td = torch.from_numpy(np.ascontiguousarray(ts)).cuda()
    res = nat.match_fused(qd, td, ratio=ratio, cross_check=cross, dist_threshold=thr, variant=variant,
                          want_keys=want_keys)
    oq, ot, od, cnt = (x.cpu().numpy() for x in res[:4])
    out = [(oq[b, :cnt[b]], ot[b, :cnt[b]], od[b, :cnt[b]]) for b in range(qs.shape[0])]
    if want_keys:
        return out, res[4].cpu().numpy().view(np.uint64)
    return out


def assert_same(got, exp, what):
    gq, gt, gd = got
    eq, et, ed = exp
    assert len(gq) == len(eq), f"{what}: {len(gq)} matches, oracle {len(eq)}"
    bad = np.flatnonzero((gq != eq) | (gt != et) | (gd != ed))
    assert bad.size == 0, f"{what}: {bad.size} of {len(eq)} matches differ, first at {bad[:5]}: " \
                          f"got {list(zip(gq[bad[:3]], gt[bad[:3]], gd[bad[:3]]))}, " \
                          f"oracle {list(zip(eq[bad[:3]], et[bad[:3]], ed[bad[:3]]))}"


def check_fused(q, t, variant, ratio=None, cross=False, thr=None, what=""):
    got = device_match(q[None], t[None], variant, ratio, cross, thr)[0]
    assert_same(got, expected(q, t, ratio, cross, thr), f"{what} {variant} ratio={ratio} cross={cross} thr={thr}")


def launch_grid(nq, nt, batch, variant):
    """(query blocks, splits, cluster) that the k-NN launch of an nq x nt problem gets."""
    from slam_experiments_b200 import _native as nat
    s = nat.describe_launch(nq, nt, batch, variant)
    m = re.search(r"grid=\((\d+),(\d+),(\d+)\) cluster=(\d+)", s)
    assert m, s
    return int(m.group(1)), int(m.group(2)), int(m.group(4))


def flip_bits(row, bits):
    out = row.copy()
    for b in bits:
        out[b >> 3] ^= np.uint8(1 << (b & 7))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# (a) the reference's goldens through the device pipeline, every core
# ---------------------------------------------------------------------------------------------------------------------
def _golden_keys(knn2):
    """[nq, 2] packed keys from the golden knn2 rows (queryIdx, trainIdx, imgIdx, distance); -1 rows are missing."""
    keys = np.full(knn2.shape[:2], NO_MATCH, np.uint64)
    ok = knn2[:, :, 0] >= 0
    keys[ok] = (knn2[:, :, 3][ok].astype(np.uint64) << np.uint64(32)) | knn2[:, :, 1][ok].astype(np.uint64)
    return keys


GOLDEN_CASES = [("ref_match", None, False, None), ("ref_match_thr30", None, False, 30.0),
                ("ref_match_thr64", None, False, 64.0), ("cross", None, True, None)] + \
               [(f"{kind}{r}", r / 100.0, kind == "pipe", None) for r in (70, 75, 80) for kind in ("ratio", "pipe")]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("path", pair_goldens(), ids=[os.path.basename(p)[:-4] for p in pair_goldens()])
def test_goldens_through_device_pipeline(path, variant):
    """``match_fused`` honours the variant at every size, so the tie-heavy small goldens reach the tensor-core top-1
    kernels, the candidate selection and the candidate pass.  With ``want_keys`` the forward pass is the k=2 kernel and
    its keys must equal the golden knnMatch(k=2)."""
    g = load_golden(path)
    q, t = g["query"][None], g["train"][None]
    gkeys = _golden_keys(g["knn2"])
    for name, ratio, cross, thr in GOLDEN_CASES:
        exp = g[name]
        exp = (exp[:, 0].astype(np.int32), exp[:, 1].astype(np.int32), exp[:, 3].astype(np.int32))
        assert_same(device_match(q, t, variant, ratio, cross, thr)[0], exp, f"{name} {variant}")
        got, keys = device_match(q, t, variant, ratio, cross, thr, want_keys=True)
        assert_same(got[0], exp, f"{name} {variant} want_keys")
        assert np.array_equal(keys[0], gkeys), f"{name} {variant}: keys differ from the golden knnMatch(k=2)"


# ---------------------------------------------------------------------------------------------------------------------
# (b) exact candidate counts
# ---------------------------------------------------------------------------------------------------------------------
CAND_NQ, CAND_NT = 20000, 3000
CAND_KS = (0, 1, 2, 255, 256, 257, 511, 512, 513, 767, 768, 769)
EDGE_KS = (1, 2, 255, 256, 257, 511, 512, 513, 769)           # the 256-row block edges, run again under clusters


def candidate_problem(k, seed=0, nq=CAND_NQ, nt=CAND_NT):
    """Exactly ``k`` train rows become candidates of the ratio test (0.75) and exactly ``k`` mutual matches survive.

    Train rows are uniform and row nt-1 is a copy of row 0; every filler query is a copy of row 0, so its two best
    distances are 0 and 0 and it fails the ratio test.  ``k`` queries are copies of ``k`` distinct other train rows
    (distance 0, second best ~90: they pass), and a few of them are copied again to other query indices, so some
    candidates are named by several rows.  Without the ratio test every row names a candidate: ``k + 1`` of them."""
    rng = np.random.default_rng(1000 * seed + k)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    t[nt - 1] = t[0]
    q = np.repeat(t[:1], nq, axis=0)
    rows = rng.choice(np.arange(1, nt - 1), k, replace=False)
    extra = min(k, 7)
    pos = rng.choice(nq, k + extra, replace=False)
    q[pos[:k]] = t[rows]
    if extra:
        q[pos[k:]] = t[rows[rng.integers(0, k, extra)]]
    return q, t


def candidate_edge_problem(nt, nq=CAND_NQ, seed=5):
    """Without the ratio test every train row that is some query's best is a candidate: here all ``nt`` of them (the
    first nt queries are copies of the train rows, the others uniform)."""
    rng = np.random.default_rng(seed + nt)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    q[rng.permutation(nq)[:nt]] = t
    return q, t


def _recipe_oracle(q, t, ratio, mutual=True):
    """Candidate count (distinct best train rows of the ratio survivors) and mutual matches from the numpy oracle,
    computed on the distinct query rows and expanded to all of them."""
    uq, inv = np.unique(q, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    idx, dist = ho.knn(uq, t, 2)
    idx, dist = idx[inv], dist[inv]
    keep = ho.ratio_test(idx, dist, ratio) if ratio is not None else np.ones(q.shape[0], bool)
    candidates = np.unique(idx[keep, 0]).size
    if not mutual:
        return candidates
    best_query = np.argmin(ho.hamming_matrix(uq, t).astype(np.uint16)[inv], axis=0)   # lowest index on ties
    return candidates, int((keep & (best_query[idx[:, 0]] == np.arange(q.shape[0]))).sum())


@pytest.mark.parametrize("k", CAND_KS)
def test_candidate_recipe_counts(k):
    """CPU: the inputs of the candidate-count tests really produce k candidates and k mutual matches (k + 1 candidates
    without the ratio test), so the device tests below cannot drift off the block edges they are meant to hit."""
    q, t = candidate_problem(k)
    assert _recipe_oracle(q, t, 0.75) == (k, k)
    assert _recipe_oracle(q, t, None, mutual=False) == k + 1
    if k in (257, 513, 769):
        q, t = candidate_edge_problem(k)
        assert _recipe_oracle(q, t, None, mutual=False) == k


def _run_candidate_cases(ks):
    """Ratio 0.75 + mutual check on the kind::mxf4 core for every k, the mutual check alone (k + 1 candidates), the
    shapes where every train row is a candidate, and one batched launch with k = 0, 257, 1, 513."""
    for k in ks:
        q, t = candidate_problem(k)
        exp = co.pipeline(q, t, 0.75, True)
        assert len(exp[0]) == k
        assert_same(device_match(q[None], t[None], "f4", 0.75, True)[0], exp, f"k={k}")
        check_fused(q, t, "f4", None, True, what=f"k={k} ({k + 1} candidates)")
    for nt in (257, 513, 769):
        q, t = candidate_edge_problem(nt)
        check_fused(q, t, "f4", None, True, what=f"all {nt} train rows candidates")
    ks_b = (0, 257, 1, 513)
    probs = [candidate_problem(k, seed=3) for k in ks_b]
    qs, ts = np.stack([p[0] for p in probs]), np.stack([p[1] for p in probs])
    got = device_match(qs, ts, "f4", 0.75, True)
    for b, k in enumerate(ks_b):
        exp = co.pipeline(qs[b], ts[b], 0.75, True)
        assert len(exp[0]) == k
        assert_same(got[b], exp, f"batched problem {b} (k={k})")


@pytest.mark.gpu
def test_candidate_counts_at_block_edges():
    """Ratio 0.75 + mutual check on the kind::mxf4 core with exactly k candidates, k at and around the 256-row blocks of
    the candidate pass (0: no candidate at all; 257: a second block with one row), without the ratio test (k + 1
    candidates, and shapes where every train row is one), and one batched launch with k = 0, 257, 1, 513."""
    qb, splits, _ = launch_grid(CAND_NT, CAND_NQ, 1, "f4")          # candidate pass: nt rows x nq columns
    assert splits > 1 and qb >= 4, (qb, splits)
    _run_candidate_cases(CAND_KS)


def _cluster_child():
    """Body of the child process of test_candidate_pass_in_cluster_pairs (HM_I8_CLUSTER=2 is read once per process)."""
    _, _, cluster = launch_grid(CAND_NT, CAND_NQ, 1, "f4")
    assert cluster == 2, "HM_I8_CLUSTER=2 did not force cluster pairs"
    _run_candidate_cases(EDGE_KS)
    print("cluster-pair candidate cases ok")


@pytest.mark.gpu
def test_candidate_pass_in_cluster_pairs():
    """The block-edge cases again with every tensor-core launch in clusters of two query blocks.  With k = 1, 2, 255,
    256 or 513 the last cluster that holds candidates has one CTA with rows and one without; with k = 512 a whole
    cluster is past the count and returns before its first cluster barrier."""
    code = ("import sys; sys.path[:0] = [{!r}, {!r}]; import test_pipeline_edges as m; m._cluster_child()"
            .format(ROOT, os.path.join(ROOT, "tests")))
    env = dict(os.environ, HM_I8_CLUSTER="2")
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"child exited with {r.returncode}\n{r.stdout[-3000:]}\n{r.stderr[-6000:]}"
    assert "cluster-pair candidate cases ok" in r.stdout


# ---------------------------------------------------------------------------------------------------------------------
# (d) ties in the swapped pass
# ---------------------------------------------------------------------------------------------------------------------
def swapped_tie_problem(seed=11, nq=CAND_NQ, nt=CAND_NT):
    """Many queries equidistant from one train row -- at distance 0 (exact copies) and at distance 3 (three different
    bits flipped each) -- in the same 8-column group, in other groups of the same 128-column tile, and in other tiles
    and splits of the swapped pass.  Only the lowest of those query indices is that train row's best query."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    j0, j1 = 17, nt - 5
    at0 = np.array([5, 6, 13, 100, 127, 200, 208, 255, 4000, 12345, nq - 1])
    at3 = np.array([131, 139, 140, 191, 255 + 128, 640, 9000, 19000])
    q[at0] = t[j0]
    for i, a in enumerate(at3):
        q[a] = flip_bits(t[j1], (3 * i, 3 * i + 100, 3 * i + 200))
    return q, t, (j0, int(at0.min())), (j1, int(at3.min()))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ("f4", "i8"))
def test_swapped_pass_ties(variant):
    q, t, (j0, q0), (j1, q1) = swapped_tie_problem()
    _, splits, _ = launch_grid(t.shape[0], q.shape[0], 1, variant)
    assert splits > 1
    for ratio in (0.75, None):
        exp = expected(q, t, ratio, True)
        pairs = set(zip(exp[0].tolist(), exp[1].tolist()))
        assert (q0, j0) in pairs and (q1, j1) in pairs                  # the lowest tied query index wins
        assert sum(tt in (j0, j1) for tt in exp[1].tolist()) == 2
        check_fused(q, t, variant, ratio, True, what="swapped-pass ties")


def low_entropy_problem(seed=12, nq=CAND_NQ, nt=CAND_NT):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 3, (nq, 32), dtype=np.uint8), rng.integers(0, 3, (nt, 32), dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ("f4", "i8"))
@pytest.mark.parametrize("kind", ("lowentropy", "alleq"))
def test_tie_heavy_pipeline_at_split_size(variant, kind):
    """Bytes in {0, 1, 2} (a handful of distinct distances, ties everywhere) and all-equal rows (every pair ties) at a
    size where the swapped pass splits its columns: mutual check alone, with ratio 0.9, and the k=1 ``match()`` path with
    the distance filter."""
    q, t = low_entropy_problem()
    if kind == "alleq":
        q[:], t[:] = 0x5A, 0x5A
    for ratio, cross, thr in ((None, True, None), (0.9, True, None), (None, False, 30.0), (None, False, 64.5)):
        check_fused(q, t, variant, ratio, cross, thr, what=kind)


# ---------------------------------------------------------------------------------------------------------------------
# (e) forward top-1 (cv2 match()) at split-launch size
# ---------------------------------------------------------------------------------------------------------------------
def forward_split_problems(nq, nt=40000, seed=77):
    """The tie-heavy inputs of test_split_launch_shared_row_thresholds for nq queries against 40000 train rows."""
    rng = np.random.default_rng(seed + nq)
    t = np.zeros((nt, 32), np.uint8)
    t[:, 5] = rng.integers(0, 4, nt)
    q = np.zeros((nq, 32), np.uint8)
    q[:, 5] = rng.integers(0, 4, nq)
    yield "one varying byte", q, t
    yield "bytes in {0,1,2}", rng.integers(0, 3, (nq, 32), dtype=np.uint8), rng.integers(0, 3, (nt, 32), dtype=np.uint8)
    yield "all train rows equal", q, np.full((nt, 32), 0x5A, np.uint8)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    where = rng.choice(nt, (3, nq), replace=False)
    for w in where:                                       # exact copies of every query early, in the middle and late
        t[w] = q
    yield "three planted copies", q, t


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ("f4", "i8"))
@pytest.mark.parametrize("nq", (300, 1, 64, 257))
def test_forward_top1_at_split_size(variant, nq):
    """cv2 ``match()`` (k = 1, no ratio, no mutual check, dist_threshold None / 30 / 64.5) runs the top-1 kernel, which
    has no shared row floors: the nearest train row of every query over many splits, ties to the lowest index."""
    _, splits, _ = launch_grid(nq, 40000, 1, variant)
    assert splits > 1
    for label, q, t in forward_split_problems(nq):
        for thr in (None, 30.0, 64.5):
            check_fused(q, t, variant, None, False, thr, what=f"{label} nq={nq}")


# ---------------------------------------------------------------------------------------------------------------------
# (f) tiny query side: the swapped pass has one ragged column tile
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("variant", ("f4", "i8"))
@pytest.mark.parametrize("nt", (300, 40000))
@pytest.mark.parametrize("nq", (1, 2, 127, 129))
def test_tiny_query_side(nq, nt, variant):
    """nq of 1, 2, 127 and 129 queries: the swapped pass (nt rows x nq columns) has a single, ragged column tile whose
    padding columns must never win.  Matchable queries with a duplicated query row (a tie in the swapped pass), and
    train rows that are all farther than 128 from every query (a padding column would be nearer)."""
    from slam_experiments_b200 import synth
    rng = np.random.default_rng(nq * 7 + nt)
    t = rng.integers(0, 256, (nt, 32), dtype=np.uint8)
    q = synth.matchable_queries(t, nq, nq + nt, flip_p=0.05, frac=0.8)
    if nq >= 2:
        q[nq - 1] = q[0]
    for ratio, cross in ((0.75, True), (None, True), (0.8, False)):
        check_fused(q, t, variant, ratio, cross, what=f"matchable {nq}x{nt}")
    far = (~q[rng.integers(0, nq, nt)]) ^ rng.integers(0, 2, (nt, 32), dtype=np.uint8)
    check_fused(q, far, variant, None, True, what=f"far {nq}x{nt}")


# ---------------------------------------------------------------------------------------------------------------------
# (g) the single-launch small-problem kernel at its eligibility edges, and the graph path one step past them
# ---------------------------------------------------------------------------------------------------------------------
SMALL_SHAPES = [(1024, 256), (256, 1024), (1024, 1), (1, 1024), (513, 511), (512, 512),
                (1025, 200), (1024, 257)]                      # the last two are past the limits: graph path
FLAG_SETS = [(ratio, cross, thr) for ratio in (None, 0.8) for cross in (False, True) for thr in (None, 12.5)]


def small_problem(nq, nt, seed):
    """Tie-heavy rows (bytes in {0, 1, 2}); half the queries are train rows with at most one bit flipped, and a few train
    rows are duplicated, so the ratio test, the mutual check and the distance filter all keep and drop rows."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 3, (nt, 32), dtype=np.uint8)
    q = rng.integers(0, 3, (nq, 32), dtype=np.uint8)
    if nt >= 4:
        t[rng.integers(0, nt, nt // 4)] = t[rng.integers(0, nt, nt // 4)]
    m = (nq + 1) // 2
    if m:
        q[:m] = t[rng.integers(0, nt, m)]
        q[:m:2, 7] ^= 1
    return q, t


@pytest.mark.gpu
@pytest.mark.parametrize("nq,nt", SMALL_SHAPES)
def test_small_kernel_edges_through_host_context(nq, nt):
    """``HostContext.match`` / ``frame_match``: AUTO takes hm_small.cu up to 1024 rows a side and 262144 pairs and the
    graph path beyond; an explicit core runs that core at every size.  Every flag combination, twice (the second call of
    a shape on the graph path is captured, later ones replay)."""
    from slam_experiments_b200 import _native as nat
    q, t = small_problem(nq, nt, nq * 31 + nt)
    ctx = nat.HostContext()
    try:
        ctx.frame_put(0, t)
        ctx.frame_put(1, q)
        for ratio, cross, thr in FLAG_SETS:
            exp = expected(q, t, ratio, cross, thr)
            for variant in ("auto", "popc", "i8", "f4"):
                what = f"{nq}x{nt} {variant} ratio={ratio} cross={cross} thr={thr}"
                for _ in range(2):
                    assert_same(ctx.match(q, t, ratio=ratio, cross_check=cross, dist_threshold=thr, variant=variant),
                                exp, what)
                assert_same(ctx.frame_match(0, 1, nq, ratio=ratio, cross_check=cross, dist_threshold=thr,
                                            variant=variant), exp, "frame " + what)
    finally:
        ctx.close()
