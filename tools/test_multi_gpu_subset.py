"""Multi-GPU parity of keyframe selections (``keyframes=``) in the keyframe database (run under torchrun, one rank per
GPU; tests/test_multi_gpu_subset.py spawns it when >= 2 GPUs are visible).  Every rank's k-NN result and match list must
equal the oracle over the concatenation of the selected keyframes, for both exchange modes and every core, including a
selection in which some rank owns no selected row, a selection that is empty on every rank, and a selection of
keyframes on shard boundaries."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
import slam_experiments_b200 as sx
from oracle import c_oracle
from oracle.hamming_oracle import NO_MATCH_KEY

COMBOS = ((None, False), (0.75, False), (None, True), (0.75, True))


def check(db, q, kfs, sel, rank, what):
    idx = np.flatnonzero(sx.keyframe_db.selection_mask(sel, len(kfs)))
    starts = db.starts
    rows = np.concatenate([np.arange(starts[i], starts[i + 1]) for i in idx] + [np.empty(0, np.int64)]).astype(np.int64)
    cat = np.concatenate(kfs)
    sub = cat[rows]
    good = True
    keys = c_oracle.knn2_keys(q, sub) if q.shape[0] else np.empty((0, 2), np.uint64)
    mapped = np.where(keys != NO_MATCH_KEY, (keys & np.uint64(0xFFFFFFFF00000000)) +
                      rows[(keys & np.uint64(0xFFFFFFFF)).astype(np.int64) * (keys != NO_MATCH_KEY)].astype(np.uint64), keys)
    if q.shape[0]:
        got = db.knn2_keys_device(torch.from_numpy(q).cuda(), keyframes=sel).cpu().numpy().view(np.uint64)
        good &= bool(np.array_equal(got, mapped))
        img, loc, d = db.knn_tensors(q, 2, keyframes=sel)
        kk = min(2, rows.size)
        g = (mapped[:, :kk] & np.uint64(0xFFFFFFFF)).astype(np.int64)
        good &= img.shape == (q.shape[0], kk) and bool(np.array_equal(starts[img] + loc, g))
    for ratio, cross in COMBOS:
        if sub.shape[0] and q.shape[0]:
            eq, et, ed = c_oracle.pipeline(q, sub, ratio, cross)
        else:
            eq = et = ed = np.empty(0, np.int32)
        qi, gi, gl, gd = db.match_tensors(q, ratio=ratio, cross_check=cross, keyframes=sel)
        ok = (np.array_equal(qi, eq) and np.array_equal(starts[gi] + gl, rows[et]) and np.array_equal(gd, ed))
        if not ok:
            print(f"rank {rank} {what} nq {q.shape[0]} ratio {ratio} cross {cross}: MISMATCH "
                  f"({len(qi)} vs {len(eq)} matches)", flush=True)
        good &= ok
    if not good:
        print(f"rank {rank} {what}: FAILED", flush=True)
    return good


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rng = np.random.default_rng(12)
    ok = True
    W = dist.group.WORLD
    nkf = 31
    sizes = rng.integers(1, 3000, nkf).tolist()
    sizes[5] = 1
    kfs = [rng.integers(0, 3, (s, 32), dtype=np.uint8) for s in sizes]
    kfs[25][:7] = kfs[2][:7]
    cat = np.concatenate(kfs)
    ranges = sx.shard_ranges(sizes, world)
    lo, hi, _, _ = ranges[rank]
    boundary = sorted({k for a, b, _, _ in ranges if b > a for k in (a, b - 1)})
    selections = {
        "first_rank_only": list(range(ranges[0][0], ranges[0][1])),      # every other rank owns no selected row
        "last_kf": [nkf - 1],
        "empty": [],
        "every_other": np.arange(0, nkf, 2),
        "boundaries": boundary,
        "all": np.ones(nkf, bool),
    }
    for mode, variant in (("fused", "f4"), ("fused", "i8"), ("fused", "popc"), ("nccl", "f4"), ("nccl", "i8"),
                          ("nccl", "popc")):
        db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange=mode,
                                        variant=variant)
        for name, sel in selections.items():
            for nq in (700, 1, 0):
                q = rng.integers(0, 3, (nq, 32), dtype=np.uint8)
                q[: nq // 2] = cat[rng.integers(0, cat.shape[0], nq // 2)]
                ok &= check(db, q, kfs, sel, rank, f"{mode}/{variant}/{name}")
        # a selection call and an unselected call share the exchange's epochs
        q = cat[rng.integers(0, cat.shape[0], 300)]
        ok &= bool(np.array_equal(db.knn2_keys_device(torch.from_numpy(q).cuda()).cpu().numpy(),
                                  db.knn2_keys_device(torch.from_numpy(q).cuda(), keyframes=np.ones(nkf, bool)).cpu().numpy()))
    # mixed shards under "auto": prepared and packed ranks, and a selection that leaves the prepared rank out
    sizes = [70000, 60000] + [900] * 3
    kfs = [rng.integers(0, 256, (s, 32), dtype=np.uint8) for s in sizes]
    lo, hi, _, _ = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange="fused",
                                    variant="auto")
    q = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    q[:200] = np.concatenate(kfs)[rng.integers(0, sum(sizes), 200)]
    for name, sel in (("big", [0, 1]), ("small", [2, 3, 4]), ("mixed", [1, 3])):
        ok &= check(db, q, kfs, sel, rank, f"mixed/{name}")

    t = torch.tensor([int(ok)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_SUBSET", "OK" if int(t) == 1 else "FAILED", f"world={world}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(t) == 1 else 1)


if __name__ == "__main__":
    main()
