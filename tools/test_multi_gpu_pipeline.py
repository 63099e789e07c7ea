"""Multi-GPU parity of the keyframe database's ratio test + mutual check (run under torchrun, one rank per GPU;
tests/test_multi_gpu_pipeline.py spawns it when >= 2 GPUs are visible).  Every rank's match list must equal the oracle
over the concatenated database, for every option combination: homogeneous shards of every core under both k-NN
exchange modes, mixed prepared / unprepared shards, a rank without rows, query rows whose best row sits on a shard
boundary or is duplicated on another shard, and a database grown with append_keyframe."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
import slam_experiments_b200 as sx
from oracle import c_oracle

COMBOS = ((None, False), (0.75, False), (None, True), (0.75, True))


def check(db, q, cat, rank, what):
    starts = db.starts
    good = True
    for ratio, cross in COMBOS:
        eq, et, ed = c_oracle.pipeline(q, cat, ratio, cross) if cat.shape[0] else (np.empty(0, np.int32),) * 3
        img = (np.searchsorted(starts, et, side="right") - 1).astype(np.int32)
        qi, gi, gl, gd = db.match_tensors(q, ratio=ratio, cross_check=cross)
        ok = (np.array_equal(qi, eq) and np.array_equal(gi, img) and np.array_equal(gl, et - starts[img])
              and np.array_equal(gd, ed))
        if not ok:
            print(f"rank {rank} {what} nq {q.shape[0]} ratio {ratio} cross {cross}: MISMATCH "
                  f"({len(qi)} vs {len(eq)} matches)", flush=True)
        good &= ok
    return good


def boundary_queries(rng, kfs, sizes, world, nq, hi=256):
    """queries whose best row is the first / last row of every shard, plus random ones"""
    cat = np.concatenate(kfs)
    rows = sorted({r for _, _, lo, h in sx.shard_ranges(sizes, world) if h > lo for r in (lo, h - 1)})
    q = rng.integers(0, hi, (nq, 32), dtype=np.uint8)
    k = min(nq, len(rows))
    q[:k] = cat[rows[:k]]
    return q


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rng = np.random.default_rng(11)
    ok = True
    W = dist.group.WORLD

    # ---- homogeneous shards, every core, both exchange modes; tie-heavy rows, cross-shard duplicates ------------
    nkf = 29
    sizes = rng.integers(50, 3000, nkf).tolist()
    kfs = [rng.integers(0, 3, (s, 32), dtype=np.uint8) for s in sizes]
    kfs[25][:7] = kfs[2][:7]                                  # duplicates on another shard: the lower global row wins
    cat = np.concatenate(kfs)
    lo, hi, _, _ = sx.shard_ranges(sizes, world)[rank]
    for mode, variant in (("fused", "f4"), ("fused", "i8"), ("fused", "popc"), ("nccl", "f4"), ("nccl", "i8"),
                          ("nccl", "popc")):
        db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange=mode,
                                        variant=variant)
        for nq in (700, 1, 2000, 0, 129):
            q = boundary_queries(rng, kfs, sizes, world, nq, hi=3)
            q[len(q) // 2: len(q) // 2 + min(nq, 7)] = kfs[2][: min(nq - len(q) // 2, 7)]
            ok &= check(db, q, cat, rank, f"homogeneous {mode}/{variant}")

    # ---- mixed shards under variant="auto": prepared (>= 65536 rows) and packed-bits shards; at world > 3 empty ranks
    sizes = [70000, 60000] + [900] * 3
    kfs = [rng.integers(0, 256, (s, 32), dtype=np.uint8) for s in sizes]
    kfs[4][:30] = kfs[0][:30]
    cat = np.concatenate(kfs)
    lo, hi, rlo, rhi = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange="fused",
                                    variant="auto")
    kinds = [None] * world
    dist.all_gather_object(kinds, (rhi - rlo, db.shard["prepared"] is not None))
    if rank == 0:
        print(f"mixed: (rows, prepared) per rank = {kinds}", flush=True)
    ok &= len({k[1] for k in kinds}) == 2
    for nq in (2000, 1, 4096):
        q = boundary_queries(rng, kfs, sizes, world, nq)
        q[-min(nq, 50):] = cat[rng.choice(cat.shape[0], min(nq, 50), replace=False)]
        ok &= check(db, q, cat, rank, "mixed/auto")

    # ---- a rank without rows: one big keyframe and empty ones behind it ------------------------------------------
    sizes = [130000] + [0] * (2 * world - 1)
    kfs = [rng.integers(0, 256, (s, 32), dtype=np.uint8) for s in sizes]
    lo, hi, rlo, rhi = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange="fused",
                                    variant="auto")
    empty = [None] * world
    dist.all_gather_object(empty, rhi == rlo)
    ok &= any(empty)
    q = rng.integers(0, 256, (1500, 32), dtype=np.uint8)
    q[:40] = kfs[0][rng.choice(130000, 40, replace=False)]
    ok &= check(db, q, kfs[0], rank, "empty rank")

    # ---- growth: the last rank's shard crosses the tensor-core threshold through append_keyframe ------------------
    sizes = [1000] * (2 * world)
    kfs = [rng.integers(0, 256, (s, 32), dtype=np.uint8) for s in sizes]
    lo, hi, _, _ = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, kfs[lo:hi], rank=rank, world_size=world, group=W, exchange="fused",
                                    variant="auto")
    q = rng.integers(0, 256, (2000, 32), dtype=np.uint8)
    q[:100] = np.concatenate(kfs)[rng.choice(sum(sizes), 100, replace=False)]
    ok &= check(db, q, np.concatenate(kfs), rank, "growth/before")
    for s in (40000, 30000):
        extra = rng.integers(0, 256, (s, 32), dtype=np.uint8)
        kfs.append(extra)
        db.append_keyframe(extra)
        q[100:150] = extra[:50]
        ok &= check(db, q, np.concatenate(kfs), rank, f"growth/+{s}")
    kinds = [None] * world
    dist.all_gather_object(kinds, db.shard["prepared"] is not None)
    ok &= kinds[-1] and not kinds[0]

    t = torch.tensor([int(ok)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_PIPELINE", "OK" if int(t) == 1 else "FAILED", f"world={world}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(t) == 1 else 1)


if __name__ == "__main__":
    main()
