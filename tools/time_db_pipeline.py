"""Cost of the keyframe database's ratio test + mutual check over its plain k-NN step, on the C4 input.

C4: 2000 queries against 4096 keyframes x 2000 rows (synth.keyframe_database(4096, 2000, 2000, seed=4096), 262 MB of
descriptors, larger than the 126 MB L2), sharded over the ranks like bench.py.  One process per GPU:

    python tools/time_db_pipeline.py                      # N = 1
    torchrun --nproc-per-node N tools/time_db_pipeline.py # N = 2, 4, 8

Before timing, every rank's pipeline result (ratio 0.75 + mutual check, through match_tensors) and the global top-2 keys
are checked against the oracle: c_oracle.knn2_keys (rows split over the ranks), then oracle.db_oracle for the mutual
check.  Then, inputs resident, `--warmup` (>= 3) untimed rounds and `--steps` (>= 100) timed rounds; each round runs the
plain k-NN step (knn2_keys_device) and the pipeline step (match_device, ratio 0.75 + mutual) one after the other, each
bracketed by its own CUDA event pair on torch's current stream.  Reported: mean and median per step on every rank and
their maximum over the ranks, with the card's name and power limit.  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

N_KF, KF_ROWS, NQ = 4096, 2000, 2000


def card(local):
    """name and power limit of this rank's GPU (nvidia-smi query; name from torch when it is unavailable)"""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={local}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"name": torch.cuda.get_device_name(local), "power_limit": f"unknown ({type(e).__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ratio", type=float, default=0.75)
    ap.add_argument("--variant", default="auto")
    args = ap.parse_args()
    if args.steps < 100 or args.warmup < 3:
        raise SystemExit("--steps >= 100 and --warmup >= 3")
    import slam_experiments_b200 as sx
    from slam_experiments_b200 import synth
    from oracle import c_oracle, db_oracle

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    query, train = synth.keyframe_database(N_KF, KF_ROWS, NQ, seed=4096)
    sizes = [KF_ROWS] * N_KF
    kf_lo, kf_hi, row_lo, row_hi = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, [train[i * KF_ROWS:(i + 1) * KF_ROWS] for i in range(kf_lo, kf_hi)],
                                    rank=rank, world_size=world, group=dist.group.WORLD if world > 1 else None,
                                    device=dev, variant=args.variant)
    q_dev = torch.from_numpy(query).to(dev)

    # ---- verification, outside the timed region ----------------------------------------------------------------
    mine = np.arange(rank, NQ, world)
    part = c_oracle.knn2_keys(query[mine], train, threads=max(1, (os.cpu_count() or 8) // world))
    parts = [None] * world
    if world > 1:
        dist.all_gather_object(parts, (mine, part))
    else:
        parts = [(mine, part)]
    keys = np.empty((NQ, 2), np.uint64)
    for idx, k in parts:
        keys[idx] = k
    ok = np.array_equal(db.knn2_keys_device(q_dev).cpu().numpy().view(np.uint64), keys)
    eq, et, ed = db_oracle.pipeline_from_keys(query, train, keys, args.ratio, True)
    qi, img, loc, d = db.match_tensors(query, ratio=args.ratio, cross_check=True)
    ok &= np.array_equal(qi, eq) and np.array_equal(img.astype(np.int64) * KF_ROWS + loc, et) and np.array_equal(d, ed)
    flag = torch.tensor([int(ok)], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag) != 1:
        raise SystemExit(f"rank {rank}: pipeline result differs from the oracle")

    # ---- timed region: alternate the plain k-NN step and the pipeline step ---------------------------------------
    def knn():
        return db.knn2_keys_device(q_dev)

    def pipeline():
        return db.match_device(q_dev, ratio=args.ratio, cross_check=True)

    for _ in range(args.warmup):
        knn()
        pipeline()
    barrier()
    ev = {name: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
          for name in ("knn", "pipeline")}
    for i in range(args.steps):
        for name, fn in (("knn", knn), ("pipeline", pipeline)):
            a, b = ev[name][i]
            a.record()
            fn()
            b.record()
    barrier()
    stats = {}
    for name in ev:
        ms = np.array([a.elapsed_time(b) for a, b in ev[name]])
        stats[name] = [float(ms.mean()), float(np.median(ms))]
    t = torch.tensor([stats["knn"][0], stats["knn"][1], stats["pipeline"][0], stats["pipeline"][1]],
                     dtype=torch.float64, device=dev)
    per_rank = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, t)
    per_rank = [p.cpu().tolist() for p in per_rank]
    cards = [None] * world
    if world > 1:
        dist.all_gather_object(cards, card(local))
    else:
        cards = [card(local)]
    if rank == 0:
        mx = np.max(np.array(per_rank), axis=0)
        print(json.dumps({
            "workload": "C4 keyframe database: 2000 queries x 4096 keyframes x 2000 rows",
            "gpus": world, "variant": args.variant, "exchange": db.exchange_mode, "ratio": args.ratio,
            "steps": args.steps, "warmup": args.warmup, "verified": True, "matches_kept": int(len(eq)),
            "knn_ms_mean_max_over_ranks": mx[0], "knn_ms_median_max_over_ranks": mx[1],
            "pipeline_ms_mean_max_over_ranks": mx[2], "pipeline_ms_median_max_over_ranks": mx[3],
            "pipeline_minus_knn_ms_mean": mx[2] - mx[0],
            "per_rank_ms": [{"knn_mean": p[0], "knn_median": p[1], "pipeline_mean": p[2], "pipeline_median": p[3]}
                            for p in per_rank],
            "card": cards[0], "cards_differ": any(c != cards[0] for c in cards),
            "timing": "CUDA events around each step on torch's current stream; the two steps alternate in one process",
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
