"""Cost of a keyframe-database query over a selection of keyframes (``keyframes=``) against the unselected query, on C4.

C4: 2000 queries against 4096 keyframes x 2000 rows (synth.keyframe_database(4096, 2000, 2000, seed=4096), 262 MB of
descriptors, larger than the 126 MB L2), sharded over the ranks like bench.py.  One process per GPU:

    python tools/time_db_subset.py                      # N = 1
    torchrun --nproc-per-node N tools/time_db_subset.py # N = 2, 4, 8

Before timing, every row of every case is checked against the C oracle (c_oracle.knn2_keys over the concatenation of
the selected keyframes, trainIdx mapped back), and the pipeline of "all but the last 64" (ratio 0.75 + mutual check,
match_tensors) against oracle.db_oracle on that concatenation.  Then, inputs resident, `--warmup` (>= 3) untimed rounds
and `--steps` (>= 100) timed rounds; each round runs, one after the other and each bracketed by its own CUDA event pair
on torch's current stream, the k-NN step (knn2_keys_device) unselected, with all keyframes selected, all but the last
64, every other keyframe and every 8th keyframe, then the pipeline step (match_device, ratio 0.75 + mutual) of "all but
the last 64".  Reported: median and mean per step (maximum over the ranks), the selected rows of each case and the
per-selected-row cost relative to the unselected step, with the card's name and power limit.  One JSON line (rank 0).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from time_db_pipeline import card  # noqa: E402  (same directory)

N_KF, KF_ROWS, NQ = 4096, 2000, 2000
CASES = {
    "all_selected": np.arange(N_KF),
    "all_but_last_64": np.arange(N_KF - 64),
    "every_other": np.arange(0, N_KF, 2),
    "every_8th": np.arange(0, N_KF, 8),
}


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
    from oracle.hamming_oracle import NO_MATCH_KEY

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
    kf_lo, kf_hi, _, _ = sx.shard_ranges(sizes, world)[rank]
    db = sx.ShardedKeyframeDatabase(sizes, [train[i * KF_ROWS:(i + 1) * KF_ROWS] for i in range(kf_lo, kf_hi)],
                                    rank=rank, world_size=world, group=dist.group.WORLD if world > 1 else None,
                                    device=dev, variant=args.variant)
    q_dev = torch.from_numpy(query).to(dev)

    # ---- verification, outside the timed region: every row of every case ---------------------------------------
    ok = True
    mine = np.arange(rank, NQ, world)
    threads = max(1, (os.cpu_count() or 8) // world)
    for name, sel in CASES.items():
        rows = (sel[:, None] * KF_ROWS + np.arange(KF_ROWS)).reshape(-1)
        sub = train[rows]
        part = c_oracle.knn2_keys(query[mine], sub, threads=threads)
        parts = [None] * world
        if world > 1:
            dist.all_gather_object(parts, (mine, part))
        else:
            parts = [(mine, part)]
        keys = np.empty((NQ, 2), np.uint64)
        for idx, k in parts:
            keys[idx] = k
        mapped = np.where(keys != NO_MATCH_KEY, (keys & np.uint64(0xFFFFFFFF00000000)) +
                          rows[(keys & np.uint64(0xFFFFFFFF)).astype(np.int64)].astype(np.uint64), keys)
        got = db.knn2_keys_device(q_dev, keyframes=sel).cpu().numpy().view(np.uint64)
        ok &= bool(np.array_equal(got, mapped))
        if name == "all_but_last_64":
            eq, et, ed = db_oracle.pipeline_from_keys(query, sub, keys, args.ratio, True)
            qi, img, loc, d = db.match_tensors(query, ratio=args.ratio, cross_check=True, keyframes=sel)
            ok &= bool(np.array_equal(qi, eq) and np.array_equal(img.astype(np.int64) * KF_ROWS + loc, rows[et])
                       and np.array_equal(d, ed))
            kept = int(len(eq))
    flag = torch.tensor([int(ok)], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag) != 1:
        raise SystemExit(f"rank {rank}: a selection's result differs from the oracle")

    # ---- timed region: the five k-NN steps and the pipeline step alternate ----------------------------------------
    steps = {"unselected": lambda: db.knn2_keys_device(q_dev)}
    for name, sel in CASES.items():
        steps[name] = (lambda s: lambda: db.knn2_keys_device(q_dev, keyframes=s))(sel)
    steps["pipeline_all_but_last_64"] = lambda: db.match_device(q_dev, ratio=args.ratio, cross_check=True,
                                                                keyframes=CASES["all_but_last_64"])
    for _ in range(args.warmup):
        for fn in steps.values():
            fn()
    barrier()
    ev = {name: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
          for name in steps}
    for i in range(args.steps):
        for name, fn in steps.items():
            a, b = ev[name][i]
            a.record()
            fn()
            b.record()
    barrier()
    names = list(steps)
    mine_stats = []
    for name in names:
        ms = np.array([a.elapsed_time(b) for a, b in ev[name]])
        mine_stats += [float(np.median(ms)), float(ms.mean())]
    t = torch.tensor(mine_stats, dtype=torch.float64, device=dev)
    per_rank = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, t)
    mx = np.max(np.array([p.cpu().tolist() for p in per_rank]), axis=0)
    cards = [None] * world
    if world > 1:
        dist.all_gather_object(cards, card(local))
    else:
        cards = [card(local)]
    if rank == 0:
        total_rows = N_KF * KF_ROWS
        res = {}
        for i, name in enumerate(names):
            rows = total_rows if name in ("unselected",) else len(CASES.get(name, CASES["all_but_last_64"])) * KF_ROWS
            res[name] = {"ms_median": mx[2 * i], "ms_mean": mx[2 * i + 1], "selected_rows": rows}
            if name in CASES:
                # cost per selected row over the unselected step's cost per row (1.0 = proportional to the rows)
                res[name]["per_row_vs_unselected"] = (mx[2 * i] / rows) / (mx[0] / total_rows)
        print(json.dumps({
            "workload": "C4 keyframe database: 2000 queries x 4096 keyframes x 2000 rows, keyframes= selections",
            "gpus": world, "variant": args.variant, "exchange": db.exchange_mode, "ratio": args.ratio,
            "steps": args.steps, "warmup": args.warmup, "verified": True, "pipeline_matches_kept": kept,
            "results_max_over_ranks": res,
            "all_selected_vs_unselected_median": mx[2 * names.index("all_selected")] / mx[0],
            "card": cards[0], "cards_differ": any(c != cards[0] for c in cards),
            "timing": "CUDA events around each step on torch's current stream; all steps alternate in one process",
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
