#!/usr/bin/env python
"""Benchmark of the Hamming brute-force matching hot path on B200.

Default workload (BASELINE.json configs[3], the one quoted at 1/2/4/8 GPUs): the
keyframe-database query -- 2000 query descriptors against 4096 keyframes x 2000 train
descriptors (8,192,000 rows), the train set sharded across the N GPUs of one box by contiguous
keyframe ranges, per-shard top-2 candidates merged in one exchange step (peer stores over NVLink inside
the k-NN kernel; `--exchange nccl` = all-gather + merge kernel).  A "step" is one
query batch against the whole database.  `value` is whole-job Gpairs/s with the database and the
query already resident in HBM; `e2e` is the same metric through the reference-facing drop-in
(`ShardedKeyframeDatabase.knnMatch`, the cv2 collection API `bf.add(...); bf.knnMatch(q, k=2)`)
with the query in host memory and DMatch tuples out.  `--dump-outputs DIR` writes the result of the last
timed step (imgIdx, trainIdx, distance of the two nearest rows per query) as .npy files; the inputs are
seeded, so two builds run with the same arguments can be compared file for file.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...

Other workloads (--workload c1|c2|c3|c5) are single-GPU lines used for DESIGN.md / profiles.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "hamming_pairs_per_sec"
UNIT = "Gpairs/s"
NQ = 2000
KF_ROWS = 2000
N_KEYFRAMES = 4096
I8_OPS_PER_PAIR = 512           # 256 MAC on the +/-1 expansion (SURVEY.md 8d)
POPC_PER_PAIR = 8


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU while the timed region runs.

    NVML (nvidia_ml_py) is polled every few milliseconds from a thread so that even a 40 ms timed
    region gets several samples; falls back to `nvidia-smi -lms 50` when NVML is unavailable.
    """

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._nvml = None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x.strip() for x in vis.split(",") if x.strip()]
            if self.gpu < len(ids) and ids[self.gpu].isdigit():
                return int(ids[self.gpu])
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self._nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self._nvml
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                if get_reasons:
                    mask = int(get_reasons(self._h))
                    for name, bit in bits.items():
                        if mask & bit:
                            self.reasons.add(name)
            except Exception:
                break
            self._stop.wait(0.004)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self._nvml is not None:
            self._stop.set()
            self.thread.join(timeout=1)
            sm = self.samples
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None,
                    "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def _load_synth():
    """slam_experiments_b200/synth.py loaded BY PATH (it only needs numpy): the reference arm must not import the
    product package, whose __init__ loads the native libraries."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_hm_synth", os.path.join(ROOT, "slam_experiments_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_c4(n_keyframes=N_KEYFRAMES, rows=KF_ROWS, nq=NQ, dist="M"):
    """C4 inputs.  "M" (default, SURVEY.md 8d): matchable queries over a uniform database; "U": uniform queries;
    "monotone": the adversarial input of SURVEY.md 7 -- near-identical queries and the database sorted by
    DEcreasing distance to them, so every CTA streams monotonically improving, massively tied distances."""
    synth = _load_synth()
    query, train = synth.keyframe_database(n_keyframes, rows, nq, seed=4096)
    if dist == "U":
        query = synth.uniform(nq, 4097)
    elif dist == "monotone":
        rng = np.random.default_rng(4098)
        base = rng.integers(0, 256, 32, dtype=np.uint8)
        d = np.bitwise_count(train ^ base).sum(axis=1, dtype=np.int32)
        train = np.ascontiguousarray(train[np.argsort(-d, kind="stable")])
        query = np.repeat(base[None, :], nq, axis=0)
        flips = rng.integers(0, 256, (nq, 3))                    # three random bit flips per query row
        for j in range(3):
            query[np.arange(nq), flips[:, j] >> 3] ^= (1 << (flips[:, j] & 7)).astype(np.uint8)
    return query, train


def mma_issue_peak(variant):
    """TOP/s of a pure tcgen05.mma issue loop on this chip, measured by tools/microbench*.cu (committed JSON)."""
    key = "mma_mxf4_n128_chip_tops" if variant == "f4" else "mma_i8_n128_chip_tops"
    for name in ("r01h_microbench_fp4_b200.json", "r01_microbench_b200.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            if key in d:
                return float(d[key]), f"profiles/{name}:{key}"
        except Exception:
            pass
    return (8838.2 if variant == "f4" else 4557.8), "fallback constant (microbench JSON missing)"


# =====================================================================================================
# reference arm: the reference's own CPU implementation of the path (cv2.BFMatcher, the engine
# /root/reference/feature_matchers.py:34,39 calls), all host threads, bounded sample per step
# =====================================================================================================
def cv2_collection_step(query, keyframes):
    import cv2
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    bf.add(keyframes)
    return bf.knnMatch(query, k=2)


def calibrate_sample(query, train, target_s: float, rows=KF_ROWS, max_kf=N_KEYFRAMES):
    """Number of keyframes whose cv2 collection query takes about `target_s` seconds."""
    n = 8
    for _ in range(3):                       # refine: tiny probes are dominated by thread start-up
        kfs = [train[i * rows:(i + 1) * rows] for i in range(n)]
        cv2_collection_step(query, kfs)
        t0 = time.perf_counter()
        cv2_collection_step(query, kfs)
        dt = max(time.perf_counter() - t0, 1e-4)
        est = int(n * target_s / dt)
        if dt >= 0.25 * target_s or n >= max_kf:
            n = est
            break
        n = max(n + 1, min(max_kf, est, n * 16))
    else:
        n = est
    return max(2, min(max_kf, n))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import cv2
    query, train = make_c4()
    # bounded sample: the whole (warmup + steps) run stays near two to three minutes whatever K is; when the full
    # database fits that budget (few steps) the step IS the full config
    per_step = max(0.05, min(8.0, 150.0 / max(1, args.steps + args.warmup)))
    n_kf = calibrate_sample(query, train, per_step)
    kfs = [train[i * KF_ROWS:(i + 1) * KF_ROWS] for i in range(n_kf)]
    for _ in range(args.warmup):
        cv2_collection_step(query, kfs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cv2_collection_step(query, kfs)
    dt = time.perf_counter() - t0
    pairs = float(NQ) * n_kf * KF_ROWS * args.steps
    value = pairs / dt / 1e9
    sample = f"{NQ} queries x {n_kf} of {N_KEYFRAMES} keyframes x {KF_ROWS} rows per step (cv2 collection API)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": dict(c4_config(args.gpus), same_config=bool(n_kf == N_KEYFRAMES)),
        "native_so_loaded": [m for m in sys.modules if m.startswith("slam_experiments_b200")],   # must stay empty
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cv2.getNumThreads(), "kind": "reference",
                         "sample": sample, "engine": f"cv2.BFMatcher {cv2.__version__}",
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def c4_config(n_gpus):
    return {"workload": "c4_keyframe_database", "queries": NQ, "keyframes": N_KEYFRAMES, "rows_per_keyframe": KF_ROWS,
            "train_rows": N_KEYFRAMES * KF_ROWS, "descriptor_bits": 256, "k": 2,
            "sharding": f"train rows over {n_gpus} GPU(s), contiguous keyframe ranges",
            "l2": "inputs larger than L2 (resident shard >= 262 MB per GPU)"}


# =====================================================================================================
# B200 arm
# =====================================================================================================
def verify_all_rows(db, q_dev, query, train, rank, world, dist, dev):
    """Correctness of what is timed, outside the timed region: EVERY row on EVERY rank.

    The keys a rank holds are compared bit for bit with rank 0's (broadcast), and the oracle's work is split over the
    ranks (rank r checks rows r::world with its share of the host threads), so all rows are checked against the
    oracle once and every rank's copy is tied to them.  At N > 1 the fused exchange is also checked against the
    NCCL all-gather + merge path on the same local candidates."""
    import torch
    from oracle import c_oracle
    keys_dev = db.knn2_keys_device(q_dev)
    keys = keys_dev.cpu().numpy().view(np.uint64)
    ok = True
    if world > 1:
        ref0 = keys_dev.clone()
        dist.broadcast(ref0, src=0)
        ok &= bool(torch.equal(ref0, keys_dev))
        local = db.ops.local_knn2(q_dev, db.shard, db.row_lo)
        merged = db.ops.merge(db.ops.all_gather(local, db.group))
        ok &= bool(torch.equal(merged, keys_dev))
    mine = np.arange(rank, query.shape[0], world)
    threads = max(1, (os.cpu_count() or 8) // world)
    ok &= bool(np.array_equal(keys[mine], c_oracle.knn2_keys(query[mine], train, threads=threads)))
    t = torch.tensor([int(ok)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(int(t) == 1)


def tensor_roofline(nat, peaks, peak_src, variant_used, nq, nt_local, kern_ms, batch=1):
    """Roofline record of the dominant tensor-core kernel.  `frac` = achieved / (2 or 4 x MEASURED bf16 BURST) -- the
    kernel is timed alone by its own event pair -- and `frac_of_mma_issue_peak` = achieved / the measured
    tcgen05.mma issue loop of this chip (the tighter, architectural ceiling)."""
    local_pairs = float(nq) * nt_local * batch
    achieved = local_pairs * I8_OPS_PER_PAIR / (kern_ms * 1e-3) / 1e12
    mult = 2.0 if variant_used == "i8" else 4.0
    issue_peak, issue_src = mma_issue_peak(variant_used)
    row_bytes = 256 if variant_used == "i8" else 128
    kind = "kind::i8" if variant_used == "i8" else "kind::mxf4"
    peak = mult * peaks["bf16_tflops"]
    launch = nat.describe_launch(nq, nt_local, batch, variant_used)
    tiles = 2.0 * (-(-nq // 256)) * (-(-nt_local // 128)) * batch     # 128 x 128 accumulator tiles
    return {"bound": "tensor", "kernel": launch.split()[0], "launch": launch, "achieved": achieved, "peak": peak,
            "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
            "note": f"+/-1 multiply-add ops (512/pair); peak = {mult:g} x bf16_tflops BURST of {peak_src} "
                    f"({kind} issues at {mult:g}x the bf16 rate; the kernel is timed alone by its own event pair)",
            "kernel_ms": kern_ms, "pairs_per_launch": local_pairs,
            "frac_of_mma_issue_peak": achieved / issue_peak, "mma_issue_peak": issue_peak,
            "mma_issue_peak_source": issue_src,
            "frac_of_sustained_bf16_x": achieved / (mult * peaks["bf16_tflops_sustained"]),
            "algorithmic_bytes": 32 * (nq + nt_local) * batch + 16 * nq * batch,
            "operand_bytes": (nt_local + nq) * row_bytes * batch,
            "hbm_gbs": (nt_local * row_bytes + nq * row_bytes) * batch / (kern_ms * 1e-3) / 1e9}


def time_c4(db, q_dev, steps, warmup, barrier, nat, torch, local_rank):
    """K timed steps, inputs resident: (ms per step, mean ms of the dominant kernel, clocks, keys of the last step)."""
    for _ in range(max(warmup, 3)):
        db.knn2_keys_device(q_dev)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    kern_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(steps):
        nat.profile_events(*kern_ev[i])
        keys = db.knn2_keys_device(q_dev)
    e1.record()
    barrier()
    nat.profile_events(None, None)
    clocks = sampler.stop()
    # what the SMs really ran at: the k-NN kernel's first CTA stamps %globaltimer and clock64 at entry and exit (NVML,
    # polled every few ms, reports the application clock even while the chip holds the tensor pipe at a lower one)
    probe = nat.clock_probe(q_dev.device)
    if probe:
        clocks["sm_mhz_effective_in_kernel"] = probe["sm_mhz_effective"]
        clocks["effective_note"] = "clock64 / %globaltimer over the first CTA of the last timed k-NN launch"
    return e0.elapsed_time(e1) / steps, float(np.mean([a.elapsed_time(b) for a, b in kern_ev])), clocks, keys


def dump_outputs(out_dir, db, keys, nat):
    """What a caller of the timed path receives, decoded as `ShardedKeyframeDatabase.knn_tensors` does: imgIdx,
    trainIdx and distance of the two nearest rows of every query, each [Nq, 2], as float64 (exact for these
    integers) so that two builds can be compared output for output."""
    gidx, dist, _ = nat.split_keys(keys.cpu().numpy())
    img, local = nat.locate_rows(db.starts, gidx)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("img_idx", img), ("train_idx", local), ("distance", dist)):
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


def run_b200(args):
    import torch
    import torch.distributed as dist
    import slam_experiments_b200 as sx
    from slam_experiments_b200 import _native as nat

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks, peak_src = measured_peaks()
    query, train = make_c4()
    sizes = [KF_ROWS] * N_KEYFRAMES
    kf_lo, kf_hi, row_lo, row_hi = sx.shard_ranges(sizes, world)[rank]

    def build_db(train_rows):
        local_kfs = [train_rows[i * KF_ROWS:(i + 1) * KF_ROWS] for i in range(kf_lo, kf_hi)]
        return sx.ShardedKeyframeDatabase(sizes, local_kfs, rank=rank, world_size=world,
                                          group=None if world == 1 else dist.group.WORLD, device=dev,
                                          variant=args.variant, exchange=args.exchange)

    db = build_db(train)
    q_dev = torch.from_numpy(query).to(dev)
    nt_local = row_hi - row_lo
    variant_used = nat.VARIANT_NAMES[db.shard["tc"]] if db.shard["prepared"] is not None else args.variant

    verified = None
    if not args.no_verify:
        verified = verify_all_rows(db, q_dev, query, train, rank, world, dist, dev)
        if not verified:
            raise SystemExit("bench: GPU result differs from the oracle")

    # ---- timed region: K steps, inputs resident ---------------------------------------------------------
    ms_per_step, kern_ms, clocks, last_keys = time_c4(db, q_dev, args.steps, args.warmup, barrier, nat, torch, local_rank)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, db, last_keys, nat)
    t = torch.tensor([ms_per_step, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step, kern_ms_max = float(t[0]), float(t[1])
    total_pairs = float(NQ) * N_KEYFRAMES * KF_ROWS
    value = total_pairs / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: through the drop-in, host buffers in, DMatch tuples out --------------------------------
    def e2e_loop(fn, steps):
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt[0]) / steps

    e2e_s = e2e_loop(lambda: db.knnMatch(query, 2), args.steps)
    e2e_arr_s = e2e_loop(lambda: db.knn_tensors(query, 2), args.steps)
    e2e_value = total_pairs / e2e_s / 1e9

    # ---- roofline of the dominant kernel (this rank's shard), from the live CUDA-event timing -----------
    if variant_used in ("i8", "f4"):
        roofline = tensor_roofline(nat, peaks, peak_src, variant_used, NQ, nt_local, kern_ms_max)
        eff = clocks.get("sm_mhz_effective_in_kernel")
        if eff:
            roofline["frac_of_mma_issue_peak_at_effective_clock"] = roofline["achieved"] / (roofline["mma_issue_peak"] * eff / 1965.0)
            roofline["effective_clock_note"] = (f"the issue peak is quoted at 1965 MHz; under this kernel the SMs ran at {eff:.0f} MHz "
                                                "(clocks.sm_mhz_effective_in_kernel)")
    else:
        sm = nat.sm_count()
        achieved = float(NQ) * nt_local * POPC_PER_PAIR / (kern_ms_max * 1e-3) / 1e12
        peak = sm * 16 * peaks["sm_max_mhz"] * 1e6 / 1e12
        roofline = {"bound": "popc", "kernel": "hm_popc_knn2_kernel", "achieved": achieved, "peak": peak,
                    "unit": "Tpopc/s", "frac": achieved / peak, "traffic": None,
                    "note": "POPC issue roofline: 8 POPC per pair; peak = SMs x 16/clk (measured 15.7) x sm_max_mhz",
                    "kernel_ms": kern_ms_max, "pairs_per_launch": float(NQ) * nt_local}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            with open(traffic_file) as f:
                roofline["traffic"] = json.load(f).get(f"c4_n{world}_{variant_used}")
        except Exception:
            pass

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "config": dict(c4_config(world), variant=variant_used, exchange=db.exchange_mode,
                                                         exchange_fallback_reason=db.exchange_fallback_reason,
                                                         distribution="M (matchable queries, uniform database)",
                                                         db_format={"i8": "train shard resident as +/-1 int8 (expanded once at add())",
                                                                    "f4": "train shard resident as +/-1 e2m1 (expanded once at add())"}.get(variant_used, "packed bits")),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": NQ * 32, "d2h_bytes_per_step": NQ * 16,
                "ms_per_step": e2e_s * 1e3, "api": "ShardedKeyframeDatabase.knnMatch(query_numpy, 2) -> DMatch tuples",
                "arrays_out_ms_per_step": e2e_arr_s * 1e3},
        # per step: the k-NN kernel (query expansion, split merge and, for N > 1, the fused exchange run inside it);
        # with the NCCL exchange one hm_merge_top2_kernel more (ncu launch list in profiles/)
        "gpu_launches": args.steps * db.ops.launches_per_step(db.shard, world, db.exchange_mode),
        "roofline": roofline,
        "verified_vs_oracle": verified,
        "verified_rows": NQ if verified else 0,
        "verified_how": "all rows vs the C oracle (rows split over ranks), every rank bit-identical to rank 0"
                        + (", fused exchange == NCCL all-gather + merge" if world > 1 else ""),
    }

    if world == 1 and not args.quick:
        # ---- north star: "report both" -- the same workload on uniform queries and on the adversarial monotone input
        others = {}
        del db
        for name in ("U", "monotone"):
            q2, t2 = make_c4(dist=name)
            db2 = build_db(t2)
            q2_dev = torch.from_numpy(q2).to(dev)
            from oracle import c_oracle
            rows = np.linspace(0, NQ - 1, 250).astype(np.int64)
            got = db2.knn2_keys_device(q2_dev).cpu().numpy().view(np.uint64)
            good = bool(np.array_equal(got[rows], c_oracle.knn2_keys(q2[rows], t2)))
            if not good:
                raise SystemExit(f"bench: C4 distribution {name}: GPU result differs from the oracle")
            ms2, k2, _, _ = time_c4(db2, q2_dev, max(10, args.steps // 4), 3, barrier, nat, torch, local_rank)
            others[name] = {"value": total_pairs / (ms2 * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms2, "kernel_ms": k2,
                            "verified_rows": int(rows.size)}
            del db2, q2_dev, t2
            torch.cuda.empty_cache()
        line["distributions"] = dict(others, M={"value": value, "unit": UNIT, "ms_per_step": ms_per_step,
                                                "kernel_ms": kern_ms_max, "verified_rows": NQ})
        # ---- the other BASELINE.json configs as sub-records of this one driver-run line ------------------------
        from tools import bench_extra
        subs = {}
        sub_steps = max(10, min(args.steps, 30))
        for key, wl, n in (("c1", "c1", 0), ("c2", "c2", 0), ("c3_16k", "c3", 16384), ("c3_64k", "c3", 65536), ("c5", "c5", 0)):
            try:
                rec = bench_extra.measure(wl, sub_steps, 3, args.variant, n, cpu_seconds=3.0)
                subs[key] = {k: rec[k] for k in ("value", "unit", "ms_per_step", "config", "e2e", "roofline", "cpu_baseline",
                                                 "verified_vs_oracle", "verified", "gpu_launches", "frame_pairs_per_s")
                             if k in rec}
            except SystemExit as e:      # a parity failure in a sub-config fails the bench
                raise
            except Exception as e:       # anything else is reported, not hidden
                subs[key] = {"error": f"{type(e).__name__}: {e}"}
        try:
            subs["orb_describe"] = bench_extra.measure_orb(sub_steps)
        except SystemExit:
            raise
        except Exception as e:
            subs["orb_describe"] = {"error": f"{type(e).__name__}: {e}"}
        line["configs"] = subs

    # ---- cpu baseline beside it (rank 0, N=1 only): cv2 on the host cores, bounded sample ----------------
    if world == 1 and not args.no_cpu_baseline:
        import cv2
        n_kf = calibrate_sample(query, train, 12.0)
        kfs = [train[i * KF_ROWS:(i + 1) * KF_ROWS] for i in range(n_kf)]
        t0 = time.perf_counter()
        cv2_collection_step(query, kfs)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {
            "value": float(NQ) * n_kf * KF_ROWS / dt / 1e9, "unit": UNIT, "cores": cv2.getNumThreads(),
            "kind": "reference",
            "sample": f"{NQ} queries x {n_kf} of {N_KEYFRAMES} keyframes x {KF_ROWS} rows, one cv2 collection knnMatch(k=2)",
            "engine": f"cv2.BFMatcher {cv2.__version__}", "host_cpus": os.cpu_count(), "seconds": dt}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", default="auto", choices=["auto", "popc", "i8", "f4"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c1", "c2", "c3", "c5"])
    ap.add_argument("--n", type=int, default=65536, help="c3: N x N")
    ap.add_argument("--exchange", default="auto", choices=["auto", "fused", "nccl"])
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--quick", action="store_true", help="C4 only: skip the other distributions and the c1/c2/c3/c5 sub-records")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="C4: write what the last timed step computed as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "c4"):
        ap.error("--dump-outputs applies to the C4 workload of the B200 arm")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload != "c4":
        from tools import bench_extra
        return bench_extra.run(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
