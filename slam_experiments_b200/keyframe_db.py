"""Keyframe-database matching with the train set sharded across the GPUs of one box.

The reference keeps keyframes in ``Map._keyframes`` (`/root/reference/backend.py:31-37`) but
never matches against them (SURVEY.md D2); the north-star workload maps onto cv2's
train-collection API, ``bf.add([kf0, kf1, ...]); bf.knnMatch(query, k=2)``, whose result is the
global stable top-k over the row concatenation reported as ``(imgIdx, trainIdx)``
(SURVEY.md E5).  Here each rank (one process per GPU) keeps a contiguous range of keyframes
resident, computes its local top-2 with global row ids, and the per-shard candidates are
merged after ONE exchange step of ``Nq x 2`` packed 64-bit keys (32 KB per rank for 2000 queries):
by default inside the k-NN kernel itself (``hm_knn2_prepared_exchange``: peer stores into symmetric
memory over NVLink + epoch flags + merge by the last CTA of each query block), else an NCCL all-gather
followed by ``hm_merge_top2``.  Unsigned min over
``(dist << 32 | global_row)`` is cv2's order because a lower global row is a lower
``(imgIdx, trainIdx)``.
"""
from __future__ import annotations

import os
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as nat
from .feature_matchers import MatcherError, _Staging, _build_dmatches, _fill_dmatches, _prealloc_dmatches


def shard_ranges(sizes: Sequence[int], world_size: int) -> List[Tuple[int, int, int, int]]:
    """Contiguous keyframe ranges balanced by row count.

    Returns, per rank, ``(kf_lo, kf_hi, row_lo, row_hi)``; ranges tile the collection in
    order, so a lower rank always holds lower global rows.
    """
    sizes = np.asarray(sizes, dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    total = int(starts[-1])
    nkf = len(sizes)
    out = []
    lo = 0
    for r in range(world_size):
        target = total * (r + 1) // world_size
        hi = int(np.searchsorted(starts, target, side="left"))
        hi = max(lo, min(hi, nkf))
        if r == world_size - 1:
            hi = nkf
        out.append((lo, hi, int(starts[lo]), int(starts[hi])))
        lo = hi
    return out


def selection_mask(keyframes, n_keyframes: int) -> np.ndarray:
    """A keyframe selection as a bool mask ``[n_keyframes]``.

    ``keyframes`` is a 1-D bool array of length ``n_keyframes`` or a 1-D sequence of integer ``imgIdx`` values (a set:
    order and duplicates do not matter; an empty sequence selects nothing).  Anything else raises ``MatcherError``."""
    if isinstance(keyframes, (list, tuple)) and len(keyframes) == 0:
        return np.zeros(n_keyframes, bool)
    try:
        a = np.asarray(keyframes)
    except Exception as e:
        raise MatcherError(f"keyframes: not an array ({e})") from None
    if a.ndim != 1:
        raise MatcherError("keyframes: expected a 1-D bool mask or a 1-D sequence of imgIdx values")
    if a.dtype == np.bool_:
        if a.shape[0] != n_keyframes:
            raise MatcherError(f"keyframes: bool mask of length {a.shape[0]}, the database has {n_keyframes} keyframes")
        return a.copy()
    if a.dtype.kind not in "iu":
        raise MatcherError(f"keyframes: expected bool or integer values, got {a.dtype}")
    if a.size and (int(a.min()) < 0 or int(a.max()) >= n_keyframes):
        raise MatcherError(f"keyframes: imgIdx outside [0, {n_keyframes})")
    mask = np.zeros(n_keyframes, bool)
    mask[a] = True
    return mask


def shard_runs(mask: np.ndarray, starts: np.ndarray, kf_lo: int, kf_hi: int, row_lo: int) -> np.ndarray:
    """The runs ``int64 [n, 2]`` of shard-local rows ``[lo, hi)`` that the selected keyframes of ``[kf_lo, kf_hi)``
    hold: maximal ranges of rows of consecutive selected keyframes (keyframes without rows hold none), ascending and
    disjoint.  O(keyframes of the shard)."""
    sel = np.flatnonzero(mask[kf_lo:kf_hi]) + kf_lo
    lo, hi = starts[sel], starts[sel + 1]
    keep = hi > lo
    lo, hi = lo[keep], hi[keep]
    if lo.size == 0:
        return np.empty((0, 2), np.int64)
    brk = np.flatnonzero(lo[1:] != hi[:-1]) + 1
    first = np.concatenate([[0], brk])
    last = np.concatenate([brk, [lo.size]]) - 1
    return (np.stack([lo[first], hi[last]], axis=1) - row_lo).astype(np.int64)


class NativeOps:
    """Device operations of the sharded path: the C ABI kernels + torch.distributed."""

    def __init__(self, device=None, variant: str = "auto"):
        self.device = nat.require_cuda(device)
        self.variant = variant
        # "in_knn": exchange folded into the k-NN kernel's last-CTA merge (one launch);
        # "separate": hm_exchange_merge as its own launch after the k-NN kernel
        self.exchange_kernel = os.environ.get("HM_EXCHANGE_KERNEL", "in_knn")
        self._staging = _Staging()
        nat.lib()

    def upload(self, a: np.ndarray) -> torch.Tensor:
        """Host -> device through a reused pinned buffer (queries); big one-off uploads go direct."""
        a = np.asarray(a)
        if a.nbytes <= (8 << 20):
            with nat.on_device(self.device):
                return self._staging.to_device("q", a, self.device)
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint8)).to(self.device)

    def make_shard(self, train: torch.Tensor):
        """Keep the shard resident; for the tensor-core variant also its prepared image."""
        nt = train.shape[0]
        tc = self._tensor_core(nt)
        prepared = nat.prepare(train, variant=tc) if (tc and nt > 0) else None
        return {"bits": train, "prepared": prepared, "tc": tc, "nt": nt, "buf": None, "pbuf": None}

    def _tensor_core(self, nt: int) -> int:
        """The tensor-core core a resident shard of ``nt`` rows is prepared for (0 = keep packed bits only)."""
        if self.variant in ("i8", "f4") or (self.variant == "auto" and nt >= 65536):
            return nat.tensor_variant(self.variant)
        return 0

    def append_rows(self, shard, rows: np.ndarray):
        """Grow the resident shard by ``rows`` (a new keyframe): amortised-doubling device buffers, one
        H2D of the new rows, and re-expansion of the touched 256-row blocks only."""
        n = rows.shape[0]
        if n == 0:
            return shard
        nt, new_nt = shard["nt"], shard["nt"] + n
        with nat.on_device(self.device):
            buf = shard.get("buf")
            if buf is None or buf.shape[0] < new_nt:
                cap = max(2 * new_nt, 4096)
                nbuf = torch.empty((cap, nat.DESC_BYTES), dtype=torch.uint8, device=self.device)
                if nt:
                    nbuf[:nt].copy_(shard["bits"])
                shard["buf"] = buf = nbuf
                shard["pbuf"] = None
            buf[nt:new_nt].copy_(torch.from_numpy(np.ascontiguousarray(rows, dtype=np.uint8)), non_blocking=False)
            shard["bits"] = buf[:new_nt]
            tc = shard.get("tc") or self._tensor_core(new_nt)
            if tc:
                row_bytes = nat.PREPARED_ROW_BYTES[tc]
                need = nat.prepared_bytes(new_nt, tc) + 512 * row_bytes
                pbuf = shard.get("pbuf")
                first = 0                                     # first row whose prepared image must be (re)written
                if pbuf is None or pbuf.numel() < need:
                    pbuf = torch.empty(max(need, nat.prepared_bytes(buf.shape[0], tc) + 512 * row_bytes),
                                       dtype=torch.uint8, device=self.device)
                    shard["pbuf"] = pbuf
                elif shard["prepared"] is not None:
                    # the partially filled block and everything after it.  hm_prepare pads to whole 256-row blocks, so
                    # starting on a 256-row boundary makes the rewritten rows end exactly at the grown image's padded
                    # end: every padding row of the image is rewritten, none keeps what the buffer held before.
                    first = (nt // nat.PREPARED_PAD_ROWS) * nat.PREPARED_PAD_ROWS
                nat.prepare(buf[first:new_nt], out=pbuf[first * row_bytes:], variant=tc)
                shard["prepared"] = pbuf
                shard["tc"] = tc
            shard["nt"] = new_nt
        return shard

    def local_knn2(self, query: torch.Tensor, shard, train_base: int) -> torch.Tensor:
        if shard["prepared"] is not None and query.shape[0] > 0:
            # resident prepared database, packed query: one launch with the f4 core (query expanded in-kernel)
            return nat.knn2_keys_resident(query, shard["prepared"], shard["nt"], train_base, variant=shard["tc"])
        return nat.knn2_keys(query, shard["bits"], train_base=train_base, variant=self.variant)

    # ---- selected keyframes: the shard's runs of selected rows (keyframe_db.shard_runs), never empty here ----
    def _runs_dev(self, runs: np.ndarray) -> torch.Tensor:
        """The run table (``_native.run_table``) on the device, through the pinned staging: 32 bytes per run, the
        row size the staging buffers are built for."""
        table = nat.run_table(runs)
        with nat.on_device(self.device):
            return self._staging.to_device("runs", table.view(np.uint8), self.device).view(torch.int64)

    def local_knn2_runs(self, query: torch.Tensor, shard, train_base: int, runs: np.ndarray) -> torch.Tensor:
        """Local top-2 over the runs: the tensor-core kernel walks them in place over a prepared image; packed bits are
        gathered (selected rows only) and searched with ``hm_knn2``."""
        runs_dev = self._runs_dev(runs)
        if shard["prepared"] is not None:
            return nat.knn2_keys_resident_runs(query, shard["prepared"], shard["nt"], runs, runs_dev, train_base,
                                               variant=shard["tc"])
        return nat.knn2_keys_runs(query, shard["bits"], runs, runs_dev, train_base, variant=self.variant)

    def local_knn2_runs_exchange(self, query: torch.Tensor, shard, train_base: int, runs: np.ndarray,
                                 group) -> torch.Tensor:
        """Local top-2 over the runs + exchange + merge.  Takes the same branch as :meth:`gather_merge` (which a rank
        without selected rows calls instead): both depend only on ``_xch`` and the query size, and both advance the
        epoch once."""
        x = getattr(self, "_xch", None)
        nq = query.shape[0]
        if x is None or not (0 < nq <= x["max_rows"]) or shard["prepared"] is None:
            return self.gather_merge(self.local_knn2_runs(query, shard, train_base, runs), group)
        x["epoch"] += 1
        return nat.knn2_keys_resident_runs(query, shard["prepared"], shard["nt"], runs, self._runs_dev(runs), train_base,
                                           variant=shard["tc"],
                                           exchange=(x["world"], x["rank"], x["ptrs"], x["max_rows"], x["epoch"]))

    def launches_per_step(self, shard, world: int, exchange_mode: str) -> int:
        """Kernels of THIS library launched per ``knn2_keys_device`` call (bench.py's ``gpu_launches``; the ncu launch
        lists under profiles/ are the evidence): the k-NN kernel for a prepared shard (query expansion, split merge and
        the fused exchange run inside it; the i8 core expands the query in a launch of its own), k-NN (+ split merge) for
        packed bits, + hm_exchange_merge or hm_merge_top2 when the exchange is a launch of its own."""
        # f4 resident shard: ONE launch (the kernel expands the query itself); i8: query expansion + k-NN;
        # packed bits: k-NN + split merge
        n = (1 if shard["tc"] == nat.VARIANT_F4 else 2) if shard["prepared"] is not None else 2
        if world > 1 and (exchange_mode != "fused" or shard["prepared"] is None or self.exchange_kernel != "in_knn"):
            n += 1
        return n

    def all_gather(self, keys: torch.Tensor, group) -> torch.Tensor:
        import torch.distributed as dist
        world = dist.get_world_size(group)
        out = torch.empty((world,) + tuple(keys.shape), dtype=keys.dtype, device=keys.device)
        dist.all_gather_into_tensor(out, keys.contiguous(), group=group)
        return out

    def merge(self, gathered: torch.Tensor) -> torch.Tensor:
        return nat.merge_top2(gathered)

    # ---- fused exchange: peer stores into symmetric memory + flags + merge, one launch, no NCCL call ----
    def setup_exchange(self, group, world: int, rank: int, max_rows: int = 4096) -> str:
        """Allocate and rendezvous the symmetric buffer of ``hm_exchange_merge``.  Returns the mode in
        use: ``"fused"`` or ``"nccl"`` (when symmetric memory cannot be set up on this system)."""
        self._xch = None
        try:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm
            nbytes = nat.exchange_bytes(max_rows, world)
            with nat.on_device(self.device):
                buf = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
                buf.zero_()
                torch.cuda.synchronize(self.device)
                handle = symm.rendezvous(buf, group if group is not None else dist.group.WORLD)
                ptrs = [int(p) for p in handle.buffer_ptrs]
                dist.barrier(group)                      # every rank's flags are zero before the first epoch
            if len(ptrs) != world or any(p == 0 for p in ptrs):
                raise RuntimeError("symmetric memory rendezvous returned no peer pointers")
            import ctypes
            self._xch = {"buf": buf, "handle": handle, "ptrs": (ctypes.c_void_p * world)(*ptrs), "max_rows": max_rows,
                         "epoch": 0, "world": world, "rank": rank}
            return "fused"
        except Exception as e:  # symmetric memory unavailable: the NCCL all-gather path still works
            self._xch_error = f"{type(e).__name__}: {e}"
            return "nccl"

    def local_knn2_exchange(self, query: torch.Tensor, shard, train_base: int, group) -> torch.Tensor:
        """Local k-NN + exchange + merge: one k-NN launch (plus the query expansion) per step.

        Which kernel carries the exchange is a per-rank choice (a rank whose shard has no prepared image -- empty,
        or below the tensor-core threshold under variant="auto" -- runs ``hm_exchange_merge`` after a plain k-NN).
        That is safe because both kernels use the same symmetric buffer, epoch and flag blocks (one per 256 query
        rows that exist); whether the symmetric path is used at all depends only on ``_xch`` (set up collectively)
        and on the query size (replicated), so every rank takes the same branch here."""
        x = getattr(self, "_xch", None)
        nq = query.shape[0]
        if x is None or not (0 < nq <= x["max_rows"]):
            return self.merge(self.all_gather(self.local_knn2(query, shard, train_base), group))
        if shard["prepared"] is None:
            return self.gather_merge(self.local_knn2(query, shard, train_base), group)
        x["epoch"] += 1
        if self.exchange_kernel == "in_knn":
            return nat.knn2_resident_exchange(query, shard["prepared"], shard["nt"], train_base, x["world"], x["rank"],
                                              x["ptrs"], x["max_rows"], x["epoch"], variant=shard["tc"])
        qprep = nat.prepare(query, variant=shard["tc"])
        ptr, groups = nat.knn2_partials_prepared(qprep, nq, shard["prepared"], shard["nt"], train_base,
                                                 variant=shard["tc"])
        return nat.exchange_merge(ptr, x["world"], x["rank"], x["ptrs"], x["max_rows"], x["epoch"], rows=nq,
                                  groups=groups, device=self.device)

    def gather_merge(self, local: torch.Tensor, group) -> torch.Tensor:
        x = getattr(self, "_xch", None)
        if x is not None and 0 < local.shape[0] <= x["max_rows"]:
            x["epoch"] += 1
            return nat.exchange_merge(local.contiguous(), x["world"], x["rank"], x["ptrs"], x["max_rows"], x["epoch"])
        return self.merge(self.all_gather(local, group))

    # ---- host-buffer query of the resident shard through the C context (one C call to enqueue, one to finish) ----
    def host_query_begin(self, query: np.ndarray, shard, train_base: int, world: int):
        """Enqueue query upload + k-NN (+ fused exchange) + key download on the context's stream; returns a token for
        :meth:`host_query_end`, or None when this path does not apply (no prepared shard, exchange over NCCL, a query
        larger than the symmetric buffer): the caller then takes the torch-level path."""
        x = getattr(self, "_xch", None)
        nq = query.shape[0]
        if shard["prepared"] is None or nq == 0 or query.dtype != np.uint8:
            return None
        if world > 1 and (x is None or self.exchange_kernel != "in_knn" or nq > x["max_rows"]):
            return None
        if getattr(self, "_hctx", None) is None:
            with nat.on_device(self.device):
                torch.cuda.synchronize(self.device)         # the shard's prepared image was written on torch's stream
                self._hctx = nat.HostContext()
        if shard.get("_host_epoch") != id(shard["prepared"]) or shard.get("_host_nt") != shard["nt"]:
            torch.cuda.synchronize(self.device)             # the shard grew / moved since the last query
            shard["_host_epoch"], shard["_host_nt"] = id(shard["prepared"]), shard["nt"]
        with nat.on_device(self.device):
            if world > 1:
                x["epoch"] += 1
                return self._hctx.resident_query_begin(query, shard["prepared"], shard["nt"], train_base, shard["tc"],
                                                       x["world"], x["rank"], x["ptrs"], x["max_rows"], x["epoch"])
            return self._hctx.resident_query_begin(query, shard["prepared"], shard["nt"], train_base, shard["tc"])

    def host_query_end(self, token) -> np.ndarray:
        with nat.on_device(self.device):
            return self._hctx.resident_query_end(token).view(np.int64)

    def to_host(self, keys: torch.Tensor) -> np.ndarray:
        with nat.on_device(self.device):
            return self._staging.to_host("keys", keys)

    # ---- ratio test + database-wide mutual check over the global top-2 (all on torch's current stream) ----
    def mutual_flags(self, keys: torch.Tensor, query: torch.Tensor, shard, row_lo: int,
                     ratio: Optional[float]) -> torch.Tensor:
        """This shard's mutual flags ``uint8 [Nq]``: 1 where the query's best row is held here and the query is that
        row's nearest query; 0 everywhere else.  The top-1 pass over the query batch uses the shard's tensor core when
        it has a prepared image (kind::mxf4 computes only the rows this shard owns), else the configured variant."""
        variant = shard["tc"] if shard.get("prepared") is not None else self.variant
        return nat.db_mutual_flags(keys, query, shard["bits"], row_lo, ratio, variant=variant)

    def all_reduce_max(self, flags: torch.Tensor, group) -> torch.Tensor:
        """Element-wise MAX of every rank's flags.  This is its own collective on the process group: it shares nothing
        with the k-NN exchange (symmetric buffer, slots, epochs).  An empty batch still joins with one zero."""
        import torch.distributed as dist
        buf = flags if flags.numel() else torch.zeros(1, dtype=torch.uint8, device=self.device)
        dist.all_reduce(buf, op=dist.ReduceOp.MAX, group=group)
        return buf

    def filter_matches(self, keys: torch.Tensor, flags: Optional[torch.Tensor], ratio: Optional[float]):
        return nat.db_filter(keys, flags, ratio)


class ShardedKeyframeDatabase:
    """Train collection sharded by contiguous keyframe ranges, one shard per rank.

    ``sizes`` (rows per keyframe) is known to every rank; ``local_keyframes`` holds only this
    rank's range ``shard_ranges(sizes, world)[rank]``.  With ``world_size == 1`` (or no process
    group) it is the single-GPU resident database.
    """

    def __init__(self, sizes: Sequence[int], local_keyframes: Sequence[np.ndarray], *, rank: int = 0,
                 world_size: int = 1, group=None, ops=None, device=None, variant: str = "auto",
                 exchange: str = "auto", max_query_rows: int = 4096):
        self.sizes = np.asarray(sizes, dtype=np.int64)
        self.starts = np.concatenate([[0], np.cumsum(self.sizes)])
        self.rank, self.world_size, self.group = rank, world_size, group
        self.ops = ops if ops is not None else NativeOps(device, variant)
        self.kf_lo, self.kf_hi, self.row_lo, self.row_hi = shard_ranges(self.sizes, world_size)[rank]
        if len(local_keyframes) != self.kf_hi - self.kf_lo:
            raise ValueError(f"rank {rank} owns keyframes [{self.kf_lo}, {self.kf_hi}) but got "
                             f"{len(local_keyframes)} arrays")
        for i, a in enumerate(local_keyframes):
            a = np.asarray(a)
            if a.dtype != np.uint8 or a.ndim != 2 or a.shape[1] != nat.DESC_BYTES:
                raise MatcherError(f"keyframe {self.kf_lo + i}: expected uint8 [N, 32] descriptors")
            if a.shape[0] != self.sizes[self.kf_lo + i]:
                raise ValueError(f"keyframe {self.kf_lo + i}: {a.shape[0]} rows, sizes says "
                                 f"{self.sizes[self.kf_lo + i]}")
        cat = (np.concatenate([np.asarray(a) for a in local_keyframes], axis=0)
               if len(local_keyframes) else np.empty((0, nat.DESC_BYTES), np.uint8))
        self.shard = self.ops.make_shard(self.ops.upload(cat))
        # exchange step: "fused" = hm_exchange_merge over symmetric memory, "nccl" = all-gather + merge
        self.exchange_mode = "none" if world_size == 1 else "nccl"
        # why "auto" ended up on the NCCL path (None = it did not): surfaced in bench.py's config so that a broken
        # symmetric-memory setup cannot silently cost the fused path's throughput
        self.exchange_fallback_reason = None
        if world_size > 1 and exchange in ("auto", "fused") and hasattr(self.ops, "setup_exchange"):
            self.exchange_mode = self.ops.setup_exchange(group, world_size, rank, max_query_rows)
            if self.exchange_mode != "fused":
                self.exchange_fallback_reason = getattr(self.ops, "_xch_error", "unknown")
                if exchange == "fused":
                    raise nat.NativeError(f"fused exchange unavailable: {self.exchange_fallback_reason}")
                import warnings
                warnings.warn(f"fused exchange unavailable, using the NCCL all-gather path: {self.exchange_fallback_reason}")

    # ---- incremental growth (Map.insert_keyframe, `/root/reference/backend.py:31-37`) -----------------
    def append_keyframe(self, descriptors: np.ndarray) -> int:
        """Add one keyframe to the resident database; returns its ``imgIdx``.

        Every rank calls this with the same array.  The keyframe joins the LAST rank's shard so that
        shards stay contiguous keyframe ranges and a lower global row stays a lower
        ``(imgIdx, trainIdx)`` -- the property the u64-min merge relies on."""
        a = np.asarray(descriptors)
        if a.size == 0:
            a = np.empty((0, nat.DESC_BYTES), np.uint8)
        if a.dtype != np.uint8 or a.ndim != 2 or a.shape[1] != nat.DESC_BYTES:
            raise MatcherError("keyframe: expected uint8 [N, 32] descriptors")
        if a.shape[0] >= (1 << 18):
            raise MatcherError("too many rows in one train image (cv2: matchers.cpp:860)")
        img = len(self.sizes)
        if img + 1 >= 8192:
            raise MatcherError("too many train images (cv2: matchers.cpp:856)")
        self.sizes = np.append(self.sizes, a.shape[0])
        self.starts = np.concatenate([[0], np.cumsum(self.sizes)])
        if self.rank == self.world_size - 1:
            self.shard = self.ops.append_rows(self.shard, a)
            self.kf_hi += 1
            self.row_hi += a.shape[0]
        return img

    # ---- selected keyframes ------------------------------------------------------------------------
    def _selection(self, keyframes):
        """Validate a ``keyframes=`` argument (before any device work): this rank's runs and the selected rows of the
        whole database."""
        mask = selection_mask(keyframes, len(self.sizes))
        return shard_runs(mask, self.starts, self.kf_lo, self.kf_hi, self.row_lo), int(self.sizes[mask].sum())

    def _knn2_keys_runs(self, query_dev: torch.Tensor, runs: np.ndarray) -> torch.Tensor:
        """Global top-2 keys over this rank's runs and every other rank's.  A rank without selected rows (or a batch
        without rows) contributes all-``NO_MATCH`` keys without a k-NN launch but still takes the same exchange as every
        other rank: which exchange runs depends only on the exchange mode and the query size, both replicated."""
        nq = query_dev.shape[0]
        if runs.shape[0] and nq:
            if self.world_size > 1 and self.exchange_mode == "fused":
                return self.ops.local_knn2_runs_exchange(query_dev, self.shard, self.row_lo, runs, self.group)
            local = self.ops.local_knn2_runs(query_dev, self.shard, self.row_lo, runs)
        else:
            local = torch.full((nq, 2), -1, dtype=torch.int64, device=query_dev.device)     # HM_NO_MATCH
        if self.world_size == 1:
            return local
        if self.exchange_mode == "fused":
            return self.ops.gather_merge(local, self.group)
        return self.ops.merge(self.ops.all_gather(local, self.group))

    # ---- device-level API ---------------------------------------------------------------------
    def knn2_keys_device(self, query_dev: torch.Tensor, keyframes=None) -> torch.Tensor:
        """Global top-2 keys ``[Nq, 2]`` (identical on every rank).  ``keyframes``: search only these keyframes (a bool
        mask over ``imgIdx`` or a sequence of ``imgIdx``; every rank passes the same); trainIdx stay global rows."""
        if keyframes is not None:
            return self._knn2_keys_runs(query_dev, self._selection(keyframes)[0])
        if self.world_size > 1 and self.exchange_mode == "fused":
            return self.ops.local_knn2_exchange(query_dev, self.shard, self.row_lo, self.group)
        local = self.ops.local_knn2(query_dev, self.shard, self.row_lo)
        if self.world_size == 1:
            return local
        gathered = self.ops.all_gather(local, self.group)
        return self.ops.merge(gathered)

    # ---- host-level API -----------------------------------------------------------------------
    def knn_tensors(self, query: np.ndarray, k: int = 2, while_running=None, *, keyframes=None):
        """``(imgIdx, trainIdx, distance)`` each ``[Nq, k']``: cv2's collection result as arrays.  With ``keyframes``
        the result over the sub-collection of the selected keyframes, ``imgIdx`` still indexing the whole database
        (``k' = min(k, selected rows)``)."""
        if k not in (1, 2):
            raise MatcherError("only k in {1, 2} is supported on the B200 path")
        runs = self._selection(keyframes)[0] if keyframes is not None else None
        q = np.asarray(query)
        if q.size == 0:
            e = np.empty((0, 0), np.int32)
            return e, e.copy(), e.copy()
        if q.dtype != np.uint8 or q.ndim != 2 or q.shape[1] != nat.DESC_BYTES:
            raise MatcherError("query: expected uint8 [N, 32] descriptors")
        token = None
        if runs is None and hasattr(self.ops, "host_query_begin") and (self.world_size == 1 or self.exchange_mode == "fused"):
            token = self.ops.host_query_begin(q, self.shard, self.row_lo, self.world_size)
        if token is None:
            qd = self.ops.upload(q)
            keys_dev = self._knn2_keys_runs(qd, runs) if runs is not None else self.knn2_keys_device(qd)  # enqueued
        if while_running is not None:
            while_running()                                       # host work that overlaps the kernels
        keys = self.ops.host_query_end(token) if token is not None else self.ops.to_host(keys_dev)
        gidx, dist, valid = nat.split_keys(keys)
        kk = min(k, int(valid[0].sum()))
        gidx, dist = gidx[:, :kk], dist[:, :kk]
        img, local = nat.locate_rows(self.starts, gidx)
        return img, local, dist

    # ---- ratio test + mutual check over the whole database ---------------------------------------------
    def _match_device(self, query_dev: torch.Tensor, ratio: Optional[float], cross_check: bool, runs):
        nq = query_dev.shape[0]
        if not nq:
            keys = torch.empty((0, 2), dtype=torch.int64, device=query_dev.device)
        else:
            keys = self._knn2_keys_runs(query_dev, runs) if runs is not None else self.knn2_keys_device(query_dev)
        flags = None
        if cross_check:
            # the best row of a kept query lies in the selection, so the swapped side needs none
            flags = self.ops.mutual_flags(keys, query_dev, self.shard, self.row_lo, ratio)
            if self.world_size > 1:
                flags = self.ops.all_reduce_max(flags, self.group)
        return self.ops.filter_matches(keys, flags, ratio)

    def match_device(self, query_dev: torch.Tensor, *, ratio: Optional[float] = None, cross_check: bool = False,
                     keyframes=None):
        """knnMatch k=2 over the whole database, then Lowe's ratio test and the database-wide mutual check.

        Returns device tensors ``(q, t, d, count)``: ``q / t / d [Nq] int32`` hold queryIdx, GLOBAL database row and
        distance of the kept queries in query order, ``count [1]`` how many there are.  A query is kept iff
        ``ratio`` is None or its two nearest rows satisfy ``d1 < ratio * d2`` (float64; a database of fewer than two rows
        drops every query), and -- with ``cross_check`` -- it is the lowest-index nearest query of its best row among
        the ``Nq`` queries of the batch.  Every rank calls it with the same arguments and gets the same list; with
        ``world_size > 1`` and ``cross_check`` there is one MAX all-reduce over ``Nq`` bytes on the process group.
        ``keyframes``: the same over the sub-collection of the selected keyframes (the top-2 inside the selection)."""
        runs = self._selection(keyframes)[0] if keyframes is not None else None
        return self._match_device(query_dev, ratio, cross_check, runs)

    def match_tensors(self, query, *, ratio: Optional[float] = None, cross_check: bool = False, keyframes=None):
        """``(queryIdx, imgIdx, trainIdx, distance)`` int32 arrays of :meth:`match_device`, ordered by queryIdx;
        ``(imgIdx, trainIdx)`` locate the best row in the keyframe collection as :meth:`knn_tensors` does."""
        runs = self._selection(keyframes)[0] if keyframes is not None else None
        q = np.asarray(query)
        if q.size == 0:
            q = np.empty((0, nat.DESC_BYTES), np.uint8)
        if q.dtype != np.uint8 or q.ndim != 2 or q.shape[1] != nat.DESC_BYTES:
            raise MatcherError("query: expected uint8 [N, 32] descriptors")
        oq, ot, od, cnt = self._match_device(self.ops.upload(q), ratio, cross_check, runs)
        host = self.ops.to_host(torch.cat([cnt.view(1), oq.view(-1), ot.view(-1), od.view(-1)]))   # one D2H
        n, nq = int(host[0]), q.shape[0]
        qi, gidx, d = host[1:1 + n], host[1 + nq:1 + nq + n], host[1 + 2 * nq:1 + 2 * nq + n]
        img, local = nat.locate_rows(self.starts, gidx.astype(np.int64))
        return qi.astype(np.int32), img, local, d.astype(np.int32)

    def match(self, query, *, ratio: Optional[float] = None, cross_check: bool = False, keyframes=None) -> tuple:
        """The kept matches of :meth:`match_tensors` as a tuple of ``cv2.DMatch`` (``imgIdx`` = keyframe index)."""
        qi, img, local, d = self.match_tensors(query, ratio=ratio, cross_check=cross_check, keyframes=keyframes)
        return tuple(_build_dmatches(qi, local, d, img))

    def knnMatch(self, queryDescriptors, k: int = 2, *, keyframes=None) -> tuple:
        """cv2 ``bf.knnMatch(query, k)`` over the whole (sharded) collection; with ``keyframes`` over the sub-collection
        of the selected keyframes (cv2's result for that collection, ``imgIdx`` mapped back to the whole database;
        ``Nq`` empty tuples when the selection holds no row)."""
        # the result has nq * min(k, rows in the collection) entries whatever the distances turn out to be, so the DMatch
        # objects are allocated while the kernels run and only filled in afterwards
        q = np.asarray(queryDescriptors)
        rows = int(self.starts[-1]) if keyframes is None else self._selection(keyframes)[1]
        kk_known = min(k, rows) if k in (1, 2) else 0
        pre = []
        if q.ndim == 2 and kk_known > 0:
            img, local, dist = self.knn_tensors(q, k, while_running=lambda: pre.append(_prealloc_dmatches(q.shape[0] * kk_known, kk_known)),
                                                keyframes=keyframes)
        else:
            img, local, dist = self.knn_tensors(queryDescriptors, k, keyframes=keyframes)
        nq, kk = img.shape
        if kk == 0:
            return tuple(() for _ in range(nq))
        qi = np.repeat(np.arange(nq, dtype=np.int32), kk)
        if pre and pre[0] is not None and kk == kk_known:
            return _fill_dmatches(pre[0], qi, local.reshape(-1), dist.reshape(-1), img.reshape(-1), rows=kk)
        return _build_dmatches(qi, local.reshape(-1), dist.reshape(-1), img.reshape(-1), rows=kk)
