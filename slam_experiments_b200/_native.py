"""ctypes binding of the C ABI in include/hm_matcher.h (libhm_matcher.so).

PyTorch is plumbing only: it owns device memory and streams; every argument
that crosses the boundary is a raw pointer, a size or a stream handle.  There
is no CPU fallback: if the library is missing or no sm_100 device is visible,
calls raise ``NativeError``.
"""
from __future__ import annotations

import contextlib
import ctypes
import os
import threading
from typing import Optional, Tuple

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("HM_MATCHER_SO") or os.path.join(HERE, "libhm_matcher.so")

HM_OK = 0
VARIANT_AUTO, VARIANT_POPC, VARIANT_I8, VARIANT_F4 = 0, 1, 2, 3
VARIANTS = {"auto": VARIANT_AUTO, "popc": VARIANT_POPC, "i8": VARIANT_I8, "f4": VARIANT_F4,
            None: VARIANT_AUTO, 0: 0, 1: 1, 2: 2, 3: 3}
VARIANT_NAMES = {VARIANT_POPC: "popc", VARIANT_I8: "i8", VARIANT_F4: "f4"}
FLAG_RATIO, FLAG_MUTUAL, FLAG_DIST_THRESHOLD = 1, 2, 4
NO_MATCH = 0xFFFFFFFFFFFFFFFF
DESC_BYTES = 32
PREPARED_ROW_BYTES = {VARIANT_I8: 256, VARIANT_F4: 128}
PREPARED_PAD_ROWS = 256         # HM_PREPARED_TILE_ROWS: prepared images are padded to whole blocks of this many rows

# every symbol include/hm_matcher.h declares (tests check the library exports all of them)
EXPORTS = (
    "hm_version", "hm_last_error", "hm_profile_events", "hm_device_sm_count", "hm_select_variant", "hm_workspace_bytes",
    "hm_describe_launch",
    "hm_knn2", "hm_knn2_batched", "hm_default_tensor_variant", "hm_prepared_bytes", "hm_prepared_workspace_bytes", "hm_prepare", "hm_knn2_prepared", "hm_knn2_prepared_partials", "hm_knn2_prepared_exchange",
    "hm_resident_workspace_bytes", "hm_knn2_resident", "hm_knn2_resident_exchange",
    "hm_runs_workspace_bytes", "hm_describe_runs_launch", "hm_knn2_resident_runs", "hm_knn2_resident_runs_exchange",
    "hm_knn2_runs",
    "hm_merge_top2", "hm_exchange_bytes", "hm_exchange_merge", "hm_filter_matches", "hm_match_fused", "hm_gather_points", "hm_rasterize_mask",
    "hm_db_mutual_workspace_bytes", "hm_db_mutual_flags", "hm_db_filter",
    "hm_context_create", "hm_context_destroy", "hm_knn2_host", "hm_match_host", "hm_frame_put", "hm_frame_match",
    "hm_resident_query_begin", "hm_resident_query_end",
    "hm_orb_workspace_bytes", "hm_orb_level_geometry", "hm_orb_angles_to_cs", "hm_orb_build_pyramid", "hm_orb_describe",
    "hm_frame_put_orb",
)


class NativeError(RuntimeError):
    """The CUDA library is missing, no B200 is visible, or a native call failed."""


_lib = None
_lock = threading.Lock()


def _declare(L):
    c = ctypes
    vp, i64, u64, sz, ci, cu = c.c_void_p, c.c_int64, c.c_uint64, c.c_size_t, c.c_int, c.c_uint
    L.hm_version.restype = ci
    L.hm_last_error.restype = c.c_char_p
    L.hm_device_sm_count.restype = ci
    L.hm_profile_events.restype = None
    L.hm_profile_events.argtypes = [vp, vp]
    L.hm_select_variant.restype = ci
    L.hm_select_variant.argtypes = [i64, i64, ci]
    L.hm_describe_launch.restype = ci
    L.hm_describe_launch.argtypes = [i64, i64, ci, ci, c.c_char_p, sz]
    L.hm_workspace_bytes.restype = sz
    L.hm_workspace_bytes.argtypes = [i64, i64, ci, ci]
    L.hm_knn2.restype = ci
    L.hm_knn2.argtypes = [vp, i64, i64, vp, i64, i64, u64, vp, ci, vp, sz, vp]
    L.hm_knn2_batched.restype = ci
    L.hm_knn2_batched.argtypes = [vp, i64, i64, i64, vp, i64, i64, i64, ci, vp, ci, vp, sz, vp]
    L.hm_default_tensor_variant.restype = ci
    L.hm_prepared_bytes.restype = sz
    L.hm_prepared_bytes.argtypes = [i64, ci]
    L.hm_prepared_workspace_bytes.restype = sz
    L.hm_prepared_workspace_bytes.argtypes = [i64, i64, ci]
    L.hm_prepare.restype = ci
    L.hm_prepare.argtypes = [vp, i64, i64, vp, ci, vp]
    L.hm_knn2_prepared.restype = ci
    L.hm_knn2_prepared.argtypes = [vp, i64, vp, i64, u64, vp, ci, vp, sz, vp]
    L.hm_resident_workspace_bytes.restype = sz
    L.hm_resident_workspace_bytes.argtypes = [i64, i64, ci]
    L.hm_knn2_resident.restype = ci
    L.hm_knn2_resident.argtypes = [vp, i64, i64, vp, i64, u64, vp, ci, vp, sz, vp]
    L.hm_knn2_resident_exchange.restype = ci
    L.hm_knn2_resident_exchange.argtypes = [vp, i64, i64, vp, i64, u64, ci, ci, vp, i64, c.c_uint32, vp, ci, vp, sz, vp]
    L.hm_runs_workspace_bytes.restype = sz
    L.hm_runs_workspace_bytes.argtypes = [i64, vp, i64, ci, ci]
    L.hm_describe_runs_launch.restype = ci
    L.hm_describe_runs_launch.argtypes = [i64, i64, vp, i64, ci, c.c_char_p, sz, vp]
    L.hm_knn2_resident_runs.restype = ci
    L.hm_knn2_resident_runs.argtypes = [vp, i64, i64, vp, i64, vp, vp, i64, u64, vp, ci, vp, sz, vp]
    L.hm_knn2_resident_runs_exchange.restype = ci
    L.hm_knn2_resident_runs_exchange.argtypes = [vp, i64, i64, vp, i64, vp, vp, i64, u64, ci, ci, vp, i64, c.c_uint32,
                                                 vp, ci, vp, sz, vp]
    L.hm_knn2_runs.restype = ci
    L.hm_knn2_runs.argtypes = [vp, i64, i64, vp, i64, i64, vp, vp, i64, u64, vp, ci, vp, sz, vp]
    L.hm_merge_top2.restype = ci
    L.hm_merge_top2.argtypes = [vp, ci, i64, vp, vp]
    L.hm_exchange_bytes.restype = sz
    L.hm_exchange_bytes.argtypes = [i64, ci]
    L.hm_exchange_merge.restype = ci
    L.hm_exchange_merge.argtypes = [vp, ci, i64, ci, ci, vp, i64, c.c_uint32, vp, vp]
    L.hm_knn2_prepared_exchange.restype = ci
    L.hm_knn2_prepared_exchange.argtypes = [vp, i64, vp, i64, u64, ci, ci, vp, i64, c.c_uint32, vp, ci, vp, sz, vp]
    L.hm_knn2_prepared_partials.restype = ci
    L.hm_knn2_prepared_partials.argtypes = [vp, i64, vp, i64, u64, ci, vp, sz, vp, c.POINTER(vp), c.POINTER(ci)]
    L.hm_filter_matches.restype = ci
    L.hm_filter_matches.argtypes = [vp, i64, vp, i64, ci, cu, vp, c.c_double, vp, vp, vp, vp, vp]
    L.hm_match_fused.restype = ci
    L.hm_match_fused.argtypes = [vp, i64, i64, i64, vp, i64, i64, i64, ci, cu, vp, c.c_double,
                                 vp, vp, vp, vp, vp, ci, vp, sz, vp]
    L.hm_db_mutual_workspace_bytes.restype = sz
    L.hm_db_mutual_workspace_bytes.argtypes = [i64, ci]
    L.hm_db_mutual_flags.restype = ci
    L.hm_db_mutual_flags.argtypes = [vp, i64, vp, i64, vp, i64, i64, u64, cu, vp, vp, ci, vp, sz, vp]
    L.hm_db_filter.restype = ci
    L.hm_db_filter.argtypes = [vp, i64, vp, cu, vp, vp, vp, vp, vp, vp]
    L.hm_gather_points.restype = ci
    L.hm_gather_points.argtypes = [vp, vp, vp, i64, ci, vp, i64, vp, i64, vp, vp, vp]
    L.hm_rasterize_mask.restype = ci
    L.hm_rasterize_mask.argtypes = [vp, i64, ci, ci, vp, ci, ci, i64, vp]
    L.hm_context_create.restype = ci
    L.hm_context_create.argtypes = [c.POINTER(vp)]
    L.hm_context_destroy.restype = None
    L.hm_context_destroy.argtypes = [vp]
    L.hm_resident_query_begin.restype = ci
    L.hm_resident_query_begin.argtypes = [vp, vp, i64, i64, vp, i64, u64, ci, ci, ci, vp, i64, c.c_uint32]
    L.hm_resident_query_end.restype = ci
    L.hm_resident_query_end.argtypes = [vp, i64, vp]
    L.hm_knn2_host.restype = ci
    L.hm_knn2_host.argtypes = [vp, vp, i64, vp, i64, vp, ci]
    L.hm_frame_put.restype = ci
    L.hm_frame_put.argtypes = [vp, ci, vp, i64, i64, vp]
    L.hm_frame_match.restype = ci
    L.hm_frame_match.argtypes = [vp, ci, ci, cu, vp, c.c_double, ci, vp, vp, vp, vp, vp, vp]
    L.hm_match_host.restype = ci
    L.hm_match_host.argtypes = [vp, vp, i64, i64, vp, i64, i64, cu, vp, c.c_double, ci, vp, vp, vp, vp]
    L.hm_orb_workspace_bytes.restype = sz
    L.hm_orb_workspace_bytes.argtypes = [ci, ci, ci]
    L.hm_orb_level_geometry.restype = ci
    L.hm_orb_level_geometry.argtypes = [ci, ci, ci, c.POINTER(ci), c.POINTER(ci), c.POINTER(c.c_float)]
    L.hm_orb_angles_to_cs.restype = ci
    L.hm_orb_angles_to_cs.argtypes = [vp, i64, vp]
    L.hm_orb_build_pyramid.restype = ci
    L.hm_orb_build_pyramid.argtypes = [vp, ci, ci, i64, ci, ci, vp, sz, vp]
    L.hm_orb_describe.restype = ci
    L.hm_orb_describe.argtypes = [vp, ci, ci, ci, vp, vp, vp, i64, vp, i64, vp]
    L.hm_frame_put_orb.restype = ci
    L.hm_frame_put_orb.argtypes = [vp, ci, vp, ci, ci, i64, ci, ci, vp, vp, vp, i64, vp, vp]


def lib():
    """Load libhm_matcher.so (built by ``python -m slam_experiments_b200.build``)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(SO_PATH):
                    raise NativeError(
                        f"{SO_PATH} not found: build it with `python -m slam_experiments_b200.build` "
                        "(there is no CPU fallback)")
                L = ctypes.CDLL(SO_PATH)
                _declare(L)
                _lib = L
    return _lib


def last_error() -> str:
    return lib().hm_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != HM_OK:
        raise NativeError(f"{what} failed with status {rc}: {last_error()}")


def require_cuda(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise NativeError("no CUDA device visible: the Hamming matcher runs on B200 only (no CPU fallback)")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise NativeError(f"device {dev} is not a CUDA device (no CPU fallback)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


_NULL_CONTEXT = contextlib.nullcontext()


def on_device(dev: torch.device):
    """Context manager that makes ``dev`` current -- a shared no-op object when it already is (torch's own
    context manager costs ~10 us per use, which is visible on the small-problem and end-to-end paths)."""
    if torch.cuda.current_device() == dev.index:
        return _NULL_CONTEXT
    return torch.cuda.device(dev)


def variant_id(variant) -> int:
    try:
        return VARIANTS[variant]
    except KeyError:
        raise ValueError(f"unknown variant {variant!r}; expected 'auto', 'popc', 'i8' or 'f4'") from None


def tensor_variant(variant="auto") -> int:
    """The tensor-core core (``VARIANT_I8`` / ``VARIANT_F4``) a prepared-operand call uses."""
    v = variant_id(variant)
    if v == VARIANT_AUTO:
        v = lib().hm_default_tensor_variant()
    if v not in (VARIANT_I8, VARIANT_F4):
        raise ValueError(f"variant {variant!r} has no prepared operand format")
    return v


# ---- workspace cache: one growing uint8 tensor per (device, stream) ---------------------------
_ws_cache = {}


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, threading.get_ident())
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


WS_CLOCK_PROBE_OFFSET = 64      # HM_WS_CLOCK_PROBE_OFFSET


def clock_probe(device) -> Optional[dict]:
    """SM clock the last tensor-core k-NN kernel on this thread / stream really ran at: the kernel's first CTA stamps
    %globaltimer and clock64 at entry and exit into its workspace header (``HM_WS_CLOCK_PROBE_OFFSET``).  Synchronises.
    Returns ``{"sm_mhz_effective", "cta0_us"}`` or None when no such kernel has run on the cached workspace."""
    device = torch.device(device)
    key = (device.index, torch.cuda.current_stream(device).cuda_stream, threading.get_ident())
    buf = _ws_cache.get(key)
    if buf is None:
        return None
    vals = buf[WS_CLOCK_PROBE_OFFSET:WS_CLOCK_PROBE_OFFSET + 32].cpu().numpy().view(np.int64)
    ns, cyc = int(vals[2] - vals[0]), int(vals[3] - vals[1])
    if ns <= 0 or cyc <= 0:
        return None
    return {"sm_mhz_effective": cyc / ns * 1e3, "cta0_us": ns / 1e3}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _check_desc(t: torch.Tensor, name: str, ndim: int = 2) -> None:
    if t.dtype != torch.uint8 or t.dim() != ndim or t.shape[-1] != DESC_BYTES or not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA uint8 tensor of shape [..., {DESC_BYTES}]")
    if t.stride(-1) != 1 or (t.numel() and (t.stride(-2) % 16 or t.data_ptr() % 16)):
        raise ValueError(f"{name} rows must be 16-byte aligned with unit element stride")


def knn2_keys(query: torch.Tensor, train: torch.Tensor, train_base: int = 0, variant="auto",
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_knn2``: packed top-2 keys ``[Nq, 2]`` (int64 storage of the uint64 keys)."""
    _check_desc(query, "query")
    _check_desc(train, "train")
    dev = query.device
    nq, nt = query.shape[0], train.shape[0]
    if out is None:
        out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    v = variant_id(variant)
    L = lib()
    with on_device(dev):
        wsb = L.hm_workspace_bytes(nq, nt, 1, v)
        ws = workspace(wsb, dev)
        check(L.hm_knn2(query.data_ptr(), nq, query.stride(0) if nq else DESC_BYTES,
                        train.data_ptr(), nt, train.stride(0) if nt else DESC_BYTES,
                        train_base, out.data_ptr(), v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_knn2")
    return out


def knn2_keys_batched(query: torch.Tensor, train: torch.Tensor, variant="auto",
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_knn2_batched`` over ``query[B, Nq, 32]`` and ``train[B, Nt, 32]`` (strided views allowed)."""
    _check_desc(query, "query", 3)
    _check_desc(train, "train", 3)
    if query.shape[0] != train.shape[0]:
        raise ValueError("batch sizes differ")
    dev = query.device
    b, nq, nt = query.shape[0], query.shape[1], train.shape[1]
    if out is None:
        out = torch.empty((b, nq, 2), dtype=torch.int64, device=dev)
    v = variant_id(variant)
    L = lib()
    with on_device(dev):
        wsb = L.hm_workspace_bytes(nq, nt, b, v)
        ws = workspace(wsb, dev)
        check(L.hm_knn2_batched(query.data_ptr(), nq, query.stride(1) if nq else DESC_BYTES, query.stride(0),
                                train.data_ptr(), nt, train.stride(1) if nt else DESC_BYTES, train.stride(0),
                                b, out.data_ptr(), v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)),
              "hm_knn2_batched")
    return out


def prepared_bytes(n: int, variant="auto") -> int:
    return int(lib().hm_prepared_bytes(n, tensor_variant(variant)))


def prepare(bits: torch.Tensor, out: Optional[torch.Tensor] = None, variant="auto") -> torch.Tensor:
    """``hm_prepare``: expand packed descriptors to the +/-1 tensor-core image of ``variant``
    (int8 for ``"i8"``, e2m1 for ``"f4"``)."""
    _check_desc(bits, "bits")
    dev = bits.device
    n = bits.shape[0]
    v = tensor_variant(variant)
    nbytes = prepared_bytes(n, v)
    if out is None:
        out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    elif out.numel() < nbytes:
        raise ValueError("prepared buffer too small")
    with on_device(dev):
        check(lib().hm_prepare(bits.data_ptr(), n, bits.stride(0) if n else DESC_BYTES, out.data_ptr(), v,
                               _stream_ptr(dev)), "hm_prepare")
    return out


def knn2_keys_prepared(query_prepared: torch.Tensor, nq: int, train_prepared: torch.Tensor, nt: int,
                       train_base: int = 0, out: Optional[torch.Tensor] = None, variant="auto") -> torch.Tensor:
    dev = query_prepared.device
    if out is None:
        out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    v = tensor_variant(variant)
    L = lib()
    with on_device(dev):
        wsb = L.hm_prepared_workspace_bytes(nq, nt, v)
        ws = workspace(wsb, dev)
        check(L.hm_knn2_prepared(query_prepared.data_ptr(), nq, train_prepared.data_ptr(), nt, train_base,
                                 out.data_ptr(), v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_knn2_prepared")
    return out


def knn2_keys_resident(query: torch.Tensor, train_prepared: torch.Tensor, nt: int, train_base: int = 0,
                       out: Optional[torch.Tensor] = None, variant="auto") -> torch.Tensor:
    """``hm_knn2_resident``: packed query descriptors against a resident prepared database -- one launch with the
    ``f4`` core (the kernel expands the query rows itself)."""
    _check_desc(query, "query")
    dev = query.device
    nq = query.shape[0]
    if out is None:
        out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    if nq == 0:
        return out
    v = tensor_variant(variant)
    L = lib()
    with on_device(dev):
        ws = workspace(L.hm_resident_workspace_bytes(nq, nt, v), dev)
        check(L.hm_knn2_resident(query.data_ptr(), nq, query.stride(0), train_prepared.data_ptr(), nt, train_base,
                                 out.data_ptr(), v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_knn2_resident")
    return out


def knn2_resident_exchange(query: torch.Tensor, train_prepared: torch.Tensor, nt: int, train_base: int, world: int,
                           rank: int, peer_ptrs, max_rows: int, epoch: int, out: Optional[torch.Tensor] = None,
                           variant="auto") -> torch.Tensor:
    """``hm_knn2_resident_exchange``: the same with the cross-GPU exchange inside the kernel's last-CTA merge."""
    _check_desc(query, "query")
    dev = query.device
    nq = query.shape[0]
    if out is None:
        out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    v = tensor_variant(variant)
    L = lib()
    with on_device(dev):
        ws = workspace(L.hm_resident_workspace_bytes(nq, nt, v), dev)
        check(L.hm_knn2_resident_exchange(query.data_ptr(), nq, query.stride(0), train_prepared.data_ptr(), nt, train_base,
                                          world, rank, peer_ptrs, max_rows, epoch, out.data_ptr(), v, ws.data_ptr(),
                                          ws.numel(), _stream_ptr(dev)), "hm_knn2_resident_exchange")
    return out


# ---- selections of train rows as runs (include/hm_matcher.h, "search a selection of the train rows") -------------
def run_table(runs: np.ndarray) -> np.ndarray:
    """The device layout of a run list ``int64 [n, 2]`` (lo, hi): ``int64 [n, 4]`` = lo, hi, the 128-row tiles and the
    rows of the runs before it."""
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    tiles = -(-runs[:, 1] // 128) - runs[:, 0] // 128
    rows = runs[:, 1] - runs[:, 0]
    out = np.empty((runs.shape[0], 4), np.int64)
    out[:, :2] = runs
    out[:, 2] = np.cumsum(tiles) - tiles
    out[:, 3] = np.cumsum(rows) - rows
    return out


def runs_workspace_bytes(nq: int, runs: np.ndarray, prepared: bool, variant="auto") -> int:
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    v = tensor_variant(variant) if prepared else variant_id(variant)
    return int(lib().hm_runs_workspace_bytes(nq, runs.ctypes.data, runs.shape[0], int(prepared), v))


def describe_runs_launch(nq: int, nt: int, runs: np.ndarray, variant="auto", pieces: bool = False):
    """``hm_describe_runs_launch`` (host arithmetic, no device needed): the resident launch of a run list as text, and
    with ``pieces`` the tile walk ``int64 [T, 4]`` = (split, physical tile, first row, end row) per virtual tile."""
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    L = lib()
    n = L.hm_describe_runs_launch(nq, nt, runs.ctypes.data, runs.shape[0], tensor_variant(variant), None, 0, None)
    if n < 0:
        raise NativeError(f"hm_describe_runs_launch failed with status {n}: {last_error()}")
    buf = ctypes.create_string_buffer(256)
    out = np.zeros((n, 4), np.int64)
    check(min(0, L.hm_describe_runs_launch(nq, nt, runs.ctypes.data, runs.shape[0], tensor_variant(variant), buf, 256,
                                           out.ctypes.data if pieces and n else None)), "hm_describe_runs_launch")
    return (buf.value.decode(), out) if pieces else buf.value.decode()


def knn2_keys_resident_runs(query: torch.Tensor, train_prepared: torch.Tensor, nt: int, runs: np.ndarray,
                            runs_dev: torch.Tensor, train_base: int = 0, variant="auto", exchange=None) -> torch.Tensor:
    """``hm_knn2_resident_runs`` (``exchange`` = (world, rank, peer_ptrs, max_rows, epoch):
    ``hm_knn2_resident_runs_exchange``): top-2 keys over the runs ``[lo, hi)`` of a resident prepared database.
    ``runs_dev`` is :func:`run_table` of ``runs`` on the device."""
    _check_desc(query, "query")
    dev = query.device
    nq = query.shape[0]
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    v = tensor_variant(variant)
    L = lib()
    with on_device(dev):
        ws = workspace(L.hm_runs_workspace_bytes(nq, runs.ctypes.data, runs.shape[0], 1, v), dev)
        if exchange is None:
            check(L.hm_knn2_resident_runs(query.data_ptr(), nq, query.stride(0), train_prepared.data_ptr(), nt,
                                          runs.ctypes.data, runs_dev.data_ptr(), runs.shape[0], train_base, out.data_ptr(),
                                          v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_knn2_resident_runs")
        else:
            world, rank, peer_ptrs, max_rows, epoch = exchange
            check(L.hm_knn2_resident_runs_exchange(query.data_ptr(), nq, query.stride(0), train_prepared.data_ptr(), nt,
                                                   runs.ctypes.data, runs_dev.data_ptr(), runs.shape[0], train_base, world,
                                                   rank, peer_ptrs, max_rows, epoch, out.data_ptr(), v, ws.data_ptr(),
                                                   ws.numel(), _stream_ptr(dev)), "hm_knn2_resident_runs_exchange")
    return out


def knn2_keys_runs(query: torch.Tensor, train: torch.Tensor, runs: np.ndarray, runs_dev: torch.Tensor,
                   train_base: int = 0, variant="auto") -> torch.Tensor:
    """``hm_knn2_runs``: top-2 keys over the runs ``[lo, hi)`` of packed train rows (gathered into the workspace)."""
    _check_desc(query, "query")
    _check_desc(train, "train")
    dev = query.device
    nq, nt = query.shape[0], train.shape[0]
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    v = variant_id(variant)
    L = lib()
    with on_device(dev):
        ws = workspace(L.hm_runs_workspace_bytes(nq, runs.ctypes.data, runs.shape[0], 0, v), dev)
        check(L.hm_knn2_runs(query.data_ptr(), nq, query.stride(0) if nq else DESC_BYTES, train.data_ptr(), nt,
                             train.stride(0) if nt else DESC_BYTES, runs.ctypes.data, runs_dev.data_ptr(), runs.shape[0],
                             train_base, out.data_ptr(), v, ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_knn2_runs")
    return out


def merge_top2(keys: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_merge_top2``: ``keys[G, rows, 2]`` -> ``[rows, 2]``."""
    if keys.dim() != 3 or keys.shape[2] != 2 or keys.dtype != torch.int64 or not keys.is_contiguous():
        raise ValueError("keys must be a contiguous int64 tensor [G, rows, 2]")
    dev = keys.device
    g, rows = keys.shape[0], keys.shape[1]
    if out is None:
        out = torch.empty((rows, 2), dtype=torch.int64, device=dev)
    with on_device(dev):
        check(lib().hm_merge_top2(keys.data_ptr(), g, rows, out.data_ptr(), _stream_ptr(dev)), "hm_merge_top2")
    return out


def exchange_bytes(max_rows: int, world: int) -> int:
    return int(lib().hm_exchange_bytes(max_rows, world))


def exchange_merge(local_keys, world: int, rank: int, peer_ptrs, max_rows: int, epoch: int,
                   out: Optional[torch.Tensor] = None, *, rows: Optional[int] = None, groups: int = 1,
                   device=None) -> torch.Tensor:
    """``hm_exchange_merge``: push local keys to every peer's symmetric buffer, flag, wait, merge.

    ``local_keys`` is a ``[rows, 2]`` tensor, or a raw device pointer to ``[groups][rows][2]`` partials
    (from :func:`knn2_partials_prepared`) together with ``rows`` / ``groups`` / ``device``."""
    if isinstance(local_keys, torch.Tensor):
        dev, rows, ptr = local_keys.device, local_keys.shape[0], local_keys.data_ptr()
    else:
        dev, ptr = device, int(local_keys)
    if out is None:
        out = torch.empty((rows, 2), dtype=torch.int64, device=dev)
    arr = peer_ptrs if isinstance(peer_ptrs, ctypes.Array) else (ctypes.c_void_p * world)(*[int(p) for p in peer_ptrs])
    with on_device(dev):
        check(lib().hm_exchange_merge(ptr, groups, rows, world, rank, arr, max_rows, epoch, out.data_ptr(),
                                      _stream_ptr(dev)), "hm_exchange_merge")
    return out


def knn2_prepared_exchange(query_prepared: torch.Tensor, nq: int, train_prepared: torch.Tensor, nt: int,
                           train_base: int, world: int, rank: int, peer_ptrs, max_rows: int, epoch: int,
                           out: Optional[torch.Tensor] = None, variant="auto") -> torch.Tensor:
    """``hm_knn2_prepared_exchange``: local k-NN + cross-GPU exchange + merge in one launch."""
    dev = query_prepared.device
    if out is None:
        out = torch.empty((nq, 2), dtype=torch.int64, device=dev)
    arr = peer_ptrs if isinstance(peer_ptrs, ctypes.Array) else (ctypes.c_void_p * world)(*[int(p) for p in peer_ptrs])
    v = tensor_variant(variant)
    L = lib()
    with on_device(dev):
        wsb = L.hm_prepared_workspace_bytes(nq, nt, v)
        ws = workspace(wsb, dev)
        check(L.hm_knn2_prepared_exchange(query_prepared.data_ptr(), nq, train_prepared.data_ptr(), nt, train_base,
                                          world, rank, arr, max_rows, epoch, out.data_ptr(), v, ws.data_ptr(),
                                          ws.numel(), _stream_ptr(dev)), "hm_knn2_prepared_exchange")
    return out


def knn2_partials_prepared(query_prepared: torch.Tensor, nq: int, train_prepared: torch.Tensor, nt: int,
                           train_base: int = 0, variant="auto"):
    """``hm_knn2_prepared_partials``: returns ``(device_ptr, groups)`` of the unmerged per-split keys,
    valid until the cached workspace is reused on this stream."""
    dev = query_prepared.device
    L = lib()
    parts, groups = ctypes.c_void_p(), ctypes.c_int(0)
    v = tensor_variant(variant)
    with on_device(dev):
        wsb = L.hm_prepared_workspace_bytes(nq, nt, v)
        ws = workspace(wsb, dev)
        check(L.hm_knn2_prepared_partials(query_prepared.data_ptr(), nq, train_prepared.data_ptr(), nt, train_base,
                                          v, ws.data_ptr(), ws.numel(), _stream_ptr(dev), ctypes.byref(parts),
                                          ctypes.byref(groups)), "hm_knn2_prepared_partials")
    return parts.value, groups.value


def ratio_lut(ratio: float) -> np.ndarray:
    """``lut[d2] = ceil(ratio * d2)`` in float64: ``d1 < ratio*d2  <=>  d1 < lut[d2]`` for integer d1."""
    import math
    lut = np.empty(257, dtype=np.uint16)
    for d2 in range(257):
        lut[d2] = min(65535, max(0, math.ceil(float(ratio) * float(d2))))
    return lut


_lut_cache = {}


def _ratio_lut_cached(ratio: float) -> np.ndarray:
    lut = _lut_cache.get(ratio)
    if lut is None:
        lut = _lut_cache[ratio] = ratio_lut(ratio)
    return lut


def match_fused(query: torch.Tensor, train: torch.Tensor, ratio: Optional[float] = None,
                cross_check: bool = False, dist_threshold: Optional[float] = None, variant="auto",
                want_keys: bool = False):
    """``hm_match_fused`` over ``[B, Nq, 32]`` / ``[B, Nt, 32]``.

    Returns ``(q, t, d, count[, keys])`` device tensors; row ``b`` holds ``count[b]`` matches
    ordered by queryIdx.
    """
    _check_desc(query, "query", 3)
    _check_desc(train, "train", 3)
    dev = query.device
    b, nq, nt = query.shape[0], query.shape[1], train.shape[1]
    flags = 0
    lut_ptr = None
    lut = None
    if ratio is not None:
        flags |= FLAG_RATIO
        lut = ratio_lut(ratio)
        lut_ptr = lut.ctypes.data
    if cross_check:
        flags |= FLAG_MUTUAL
    thr = 0.0
    if dist_threshold:
        flags |= FLAG_DIST_THRESHOLD
        thr = float(dist_threshold)
    oq = torch.empty((b, nq), dtype=torch.int32, device=dev)
    ot = torch.empty((b, nq), dtype=torch.int32, device=dev)
    od = torch.empty((b, nq), dtype=torch.int32, device=dev)
    cnt = torch.empty((b,), dtype=torch.int32, device=dev)
    keys = torch.empty((b, nq, 2), dtype=torch.int64, device=dev) if want_keys else None
    v = variant_id(variant)
    L = lib()
    with on_device(dev):
        wsb = L.hm_workspace_bytes(nq, nt, b, v)
        ws = workspace(wsb, dev)
        check(L.hm_match_fused(query.data_ptr(), nq, query.stride(1) if nq else DESC_BYTES, query.stride(0),
                               train.data_ptr(), nt, train.stride(1) if nt else DESC_BYTES, train.stride(0),
                               b, flags, lut_ptr, thr, oq.data_ptr(), ot.data_ptr(), od.data_ptr(), cnt.data_ptr(),
                               keys.data_ptr() if keys is not None else None, v, ws.data_ptr(), ws.numel(),
                               _stream_ptr(dev)), "hm_match_fused")
    del lut
    return (oq, ot, od, cnt, keys) if want_keys else (oq, ot, od, cnt)


def _check_keys(keys: torch.Tensor) -> None:
    if keys.dtype != torch.int64 or keys.dim() != 2 or keys.shape[1] != 2 or not keys.is_cuda or not keys.is_contiguous():
        raise ValueError("keys must be a contiguous CUDA int64 tensor [Nq, 2]")


def db_mutual_workspace_bytes(nq: int, variant="auto") -> int:
    return int(lib().hm_db_mutual_workspace_bytes(nq, variant_id(variant)))


def db_mutual_flags(keys: torch.Tensor, query: torch.Tensor, shard_bits: torch.Tensor, row_lo: int,
                    ratio: Optional[float] = None, variant="auto", out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_db_mutual_flags``: ``uint8 [Nq]`` mutual flags of one shard of a keyframe database.

    ``keys`` are the global top-2 keys of ``query`` over the whole database; ``shard_bits`` holds the database rows
    ``[row_lo, row_lo + len(shard_bits))``.  ``flags[q] = 1`` iff the best row of ``q`` lies in this shard (and passes
    the ratio test when ``ratio`` is given) and ``q`` is the lowest-index nearest query of that row; every other entry
    is 0, so the element-wise maximum over all shards is the database-wide mutual check."""
    _check_keys(keys)
    _check_desc(query, "query")
    _check_desc(shard_bits, "shard_bits")
    nq, rows = query.shape[0], shard_bits.shape[0]
    if keys.shape[0] != nq:
        raise ValueError("keys and query differ in rows")
    dev = query.device
    if out is None:
        out = torch.empty(nq, dtype=torch.uint8, device=dev)
    flags, lut = (FLAG_MUTUAL | FLAG_RATIO, _ratio_lut_cached(float(ratio))) if ratio is not None else (FLAG_MUTUAL, None)
    v = variant_id(variant)
    L = lib()
    with on_device(dev):
        ws = workspace(L.hm_db_mutual_workspace_bytes(nq, v), dev)
        check(L.hm_db_mutual_flags(keys.data_ptr(), nq, query.data_ptr(), query.stride(0) if nq else DESC_BYTES,
                                   shard_bits.data_ptr(), rows, shard_bits.stride(0) if rows else DESC_BYTES, row_lo,
                                   flags, lut.ctypes.data if lut is not None else None, out.data_ptr(), v,
                                   ws.data_ptr(), ws.numel(), _stream_ptr(dev)), "hm_db_mutual_flags")
    return out


def db_filter(keys: torch.Tensor, mutual_flags: Optional[torch.Tensor] = None, ratio: Optional[float] = None):
    """``hm_db_filter``: ratio test and (with ``mutual_flags``) the mutual check on global top-2 keys, compacted in
    query order.  Returns ``(q, t, d, count)`` device tensors: ``q / t / d [Nq] int32`` (queryIdx, global database row,
    distance), valid up to ``count [1]``."""
    _check_keys(keys)
    nq = keys.shape[0]
    dev = keys.device
    flags, lut = (FLAG_RATIO, _ratio_lut_cached(float(ratio))) if ratio is not None else (0, None)
    if mutual_flags is not None:
        if mutual_flags.dtype != torch.uint8 or not mutual_flags.is_cuda or mutual_flags.numel() < nq:
            raise ValueError("mutual_flags must be a CUDA uint8 tensor of at least Nq entries")
        flags |= FLAG_MUTUAL
    out = torch.empty((3, nq), dtype=torch.int32, device=dev)
    cnt = torch.empty(1, dtype=torch.int32, device=dev)
    with on_device(dev):
        check(lib().hm_db_filter(keys.data_ptr(), nq, mutual_flags.data_ptr() if mutual_flags is not None else None, flags,
                                 lut.ctypes.data if lut is not None else None, out[0].data_ptr(), out[1].data_ptr(),
                                 out[2].data_ptr(), cnt.data_ptr(), _stream_ptr(dev)), "hm_db_filter")
    return out[0], out[1], out[2], cnt


def gather_points(q_idx: torch.Tensor, t_idx: torch.Tensor, count: torch.Tensor, query_pts: torch.Tensor,
                  train_pts: torch.Tensor):
    """``hm_gather_points``: packed matched-point arrays from a device match list.

    ``q_idx`` / ``t_idx`` ``[B, nq]`` int32 and ``count`` ``[B]`` as returned by :func:`match_fused`;
    ``query_pts`` ``[B, nq, 2]`` / ``train_pts`` ``[B, nt, 2]`` int32.  Returns ``(out_query, out_train)``
    ``[B, nq, 2]`` int32; rows ``>= count[b]`` are undefined."""
    for t, name in ((query_pts, "query_pts"), (train_pts, "train_pts")):
        if t.dtype != torch.int32 or t.dim() != 3 or t.shape[2] != 2 or not t.is_cuda or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous CUDA int32 tensor [B, N, 2]")
    b, stride = q_idx.shape
    dev = q_idx.device
    oq = torch.empty((b, stride, 2), dtype=torch.int32, device=dev)
    ot = torch.empty((b, stride, 2), dtype=torch.int32, device=dev)
    with on_device(dev):
        check(lib().hm_gather_points(q_idx.data_ptr(), t_idx.data_ptr(), count.data_ptr(), stride, b,
                                     query_pts.data_ptr(), query_pts.shape[1], train_pts.data_ptr(), train_pts.shape[1],
                                     oq.data_ptr(), ot.data_ptr(), _stream_ptr(dev)), "hm_gather_points")
    return oq, ot


def rasterize_mask(points: torch.Tensor, shape, radius: int, inner: bool = True,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_rasterize_mask``: the detection mask of `utils.py:58-74` as a ``[h, w] uint8`` CUDA tensor;
    ``points`` is a contiguous CUDA int32 ``[N, 2]`` tensor of (x, y) pixel positions."""
    if points.dtype != torch.int32 or points.dim() != 2 or points.shape[1] != 2 or not points.is_cuda or not points.is_contiguous():
        raise ValueError("points must be a contiguous CUDA int32 tensor [N, 2]")
    h, w = int(shape[0]), int(shape[1])
    dev = points.device
    if out is None:
        out = torch.empty((h, w), dtype=torch.uint8, device=dev)
    with on_device(dev):
        check(lib().hm_rasterize_mask(points.data_ptr(), points.shape[0], int(radius), 1 if inner else 0,
                                      out.data_ptr(), h, w, out.stride(0) if h else w, _stream_ptr(dev)), "hm_rasterize_mask")
    return out


# ---- ORB descriptor stage (hm_orb.cu) --------------------------------------------------------------------
def orb_level_geometry(rows: int, cols: int, level: int):
    """``(rows, cols, 1 / scale)`` of pyramid level ``level`` -- host arithmetic, no device needed."""
    r, c_, inv = ctypes.c_int(), ctypes.c_int(), ctypes.c_float()
    check(lib().hm_orb_level_geometry(int(rows), int(cols), int(level), ctypes.byref(r), ctypes.byref(c_), ctypes.byref(inv)),
          "hm_orb_level_geometry")
    return r.value, c_.value, inv.value


def orb_angles_to_cs(angles_deg: np.ndarray) -> np.ndarray:
    """``[n, 2] float32`` (cos, sin) of keypoint angles in degrees, computed the way cv2 computes them."""
    a = np.ascontiguousarray(angles_deg, dtype=np.float32).reshape(-1)
    out = np.empty((a.shape[0], 2), np.float32)
    check(lib().hm_orb_angles_to_cs(a.ctypes.data if a.shape[0] else None, a.shape[0], out.ctypes.data if a.shape[0] else None),
          "hm_orb_angles_to_cs")
    return out


def orb_build_pyramid(image: torch.Tensor, n_levels: int = 8, workspace: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_orb_build_pyramid``: CUDA uint8 image ``[h, w]`` (gray) or ``[h, w, 3]`` (BGR) -> the workspace tensor that
    holds the framed, blurred scale pyramid (input of :func:`orb_describe`)."""
    if image.dtype != torch.uint8 or not image.is_cuda or image.dim() not in (2, 3) or (image.dim() == 3 and image.shape[2] != 3):
        raise ValueError("image must be a CUDA uint8 tensor [h, w] or [h, w, 3]")
    if image.stride(-1) != 1 or (image.dim() == 3 and image.stride(1) != 3):
        image = image.contiguous()
    h, w, ch = int(image.shape[0]), int(image.shape[1]), (3 if image.dim() == 3 else 1)
    need = lib().hm_orb_workspace_bytes(h, w, int(n_levels))
    if not need:
        raise NativeError(f"hm_orb_workspace_bytes failed: {last_error()}")
    dev = image.device
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    with on_device(dev):
        check(lib().hm_orb_build_pyramid(image.data_ptr(), h, w, image.stride(0), ch, int(n_levels), workspace.data_ptr(),
                                         workspace.numel(), _stream_ptr(dev)), "hm_orb_build_pyramid")
    return workspace


def orb_describe(workspace: torch.Tensor, shape, n_levels: int, xy: torch.Tensor, cs: torch.Tensor, octave: torch.Tensor,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``hm_orb_describe``: ``[n, 32] uint8`` rBRIEF descriptors of ``n`` keypoints (``xy`` / ``cs`` float32 ``[n, 2]``,
    ``octave`` int32 ``[n]``, all contiguous CUDA tensors) from a pyramid built for an image of ``shape``."""
    n = int(xy.shape[0])
    dev = workspace.device
    for t, dt in ((xy, torch.float32), (cs, torch.float32), (octave, torch.int32)):
        if t.dtype != dt or not t.is_cuda or not t.is_contiguous() or t.shape[0] != n:
            raise ValueError("xy / cs must be contiguous CUDA float32 [n, 2], octave int32 [n]")
    if out is None:
        out = torch.empty((n, DESC_BYTES), dtype=torch.uint8, device=dev)
    with on_device(dev):
        check(lib().hm_orb_describe(workspace.data_ptr(), int(shape[0]), int(shape[1]), int(n_levels), xy.data_ptr(), cs.data_ptr(),
                                    octave.data_ptr(), n, out.data_ptr(), out.stride(0) if n else DESC_BYTES, _stream_ptr(dev)),
              "hm_orb_describe")
    return out


def profile_events(start: Optional[torch.cuda.Event], stop: Optional[torch.cuda.Event]) -> None:
    """``hm_profile_events``: record ``start``/``stop`` around the dominant kernel of later calls
    made from this thread (events must have been created with ``enable_timing=True``)."""
    if start is None or stop is None:
        lib().hm_profile_events(None, None)
        return
    for e in (start, stop):          # torch creates the cudaEvent lazily on first record
        if not e.cuda_event:
            e.record()
    lib().hm_profile_events(start.cuda_event, stop.cuda_event)


def describe_launch(nq: int, nt: int, batch: int = 1, variant="auto") -> str:
    """``hm_describe_launch``: kernel name and grid the k-NN call would use for this shape."""
    buf = ctypes.create_string_buffer(256)
    check(lib().hm_describe_launch(nq, nt, batch, variant_id(variant), buf, 256), "hm_describe_launch")
    return buf.value.decode()


def sm_count() -> int:
    n = lib().hm_device_sm_count()
    if n < 0:
        raise NativeError(f"hm_device_sm_count failed with status {n}: {last_error()}")
    return n


def select_variant(nq: int, nt: int, batch: int = 1) -> str:
    return VARIANT_NAMES[lib().hm_select_variant(nq, nt, batch)]


def split_keys(keys: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Host-side decode of packed keys: ``(idx int64, dist int32, valid bool)``."""
    k = np.asarray(keys).view(np.uint64)
    valid = k != np.uint64(NO_MATCH)
    return (k & np.uint64(0xFFFFFFFF)).astype(np.int64), (k >> np.uint64(32)).astype(np.int32), valid


def locate_rows(starts: np.ndarray, gidx: np.ndarray):
    """Global train rows -> ``(imgIdx, trainIdx)`` of cv2's collection API, given the first global row of
    every train image (``starts``, length n_images + 1).  Equal-sized images (the usual fixed ORB budget)
    are located by one division instead of a binary search (0.25 ms per 4000 rows against 4096 images)."""
    n = len(starts) - 1
    size = int(starts[1] - starts[0]) if n > 0 else 0
    if size > 0 and int(starts[-1]) == size * n and _uniform_starts(starts, size):
        img = gidx // size
        return img.astype(np.int32), (gidx - img * size).astype(np.int32)
    img = np.searchsorted(starts, gidx, side="right") - 1
    return img.astype(np.int32), (gidx - starts[img]).astype(np.int32)


_uniform_cache = {}


def _uniform_starts(starts: np.ndarray, size: int) -> bool:
    key = (starts.ctypes.data, len(starts), size)
    hit = _uniform_cache.get(key)
    if hit is None or hit[0] is not starts:
        ok = bool((np.diff(starts) == size).all())
        _uniform_cache.clear()
        _uniform_cache[key] = hit = (starts, ok)
    return hit[1]


class HostContext:
    """``hm_context``: numpy in / numpy out through the C ABI alone (no torch tensors)."""

    def __init__(self):
        require_cuda()
        self._h = ctypes.c_void_p()
        check(lib().hm_context_create(ctypes.byref(self._h)), "hm_context_create")

    def knn2_keys(self, query: np.ndarray, train: np.ndarray, variant="auto") -> np.ndarray:
        q = np.ascontiguousarray(query, dtype=np.uint8)
        t = np.ascontiguousarray(train, dtype=np.uint8)
        out = np.empty((q.shape[0], 2), dtype=np.uint64)
        check(lib().hm_knn2_host(self._h, q.ctypes.data, q.shape[0], t.ctypes.data, t.shape[0],
                                 out.ctypes.data, variant_id(variant)), "hm_knn2_host")
        return out

    def match(self, query: np.ndarray, train: np.ndarray, ratio: Optional[float] = None,
              cross_check: bool = False, dist_threshold: Optional[float] = None, variant="auto"):
        """``hm_match_host``: fused pipeline, numpy in -> ``(q, t, d)`` int32 arrays out."""
        q, t = query, train
        if q.strides[1] != 1 or q.strides[0] < DESC_BYTES:
            q = np.ascontiguousarray(q)
        if t.strides[1] != 1 or t.strides[0] < DESC_BYTES:
            t = np.ascontiguousarray(t)
        nq = q.shape[0]
        flags, lut_ptr, lut, thr = 0, None, None, 0.0
        if ratio is not None:
            flags |= FLAG_RATIO
            lut = _ratio_lut_cached(float(ratio))
            lut_ptr = lut.ctypes.data
        if cross_check:
            flags |= FLAG_MUTUAL
        if dist_threshold:
            flags |= FLAG_DIST_THRESHOLD
            thr = float(dist_threshold)
        out = np.empty((3, max(nq, 1)), dtype=np.int32)
        cnt = ctypes.c_int32(0)
        check(lib().hm_match_host(self._h, q.ctypes.data, nq, q.strides[0], t.ctypes.data, t.shape[0], t.strides[0],
                                  flags, lut_ptr, thr, variant_id(variant), out[0].ctypes.data, out[1].ctypes.data,
                                  out[2].ctypes.data, ctypes.byref(cnt)), "hm_match_host")
        n = cnt.value
        return out[0, :n], out[1, :n], out[2, :n]

    # ---- resident prepared database queried from host memory (hm_resident_query_begin / _end) ----
    def resident_query_begin(self, query: np.ndarray, train_prepared: torch.Tensor, nt: int, train_base: int = 0,
                             variant="auto", world: int = 1, rank: int = 0, peer_ptrs=None, max_rows: int = 0,
                             epoch: int = 0) -> int:
        q = query
        if q.strides[1] != 1 or q.strides[0] < DESC_BYTES:
            q = np.ascontiguousarray(q)
        check(lib().hm_resident_query_begin(self._h, q.ctypes.data, q.shape[0], q.strides[0], train_prepared.data_ptr(), nt,
                                            train_base, tensor_variant(variant), world, rank, peer_ptrs, max_rows, epoch),
              "hm_resident_query_begin")
        return q.shape[0]

    def resident_query_end(self, nq: int) -> np.ndarray:
        out = np.empty((nq, 2), dtype=np.uint64)
        check(lib().hm_resident_query_end(self._h, nq, out.ctypes.data), "hm_resident_query_end")
        return out

    # ---- resident frames (hm_frame_put / hm_frame_match) ----
    FRAME_SLOTS = 16

    def frame_put(self, slot: int, descriptors: np.ndarray, positions: Optional[np.ndarray] = None) -> None:
        d = descriptors
        if d.shape[0] and (d.strides[1] != 1 or d.strides[0] < DESC_BYTES):
            d = np.ascontiguousarray(d)
        p_ptr = None
        if positions is not None:
            positions = np.ascontiguousarray(positions, dtype=np.int32)
            p_ptr = positions.ctypes.data
        check(lib().hm_frame_put(self._h, slot, d.ctypes.data if d.shape[0] else None, d.shape[0],
                                 d.strides[0] if d.shape[0] else DESC_BYTES, p_ptr), "hm_frame_put")

    def frame_put_orb(self, slot: int, image: np.ndarray, xy: np.ndarray, angles_deg: np.ndarray, octaves: np.ndarray,
                      n_levels: int = 8, positions: Optional[np.ndarray] = None, want_descriptors: bool = False):
        """``hm_frame_put_orb``: the frame's descriptors are computed on the device from the image and cv2's keypoints and
        stored in ``slot``; returns them as ``[n, 32] uint8`` only when ``want_descriptors``."""
        img = image
        if img.dtype != np.uint8 or img.ndim not in (2, 3) or (img.ndim == 3 and img.shape[2] != 3):
            raise ValueError("image must be uint8 [h, w] or [h, w, 3]")
        if img.strides[-1] != 1 or (img.ndim == 3 and img.strides[1] != 3) or img.strides[0] < img.shape[1] * (3 if img.ndim == 3 else 1):
            img = np.ascontiguousarray(img)
        xy = np.ascontiguousarray(xy, dtype=np.float32).reshape(-1, 2)
        ang = np.ascontiguousarray(angles_deg, dtype=np.float32).reshape(-1)
        octv = np.ascontiguousarray(octaves, dtype=np.int32).reshape(-1)
        n = xy.shape[0]
        if ang.shape[0] != n or octv.shape[0] != n:
            raise ValueError("xy, angles and octaves must have one entry per keypoint")
        p_ptr = None
        if positions is not None:
            positions = np.ascontiguousarray(positions, dtype=np.int32)
            p_ptr = positions.ctypes.data
        out = np.empty((n, DESC_BYTES), np.uint8) if want_descriptors else None
        check(lib().hm_frame_put_orb(self._h, slot, img.ctypes.data, img.shape[0], img.shape[1], img.strides[0],
                                     3 if img.ndim == 3 else 1, int(n_levels), xy.ctypes.data if n else None,
                                     ang.ctypes.data if n else None, octv.ctypes.data if n else None, n, p_ptr,
                                     out.ctypes.data if (want_descriptors and n) else None), "hm_frame_put_orb")
        return out

    def frame_match(self, train_slot: int, query_slot: int, nq: int, ratio: Optional[float] = None,
                    cross_check: bool = False, dist_threshold: Optional[float] = None, variant="auto",
                    want_indices: bool = True, want_points: bool = False):
        """Match two resident frames.  Returns ``(q, t, d)`` int32 arrays and/or ``(query_pts, train_pts)``
        ``(M, 2)`` int32 arrays, depending on ``want_indices`` / ``want_points``."""
        flags, lut_ptr, lut, thr = 0, None, None, 0.0
        if ratio is not None:
            flags |= FLAG_RATIO
            lut = _ratio_lut_cached(float(ratio))
            lut_ptr = lut.ctypes.data
        if cross_check:
            flags |= FLAG_MUTUAL
        if dist_threshold:
            flags |= FLAG_DIST_THRESHOLD
            thr = float(dist_threshold)
        m = max(nq, 1)
        idx = np.empty((3, m), dtype=np.int32) if want_indices else None
        pts = np.empty((2, m, 2), dtype=np.int32) if want_points else None
        cnt = ctypes.c_int32(0)
        check(lib().hm_frame_match(self._h, train_slot, query_slot, flags, lut_ptr, thr, variant_id(variant),
                                   idx[0].ctypes.data if want_indices else None, idx[1].ctypes.data if want_indices else None,
                                   idx[2].ctypes.data if want_indices else None,
                                   pts[0].ctypes.data if want_points else None, pts[1].ctypes.data if want_points else None,
                                   ctypes.byref(cnt)), "hm_frame_match")
        n = cnt.value
        out = ()
        if want_indices:
            out += (idx[0, :n], idx[1, :n], idx[2, :n])
        if want_points:
            out += (pts[0, :n], pts[1, :n])
        return out

    def close(self):
        if self._h:
            lib().hm_context_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
