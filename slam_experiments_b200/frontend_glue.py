"""Host-side mirror of the reference code either side of the matcher call (SURVEY.md 8a rows a5-a7,
8f ranks 1-2): descriptor packing, the `_match_features` call site, and the consumers of
``queryIdx`` / ``trainIdx``.

The reference's own versions are Python loops over ``Feature`` objects:

* ``Frame.get_descriptors`` (`/root/reference/primitives.py:200-205`) copies each feature's 32-byte
  descriptor into a fresh ``(N, 32) uint8`` array on every call (0.7 ms at 2,000 features) and
  returns ``np.array([])`` -- shape ``(0,)``, float64 -- for a frame without features;
* ``Frontend._match_features`` (`/root/reference/frontend.py:181-187`) packs the last and the
  current frame and calls ``matcher.match(desc_last, desc_cur)`` (train = last frame);
* the consumers (`frontend.py:174-177,194,205-207`; `utils.py:13-19,41-47`) only index
  ``last.features[m.trainIdx]`` and ``current.features[m.queryIdx]``.

``get_descriptors`` / ``match_features`` / ``propagate_map_points`` reproduce those semantics
exactly and work on the reference's own ``Frame`` / ``Feature`` objects (duck-typed: anything with
``.features`` whose items have ``.descriptor``, ``.keypoint.pt`` / ``.position`` and ``.map_point``).
``FrameDescriptorStore`` is the device-resident replacement for the per-call repacking: every
frame's descriptors are uploaded once when the frame is created, so frame-to-frame tracking moves
only the new frame (64 KB at 2,000 features) and the train side is already in HBM.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Any, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as nat
from .feature_matchers import BruteForceFeatureMatcher, MatcherError, _build_dmatches


def get_descriptors(features: Sequence[Any]) -> np.ndarray:
    """``Frame.get_descriptors`` (`primitives.py:200-205`): ``np.array([f.descriptor for f in features])``;
    an empty feature list gives ``np.array([])`` exactly like the reference."""
    return np.array([f.descriptor for f in features])


def match_features(feature_matcher, last_frame, current_frame, dist_threshold: Optional[float] = None):
    """``Frontend._match_features`` (`frontend.py:181-187`): train = last frame, query = current frame."""
    desc_last = last_frame.get_descriptors() if hasattr(last_frame, "get_descriptors") else get_descriptors(last_frame.features)
    desc_cur = current_frame.get_descriptors() if hasattr(current_frame, "get_descriptors") else get_descriptors(current_frame.features)
    if dist_threshold is None:
        return feature_matcher.match(desc_last, desc_cur)
    return feature_matcher.match(desc_last, desc_cur, dist_threshold)


def propagate_map_points(matches, last_features: Sequence[Any], current_features: Sequence[Any]) -> int:
    """The consumer loop of `frontend.py:174-177`: copy ``map_point`` from the matched feature of the
    last frame to the current frame's feature.  ``matches`` is a DMatch sequence or a
    ``(queryIdx, trainIdx, ...)`` tuple of arrays.  Returns the number of propagated points."""
    if isinstance(matches, tuple) and len(matches) >= 2 and isinstance(matches[0], np.ndarray):
        pairs = zip(matches[0].tolist(), matches[1].tolist())
    else:
        pairs = ((m.queryIdx, m.trainIdx) for m in matches)
    n = 0
    for q, t in pairs:
        map_point = last_features[t].map_point
        if map_point:
            current_features[q].map_point = map_point
            n += 1
    return n


def keypoint_array(features: Sequence[Any]) -> np.ndarray:
    """``(N, 2) int32`` pixel positions, as ``Feature.position`` (`primitives.py:108-110`) truncates them."""
    if len(features) == 0:
        return np.empty((0, 2), np.int32)
    return np.array([f.keypoint.pt for f in features], dtype=np.float64).astype(np.int32)


def matched_point_arrays(q_idx: np.ndarray, t_idx: np.ndarray, source_positions: np.ndarray,
                         query_positions: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Packed ``(M, 2)`` arrays for ``cv2.findEssentialMat`` / ``triangulatePoints``: the two
    list-building loops of `utils.py:13-19` and `:41-47` as two gathers (source = train frame)."""
    return source_positions[np.asarray(t_idx)], query_positions[np.asarray(q_idx)]


def get_featured_detection_mask(shape, features_or_positions, radius: int, inner: bool = True, device=None) -> np.ndarray:
    """``utils.get_featured_detection_mask`` (`utils.py:58-74`): a ``shape`` uint8 mask, 0 (``inner``) or 255
    everywhere, with the filled square of half-width ``radius`` around every feature set to 255 / 0.  The
    reference draws the squares with one ``cv2.rectangle`` call per feature from Python; here the positions
    (``Feature.position`` of each feature, or an ``[N, 2]`` array -- e.g. the re-projected map points of the
    reference's ``camera`` branch, computed by the caller) are rasterised by ``hm_rasterize_mask``."""
    dev = nat.require_cuda(device)
    if isinstance(features_or_positions, np.ndarray):
        pos = features_or_positions.reshape(-1, 2).astype(np.int32)
    elif len(features_or_positions) == 0:
        pos = np.empty((0, 2), np.int32)
    else:
        pos = np.array([f.position for f in features_or_positions], dtype=np.int32).reshape(-1, 2)
    with torch.cuda.device(dev):
        pts = torch.from_numpy(np.ascontiguousarray(pos)).to(dev)
        return nat.rasterize_mask(pts, shape, radius, inner).cpu().numpy()


class FrameDescriptorStore:
    """Device-resident descriptors of recent frames (SURVEY.md 8f rank 1).

    ``put(frame_id, descriptors)`` uploads a frame once (pinned staging, async copy); ``match(last_id,
    current_id)`` runs the fused pipeline on the two resident arrays -- no host repacking, no H2D for
    the train side.  Keeps at most ``capacity`` frames (oldest evicted), like the reference's 7 active
    keyframes (`backend.py:11`).

    numpy frames live in the frame slots of an ``hm_context`` (``hm_frame_put`` / ``hm_frame_match``): one C
    call per upload and one per match, nothing torch-level on the path.  Frames given as CUDA tensors stay
    torch tensors and are matched through the device-pointer entry points.
    """

    def __init__(self, capacity: int = 8, *, ratio: Optional[float] = None, cross_check: bool = False,
                 device=None, variant: str = "auto"):
        self.device = nat.require_cuda(device)
        self.capacity = int(capacity)
        self.ratio, self.cross_check, self.variant = ratio, bool(cross_check), variant
        self._frames: "OrderedDict[Any, torch.Tensor]" = OrderedDict()
        self._points: dict = {}                                   # frame_id -> [N, 2] int32 pixel positions on the device
        # numpy frames: frame_id -> (slot, rows, has_positions) in the C context
        self._slots: "OrderedDict[Any, Tuple[int, int, bool]]" = OrderedDict()
        self._free_slots = list(range(min(self.capacity, nat.HostContext.FRAME_SLOTS)))[::-1]
        self._ctx: Optional[nat.HostContext] = None

    def __contains__(self, frame_id) -> bool:
        return frame_id in self._frames or frame_id in self._slots

    def __len__(self) -> int:
        return len(self._frames) + len(self._slots)

    def _put_slot(self, frame_id, a: np.ndarray, positions) -> None:
        if self._ctx is None:
            with nat.on_device(self.device):
                self._ctx = nat.HostContext()
        pos = None                                                 # validate before any slot changes hands
        if positions is not None:
            pos = np.asarray(positions)
            if pos.size == 0:
                pos = np.empty((0, 2), np.int32)
            if pos.ndim != 2 or pos.shape[1] != 2 or pos.shape[0] != a.shape[0]:
                raise MatcherError(f"positions: expected [{a.shape[0]}, 2], got {pos.shape}")
            pos = pos.astype(np.int32, copy=False)
        if frame_id in self._slots:
            slot = self._slots.pop(frame_id)[0]
        elif self._free_slots:
            slot = self._free_slots.pop()
        else:                                                      # evict the oldest resident frame
            _, (slot, _, _) = self._slots.popitem(last=False)
        try:
            with nat.on_device(self.device):
                self._ctx.frame_put(slot, a, pos)
        except Exception:
            self._free_slots.append(slot)                          # the slot is empty again (hm_frame_put clears it)
            raise
        self._slots[frame_id] = (slot, a.shape[0], pos is not None)
        if frame_id in self._frames:
            del self._frames[frame_id]
            self._points.pop(frame_id, None)

    def put_image(self, frame_id, image: np.ndarray, keypoints, n_levels: Optional[int] = None, with_positions: bool = True,
                  want_descriptors: bool = False):
        """Store a frame from its IMAGE and cv2 keypoints: the ORB descriptors are computed on the device
        (``hm_frame_put_orb``, SURVEY.md 8f rank 3) and written into the frame's slot without visiting the host.
        ``n_levels=None`` builds ``max(octave) + 1`` pyramid levels, as ``cv2.ORB.compute`` does for given keypoints.
        Returns the descriptors only when ``want_descriptors``."""
        from .feature_detectors import keypoint_arrays, pyramid_levels
        if self._ctx is None:
            with nat.on_device(self.device):
                self._ctx = nat.HostContext()
        xy, ang, octv = keypoint_arrays(keypoints)
        if n_levels is None:
            n_levels = pyramid_levels(octv)
        pos = xy.astype(np.int32) if with_positions else None      # Feature.position: int() of the keypoint coordinates
        if frame_id in self._slots:
            slot = self._slots.pop(frame_id)[0]
        elif self._free_slots:
            slot = self._free_slots.pop()
        else:
            _, (slot, _, _) = self._slots.popitem(last=False)
        try:
            with nat.on_device(self.device):
                out = self._ctx.frame_put_orb(slot, image, xy, ang, octv, n_levels, pos, want_descriptors)
        except Exception:
            self._free_slots.append(slot)
            raise
        self._slots[frame_id] = (slot, xy.shape[0], pos is not None)
        if frame_id in self._frames:
            del self._frames[frame_id]
            self._points.pop(frame_id, None)
        return out

    def put(self, frame_id, descriptors, positions=None) -> torch.Tensor:
        """Upload a frame once.  ``positions`` (optional ``[N, 2]`` pixel coordinates, truncated to int32 like
        ``Feature.position``) stay resident too, so that :meth:`matched_points` can gather on the device."""
        a = np.asarray(descriptors) if not isinstance(descriptors, torch.Tensor) else descriptors
        if isinstance(a, np.ndarray):
            if a.size == 0:
                a = np.empty((0, nat.DESC_BYTES), np.uint8)       # a frame without features
            if a.dtype != np.uint8 or a.ndim != 2 or a.shape[1] != nat.DESC_BYTES:
                raise MatcherError(f"descriptors: expected uint8 [N, {nat.DESC_BYTES}], got {a.dtype} {a.shape}")
            self._put_slot(frame_id, a, positions)                   # the C-context path (at most 16 resident frames)
            return None
        t = a.to(self.device).contiguous()
        if frame_id in self._slots:
            self._free_slots.append(self._slots.pop(frame_id)[0])
        self._frames[frame_id] = t
        self._frames.move_to_end(frame_id)
        self._points.pop(frame_id, None)
        if positions is not None:
            p = np.asarray(positions)
            if p.size == 0:
                p = np.empty((0, 2), np.int32)
            if p.ndim != 2 or p.shape[1] != 2 or p.shape[0] != t.shape[0]:
                raise MatcherError(f"positions: expected [{t.shape[0]}, 2], got {p.shape}")
            with nat.on_device(self.device):
                self._points[frame_id] = torch.from_numpy(np.ascontiguousarray(p.astype(np.int32))).to(self.device)
        while len(self._frames) > self.capacity:
            old, _ = self._frames.popitem(last=False)
            self._points.pop(old, None)
        return t

    def get(self, frame_id) -> torch.Tensor:
        return self._frames[frame_id]

    def _slot_match(self, last_id, current_id, dist_threshold, want_indices, want_points):
        (ts, nt, tp), (qs, nq, qp) = self._slots[last_id], self._slots[current_id]
        if want_points and not (tp and qp):
            raise MatcherError("matched_points needs both frames stored with positions")
        with nat.on_device(self.device):
            return self._ctx.frame_match(ts, qs, nq, ratio=self.ratio, cross_check=self.cross_check,
                                         dist_threshold=dist_threshold if dist_threshold else None, variant=self.variant,
                                         want_indices=want_indices, want_points=want_points)

    def match_tensors(self, last_id, current_id, dist_threshold: Optional[float] = None):
        """``(queryIdx, trainIdx, distance)`` int32 arrays; query = current frame, train = last frame."""
        if last_id in self._slots and current_id in self._slots:
            return self._slot_match(last_id, current_id, dist_threshold, True, False)
        t, q = self._frames[last_id], self._frames[current_id]
        if q.shape[0] == 0 or t.shape[0] == 0:
            e = np.empty(0, np.int32)
            return e, e.copy(), e.copy()
        oq, ot, od, cnt = nat.match_fused(q.unsqueeze(0), t.unsqueeze(0), ratio=self.ratio, cross_check=self.cross_check,
                                          dist_threshold=dist_threshold if dist_threshold else None, variant=self.variant)
        packed = torch.cat([cnt.view(1), oq.view(-1), ot.view(-1), od.view(-1)]).cpu().numpy()
        n, nq = int(packed[0]), q.shape[0]
        return packed[1:1 + n].copy(), packed[1 + nq:1 + nq + n].copy(), packed[1 + 2 * nq:1 + 2 * nq + n].copy()

    def matched_points(self, last_id, current_id, dist_threshold: Optional[float] = None):
        """``(source_pts, query_pts)``, two packed ``(M, 2) int32`` arrays: the inputs `utils.py:13-19` and
        `:41-47` build for ``cv2.findEssentialMat`` / ``triangulatePoints`` with a Python loop over the matches
        (source = last frame = train side).  Matching, filtering and the gather (``hm_gather_points``) run on the
        device; one D2H brings back the count and both arrays -- no DMatch objects, no index arrays."""
        if last_id in self._slots and current_id in self._slots:
            qp, tp = self._slot_match(last_id, current_id, dist_threshold, False, True)
            return tp, qp
        t, q = self._frames[last_id], self._frames[current_id]
        if last_id not in self._points or current_id not in self._points:
            raise MatcherError("matched_points needs both frames stored with positions")
        if q.shape[0] == 0 or t.shape[0] == 0:
            e = np.empty((0, 2), np.int32)
            return e, e.copy()
        oq, ot, _, cnt = nat.match_fused(q.unsqueeze(0), t.unsqueeze(0), ratio=self.ratio, cross_check=self.cross_check,
                                         dist_threshold=dist_threshold if dist_threshold else None, variant=self.variant)
        pq, pt = nat.gather_points(oq, ot, cnt, self._points[current_id].unsqueeze(0), self._points[last_id].unsqueeze(0))
        packed = torch.cat([cnt.view(1), pq.view(-1), pt.view(-1)]).cpu().numpy()
        n, nq = int(packed[0]), q.shape[0]
        return packed[1 + 2 * nq:1 + 2 * nq + 2 * n].reshape(n, 2).copy(), packed[1:1 + 2 * n].reshape(n, 2).copy()

    def match(self, last_id, current_id, dist_threshold: Optional[float] = None):
        """DMatch sequence with the reference's return convention (tuple, or list when filtered)."""
        q, t, d = self.match_tensors(last_id, current_id, dist_threshold)
        matches = _build_dmatches(q, t, d, 0)
        if dist_threshold and len(matches) != 0:
            return matches
        return tuple(matches)


class KeyframeWindow:
    """A local window of keyframes resident in ONE device buffer, matched against the current frame in one batched
    call (BASELINE config C5: 32 train frames x 10,000 rows, ratio test + mutual check).

    The reference keeps its active keyframes in the backend's map (`/root/reference/backend.py:11`, 7 of them) and
    would match them one ``match()`` call at a time, re-packing and re-sending both sides each time
    (`frontend.py:181-187`).  Here ``put(i, descriptors)`` uploads a keyframe once into ring position ``i``;
    ``match(query)`` sends only the current frame's descriptors (or one query per keyframe), runs ONE fused pipeline
    launch over all resident frames -- forward k-NN with the ratio test inside, candidate pass of the mutual check,
    filter -- and brings every match list back with one D2H.  All frames of a window share one row count (the batched
    kernels take one shape per launch; ORB returns exactly ``n_features`` on ordinary content)."""

    def __init__(self, capacity: int = 32, *, ratio: Optional[float] = None, cross_check: bool = False, device=None,
                 variant: str = "auto"):
        self.device = nat.require_cuda(device)
        self.capacity = int(capacity)
        self.ratio, self.cross_check, self.variant = ratio, bool(cross_check), variant
        self._buf: Optional[torch.Tensor] = None          # [capacity, rows, 32]
        self._present = [False] * self.capacity
        from .feature_matchers import _Staging
        self._staging = _Staging()

    @property
    def rows(self) -> int:
        return 0 if self._buf is None else int(self._buf.shape[1])

    def put(self, index: int, descriptors: np.ndarray) -> None:
        a = np.asarray(descriptors)
        if a.dtype != np.uint8 or a.ndim != 2 or a.shape[1] != nat.DESC_BYTES or a.shape[0] == 0:
            raise MatcherError(f"descriptors: expected non-empty uint8 [N, {nat.DESC_BYTES}], got {a.dtype} {a.shape}")
        if not 0 <= index < self.capacity:
            raise MatcherError(f"window index {index} out of range 0..{self.capacity - 1}")
        with nat.on_device(self.device):
            if self._buf is None:
                self._buf = torch.empty((self.capacity, a.shape[0], nat.DESC_BYTES), dtype=torch.uint8, device=self.device)
            if a.shape[0] != self._buf.shape[1]:
                raise MatcherError(f"every keyframe of a window has the same row count ({self._buf.shape[1]}), got {a.shape[0]}")
            self._buf[index].copy_(self._staging.to_device("kf", a, self.device), non_blocking=True)
        self._present[index] = True

    def match_tensors(self, query: np.ndarray, dist_threshold: Optional[float] = None):
        """``query``: ``[Nq, 32]`` (the current frame against every resident keyframe) or ``[B, Nq, 32]`` (one query per
        resident keyframe, in ring order).  Returns a list with one ``(queryIdx, trainIdx, distance)`` triple of int32
        arrays per resident keyframe, in ring order."""
        idx = [i for i, p in enumerate(self._present) if p]
        if not idx:
            return []
        q = np.asarray(query)
        if q.dtype != np.uint8 or q.shape[-1] != nat.DESC_BYTES or q.ndim not in (2, 3) or (q.ndim == 3 and q.shape[0] != len(idx)):
            raise MatcherError(f"query: expected uint8 [Nq, 32] or [{len(idx)}, Nq, 32], got {q.dtype} {q.shape}")
        nq = q.shape[-2]
        if nq == 0:
            e = np.empty(0, np.int32)
            return [(e, e.copy(), e.copy()) for _ in idx]
        with nat.on_device(self.device):
            train = self._buf if len(idx) == self.capacity else self._buf[torch.tensor(idx, device=self.device)]
            qd = self._staging.to_device("wq", q.reshape(-1, nat.DESC_BYTES), self.device)
            qd = qd.view(len(idx), nq, nat.DESC_BYTES) if q.ndim == 3 else qd.unsqueeze(0).expand(len(idx), nq, nat.DESC_BYTES)
            oq, ot, od, cnt = nat.match_fused(qd, train, ratio=self.ratio, cross_check=self.cross_check,
                                              dist_threshold=dist_threshold if dist_threshold else None, variant=self.variant)
            host = self._staging.to_host("wm", torch.cat([cnt.view(-1), oq.view(-1), ot.view(-1), od.view(-1)]))
        b = len(idx)
        counts = host[:b]
        body = host[b:].reshape(3, b, nq)
        return [(body[0, i, :counts[i]].copy(), body[1, i, :counts[i]].copy(), body[2, i, :counts[i]].copy()) for i in range(b)]

    def match(self, query: np.ndarray, dist_threshold: Optional[float] = None):
        """DMatch tuples per resident keyframe (``imgIdx`` = ring position)."""
        idx = [i for i, p in enumerate(self._present) if p]
        return [tuple(_build_dmatches(q, t, d, i)) for i, (q, t, d) in zip(idx, self.match_tensors(query, dist_threshold))]
