"""Feature detector plugin with the descriptor stage on the device -- host-side mirror of
`/root/reference/feature_detectors.py:9-26` (same class names, constructor and method signatures).

The reference's ``OrbFeatureDetector`` is two cv2 calls: ``ORB.detect`` and ``ORB.detectAndCompute``.  Here keypoint
DETECTION stays with cv2 on the host (FAST + Harris + per-level retainBest: not on the matcher's path, SURVEY.md 8f rank 3
asks for the descriptor stage), and the DESCRIPTORS -- scale pyramid, blur, 256 steered-BRIEF comparisons -- are computed
by ``csrc/hm_orb.cu``, bit-identical to ``cv2.ORB.compute`` for the same keypoints (oracle/orb_oracle.py, tests/test_orb.py).
``detect_and_compute`` keeps the reference's return value; ``detect_and_store`` writes the descriptors straight into a
:class:`~slam_experiments_b200.frontend_glue.FrameDescriptorStore` slot so that they never visit the host.
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from typing import Optional, Sequence

import numpy as np
import torch
from cv2 import KeyPoint, KeyPoint_convert, ORB

from . import _native as nat


class FeatureDetector(ABC):
    """`feature_detectors.py:9-16`."""

    @abstractmethod
    def detect(self, img: np.ndarray, mask: np.ndarray = None) -> Sequence[KeyPoint]:
        raise NotImplementedError

    @abstractmethod
    def detect_and_compute(self, img: np.ndarray, mask: np.ndarray = None) -> tuple[Sequence[KeyPoint], np.ndarray]:
        raise NotImplementedError


def keypoint_arrays(keypoints: Sequence[KeyPoint]):
    """``(xy float32 [n, 2], angle float32 [n], octave int32 [n])`` of a cv2 keypoint sequence (positions through
    ``cv2.KeyPoint_convert``, one C++ call; the other two fields have no bulk accessor)."""
    n = len(keypoints)
    if n == 0:
        return np.empty((0, 2), np.float32), np.empty(0, np.float32), np.empty(0, np.int32)
    xy = np.ascontiguousarray(KeyPoint_convert(keypoints), dtype=np.float32).reshape(n, 2)
    ang = np.fromiter((k.angle for k in keypoints), np.float32, n)
    octv = np.fromiter((k.octave for k in keypoints), np.int32, n)
    return xy, ang, octv


def pyramid_levels(octaves: np.ndarray) -> int:
    """Levels of the pyramid the descriptors of these keypoints need: ``max(octave) + 1``, as ``cv2.ORB.compute`` builds
    it for keypoints passed in (1 for none).  On a small image cv2's detector stops short of its 8 levels, and the
    levels it never reached may be too small to hold the 32-pixel frame."""
    return int(octaves.max()) + 1 if octaves.size else 1


class OrbFeatureDetector(FeatureDetector):
    """`feature_detectors.py:18-26`, descriptors on the device."""

    def __init__(self, n_features: int = 500, device=None) -> None:
        self.orb = ORB.create(nfeatures=n_features)
        self.device = nat.require_cuda(device)
        self._workspace: Optional[torch.Tensor] = None

    def detect(self, img: np.ndarray, mask: np.ndarray = None) -> Sequence[KeyPoint]:
        return self.orb.detect(img, mask)

    def compute(self, img: np.ndarray, keypoints: Sequence[KeyPoint]) -> Optional[np.ndarray]:
        """``cv2.ORB.compute`` for keypoints that came out of :meth:`detect` (sorted by octave, 31 pixels inside their
        level): ``[n, 32] uint8``, or ``None`` for an empty keypoint list like cv2."""
        if len(keypoints) == 0:
            return None
        return self.compute_device(img, keypoints).cpu().numpy()

    def compute_device(self, img: np.ndarray, keypoints: Sequence[KeyPoint]) -> torch.Tensor:
        """The same descriptors as a ``[n, 32] uint8`` CUDA tensor (no D2H)."""
        xy, ang, octv = keypoint_arrays(keypoints)
        n_levels = pyramid_levels(octv)
        with nat.on_device(self.device):
            image = torch.from_numpy(np.ascontiguousarray(img)).to(self.device)
            self._workspace = nat.orb_build_pyramid(image, n_levels, self._workspace)
            pack = torch.from_numpy(np.concatenate([xy.reshape(-1), nat.orb_angles_to_cs(ang).reshape(-1)])).to(self.device)
            n = xy.shape[0]
            return nat.orb_describe(self._workspace, img.shape[:2], n_levels, pack[:2 * n].view(n, 2),
                                    pack[2 * n:].view(n, 2), torch.from_numpy(octv).to(self.device))

    def detect_and_compute(self, img: np.ndarray, mask: np.ndarray = None) -> tuple[Sequence[KeyPoint], np.ndarray]:
        keypoints = self.orb.detect(img, mask)
        return keypoints, self.compute(img, keypoints)

    def detect_and_store(self, img: np.ndarray, store, frame_id, mask: np.ndarray = None, with_positions: bool = True):
        """Detect on the host, describe on the device straight into ``store`` (a ``FrameDescriptorStore``) under
        ``frame_id``; returns the keypoints.  Positions (truncated to int32 like ``Feature.position``,
        `/root/reference/primitives.py`) are stored with the frame so that matched points can be gathered on the
        device."""
        keypoints = self.orb.detect(img, mask)
        store.put_image(frame_id, img, keypoints, with_positions=with_positions)
        return keypoints
