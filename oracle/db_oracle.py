"""Keyframe-database pipeline at full size: knnMatch k=2 -> Lowe ratio -> mutual check over the concatenated database.

TEST INFRASTRUCTURE ONLY - see oracle/hamming_oracle.py for the policy.

``hamming_oracle.pipeline`` / ``c_oracle.pipeline`` compute the mutual check from the column minimum over EVERY train
row, which at C4 size (8.19 M rows) is a CPU pass as long as the forward one.  The check only ever asks about the best
row ``t1`` of a query that survived the ratio test, so this restatement computes the nearest query of those rows alone:
a brute-force top-1 of the (few thousand) rows ``t1`` against the query batch, lowest query index on ties.  The result
is the same ``(q, t, d)`` as ``pipeline`` (tests/test_keyframe_db_pipeline.py checks it on small inputs).
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import c_oracle
from .hamming_oracle import NO_MATCH_KEY, ratio_lut


def pipeline_from_keys(query: np.ndarray, train: np.ndarray, keys: np.ndarray, ratio: Optional[float] = 0.75,
                       cross_check: bool = True, threads: int = 0):
    """``(q, t, d)`` int32 arrays of the pipeline, given the forward top-2 ``keys`` of ``query`` over ``train``
    (``c_oracle.knn2_keys(query, train)``)."""
    keys = np.asarray(keys).view(np.uint64).reshape(-1, 2)
    nq = keys.shape[0]
    d1 = (keys[:, 0] >> np.uint64(32)).astype(np.int64)
    t1 = (keys[:, 0] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    keep = keys[:, 0] != NO_MATCH_KEY
    if ratio is not None:
        has2 = keys[:, 1] != NO_MATCH_KEY
        d2 = np.where(has2, (keys[:, 1] >> np.uint64(32)).astype(np.int64), 0)
        keep &= has2 & (d1 < ratio_lut(ratio)[np.clip(d2, 0, 256)])
    if cross_check and keep.any():
        rows = np.unique(t1[keep])
        back = c_oracle.knn2_keys(np.asarray(train)[rows], query, threads=threads)      # rows x queries, stable top-2
        best_q = dict(zip(rows.tolist(), (back[:, 0] & np.uint64(0xFFFFFFFF)).astype(np.int64).tolist()))
        idx = np.nonzero(keep)[0]
        keep[idx] = np.array([best_q[t] for t in t1[idx].tolist()]) == idx
    qi = np.nonzero(keep)[0]
    return qi.astype(np.int32), t1[qi].astype(np.int32), d1[qi].astype(np.int32)


def pipeline(query: np.ndarray, train: np.ndarray, ratio: Optional[float] = 0.75, cross_check: bool = True,
             threads: int = 0):
    """The same from scratch: forward keys from ``c_oracle.knn2_keys`` first."""
    if np.asarray(query).size == 0 or np.asarray(train).shape[0] == 0:
        e = np.empty(0, np.int32)
        return e, e.copy(), e.copy()
    return pipeline_from_keys(query, train, c_oracle.knn2_keys(query, train, threads=threads), ratio, cross_check, threads)
