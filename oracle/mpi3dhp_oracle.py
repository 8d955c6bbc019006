"""CPU oracle for the MPI-INF-3DHP PCK / AUC counts of ``d3d_pck_accumulate`` (numpy).

TEST INFRASTRUCTURE ONLY, like ``diff3d_oracle``: nothing under ``diff3dhpe_b200/`` imports this file.

The protocol is the MPI-INF-3DHP test set's own MATLAB evaluation (``mpii_compute_3d_pck.m``), not a line of the
reference, which dumps its predictions to a ``.mat`` file for that script: the per-joint Euclidean error is taken as
given, PCK is the share of errors strictly below 150 mm, AUC the mean PCK over the thresholds 0, 5, ..., 150 mm, and
pooled rows sum the counts before dividing.
"""
from __future__ import annotations

import numpy as np


def joint_errors_fp32(pred, gt) -> np.ndarray:
    """[N, J] float32 joint errors sqrt((dx*dx + dy*dy) + dz*dz), every operation rounded to float32 (numpy applies no
    FMA, and its float32 sqrt is correctly rounded): bit for bit the expression of d3d_pck_accumulate."""
    d = np.asarray(pred, dtype=np.float32) - np.asarray(gt, dtype=np.float32)
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    return np.sqrt((dx * dx + dy * dy) + dz * dz)


def pck_counts(err, thresholds, frame_index=None, frame_group=None, n_groups: int = 1):
    """d3d_pck_accumulate restated from [N, J] float32 errors: (counts int64 [G, J, n_thr] of errors < threshold, both
    float32; err_sum fp64 [G, J]; frames int64 [G]) over the listed rows (None = all; a repeated row counts again), the
    group of a row being frame_group[row] (None = 0); rows whose group lies outside [0, G) are skipped."""
    err = np.asarray(err, dtype=np.float32)
    thr = np.asarray(thresholds, dtype=np.float32)
    rows = np.arange(err.shape[0]) if frame_index is None else np.asarray(frame_index, dtype=np.int64)
    grp = np.zeros(rows.size, np.int64) if frame_group is None else np.asarray(frame_group, dtype=np.int64)[rows]
    J = err.shape[1]
    counts = np.zeros((n_groups, J, thr.size), np.int64)
    err_sum = np.zeros((n_groups, J), np.float64)
    frames = np.zeros(n_groups, np.int64)
    for g in range(n_groups):
        e = err[rows[grp == g]]
        frames[g] = e.shape[0]
        err_sum[g] = e.astype(np.float64).sum(axis=0)
        counts[g] = (e[:, :, None] < thr[None, None, :]).sum(axis=0)
    return counts, err_sum, frames


def pck_auc(err, thresholds, joints, pck_threshold):
    """(PCK %, AUC %, mean error) straight from [N, J] float32 errors over the listed joints, in fp64: PCK = 100 x the
    share of errors < pck_threshold, AUC = the mean of that share over the thresholds (all compared in float32)."""
    e = np.asarray(err, dtype=np.float32)[:, list(joints)]
    if e.size == 0:
        return float("nan"), float("nan"), float("nan")
    share = [100.0 * np.count_nonzero(e < np.float32(t)) / e.size for t in thresholds]
    pck = 100.0 * np.count_nonzero(e < np.float32(pck_threshold)) / e.size
    return float(pck), float(np.mean(share)), float(e.astype(np.float64).mean())
