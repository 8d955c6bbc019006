"""CPU oracle for the Human3.6M per-action table of ``evaluate.h36m_metrics``.

TEST INFRASTRUCTURE ONLY, like ``diff3d_oracle``: nothing under ``diff3dhpe_b200/`` imports this file.

A restatement of the reference's loop, sharing no code with the product's run planning.  The reference evaluates
Human3.6M action by action: a new DataLoader over the action's sequences (shuffle off) per action (RUN:730-736), and in
evaluate() every batch of windows adds ``N_b * metric(batch)`` over its masked frames, N_b of them, flattened in window
order, for MPJPE, N-MPJPE, P-MPJPE and the velocity error (RUN:602-614); the sums are divided by sum N_b.  The windows and
their target masks come from the generator's own rule (``chunk_windows``, ``window_batch``) and the metrics are the
``diff3d_oracle`` functions pinned to the reference's ``common/loss.py``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import diff3d_oracle as ora

METRICS = ("mpjpe", "p_mpjpe", "n_mpjpe", "velocity")


def action_table(pred, gt, seq_lengths, seq_action, n_actions: int, F: int, batch_size: int):
    """pred / gt: packed [N, J, 3] float32 (sequences back to back).  Returns {'actions': [row of action 0, ...],
    'action_mean': row}, a row being {'mpjpe', 'p_mpjpe', 'n_mpjpe', 'velocity', 'frames'} in the poses' units; an
    action without frames has NaN metrics, and the mean runs over the actions that have frames."""
    pred = torch.from_numpy(np.ascontiguousarray(pred, dtype=np.float32))
    gt = torch.from_numpy(np.ascontiguousarray(gt, dtype=np.float32))
    offsets = np.concatenate([[0], np.cumsum(seq_lengths)]).astype(np.int64)
    rows = []
    for a in range(n_actions):
        windows = []                                         # the action's loader: its sequences in order
        for s in range(len(seq_lengths)):
            if seq_action[s] != a:
                continue
            seq_p, seq_g = pred[offsets[s]:offsets[s + 1]], gt[offsets[s]:offsets[s + 1]]
            for start, start_target in zip(*ora.chunk_windows(int(seq_lengths[s]), F)):
                p, mask = ora.window_batch(seq_p, start, F, start_target, flip=False)
                g, _ = ora.window_batch(seq_g, start, F, start_target, flip=False)
                windows.append((p, g, mask))
        sums = dict.fromkeys(METRICS, 0.0)
        n = 0
        for b in range(0, len(windows), batch_size):
            batch = windows[b:b + batch_size]
            mask = torch.stack([w[2] for w in batch])
            p = torch.stack([w[0] for w in batch])[mask]         # [N_b, J, 3], window-major
            g = torch.stack([w[1] for w in batch])[mask]
            n_b = p.shape[0]
            sums["mpjpe"] += n_b * ora.mpjpe(p.unsqueeze(1), g.unsqueeze(1)).item()
            sums["n_mpjpe"] += n_b * ora.n_mpjpe(p.unsqueeze(1), g.unsqueeze(1)).item()
            sums["p_mpjpe"] += n_b * ora.p_mpjpe(p.numpy(), g.numpy())
            sums["velocity"] += n_b * ora.mean_velocity_error(p.numpy(), g.numpy())
            n += n_b
        row = {k: (sums[k] / n if n else float("nan")) for k in METRICS}
        row["frames"] = n
        rows.append(row)
    have = [r for r in rows if r["frames"]]
    mean = {k: (float(np.mean([r[k] for r in have])) if have else float("nan")) for k in METRICS}
    mean["frames"] = sum(r["frames"] for r in have)
    return {"actions": rows, "action_mean": mean}
