"""Sharded flip-TTA evaluation: the device-side equivalent of the reference's `evaluate()` inner loop
(RUN:557-606) with `nn.DataParallel` (RUN:216-218) replaced by one process per GPU.

Clips are independent, so rank r of R owns a contiguous block of clips (both flip variants of a clip stay on
the same rank); nothing is communicated inside the sampler.  One exchange step at the end: gather of the merged
predictions and an all-reduce of the fp64 (sum of joint errors, joint count) pair -- NCCL on GPUs, gloo in the
CPU tests of this plumbing.  Sweeps over raw packed sequences gather with `gather_packed` (frame counts differ per
rank) and build the Human3.6M per-action table with `h36m_metrics` on the gathered array.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import synthetic
from .engine import Engine

# The MPI-INF-3DHP test protocol, as the dataset's MATLAB evaluation (mpii_compute_3d_pck.m) defines it: PCK at 150 mm
# and AUC over 0, 5, ..., 150 mm of the 14 joints 0..13 of the MPI 17-joint order (head-top, neck, then right and left
# shoulder, elbow, wrist, hip, knee, ankle; pelvis 14, spine 15 and head 16 are not evaluated), and its joint groups.
MPI3DHP_PCK_JOINTS = tuple(range(14))
MPI3DHP_JOINT_GROUPS = {"Head": (0,), "Neck": (1,), "Shoulder": (2, 5), "Elbow": (3, 6), "Wrist": (4, 7),
                        "Hip": (8, 11), "Knee": (9, 12), "Ankle": (10, 13)}


def shard_range(n_clips: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block partition: returns (start, count) of rank's clips; counts differ by at most one."""
    base, rem = divmod(n_clips, world)
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


def window_starts(n_frames: int, F: int) -> Sequence[Tuple[int, int]]:
    """Windowing rule of ChunkedGenerator (common/nosiy_generators.py:27-48) for one sequence of n_frames with
    stride == F: non-overlapping windows, the last one shifted back to end at the sequence end.  Returns
    (start_frame, first_valid_offset) per window: frames before first_valid_offset were already predicted by the
    previous window and are masked out (`target_mask`)."""
    if n_frames < F:
        raise ValueError("sequence shorter than one window")
    out = []
    n_full = n_frames // F
    for w in range(n_full):
        out.append((w * F, 0))
    if n_frames % F:
        start = n_frames - F
        out.append((start, n_full * F - start))
    return out


def plan_windows(seq_lengths: Sequence[int], F: int):
    """Window plan of a set of sequences packed back to back: (win_start int64 [n_win] = first PACKED frame of every
    window, first_valid int32 [n_win], seq_id int32 [n_win]) following `window_starts` per sequence, in the
    generator's order (sequence by sequence, windows in time order; nosiy_generators.py:27-48)."""
    starts, valid, sid = [], [], []
    base = 0
    for s, n in enumerate(seq_lengths):
        for st, fv in window_starts(int(n), F):
            starts.append(base + st)
            valid.append(fv)
            sid.append(s)
        base += int(n)
    return (torch.tensor(starts, dtype=torch.int64), torch.tensor(valid, dtype=torch.int32),
            torch.tensor(sid, dtype=torch.int32))


def loader_batch_runs(seq_lengths: Sequence[int], seq_group: Sequence[int], F: int, batch_size: int):
    """The reference's per-action batching (a new DataLoader per action, RUN:730-736) as runs of packed frames.  The
    windows of `plan_windows` are cut, in generator order, into batches of `batch_size` consecutive windows that restart
    at every change of group (seq_group: one id per sequence).  The masked frames of such a batch, flattened window-major
    as evaluate() flattens them (RUN:589-596), are the packed frames [run_start[r], run_start[r + 1]): the windows do
    not overlap once the back-shifted last window's target_mask is applied, and sequences are packed back to back.
    Returns (run_start int64 [R + 1], run_group int32 [R]); the runs tile [0, N).  Raises ValueError when the
    sequences of a group are not consecutive: the reference never batches such sequences together."""
    if batch_size < 1:
        raise ValueError("batch_size must be positive")
    grp = torch.as_tensor(seq_group, dtype=torch.int64).reshape(-1)
    if grp.numel() != len(seq_lengths):
        raise ValueError("seq_group must have one entry per sequence")
    if grp.numel():
        first = torch.ones(grp.numel(), dtype=torch.bool)
        first[1:] = grp[1:] != grp[:-1]
        if torch.unique(grp[first]).numel() != int(first.sum()):
            raise ValueError("the sequences of a group must be consecutive in the packing")
    ws, fv, sid = plan_windows(seq_lengths, F)
    n_win = ws.numel()
    wg = grp[sid.long()]
    idx = torch.arange(n_win)
    new_block = torch.ones(n_win, dtype=torch.bool)
    new_block[1:] = wg[1:] != wg[:-1]
    block_start = torch.cummax(torch.where(new_block, idx, torch.zeros_like(idx)), 0).values if n_win else idx
    head = (idx - block_start) % batch_size == 0                     # first window of every batch
    n_total = int(sum(int(n) for n in seq_lengths))
    run_start = torch.cat([ws[head] + fv[head].long(), torch.tensor([n_total], dtype=torch.int64)])
    return run_start, wg[head].to(torch.int32)


class DeviceSampler:
    """Adapter: (x2d [n,F,J,2] device, y_T, step_noise) -> y0, running GaussianDiffusion.ddim_sample_loop."""

    def __init__(self, diffusion):
        self.diffusion = diffusion

    def __call__(self, x2d, y_T, step_noise):
        return self.diffusion.ddim_sample_loop(x2d, list(y_T.shape), noise=(y_T, step_noise))

    def merge(self, y, y_flip, left, right, scale):
        return self.diffusion.model.engine(y.shape[0]).tta_merge(y, y_flip, left, right, scale)

    def mpjpe(self, pred, gt, acc, mask):
        return self.diffusion.model.engine(1).mpjpe_accumulate(pred, gt, acc, mask)


def evaluate_shard(sampler, x2d: torch.Tensor, gt: Optional[torch.Tensor], noise_fn: Callable, *, device,
                   batch_clips: int = 256, tta: bool = True, left=synthetic.H36M_JOINTS_LEFT,
                   right=synthetic.H36M_JOINTS_RIGHT, scale: float = 1.0, frame_mask: Optional[torch.Tensor] = None,
                   clip_offset: int = 0) -> Dict[str, torch.Tensor]:
    """Runs this rank's clips.  x2d/gt/frame_mask are HOST tensors of the local shard ([n,F,J,2], [n,F,J,3],
    [n,F] uint8); `noise_fn(global_clip_ids, flip) -> (y_T, step_noise|None)` returns device noise.
    Returns {'pred': [n,F,J,3] (device), 'acc': fp64[2] (device)}."""
    n, F, J, _ = x2d.shape
    pred = torch.empty((n, F, J, 3), device=device, dtype=torch.float32)
    acc = torch.zeros(2, device=device, dtype=torch.float64)
    for s in range(0, n, batch_clips):
        e = min(n, s + batch_clips)
        ids = torch.arange(clip_offset + s, clip_offset + e)
        xb = x2d[s:e].to(device, non_blocking=True)
        y_T, sn = noise_fn(ids, False)
        if tta:
            # orig || flip as one 2B batch (clips are independent, SURVEY.md 8e), then un-flip + average (RUN:583-588)
            xf = synthetic.flip_2d(xb, left, right)
            yf_T, snf = noise_fn(ids, True)
            y_all = sampler(torch.cat([xb, xf]), torch.cat([y_T, yf_T]),
                            None if sn is None else torch.cat([sn, snf], dim=1))
            b = e - s
            out = sampler.merge(y_all[:b].contiguous(), y_all[b:].contiguous(), left, right, scale)
        else:
            out = sampler(xb, y_T, sn)
            if scale != 1.0:
                out = out * scale
        pred[s:e] = out
        if gt is not None:
            gb = gt[s:e].to(device, non_blocking=True)
            mb = None if frame_mask is None else frame_mask[s:e].to(device).reshape(-1).contiguous()
            sampler.mpjpe(out.contiguous(), gb.contiguous(), acc, mb)
    return {"pred": pred, "acc": acc}


def evaluate_sequences(sampler, seq2d: torch.Tensor, gt3d: Optional[torch.Tensor], seq_lengths: Sequence[int],
                       noise_fn: Callable, *, device, F: int, batch_clips: int = 256,
                       left=synthetic.H36M_JOINTS_LEFT, right=synthetic.H36M_JOINTS_RIGHT, scale: float = 1.0,
                       window_offset: int = 0) -> Dict[str, torch.Tensor]:
    """The evaluate() inner loop from RAW packed sequences (SURVEY.md 8f N3): seq2d [N, J, 2] / gt3d [N, J, 3] are HOST
    tensors holding this rank's sequences back to back.  The F-frame windows and their flipped copies
    (nosiy_generators.py:27-48, 264-276) are built on the device, sampled with flip-TTA, merged (RUN:583-588) and written
    back into packed frame order with the overlap of each back-shifted last window masked (RUN:589-596).
    Returns {'pred': [N, J, 3] (device), 'acc': fp64[2] (device), 'n_windows': int}."""
    ws, fv, _ = plan_windows(seq_lengths, F)
    n_win = ws.numel()
    N, J, _ = seq2d.shape
    eng = sampler.diffusion.model.engine(2 * min(batch_clips, n_win))
    seq_d = seq2d.to(device, non_blocking=True)
    ws_d, fv_d = ws.to(device), fv.to(device)
    out = torch.zeros((N, J, 3), device=device, dtype=torch.float32)
    for s in range(0, n_win, batch_clips):
        e = min(n_win, s + batch_clips)
        ids = torch.arange(window_offset + s, window_offset + e)
        xb, xf = eng.window_gather(seq_d, ws_d[s:e].contiguous(), left, right)
        y_T, sn = noise_fn(ids, False)
        yf_T, snf = noise_fn(ids, True)
        y_all = sampler(torch.cat([xb, xf]), torch.cat([y_T, yf_T]), None if sn is None else torch.cat([sn, snf], dim=1))
        b = e - s
        merged = sampler.merge(y_all[:b].contiguous(), y_all[b:].contiguous(), left, right, scale)
        eng.window_scatter(merged, ws_d[s:e].contiguous(), fv_d[s:e].contiguous(), out)
    acc = torch.zeros(2, device=device, dtype=torch.float64)
    if gt3d is not None:
        sampler.mpjpe(out, gt3d.to(device, non_blocking=True).contiguous(), acc, None)
    return {"pred": out, "acc": acc, "n_windows": n_win}


def mpi3dhp_thresholds(mm_per_unit: float):
    """The 31 PCK thresholds 0, 5, ..., 150 mm of the MPI-INF-3DHP protocol in the poses' units: mm_per_unit = 1000 for
    poses in metres, 1 for poses in millimetres.  The last one is the PCK threshold."""
    if not mm_per_unit > 0:
        raise ValueError("mm_per_unit must be positive")
    return [5.0 * k / mm_per_unit for k in range(31)]


def mpi3dhp_metrics(engine: Engine, pred: torch.Tensor, gt: torch.Tensor, *, mm_per_unit: float,
                    frame_group: Optional[torch.Tensor] = None, n_groups: int = 1, group_names: Optional[Sequence] = None,
                    frame_index: Optional[torch.Tensor] = None) -> Dict:
    """The MPI-INF-3DHP PCK / AUC / MPJPE table on the device: one `Engine.pck_accumulate` call over pred / gt ([N, 17, 3]
    in the MPI joint order, e.g. the packed 'pred' of `evaluate_sequences` and its ground truth), then the host-side table.
    Errors are taken as given (no root alignment).  frame_group: int32 [N] group id per frame (per sequence, e.g.
    `seq_id.repeat_interleave(F - first_valid)` from `plan_windows`, or per activity); frames outside [0, n_groups) are
    left out.  frame_index: the frames to evaluate (int64, None = all).
    Returns {'overall': row, 'groups': {name: row}, 'joint_groups': {'Head': row, ...}}, where a row holds 'pck' and
    'auc' (%) and 'mpjpe' (mm) over the 14 evaluated joints (of that joint group in 'joint_groups', over all groups of
    frames) and 'frames'; 'overall' and 'groups' rows also hold 'mpjpe_all_joints' (mm, all 17 joints)."""
    if engine.J != 17:
        raise ValueError("the MPI-INF-3DHP protocol needs poses in the 17-joint MPI order")
    names = list(range(n_groups)) if group_names is None else list(group_names)
    if len(names) != n_groups:
        raise ValueError("group_names must have n_groups entries")
    thr = mpi3dhp_thresholds(mm_per_unit)
    dev = engine.device
    counts = torch.zeros((n_groups, engine.J, len(thr)), device=dev, dtype=torch.int64)
    err_sum = torch.zeros((n_groups, engine.J), device=dev, dtype=torch.float64)
    frames = torch.zeros(n_groups, device=dev, dtype=torch.int64)
    if frame_group is not None:
        frame_group = frame_group.to(device=dev, dtype=torch.int32).contiguous()
    if frame_index is not None:
        frame_index = frame_index.to(device=dev, dtype=torch.int64).contiguous()
    engine.pck_accumulate(pred.contiguous(), gt.to(dev).contiguous(), counts, err_sum, frames, thr, frame_index,
                          frame_group)
    counts, err_sum, frames = counts.cpu(), err_sum.cpu(), frames.cpu()

    def table(joints):
        return Engine.pck_table(counts, err_sum, frames, thr, joints, thr[-1])

    def in_mm(row, every=None):
        out = dict(row, mpjpe=row["mpjpe"] * mm_per_unit)
        if every is not None:
            out["mpjpe_all_joints"] = every["mpjpe"] * mm_per_unit
        return out

    main, every = table(MPI3DHP_PCK_JOINTS), table(range(engine.J))
    return {"overall": in_mm(main["all"], every["all"]),
            "groups": {n: in_mm(r, a) for n, r, a in zip(names, main["groups"], every["groups"])},
            "joint_groups": {name: in_mm(table(joints)["all"]) for name, joints in MPI3DHP_JOINT_GROUPS.items()}}


def h36m_metrics(engine: Engine, pred: torch.Tensor, gt: torch.Tensor, seq_lengths: Sequence[int],
                 seq_action: Sequence[int], *, F: int, batch_size: int, mm_per_unit: float,
                 action_names: Optional[Sequence] = None) -> Dict:
    """The Human3.6M per-action table (RUN:730-736, 602-614) on the device, from the packed pred / gt [N, J, 3] of
    `evaluate_sequences` (sequences back to back, N = sum(seq_lengths)).  seq_action: the action id of every sequence,
    in [0, G), G = len(action_names) (default: max id + 1, names 0..G-1); an action's sequences must be consecutive.
    Every batch the reference's per-action loader would form (`loader_batch_runs`, `batch_size` windows of F frames) is
    one `Engine.pose_metrics_accumulate` call on its run of frames into the action's fp64 accumulator, so MPJPE,
    N-MPJPE, P-MPJPE and the velocity error carry evaluate()'s `N_b` weighting; all calls are enqueued on the current
    stream and the accumulators come back in one copy.  mm_per_unit: 1000 for poses in metres, 1 for millimetres.
    Returns {'actions': {name: row}, 'action_mean': row, 'pooled': row}, a row being {'mpjpe', 'p_mpjpe', 'n_mpjpe',
    'velocity'} in mm and 'frames'.  'action_mean' is the unweighted mean of the rows of the actions that have frames
    (the reference's mean over its actions), 'pooled' sums the accumulators before dividing.  A row without frames
    is NaN.  A batch of a single frame adds no velocity term (the reference's numpy mean over no difference is NaN)."""
    if not mm_per_unit > 0:
        raise ValueError("mm_per_unit must be positive")
    act = torch.as_tensor(seq_action, dtype=torch.int64).reshape(-1)
    G = len(action_names) if action_names is not None else (int(act.max()) + 1 if act.numel() else 0)
    names = list(range(G)) if action_names is None else list(action_names)
    if act.numel() and (int(act.min()) < 0 or int(act.max()) >= G):
        raise ValueError("seq_action must lie in [0, number of actions)")
    run_start, run_group = loader_batch_runs(seq_lengths, act, F, batch_size)
    N = int(run_start[-1])
    if tuple(pred.shape) != (N, engine.J, 3):
        raise ValueError(f"pred must have shape {(N, engine.J, 3)} (sum of seq_lengths frames), got {tuple(pred.shape)}")
    dev = engine.device
    pred, gt = pred.contiguous(), gt.to(dev).contiguous()
    acc = torch.zeros((G, 6), device=dev, dtype=torch.float64)
    bounds = run_start.tolist()
    for r, g in enumerate(run_group.tolist()):
        a, b = bounds[r], bounds[r + 1]
        engine.pose_metrics_accumulate(pred[a:b], gt[a:b], acc[g])
    acc = acc.cpu()

    def row(a):
        if a[5].item() == 0:
            vals = (float("nan"),) * 4
        else:
            vals = tuple(v * mm_per_unit for v in Engine.pose_metrics(a))
        return dict(zip(("mpjpe", "p_mpjpe", "n_mpjpe", "velocity"), vals), frames=int(a[5].item()))

    rows = [row(acc[g]) for g in range(G)]
    have = [r for r in rows if r["frames"]]
    keys = ("mpjpe", "p_mpjpe", "n_mpjpe", "velocity")
    mean = {k: (sum(r[k] for r in have) / len(have) if have else float("nan")) for k in keys}
    return {"actions": dict(zip(names, rows)), "action_mean": dict(mean, frames=sum(r["frames"] for r in have)),
            "pooled": row(acc.sum(dim=0))}


def gather_results(local_pred: torch.Tensor, acc: torch.Tensor, n_total: int, group=None):
    """The single exchange step: all-gather of the (padded) prediction shards + all-reduce(sum) of the fp64
    (error sum, joint count) pair.  Returns (pred [n_total,F,J,3] on every rank, mpjpe float)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        cnt = acc[1].item()
        return local_pred, (acc[0].item() / cnt if cnt else float("nan"))
    world = dist.get_world_size(group)
    per = (n_total + world - 1) // world
    pad = torch.zeros((per,) + tuple(local_pred.shape[1:]), device=local_pred.device, dtype=local_pred.dtype)
    pad[: local_pred.shape[0]] = local_pred
    bucket = torch.empty((world * per,) + tuple(local_pred.shape[1:]), device=local_pred.device,
                         dtype=local_pred.dtype)
    dist.all_gather_into_tensor(bucket, pad, group=group) if bucket.is_cuda else dist.all_gather(
        list(bucket.view(world, per, *local_pred.shape[1:]).unbind(0)), pad, group=group)
    dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
    parts = []
    for r in range(world):
        _, c = shard_range(n_total, r, world)
        parts.append(bucket[r * per: r * per + c])
    cnt = acc[1].item()
    return torch.cat(parts), (acc[0].item() / cnt if cnt else float("nan"))


def _all_gather(bucket: torch.Tensor, local: torch.Tensor, group):
    world = dist.get_world_size(group)
    if bucket.is_cuda:
        dist.all_gather_into_tensor(bucket, local, group=group)
    else:
        dist.all_gather(list(bucket.view(world, *local.shape).unbind(0)), local, group=group)


def gather_packed(local_pred: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather of packed predictions [n_r, ...] whose frame count n_r differs per rank (each rank's sequences of
    `evaluate_sequences`): the counts first, then every shard padded to the largest, gathered and unpadded in rank
    order.  When rank r owns a contiguous block of whole sequences (`shard_range` over sequences) the result is the
    global packed array, on every rank.  NCCL on GPUs, gloo for CPU tensors."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local_pred
    world = dist.get_world_size(group)
    n = torch.tensor([local_pred.shape[0]], device=local_pred.device, dtype=torch.int64)
    counts = torch.empty(world, device=local_pred.device, dtype=torch.int64)
    _all_gather(counts, n, group)
    counts = counts.tolist()
    per, tail = max(counts), tuple(local_pred.shape[1:])
    if per == 0:
        return local_pred
    pad =torch.zeros((per,) + tail, device=local_pred.device, dtype=local_pred.dtype)
    pad[: local_pred.shape[0]] = local_pred
    bucket = torch.empty((world * per,) + tail, device=local_pred.device, dtype=local_pred.dtype)
    _all_gather(bucket, pad, group)
    return torch.cat([bucket[r * per: r * per + c] for r, c in enumerate(counts)])
