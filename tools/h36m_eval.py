#!/usr/bin/env python
"""The Human3.6M per-action table of a full-test-set-sized sweep, with the wall time of every stage:

    python tools/h36m_eval.py [--sequences 240] [--actions 15] [--out DIR]                  # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tools/h36m_eval.py                                                                  # sequences sharded over N ranks

The cfg5 shape: 240 synthetic sequences x 2250 frames (seeded; poses in metres), F = 243, S = 9, flip-TTA, batches of
256 windows, 15 actions of 16 consecutive sequences each.  Stages, timed on the host around work that ends in a device
synchronise, after one untimed warm-up sweep:
  sweep   evaluate.evaluate_sequences over this rank's contiguous block of whole sequences (slowest rank);
  gather  evaluate.gather_packed (skipped on one GPU);
  table   evaluate.h36m_metrics on the gathered array: one d3d_pose_metrics_accumulate call per reference batch of 256
          windows (--table-batch), one device-to-host copy; mean of --table-reps calls;
  host    the reference's host path on the same frames and batches: per batch a device-to-host copy of the predictions,
          then numpy P-MPJPE and velocity error (common/loss.py, restated in oracle/diff3d_oracle.py), as evaluate()
          does at RUN:602-614.
Prints the table and one JSON line on rank 0, with the card's name, power limit and max SM clock read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from diff3dhpe_b200 import evaluate, synthetic  # noqa: E402
from oracle import diff3d_oracle as oracle  # noqa: E402

J, F, S, SEQ_LEN = 17, 243, 9, 2250
MM_PER_UNIT = 1000.0


def gpu_info(dev):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(dev.index)], capture_output=True, text=True, timeout=30).stdout
        return out.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name(dev) + ", power limit unknown"


def synchronise(world, dev):
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()


def host_reference(pred_d, gt_h, run_start, run_group, n_actions):
    """evaluate()'s host tail per batch (RUN:602-614): copy the batch's predictions to the host, numpy P-MPJPE and
    velocity error, N_b-weighted sums per action.  Returns (seconds, per-action P-MPJPE, per-action velocity)."""
    sums = np.zeros((n_actions, 3))
    bounds = run_start.tolist()
    t0 = time.perf_counter()
    for r, g in enumerate(run_group.tolist()):
        a, b = bounds[r], bounds[r + 1]
        p = pred_d[a:b].cpu().numpy()
        t = gt_h[a:b]
        sums[g] += (b - a) * np.array([oracle.p_mpjpe(p, t), oracle.mean_velocity_error(p, t), 1.0])
    dt = time.perf_counter() - t0
    return dt, sums[:, 0] / sums[:, 2], sums[:, 1] / sums[:, 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sequences", type=int, default=240)
    ap.add_argument("--actions", type=int, default=15)
    ap.add_argument("--batch", type=int, default=256, help="windows per sampler batch (x2 with the flipped copies)")
    ap.add_argument("--table-batch", type=int, default=256, help="windows per reference loader batch")
    ap.add_argument("--table-reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON line to DIR/h36m_eval.jsonl")
    args = ap.parse_args()
    if min(args.sequences, args.actions, args.batch, args.table_batch, args.table_reps) < 1:
        ap.error("all counts must be positive")
    if args.sequences % args.actions:
        ap.error("--sequences must be a multiple of --actions")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_seq = args.sequences
    lengths = [SEQ_LEN] * n_seq
    actions = [s // (n_seq // args.actions) for s in range(n_seq)]
    names = [f"A{a + 1:02d}" for a in range(args.actions)]
    g = torch.Generator().manual_seed(2000)
    seq2d = (0.3 * torch.randn(n_seq * SEQ_LEN, J, 2, generator=g)).clamp_(-1, 1)
    gt = 0.3 * torch.randn(n_seq * SEQ_LEN, J, 3, generator=g)
    gt = gt - gt[:, :1]
    start, count = evaluate.shard_range(n_seq, rank, world)
    frames = slice(start * SEQ_LEN, (start + count) * SEQ_LEN)
    local_2d, local_gt = seq2d[frames].pin_memory(), gt[frames].pin_memory()
    window_offset = evaluate.plan_windows(lengths[:start], F)[0].numel()

    model = synthetic.make_model(F).to(dev)
    model.max_clips_hint = 2 * args.batch
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).to(dev).eval()
    sampler = evaluate.DeviceSampler(diff)

    def noise_fn(ids, flip):
        return diff.draw_noise([len(ids), F, J, 3], dev)

    def sweep():
        return evaluate.evaluate_sequences(sampler, local_2d, local_gt, lengths[start:start + count], noise_fn,
                                           device=dev, F=F, batch_clips=args.batch, window_offset=window_offset)

    sweep()                                                       # warm-up: weight upload, graph capture
    synchronise(world, dev)
    t0 = time.perf_counter()
    res = sweep()
    torch.cuda.synchronize(dev)
    t_sweep = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_sweep, op=dist.ReduceOp.MAX)
    synchronise(world, dev)
    t0 = time.perf_counter()
    pred = evaluate.gather_packed(res["pred"])
    synchronise(world, dev)
    t_gather = time.perf_counter() - t0
    assert pred.shape == (n_seq * SEQ_LEN, J, 3)

    if rank == 0:
        eng = model.engine(1)
        gt_d = gt.to(dev)
        kw = dict(F=F, batch_size=args.table_batch, mm_per_unit=MM_PER_UNIT, action_names=names)
        table = evaluate.h36m_metrics(eng, pred, gt_d, lengths, actions, **kw)          # warm-up
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(args.table_reps):
            table = evaluate.h36m_metrics(eng, pred, gt_d, lengths, actions, **kw)
        t_table = (time.perf_counter() - t0) / args.table_reps
        run_start, run_group = evaluate.loader_batch_runs(lengths, actions, F, args.table_batch)
        t_host, host_p, host_v = host_reference(pred, gt.numpy(), run_start, run_group, args.actions)
        dev_p = np.array([table["actions"][n]["p_mpjpe"] for n in names])
        dev_v = np.array([table["actions"][n]["velocity"] for n in names])
        info = gpu_info(dev)
        print(f"{'action':<8}{'frames':>9}{'MPJPE':>10}{'P-MPJPE':>10}{'N-MPJPE':>10}{'MPJVE':>10}   (mm)")
        rows = list(table["actions"].items()) + [("mean", table["action_mean"]), ("pooled", table["pooled"])]
        for name, r in rows:
            print(f"{name:<8}{r['frames']:>9}{r['mpjpe']:>10.3f}{r['p_mpjpe']:>10.3f}{r['n_mpjpe']:>10.3f}"
                  f"{r['velocity']:>10.3f}")
        line = {"tool": "h36m_eval", "n_gpus": world, "sequences": n_seq, "frames": n_seq * SEQ_LEN, "F": F, "S": S,
                "tta": True, "actions": args.actions, "sampler_batch": args.batch, "table_batch": args.table_batch,
                "table_runs": run_group.numel(), "sweep_s": round(t_sweep.item(), 3),
                "gather_s": round(t_gather, 4) if world > 1 else None, "table_s": round(t_table, 5),
                "table_share_of_sweep": round(t_table / t_sweep.item(), 7), "host_reference_s": round(t_host, 3),
                "host_vs_device_max_abs_mm": {"p_mpjpe": float(np.abs(host_p * MM_PER_UNIT - dev_p).max()),
                                              "velocity": float(np.abs(host_v * MM_PER_UNIT - dev_v).max())},
                "action_mean_mpjpe_mm": table["action_mean"]["mpjpe"], "gpu": info}
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "h36m_eval.jsonl"), "a") as f:
                f.write(json.dumps(line) + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    model._engine.close()


if __name__ == "__main__":
    main()
