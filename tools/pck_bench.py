#!/usr/bin/env python
"""Device time of d3d_pck_accumulate (the MPI-INF-3DHP PCK / AUC histogram) at the size of a full-test-set sweep:

    python tools/pck_bench.py [--frames 540000] [--iters 20] [--out DIR]

Seeded synthetic poses in mm (errors uniform in 0-300 mm), the 31 protocol thresholds, no frame index.  One JSON line
per group count: 1 group (shared-memory histogram) and 4096 groups (global atomics), each the mean of --iters calls
timed with CUDA events after one warm-up call, with the card's name, power limit and max SM clock read in the same
run.  The inputs (2 x frames x 17 x 3 fp32, 220 MB at 540 k frames) are larger than the L2, so every call reads HBM.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from diff3dhpe_b200 import evaluate  # noqa: E402
from diff3dhpe_b200.engine import Engine  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip()
    except (OSError, subprocess.TimeoutExpired):
        return torch.cuda.get_device_name() + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=540_000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/pck_bench.jsonl")
    args = ap.parse_args()
    if args.frames < 1 or args.iters < 1:
        ap.error("--frames and --iters must be positive")
    J, n = 17, args.frames
    g = torch.Generator().manual_seed(0)
    gt = 300.0 * torch.randn(n, J, 3, generator=g)
    d = torch.randn(n, J, 3, generator=g)
    pred = gt + d / d.norm(dim=-1, keepdim=True) * 300.0 * torch.rand(n, J, 1, generator=g)
    pred, gt = pred.cuda().contiguous(), gt.cuda().contiguous()
    eng = Engine(27, max_clips=1)
    thr = evaluate.mpi3dhp_thresholds(1.0)
    info = gpu_info()
    lines = []
    for G in (1, 4096):
        grp = (torch.arange(n, device="cuda") * G // n).to(torch.int32)       # G contiguous runs of frames
        counts = torch.zeros((G, J, len(thr)), dtype=torch.int64, device="cuda")
        err_sum = torch.zeros((G, J), dtype=torch.float64, device="cuda")
        frames = torch.zeros(G, dtype=torch.int64, device="cuda")
        eng.pck_accumulate(pred, gt, counts, err_sum, frames, thr, None, grp)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.iters):
            eng.pck_accumulate(pred, gt, counts, err_sum, frames, thr, None, grp)
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b) / args.iters
        assert int(frames.sum()) == (args.iters + 1) * n
        lines.append(json.dumps({"tool": "pck_bench", "frames": n, "joints": J, "thresholds": len(thr), "groups": G,
                                 "ms_per_call": round(ms, 4), "gb_per_s": round(2 * n * J * 3 * 4 / ms / 1e6, 1),
                                 "iters": args.iters, "gpu": info}))
        print(lines[-1], flush=True)
    eng.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "pck_bench.jsonl"), "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
