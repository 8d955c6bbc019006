#!/usr/bin/env python
"""The reference's evaluate() inner loop (RUN:577-588) under nn.DataParallel, at the three published evaluation commands
(Experiments.sh:5, :11, :17), on seeded synthetic inputs:

    python tools/dataparallel_eval.py [--batches 2] [--warmup 1] [--seed 0] [--bench] [--out DIR]

Per batch: an original and a flipped `forward(..., output_loss=...)` call of nn.DataParallel(GaussianDiffusion), then
un-flip and average on the first device.  Each command runs at 1 GPU and at its published GPU count; a count above the
visible devices prints a "skipped" line.  One JSON line per run:
  - pose_frames_per_s: clips x F (a flip pair counts once) over the wall time of the timed batches;
  - outside_engine_share: 1 - (engine time of the busiest device) / wall time, where engine time is the sampler and
    p_losses denoiser calls timed with CUDA events on each device; the rest is replicate / scatter / gather / Python /
    un-flip.  Every call re-broadcasts the ~175 MB of fp32 parameters to each extra device; that cost is inside this
    share and is not measured on its own;
  - pred_sha256: digest of every merged prediction (bit-identical across runs with the same seeds);
  - gpu: card name, power limit and max SM clock, read in the same run.
--bench adds the same-session `bench.py --gpus N` weak-scaling line (cfg3: F = 243, S = 9, 256 clips per GPU plus
their flipped copies) for each GPU count that can run.  --out DIR also writes the last batch's merged predictions.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402
from torch import nn  # noqa: E402

# Experiments.sh:5 (h36m_cpn, F = 81), :11 (h36m_gt, F = 243), :17 (3dhp_gt, F = 27, no time embedding, output_loss)
COMMANDS = [
    dict(name="h36m_cpn_f81", F=81, S=9, batch=256, gpus=4, time_emb=True, output_loss=False, lists="h36m"),
    dict(name="h36m_gt_f243", F=243, S=6, batch=256, gpus=8, time_emb=True, output_loss=False, lists="h36m"),
    dict(name="3dhp_gt_f27", F=27, S=7, batch=512, gpus=4, time_emb=False, output_loss=True, lists="3dhp"),
]


def gpu_info(n):
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                              ",".join(str(i) for i in range(n))], capture_output=True, text=True, timeout=30).stdout
        return [line.strip() for line in out.strip().splitlines()]
    except (OSError, subprocess.TimeoutExpired):
        return [torch.cuda.get_device_name(i) + ", power limit unknown" for i in range(n)]


class EngineTimer:
    """CUDA events around every Engine.ddim_sample / forward_denoise, on the stream of the calling device."""

    def __init__(self):
        from diff3dhpe_b200.engine import Engine
        self.events, self.lock, self.on = [], threading.Lock(), False
        for name in ("ddim_sample", "forward_denoise"):
            real = getattr(Engine, name)

            def timed(eng, *a, _real=real, **kw):
                if not self.on:
                    return _real(eng, *a, **kw)
                st = torch.cuda.current_stream(eng.device)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                out = _real(eng, *a, **kw)
                e1.record(st)
                with self.lock:
                    self.events.append((eng.device.index, e0, e1))
                return out
            setattr(Engine, name, timed)

    def busy_ms(self):
        """Engine time of the busiest device, in ms (one thread per device: a device's calls never overlap)."""
        per_dev = {}
        for dev, e0, e1 in self.events:
            per_dev[dev] = per_dev.get(dev, 0.0) + e0.elapsed_time(e1)
        return max(per_dev.values()) if per_dev else 0.0


def unflip(pred, left, right):
    p = pred.clone()
    p[..., 0] *= -1
    p[:, :, left + right] = p[:, :, right + left]
    return p


def run_command(cmd, n, args, timer):
    from diff3dhpe_b200 import synthetic
    F, S, B = cmd["F"], cmd["S"], cmd["batch"]
    left, right = ((synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT) if cmd["lists"] == "h36m"
                   else (synthetic.MPI3DHP_JOINTS_LEFT, synthetic.MPI3DHP_JOINTS_RIGHT))
    model = synthetic.make_model(F, with_time_emb=cmd["time_emb"], seed=args.seed).cuda(0)
    model.max_clips_hint = -(-B // n)                   # each replica samples its own chunk
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).cuda(0).eval()
    dp = nn.DataParallel(diff, device_ids=list(range(n)))
    batches = []
    for i in range(args.warmup + args.batches):
        x2d, gt = synthetic.make_inputs(B, F, seed=1000 * args.seed + i)
        batches.append((x2d.cuda(0), synthetic.flip_2d(x2d, left, right).cuda(0), gt.cuda(0)))
    digest = hashlib.sha256()
    merged = []

    def one_batch(i):
        x2d, xf, gt = batches[i]
        torch.cuda.manual_seed_all(args.seed * 7919 + i)
        _, pred = dp(gt, x2d, output_loss=cmd["output_loss"])
        _, pred_f = dp(gt, xf, output_loss=cmd["output_loss"])
        return (pred + unflip(pred_f, left, right)) / 2

    def sync():
        for d in range(n):
            torch.cuda.synchronize(d)

    for i in range(args.warmup):
        digest.update(one_batch(i).cpu().numpy().tobytes())
    sync()
    timer.events.clear()
    timer.on = True
    t0 = time.perf_counter()
    for i in range(args.warmup, args.warmup + args.batches):
        merged.append(one_batch(i))
    sync()
    wall = time.perf_counter() - t0
    timer.on = False
    busy = timer.busy_ms() / 1000.0
    for m in merged:                    # digested after the timed region: no host copies inside it
        digest.update(m.cpu().numpy().tobytes())
    if args.out:
        import numpy as np
        os.makedirs(args.out, exist_ok=True)
        np.save(os.path.join(args.out, f"{cmd['name']}_gpus{n}.npy"), merged[-1].cpu().numpy())
    engines = [diff.model._shared.peek(torch.device("cuda", d)) for d in range(n)]
    del dp, diff, model
    return {"command": cmd["name"], "F": F, "S": S, "batch": B, "n_gpus": n, "output_loss": cmd["output_loss"],
            "time_emb": cmd["time_emb"], "batches_timed": args.batches, "wall_s": wall,
            "pose_frames_per_s": args.batches * B * F / wall, "engine_busy_s": busy,
            "outside_engine_share": max(0.0, 1.0 - busy / wall), "engines": sum(e is not None for e in engines),
            "pred_sha256": digest.hexdigest()}


def bench_line(n, args):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--steps", str(args.bench_steps),
           "--warmup", "1"]
    if n > 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
               "--master-addr", "127.0.0.1", "--master-port", "29517"] + cmd[1:]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    if out.returncode != 0 or not lines:
        return {"bench_gpus": n, "status": "failed", "stderr_tail": out.stderr[-2000:]}
    r = json.loads(lines[-1])
    return {"bench_gpus": n, "value": r["value"], "unit": r["unit"], "ms_per_step": r["ms_per_step"],
            "per_gpu_batch": "256 clips + 256 flipped copies (cfg3, F = 243, S = 9)"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batches", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--only", default=None, help="comma-separated command names")
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--bench-steps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.batches < 1 or args.warmup < 0:
        raise SystemExit("--batches must be >= 1 and --warmup >= 0")
    if not torch.cuda.is_available():
        raise SystemExit("dataparallel_eval.py needs B200 GPUs: there is no CPU fallback")
    visible = torch.cuda.device_count()
    print(json.dumps({"gpu": gpu_info(visible), "visible_gpus": visible, "torch": torch.__version__}), flush=True)
    timer = EngineTimer()
    for cmd in COMMANDS:
        if args.only and cmd["name"] not in args.only.split(","):
            continue
        for n in sorted({1, cmd["gpus"]}):
            if n > visible:
                print(json.dumps({"command": cmd["name"], "n_gpus": n, "status": "skipped",
                                  "reason": f"{n} GPUs requested, {visible} visible"}), flush=True)
                continue
            print(json.dumps(run_command(cmd, n, args, timer)), flush=True)
            torch.cuda.empty_cache()
    if args.bench:
        for n in sorted({1} | {c["gpus"] for c in COMMANDS}):
            if n > visible:
                print(json.dumps({"bench_gpus": n, "status": "skipped", "reason": f"{visible} GPUs visible"}), flush=True)
                continue
            print(json.dumps(bench_line(n, args)), flush=True)


if __name__ == "__main__":
    main()
