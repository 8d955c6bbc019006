"""Throughput of the sampler at a given model width (embed_dim 256 or 512) on one GPU: F = 243, S = 9 DDIM steps,
flip-TTA, `--clips` clips per step (each clip and its flipped copy sampled as one batch of 2 * clips).

Reports pose-frames/s of the resident step (ddim_sample of the batch + TTA merge, inputs already on the device), the
per-class device time of one un-graphed step (d3d_profile_*), the GEMM class's algorithmic TFLOP/s for width C
(qkv + proj + fc1 + fc2 = 16 C^2 FLOPs per token and block, 16 blocks) as a fraction of the dense fp16 data-sheet peak,
and the card's name and power limit read in the same run.  Prints one JSON line.

    python tools/width_bench.py --embed-dim 256 [--clips 512 --steps 3 --warmup 1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from diff3dhpe_b200 import _lib, synthetic  # noqa: E402

FP16_DENSE_PEAK_TFLOPS = 2250.0   # HGX B200 data sheet, one GPU, dense fp16 / bf16, at a 1000 W limit


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:       # noqa: BLE001 -- the numbers stay valid, the card is just unnamed
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--embed-dim", type=int, default=256)
    ap.add_argument("--frames", type=int, default=243)
    ap.add_argument("--clips", type=int, default=512)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("width_bench.py needs a B200")
    C, F, B, S, J = args.embed_dim, args.frames, args.clips, 9, 17
    L, R = synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT
    dev = torch.device("cuda", 0)
    model = synthetic.make_model(F, embed_dim=C).to(dev)
    model.gemm_mode, model.max_clips_hint = _lib.GEMM_TC_F4C, 2 * B
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).to(dev).eval()
    eng = diff._engine(2 * B)
    x2d, _ = synthetic.make_inputs(B, F)
    x2d = x2d.to(dev)
    xs = torch.cat([x2d, synthetic.flip_2d(x2d, L, R)]).contiguous()
    ys = torch.randn(2 * B, F, J, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(99))

    def step():
        raw = eng.ddim_sample(xs, ys)
        return eng.tta_merge(raw[:B], raw[B:], L, R, 1.0)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1000.0 / args.steps
    assert torch.isfinite(out).all()

    eng.profile_begin()
    step()
    prof = eng.profile_end()
    tokens = 2 * B * F * J
    gemm_ms = prof["gemm"][0]
    gemm_flops = tokens * S * 16 * (16 * C * C)
    tflops = gemm_flops / (gemm_ms / 1000.0) / 1e12
    print(json.dumps({
        "embed_dim": C, "F": F, "S": S, "clips_per_step": B, "tta": True,
        "step_ms": round(ms, 2), "pose_frames_per_s": round(B * F / (ms / 1000.0), 1),
        "profile_ms": {k: round(v[0], 2) for k, v in prof.items()},
        "profile_launches": {k: v[1] for k, v in prof.items()},
        "gemm_algorithmic_tflops": round(tflops, 1),
        "gemm_frac_of_fp16_datasheet_peak": round(tflops / FP16_DENSE_PEAK_TFLOPS, 3),
        "gemm_flops_note": "16 C^2 FLOPs per token and block (qkv 6 C^2, proj 2 C^2, fc1 4 C^2, fc2 4 C^2), 16 blocks, "
                           "S steps, orig + flipped clips; peak = dense fp16 data-sheet rate (1000 W card)",
        "card": card(),
    }))


if __name__ == "__main__":
    main()
