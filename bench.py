#!/usr/bin/env python
"""Benchmark of the Diff3DHPE DDIM/MixSTE sampler hot path on B200 (see BASELINE.json / SURVEY.md 8d).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference algorithm's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's predictions to DIR/pred.npy

Workload ("step"): cfg3 of BASELINE.json -- MixSTE s2s h36m_gt config, F=243 frames, 9 DDIM steps, flip
test-time augmentation, 256 clips per GPU (weak scaling): one step = DDIM-sample the 256 clips and their 256
flipped copies (one 512-clip batch, 2.1 M tokens), un-flip + average.  Metric: denoised pose-frames/s
(a flip pair counts once) = n_gpus * 256 * 243 / step time.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree, which may be read-only

import torch  # noqa: E402

F_FRAMES, J, S_STEPS = 243, 17, 9
METRIC, UNIT = "denoised_pose_frames_per_s", "pose-frames/s"
DUMP_BYTES = 60 * 2 ** 20           # --dump-outputs: keeps the files under 64 MB

# BASELINE.json configs.  cfg3 is the configuration the metric is quoted on (the default, and what the driver runs);
# the others are selectable with --config so that their lines come from the same harness (profiles/).
#   clips: per GPU (weak scaling) -- or the TOTAL number of windows for the strong-scaling cfg5 sweep
WORKLOADS = {
    "cfg2": dict(F=81, S=9, clips=256, tta=False, time_emb=True, lists="h36m", scaling="weak",
                 name="cfg2: Diff3DHPE-MixSTE s2s h36m_cpn, F=81, S=9 DDIM steps, no flip pass, 256 clips on 1 B200"),
    "cfg3": dict(F=243, S=9, clips=256, tta=True, time_emb=True, lists="h36m", scaling="weak", name=None),
    "cfg4": dict(F=27, S=9, clips=2048, tta=True, time_emb=False, lists="3dhp", scaling="weak",
                 name="cfg4: Diff3DHPE-MixSTE s2s 3dhp_gt, F=27, no time embedding (Experiments.sh:17), flip-TTA with the "
                      "MPI-INF-3DHP joint lists, 2048 clips/GPU"),
    "cfg5": dict(F=243, S=9, clips=2400, tta=True, time_emb=True, lists="h36m", scaling="strong",
                 name="cfg5: full-test-set-sized sweep, 240 sequences x 2250 frames = 540 000 frames -> 2400 windows of "
                      "F=243 (last window of a sequence back-shifted, overlap masked), S=9, flip-TTA, windows sharded over "
                      "the ranks in batches of 256 (+ a partial last batch), gather of predictions + MPJPE all-reduce"),
}


def workload_name(clips):
    return (f"cfg3: Diff3DHPE-MixSTE s2s h36m_gt, F={F_FRAMES}, S={S_STEPS} DDIM steps, flip-TTA, "
            f"{clips} clips/GPU (x2 flip copies in one batch), depth 8, dim 512, random-init weights")


def flops_per_token_call(F):
    """SURVEY.md 8(d): algorithmic FLOPs per token per denoiser call."""
    return 67395584 + 16384 * F


GEMM_FLOPS_PER_TOKEN_CALL = 16 * 4194304      # qkv + proj + fc1 + fc2, 16 blocks


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"], "hbm_gbs": d["hbm_gbs"],
                "source": "MEASURED_PEAKS.json"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "200", "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        busy = [s for s in sm if s > 500] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference arm
def resolve_workload(args):
    wl = dict(WORKLOADS[args.config])
    if args.clips:
        wl["clips"] = args.clips
    if args.sampling_timesteps:
        wl["S"] = args.sampling_timesteps
    if wl["name"] is None or args.clips or args.sampling_timesteps:
        if args.config == "cfg3":
            wl["name"] = workload_name(wl["clips"]).replace(f"S={S_STEPS} ", f"S={wl['S']} ")
        else:
            wl["name"] += f" [overrides: clips={wl['clips']}, S={wl['S']}]"
    from diff3dhpe_b200 import synthetic
    wl["left"], wl["right"] = ((synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT) if wl["lists"] == "h36m" else
                               (synthetic.MPI3DHP_JOINTS_LEFT, synthetic.MPI3DHP_JOINTS_RIGHT))
    return wl


def cpu_sample(wl, n_clips=1, threads=None, keep=None):
    """The reference algorithm's CPU path (oracle port: fp32 torch-CPU restatement, bit-identical to the imported
    reference in the build container) on a bounded sample of the SAME workload: n_clips clips of the workload's F, S,
    time-embedding setting and (with flip-TTA) two sampler passes + merge.  Returns (pose-frames/s, seconds, threads)."""
    from diff3dhpe_b200 import synthetic
    from oracle import diff3d_oracle as oracle
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    F, S = wl["F"], wl["S"]
    m = synthetic.make_model(F, with_time_emb=wl["time_emb"])
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    x2d, gt = synthetic.make_inputs(n_clips, F)
    n1, n2 = synthetic.make_noise(n_clips, F, S, seed=1), synthetic.make_noise(n_clips, F, S, seed=2)
    t0 = time.perf_counter()
    with torch.no_grad():
        if wl["tta"]:
            y = oracle.ddim_sample_loop(sd, x2d, *n1, sampling_timesteps=S)
            yf = oracle.ddim_sample_loop(sd, oracle.flip_2d(x2d, wl["left"], wl["right"]), *n2, sampling_timesteps=S)
            ref = oracle.tta_merge(y, yf, 1.0, wl["left"], wl["right"])
        else:
            ref = oracle.ddim_sample_loop(sd, x2d, *n1, sampling_timesteps=S)
    dt = time.perf_counter() - t0
    if keep is not None:
        keep.update(ref=ref, x2d=x2d, gt=gt, n1=n1, n2=n2)
    return n_clips * F / dt, dt, threads


def sample_desc(wl, n=1):
    return (f"{n} clip x {wl['F']} frames, S={wl['S']}, " + ("flip-TTA (2 sampler passes + merge)" if wl["tta"] else "one sampler pass") +
            ", fp32 torch-CPU oracle port")


def parity_on_sample(wl, keep, gemm_mode):
    """The CPU sample's clip through the CUDA path (same weights, 2D input and noise seeds; drop-in module -> C ABI) and
    the two numbers BASELINE.json's metric asks for next to the throughput: per-joint max-abs error (pose scale 1,
    bar 1e-2) and |MPJPE(ours) - MPJPE(reference port)| (bar 1e-4 = 0.1 mm).  The oracle is the checker here."""
    from diff3dhpe_b200 import synthetic
    from oracle import diff3d_oracle as oracle
    F, S = wl["F"], wl["S"]
    n = keep["x2d"].shape[0]
    mult = 2 if wl["tta"] else 1
    model = synthetic.make_model(F, with_time_emb=wl["time_emb"]).cuda()
    model.gemm_mode, model.max_clips_hint = gemm_mode, mult * n
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).cuda().eval()
    if wl["tta"]:
        x = torch.cat([keep["x2d"], synthetic.flip_2d(keep["x2d"], wl["left"], wl["right"])]).cuda()
        y = diff.ddim_sample_loop(x, [2 * n, F, 17, 3], noise=(torch.cat([keep["n1"][0], keep["n2"][0]]).cuda(), None))
        merged = diff._engine(2 * n).tta_merge(y[:n], y[n:], wl["left"], wl["right"], 1.0).cpu()
    else:
        merged = diff.ddim_sample_loop(keep["x2d"].cuda(), [n, F, 17, 3], noise=(keep["n1"][0].cuda(), None)).cpu()
    model._engine.close()
    ref, gt = keep["ref"], keep["gt"]
    return {"max_abs_err": (merged - ref).abs().max().item(), "max_abs_bar": 1e-2,
            "mpjpe_delta": abs(oracle.mpjpe(merged, gt).item() - oracle.mpjpe(ref, gt).item()), "mpjpe_delta_bar": 1e-4,
            "sample": sample_desc(wl, n) + "; same weights / inputs / noise seeds as the CPU arm"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = resolve_workload(args)
    times = []
    for i in range(args.warmup + args.steps):
        fps, dt, threads = cpu_sample(wl, 1)
        if i >= args.warmup:
            times.append(dt)
    ms = 1000.0 * sum(times) / len(times)
    value = wl["F"] / (ms / 1000.0)
    sample = sample_desc(wl) + " per step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["name"], "sample": sample,
                   "note": "the reference is pure Python/PyTorch, is not pip-installable and cannot travel to the GPU box; "
                           "this arm times the oracle port (kind 'port'), which tools/make_golden.py proves bit-identical "
                           "to the imported reference in the build container"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def dump_outputs(out_dir, pred):
    """Writes pred [clips, F, J, 3] as out_dir/pred.npy (float32).  Beyond DUMP_BYTES it keeps a sample of clips drawn
    with a fixed seed, in clip order, so two builds run with the same arguments dump the same clips."""
    import numpy as np
    keep = DUMP_BYTES // (pred[0].numel() * 4)
    if pred.shape[0] > keep:
        idx = torch.randperm(pred.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        pred = pred[idx.to(pred.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pred.npy"), pred.detach().to("cpu", torch.float32).numpy())


def run_ours(args):
    import torch.distributed as dist
    from diff3dhpe_b200 import _lib, evaluate, synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stdout_fd = None
    if world > 1:
        # stdout must carry exactly ONE JSON line: NCCL prints its version banner on fd 1 from C (NCCL_DEBUG_FILE does not
        # catch it on this image), so fd 1 points at stderr until the line is printed
        sys.stdout.flush()
        stdout_fd = os.dup(1)
        os.dup2(2, 1)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    wl = resolve_workload(args)
    F, S, tta, L, R = wl["F"], wl["S"], wl["tta"], wl["left"], wl["right"]
    mult = 2 if tta else 1
    strong = wl["scaling"] == "strong"
    if strong:       # cfg5: a FIXED total of windows, sharded contiguously; batches of args.batch + a partial last batch
        n_total = wl["clips"]
        shard_start, B = evaluate.shard_range(n_total, rank, world)
        batch = min(args.batch, B)
    else:            # weak scaling: every GPU owns wl["clips"] clips, sampled as one batch
        B = wl["clips"]
        n_total, shard_start, batch = world * B, rank * B, B
    gemm_mode = {"split3": _lib.GEMM_TC_SPLIT3, "fp16": _lib.GEMM_TC_FP16, "f8c": _lib.GEMM_TC_F8C,
                 "f4c": _lib.GEMM_TC_F4C}[args.gemm]

    model = synthetic.make_model(F, with_time_emb=wl["time_emb"]).to(dev)
    model.gemm_mode, model.max_clips_hint = gemm_mode, mult * batch
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).to(dev).eval()
    eng = diff._engine(mult * batch)

    # ---- synthetic inputs of this rank's clips (distinct per rank), resident in HBM for `value`
    x2d_h, gt_h = synthetic.make_inputs(B, F, seed=1234 + rank)
    x2d_h, gt_h = x2d_h.pin_memory(), gt_h.pin_memory()
    mask_h, valid_frames = None, n_total * F
    if strong:       # the back-shifted last window of every 2250-frame sequence repeats 180 frames: masked (GEN:27-48)
        wins = evaluate.window_starts(2250, F)
        mask_h = torch.ones(B, F, dtype=torch.uint8)
        for i in range(B):
            mask_h[i, :wins[(shard_start + i) % len(wins)][1]] = 0
        mask_h = mask_h.pin_memory()
        valid_frames = (n_total // len(wins)) * 2250
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    spans = [(s0, min(B, s0 + batch)) for s0 in range(0, B, batch)]
    x_dev = x2d_h.to(dev)
    xs, ys = [], []
    for s0, e0 in spans:
        xb = x_dev[s0:e0]
        xs.append(torch.cat([xb, synthetic.flip_2d(xb, L, R)]).contiguous() if tta else xb.contiguous())
        ys.append(torch.randn(mult * (e0 - s0), F, J, 3, device=dev, generator=gen))
    stream = torch.cuda.current_stream(dev)
    raw = [None] * len(spans)

    def step_resident():
        outs = []
        for i, (s0, e0) in enumerate(spans):
            n = e0 - s0
            raw[i] = eng.ddim_sample(xs[i], ys[i])
            outs.append(eng.tta_merge(raw[i][:n], raw[i][n:], L, R, 1.0) if tta else raw[i])
        return outs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    for _ in range(args.warmup):
        outs = step_resident()
    barrier()
    launches0 = eng.launch_count()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0_.record(stream)
    for _ in range(args.steps):
        outs = step_resident()
    e1_.record(stream)
    barrier()
    ms_total = max_over_ranks(e0_.elapsed_time(e1_))
    clk = clocks.stop() if rank == 0 else None
    gpu_launches = eng.launch_count() - launches0
    ms_step = ms_total / args.steps
    value = valid_frames / (ms_step / 1000.0)

    # ---- the timed output itself is checked, at the timed size: finite, inside the clamp range, and the first, middle
    #      and last clips of the timed batch BIT-EQUAL to the same clips sampled alone (clips are independent, RUN:577-588;
    #      tests/test_gpu_sampler.py::test_batch_split_invariance... asserts the same property small).  This is what pins
    #      the 2.1 M-token launches (byte offsets > 2^32, TMA coordinates, tile order) to the parity-tested small ones.
    y_timed = raw[0]
    n0 = y_timed.shape[0]
    assert all(torch.isfinite(o).all() and o.abs().max().item() <= 1.0 + 1e-6 for o in outs)
    picks = sorted({0, n0 // mult - 1, n0 // 2, n0 - 1})
    mismatched = []
    for i in picks:
        one = eng.ddim_sample(xs[0][i:i + 1].contiguous(), ys[0][i:i + 1].contiguous())
        if not torch.equal(one[0], y_timed[i]):
            mismatched.append(i)
    timed_check = {"clips_resampled_alone": picks, "bit_equal": not mismatched, "mismatched": mismatched,
                   "batch_clips": n0, "tokens": n0 * F * J}
    assert not mismatched, f"timed batch disagrees with single-clip runs at clips {mismatched}"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch.cat(outs))

    # ---- e2e: the public API with HOST buffers: pinned x2d/gt -> device, flip, sampler (noise drawn on the device in the
    #      reference's order), un-flip/average, MPJPE, then the ONE exchange step of the sharded path -- all-gather of the
    #      prediction shards + all-reduce of the fp64 (error sum, joint count) pair (evaluate.gather_results; what replaces
    #      DataParallel's gather, RUN:217) -- and the gathered predictions + metric back on the host
    sampler = evaluate.DeviceSampler(diff)
    pred_h = torch.empty(n_total if world > 1 else B, F, J, 3).pin_memory()

    def noise_fn(ids, flip):
        return diff.draw_noise([len(ids), F, J, 3], dev)

    def step_e2e():
        res = evaluate.evaluate_shard(sampler, x2d_h, gt_h, noise_fn, device=dev, batch_clips=batch, tta=tta, left=L, right=R,
                                      frame_mask=mask_h)
        pred, mp = evaluate.gather_results(res["pred"], res["acc"], n_total)     # .item() inside: device -> host sync
        if rank == 0 or world == 1:
            pred_h.copy_(pred, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return mp

    for _ in range(0 if args.lean else min(args.warmup, 2)):
        mp = step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        mp = step_e2e()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1000.0) / args.steps
    e2e_value = valid_frames / (e2e_ms / 1000.0)
    h2d = x2d_h.numel() * 4 + gt_h.numel() * 4 + (mask_h.numel() if mask_h is not None else 0)
    d2h = pred_h.numel() * 4 + 16
    gathered = n_total * F * J * 3 * 4 if world > 1 else 0

    # ---- roofline of the dominant kernel (tcgen05 GEMM): one extra un-graphed step with CUDA events around
    #      every launch on the launch stream
    eng.profile_begin()
    if args.lean:        # scaling exhibits of the long cfg5 sweep: one batch instead of the whole shard
        raw[0] = eng.ddim_sample(xs[0], ys[0])
    else:
        step_resident()
    prof = eng.profile_end()
    tokens = mult * ((spans[0][1] - spans[0][0]) if args.lean else B) * F * J       # tokens the profiled launches covered
    gemm_ms, gemm_n = prof["gemm"]
    total_prof_ms = sum(v[0] for v in prof.values())
    peaks = measured_peaks()
    gemm_flops = tokens * GEMM_FLOPS_PER_TOKEN_CALL * S
    achieved = gemm_flops / (gemm_ms / 1000.0) / 1e12
    passes = {"split3": 3, "f8c": 2, "fp16": 1, "f4c": 1.5}[args.gemm]
    roofline = {
        "bound": "tensor",
        "kernel": {"f4c": "gemm_tc_kernel (tcgen05.mma cta_group::2 kind::f16 + kind::mxf4.block_scale, tcgen05.cp scale factors, TMA, TMEM)",
                   "f8c": "gemm_tc_kernel (tcgen05.mma cta_group::2 kind::f16 + kind::f8f6f4, TMA, TMEM)"}.get(
                       args.gemm, "gemm_tc_kernel (tcgen05.mma cta_group::2 kind::f16, TMA, TMEM)"),
        "achieved": achieved, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops_sustained"],
        "traffic": None, "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step)",
        "executed_tflops": achieved * passes, "executed_frac": achieved * passes / peaks["tflops_sustained"],
        "mma_passes": passes, "executed_note": "fp16-equivalent tensor-pipe units per algorithmic FLOP (f4c: 1 fp16 pass + 2 "
                                                "block-scaled e2m1 passes at four times the rate = 1.5; f8c: 1 + 2 e5m2 passes "
                                                "at twice the rate = 2)", "launches": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1),
        "share_of_step": gemm_ms / total_prof_ms,
        "per_class_ms": {k: round(v[0], 3) for k, v in prof.items()},
        "algorithmic_flops_per_launch": gemm_flops / max(gemm_n, 1),
        "note": "frac = ALGORITHMIC FLOPs over the measured sustained bf16 peak; the shipped precision mode (f4c) executes 1.5 "
                "tensor-pipe units per algorithmic FLOP (ceiling 0.667) and moves 3.06 B per operand element: all four GEMMs "
                "sit on the L2->SM operand feed (~42.6 B/clk/SM: 400 KB per CTA and 256x256x512 tile against 6144 tensor "
                "cycles); the residual update of proj / fc2 is a TMA reduction so that X never enters the SM (DESIGN.md 4.1)",
    }
    step_tokens = mult * B * F * J
    total_flops = step_tokens * flops_per_token_call(F) * S
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (profiles/), if it matches the mode
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        t = json.load(open(tpath))
        if t.get("gemm") == args.gemm and t.get("tokens_per_launch") == tokens:
            roofline["traffic"] = t["dram_bytes_per_launch_avg"]
            roofline["traffic_source"] = t.get("source")
            roofline["algorithmic_hbm_bytes_per_launch"] = t.get("algorithmic_bytes_per_launch_avg")
    # memory-bound kernel classes against the measured HBM copy bandwidth (SURVEY.md 8d byte counts + operand writes)
    depth2 = 16
    opb = {"f4c": 1568}.get(args.gemm, 2048)                               # bytes of one 512-wide A operand row (hi + second part)
    ln_bytes = tokens * S * (depth2 * (2048 + opb) + (depth2 - 1) * (4096 + opb))   # norm2: r X, w A; post-norm+norm1: r X, w X, w A
    attn_bytes = tokens * S * depth2 * (4096 + opb)                        # r q|k|v_hi|v_lo, w A operand
    hbm = {}
    for name, ms, nbytes in (("ln", prof["ln"][0], ln_bytes),
                             ("attention", prof["attn_spatial"][0] + prof["attn_temporal"][0], attn_bytes),
                             ("lift", prof["lift"][0], tokens * S * (20 + 2048 + opb)),
                             ("head_ddim", prof["head_ddim"][0], tokens * S * (2048 + 24))):
        gbs = nbytes / (ms / 1000.0) / 1e9
        hbm[name] = {"achieved_gbs": round(gbs, 1), "frac_of_measured_hbm": round(gbs / peaks["hbm_gbs"], 3)}
    roofline["hbm_bound_kernels"] = hbm
    roofline["hbm_peak_gbs"] = peaks["hbm_gbs"]

    cpu_baseline = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        keep = {}
        fps, dt, threads = cpu_sample(wl, 1, keep=keep)
        cpu_baseline = {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": sample_desc(wl) + f", {dt:.1f} s",
                        "note": "kind 'port' = the oracle restatement, not the imported reference (which cannot travel to "
                                "the GPU box); tools/make_golden.py asserts the two bit-identical in the build container"}
        try:
            parity = parity_on_sample(wl, keep, gemm_mode)
        except Exception as e:      # the throughput line must survive a failure of the checker
            parity = {"error": f"{type(e).__name__}: {e}"}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if stdout_fd is not None:
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        os.close(stdout_fd)
    if rank != 0:
        return
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
        "dtype": {"split3": "fp16x3-split operands, fp32 accumulate",
                  "f8c": "fp16 main + e5m2 correction products (2 tensor-pipe units), fp32 accumulate",
                  "f4c": "fp16 main + block-scaled e2m1 (mxfp4) correction products (1.5 tensor-pipe units), fp32 accumulate",
                  "fp16": "fp16 operands, fp32 accumulate"}[args.gemm],
        "data": "synthetic",
        "config": {"workload": wl["name"], "clips_per_gpu": B, "frames": F, "sampling_timesteps": S,
                   "tokens_per_step": step_tokens, "batches_per_step": len(spans), "clips_total": n_total,
                   "frames_counted": valid_frames,
                   "parallelism": f"clip-sharded x{world}, no data-path collective inside the sampler; one all-gather of "
                                  f"predictions + one fp64 all-reduce per sweep (timed in e2e)",
                   "l2": "activation workspace (16 KB/token) >> 126 MB L2: every kernel streams from HBM",
                   "cuda_graph": True, "gemm_mode": args.gemm},
        "algorithmic_tflops": total_flops / (ms_step / 1000.0) / 1e12 * 1.0,
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "gathered_bytes_per_step": gathered, "mpjpe_vs_synthetic_gt": mp,
                "api": "evaluate.evaluate_shard -> GaussianDiffusion.ddim_sample_loop -> d3d_ddim_sample (C ABI) -> "
                       "evaluate.gather_results (all_gather_into_tensor + all_reduce over NCCL when n_gpus > 1)"},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "parity": parity,
        "timed_output_check": timed_check,
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(WORKLOADS),
                    help="BASELINE.json configuration (default cfg3, the one the metric is quoted on)")
    ap.add_argument("--clips", type=int, default=0, help="override: clips per GPU (cfg5: total windows)")
    ap.add_argument("--sampling-timesteps", type=int, default=0, help="override: DDIM steps (cfg4 sweep 1/9/25/50)")
    ap.add_argument("--batch", type=int, default=256, help="cfg5: clips per sampler batch (x2 with the flip copies)")
    ap.add_argument("--gemm", default="f4c", choices=["split3", "f8c", "fp16", "f4c"],
                    help="GEMM arithmetic: f4c (default; fp16 main + block-scaled e2m1 correction products, 1.5 tensor-pipe "
                         "units), f8c (fp16 main + e5m2 correction products, 2 units), split3 (3 fp16 passes), fp16 (1 pass, "
                         "outside the parity bar)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the predictions of the last timed step (rank 0's clips; flip-TTA merged) to DIR/pred.npy")
    ap.add_argument("--lean", action="store_true",
                    help="scaling exhibits (tools/gpu_scaling.sh): no e2e warm-up pass, per-class profile on the first batch only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the CUDA path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
