"""ORACLE-GENERATED fixtures of the 256-wide denoiser (embed_dim 256, 8 heads of 32, depth 8): tests/golden/w256_*.npz.

The reference tree is not importable here, so unlike tools/make_golden.py these vectors come from the in-repo oracle
(oracle/diff3d_oracle.py), which has no width constant (attention_core derives hd = C // heads) and is bit-identical to
the reference at embed_dim 512.  Synthetic recipe of diff3dhpe_b200.synthetic: weights under torch.manual_seed(0),
pos-embeds N(0, 0.02^2), 2D keypoints 0.3 N(0, 1), explicit DDIM noise.  tests/test_width256_golden.py regenerates every
case on the CPU and requires the committed arrays bit for bit.

    python tools/make_golden_width256.py
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as Fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from diff3dhpe_b200 import synthetic  # noqa: E402
from oracle import diff3d_oracle as oracle  # noqa: E402

C = 256
OUT = os.path.join(ROOT, "tests", "golden")

# name -> (F, B, S, eta, clip, with_time_emb, trace)
SAMPLER_CASES = {
    "w256_sampler_f27_b2_s9_notime": (27, 2, 9, 0.0, True, False, False),
    "w256_sampler_f81_b1_s9_clip": (81, 1, 9, 0.0, True, True, False),
    "w256_sampler_f243_b1_s9_clip": (243, 1, 9, 0.0, True, True, False),
    "w256_sampler_f27_b2_s3_eta_trace": (27, 2, 3, 0.5, True, True, True),
}
DENOISE_T = [3, 421, 998]     # per-sample timesteps of w256_denoise_f27_b3 (and the rows of its time table)


def state_dict(F, with_time_emb=True):
    m = synthetic.make_model(F, with_time_emb=with_time_emb, embed_dim=C)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def sampler_case(F, B, S, eta, clip, with_time_emb, trace):
    sd = state_dict(F, with_time_emb)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, steps = synthetic.make_noise(B, F, S)
    with torch.no_grad():
        o = oracle.ddim_sample_loop(sd, x2d, y_T, steps, timesteps=1000, sampling_timesteps=S, eta=eta,
                                    clip_denoised=clip, trace=trace)
    out = dict(F=F, B=B, S=S, eta=eta, clip=int(clip), with_time_emb=int(with_time_emb), oracle_generated=1)
    if trace:
        y, rev, x0s = o
        out.update(pred=y.numpy(), rev=rev.numpy(), x0s=x0s.numpy())
    else:
        out.update(pred=o.numpy())
    return out


def denoise_case():
    F, B = 27, 3
    sd = state_dict(F)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, 1)
    t = torch.tensor(DENOISE_T, dtype=torch.long)
    with torch.no_grad():
        out = oracle.forward_denoise(sd, torch.cat([x2d, y_T], -1), t)
        t_emb = oracle.time_mlp(sd, t, C)
        table = torch.stack([Fn.linear(Fn.silu(t_emb), sd[f"{kind}.{i}.time_mlp.1.weight"], sd[f"{kind}.{i}.time_mlp.1.bias"])
                             for i in range(8) for kind in ("STEblocks", "TTEblocks")], dim=1)
    return dict(F=F, B=B, t=t.numpy(), out=out.numpy(), time_table=table.numpy(), oracle_generated=1)


def all_cases():
    """name -> dict of arrays, computed on the CPU in a fixed order with a fixed thread count."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        cases = {name: sampler_case(*args) for name, args in SAMPLER_CASES.items()}
        cases["w256_denoise_f27_b3"] = denoise_case()
    finally:
        torch.set_num_threads(threads)
    return cases


if __name__ == "__main__":
    for name, arrays in all_cases().items():
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrays)
        print(name, {k: np.asarray(v).shape for k, v in arrays.items()})
