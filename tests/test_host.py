"""CPU: host-side mirror of the reference interface (module/diffusion drop-ins, registry, sharding plumbing)."""
import os
import subprocess
import sys

import pytest
import torch

import diff3dhpe_b200 as d3d
from diff3dhpe_b200 import evaluate, synthetic
from oracle import diff3d_oracle as oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_state_dict_contract_matches_reference():
    """Keys, order and shapes of the reference's GaussianDiffusion state dict (254 entries, SURVEY.md 8b)."""
    want = open(os.path.join(ROOT, "tests", "golden", "state_dict_keys.txt")).read().strip().split("\n")
    m = d3d.HPE_model("ConditionalDiffusionMixSTES2SGRANDLinLift")(
        num_frame=27, num_joints=17, in_chans=2, embed_dim=512, depth=8, num_heads=8, mlp_ratio=2., qkv_bias=True,
        drop_path_rate=0.1, with_time_emb=True)
    diff = synthetic.make_diffusion(m)
    got = [f"{k} {tuple(v.shape)}" for k, v in diff.state_dict().items()]
    assert len(got) == 254 and got == want


def test_checkpoint_roundtrip_with_dataparallel_prefix():
    """RUN:226-235: keys carry 'module.' under DataParallel, 'alphas' keys are dropped, strict=False."""
    m = synthetic.make_model(9)
    diff = synthetic.make_diffusion(m)
    ckpt = {"module." + k: v.clone() for k, v in diff.state_dict().items()}
    ckpt = {k: v for k, v in ckpt.items() if "alphas" not in k}
    m2 = synthetic.make_model(9, seed=5)
    diff2 = synthetic.make_diffusion(m2)
    res = diff2.load_state_dict({k[len("module."):]: v for k, v in ckpt.items()}, strict=False)
    assert not res.unexpected_keys and all("alphas" in k for k in res.missing_keys)
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_schedule_buffers_match_oracle():
    diff = synthetic.make_diffusion(synthetic.make_model(9), sampling_timesteps=9)
    b = oracle.schedule_buffers(1000)
    assert torch.equal(diff.alphas_cumprod, b["alphas_cumprod"])
    assert torch.equal(diff.sqrt_one_minus_alphas_cumprod, b["sqrt_one_minus_alphas_cumprod"])
    assert diff.ddim_times() == oracle.ddim_times(1000, 9)


def test_registry_and_loud_failures():
    with pytest.raises(KeyError):
        d3d.HPE_model("ConditionalDiffusionMixSTES2FGRANDLinLift")
    m = synthetic.make_model(9)
    x5 = torch.zeros(1, 9, 17, 5)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):      # product path never falls back to CPU
            m.forward_denoise(x5, torch.zeros(1, dtype=torch.long))
    m.train()
    with pytest.raises(NotImplementedError):
        m.forward_denoise(x5, torch.zeros(1, dtype=torch.long))
    diff = synthetic.make_diffusion(m).train()
    with pytest.raises(NotImplementedError):
        diff(x5[..., :3], x5[..., :2])


def test_product_package_does_not_import_oracle():
    import pathlib
    for f in pathlib.Path(ROOT, "diff3dhpe_b200").rglob("*.py"):
        src = f.read_text()
        assert "oracle" not in src.replace("# oracle", ""), f"{f} references the oracle"


def test_shard_range_partitions():
    for n in (0, 1, 7, 8, 2400, 2223):
        for w in (1, 2, 3, 8):
            spans = [evaluate.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == n
            assert all(spans[i][0] + spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1


def test_plan_windows_matches_generator_rule(golden):
    """evaluate.plan_windows (host side of the device windowing) against the oracle restatement of the generator rule
    for every length up to 5 windows, and against the reference generator's golden windows."""
    for F in (1, 9, 27):
        for n in range(F, 5 * F + 2):
            starts, targets = oracle.chunk_windows(n, F)
            ws, fv, sid = evaluate.plan_windows([n], F)
            assert ws.tolist() == starts and fv.tolist() == [s - t for s, t in zip(starts, targets)]
            covered = torch.zeros(n, dtype=torch.int32)             # every frame predicted exactly once
            for s, v in zip(ws.tolist(), fv.tolist()):
                covered[s + v:s + F] += 1
            assert bool((covered == 1).all())
    g = golden("windows_f9")
    ws, fv, sid = evaluate.plan_windows(g["lens"].tolist(), int(g["F"]))
    assert ws.tolist() == g["win_start"].tolist() and sid.tolist() == g["seq_id"].tolist()
    assert fv.tolist() == [int((~m).sum()) for m in g["mask"]]
    with pytest.raises(ValueError):
        evaluate.plan_windows([5], 9)


def test_window_rule():
    """ChunkedGenerator windowing (nosiy_generators.py:27-48): 2250 frames, F=243 -> 10 windows, last shifted back."""
    w = evaluate.window_starts(2250, 243)
    assert len(w) == 10 and w[0] == (0, 0) and w[8] == (1944, 0)
    assert w[9] == (2250 - 243, 9 * 243 - (2250 - 243))       # 180 frames of overlap are masked
    assert evaluate.window_starts(486, 243) == [(0, 0), (243, 0)]
    with pytest.raises(ValueError):
        evaluate.window_starts(100, 243)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the whole prediction tensor as float32 when it fits, otherwise the same seeded sample of
    clips, in clip order, on every call."""
    import numpy as np
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)     # importing bench sets it
    import bench
    pred = torch.randn(10, 3, 17, 3, generator=torch.Generator().manual_seed(0))
    bench.dump_outputs(str(tmp_path / "all"), pred)
    got = np.load(tmp_path / "all" / "pred.npy")
    assert got.dtype == np.float32 and np.array_equal(got, pred.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * pred[0].numel() * 4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), pred)
    a, b = np.load(tmp_path / "a" / "pred.npy"), np.load(tmp_path / "b" / "pred.npy")
    assert a.shape == (4, 3, 17, 3) and np.array_equal(a, b)
    rows = [next(i for i in range(10) if np.array_equal(r, pred[i].numpy())) for r in a]
    assert rows == sorted(set(rows))


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from diff3dhpe_b200 import evaluate, synthetic
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["MASTER_PORT"], rank=rank, world_size=world)

class FakeSampler:          # stands in for the CUDA sampler: any per-clip function exercises the plumbing
    def __call__(self, x2d, y_T, sn):
        return torch.cat([x2d * 2.0, x2d[..., :1] - 1.0], -1) + 0.5 * y_T
    def merge(self, y, yf, left, right, scale):
        return (y + synthetic.flip_2d(yf, left, right)) / 2.0 * scale
    def mpjpe(self, pred, gt, acc, mask):
        e = torch.norm(pred - gt, dim=-1).double()
        if mask is not None:
            e = e.reshape(-1, e.shape[-1])[mask.bool()]
        acc[0] += e.sum(); acc[1] += e.numel()
        return acc

N, F = 7, 5
x2d, gt = synthetic.make_inputs(N, F)
noise = torch.Generator().manual_seed(9)
full_noise = torch.randn(2, N, F, 17, 3, generator=noise)
def noise_fn(ids, flip):
    return full_noise[int(flip)][ids], None
s, c = evaluate.shard_range(N, rank, world)
res = evaluate.evaluate_shard(FakeSampler(), x2d[s:s + c], gt[s:s + c], noise_fn, device="cpu", batch_clips=2,
                              clip_offset=s)
pred, mp = evaluate.gather_results(res["pred"], res["acc"], N)
ref = evaluate.evaluate_shard(FakeSampler(), x2d, gt, noise_fn, device="cpu", batch_clips=3)
assert pred.shape == (N, F, 17, 3)
assert torch.equal(pred, ref["pred"]), "sharded result differs from the single-process result"
assert abs(mp - (ref["acc"][0] / ref["acc"][1]).item()) < 1e-12
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
'''


def test_sharded_evaluate_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0 and "OK" in out, out
