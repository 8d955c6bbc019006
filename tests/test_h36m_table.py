"""Human3.6M per-action table: evaluate.loader_batch_runs (the reference's per-action loader batches as runs of packed
frames), evaluate.h36m_metrics and evaluate.gather_packed.  The CPU tests check the run planning against a brute-force
restatement built from the generator's windows and masks, the table arithmetic and the gather over gloo; the GPU tests
(-m gpu) check the table against the oracle's restatement of the reference's per-action loop."""
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from diff3dhpe_b200 import evaluate, synthetic
from oracle import diff3d_oracle as oracle
from oracle import h36m_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
J = 17
KEYS = ("mpjpe", "p_mpjpe", "n_mpjpe", "velocity")


def _brute_force_batches(seq_lengths, seq_group, F, batch_size):
    """[(group, packed frame indices of the batch's masked frames, window-major)] of the reference's loaders: one per
    group in order of appearance, over the group's sequences, windows and masks from the generator's own rule."""
    offsets = np.concatenate([[0], np.cumsum(seq_lengths)]).astype(np.int64)
    order = list(dict.fromkeys(seq_group))
    out = []
    for grp in order:
        windows = []
        for s, n in enumerate(seq_lengths):
            if seq_group[s] != grp:
                continue
            seq_idx = torch.arange(offsets[s], offsets[s + 1]).view(-1, 1, 1)
            for start, start_target in zip(*oracle.chunk_windows(n, F)):
                w, mask = oracle.window_batch(seq_idx, start, F, start_target, flip=False)
                windows.append(w[:, 0, 0][mask])
        for b in range(0, len(windows), batch_size):
            out.append((grp, torch.cat(windows[b:b + batch_size])))
    return out


RUN_CASES = {
    # lengths equal to F, multiples of F and not; a batch of 2 straddles sequences; group 0 has 3 windows (odd)
    "mixed_bs2": (9, [9, 18, 20, 9, 30, 11, 45], [0, 0, 1, 1, 1, 2, 2], 2),
    "mixed_bs1": (9, [9, 18, 20, 9, 30, 11, 45], [0, 0, 1, 1, 1, 2, 2], 1),
    "mixed_bs3": (9, [9, 18, 20, 9, 30, 11, 45], [0, 0, 1, 1, 1, 2, 2], 3),
    "one_batch_per_group": (9, [9, 18, 20, 9, 30, 11, 45], [0, 0, 1, 1, 1, 2, 2], 100),
    "arbitrary_ids": (5, [7, 5, 13, 10, 6], [4, 4, 1, 9, 9], 2),
    "one_sequence": (27, [100], [0], 2),
    "one_group": (9, [10, 19, 27, 9], [3, 3, 3, 3], 4),
    "h36m_shaped": (27, None, None, 3),
}


def _h36m_shaped(F=27, n_actions=15, seed=4):
    """15 actions of 2-3 sequences, lengths F..5F (mostly not multiples of F: back-shifted last windows)."""
    rng = np.random.default_rng(seed)
    per = rng.integers(2, 4, n_actions)
    lengths = [int(v) for v in rng.integers(F, 5 * F, int(per.sum()))]
    lengths = [n + 1 if n % F == 1 else n for n in lengths]      # no single-frame last window (see h36m_metrics)
    return lengths, np.repeat(np.arange(n_actions), per).tolist()


def _poses(N, seed):
    """As tests/golden/metrics.npz: root-relative gt ~ 0.3 N(0, 1), pred = gt + 0.05 N(0, 1), some frames mirrored
    (det(R) < 0 before the reflection fix of p_mpjpe)."""
    rng = np.random.RandomState(seed)
    gt = (0.3 * rng.randn(N, J, 3)).astype(np.float32)
    gt -= gt[:, :1]
    pred = (gt + 0.05 * rng.randn(N, J, 3)).astype(np.float32)
    pred[::37, :, 0] *= -1
    return pred, gt


@pytest.mark.parametrize("case", list(RUN_CASES))
def test_loader_batch_runs_match_brute_force(case):
    F, lengths, groups, bs = RUN_CASES[case]
    if lengths is None:
        lengths, groups = _h36m_shaped(F)
    run_start, run_group = evaluate.loader_batch_runs(lengths, groups, F, bs)
    N = sum(lengths)
    assert run_start.dtype == torch.int64 and run_group.dtype == torch.int32
    assert run_start[0] == 0 and run_start[-1] == N and bool((run_start[1:] > run_start[:-1]).all())   # tiles [0, N)
    ref = _brute_force_batches(lengths, groups, F, bs)
    assert len(ref) == run_group.numel()
    for r, (grp, frames) in enumerate(ref):
        assert run_group[r].item() == grp
        assert torch.equal(frames, torch.arange(run_start[r], run_start[r + 1])), (case, r)


def test_loader_batch_runs_batches_straddle_and_restart():
    """mixed_bs2 worked by hand, as (first frame, masked frames) per window.  Group 0: (0, 9) | (9, 9) (18, 9): a batch
    of 2 then 1 window.  Group 1 restarts at frame 27: (27, 9) (36, 9) | (45, 2: back-shifted) (47, 9: next sequence)
    | (56, 9) (65, 9) | (74, 9) (83, 3).  Group 2: (86, 9) (95, 2) | (97, 9) (106, 9) | (115, 9) (124, 9) | (133, 9)."""
    run_start, run_group = evaluate.loader_batch_runs([9, 18, 20, 9, 30, 11, 45], [0, 0, 1, 1, 1, 2, 2], 9, 2)
    assert run_start.tolist() == [0, 18, 27, 45, 56, 74, 86, 97, 115, 133, 142]
    assert run_group.tolist() == [0, 0, 1, 1, 1, 1, 2, 2, 2, 2]


def test_loader_batch_runs_rejects_bad_input():
    with pytest.raises(ValueError, match="consecutive"):
        evaluate.loader_batch_runs([9, 9, 9], [0, 1, 0], 9, 2)
    with pytest.raises(ValueError, match="consecutive"):
        evaluate.loader_batch_runs([9, 9, 9, 9], [2, 2, 5, 2], 9, 1)
    with pytest.raises(ValueError):
        evaluate.loader_batch_runs([9, 9], [0], 9, 2)
    with pytest.raises(ValueError):
        evaluate.loader_batch_runs([9, 9], [0, 0], 9, 0)
    with pytest.raises(ValueError):
        evaluate.loader_batch_runs([5], [0], 9, 1)                 # shorter than one window
    run_start, run_group = evaluate.loader_batch_runs([], [], 9, 2)
    assert run_start.tolist() == [0] and run_group.numel() == 0


class _FakeEngine:
    """Stands in for Engine in h36m_metrics.  Every call adds, per frame, x of joint 0 to the three error sums (times 1,
    2, 3 for MPJPE, N-MPJPE, P-MPJPE: every joint is given that error), J joints, and a velocity term of n * n (the
    call's 'mean velocity error' is its frame count n), n frames."""
    J = J
    device = torch.device("cpu")

    def __init__(self):
        self.calls = []

    def pose_metrics_accumulate(self, pred, gt, acc, frame_index=None):
        n = pred.shape[0]
        e = pred[:, 0, 0].double().sum().item() * J
        acc += torch.tensor([e, 2 * e, 3 * e, n * J, n * n, n], dtype=torch.float64)
        self.calls.append(n)
        return acc


def test_h36m_metrics_table_arithmetic():
    """F = 4, sequences [4, 8 | 6] of actions [0, 0 | 1], batches of 2 windows: action 0 = batches of 8 and 4 frames,
    action 1 = one batch of 4 + 2 masked frames.  A third action has no sequences.  Frame errors: 62.5 mm in action 0,
    500 mm in action 1 (poses in metres, exact in fp32)."""
    F, lengths, actions = 4, [4, 8, 6], [0, 0, 1]
    pred = torch.zeros(18, J, 3)
    pred[:12, :, 0] = 0.0625
    pred[12:, :, 0] = 0.5
    eng = _FakeEngine()
    out = evaluate.h36m_metrics(eng, pred, torch.zeros_like(pred), lengths, actions, F=F, batch_size=2,
                                mm_per_unit=1000.0, action_names=["Walk", "Sit", "Eat"])
    assert eng.calls == [8, 4, 6]
    assert list(out["actions"]) == ["Walk", "Sit", "Eat"]
    walk, sit, eat = (out["actions"][k] for k in ("Walk", "Sit", "Eat"))
    assert list(walk) == ["mpjpe", "p_mpjpe", "n_mpjpe", "velocity", "frames"]
    assert walk["frames"] == 12 and sit["frames"] == 6 and eat["frames"] == 0
    assert walk["mpjpe"] == pytest.approx(62.5, rel=1e-12) and walk["p_mpjpe"] == pytest.approx(187.5, rel=1e-12)
    assert walk["n_mpjpe"] == pytest.approx(125.0, rel=1e-12)
    assert sit["mpjpe"] == pytest.approx(500.0, rel=1e-12) and sit["p_mpjpe"] == pytest.approx(1500.0, rel=1e-12)
    assert walk["velocity"] == pytest.approx((8 * 8 + 4 * 4) / 12 * 1000.0, rel=1e-12)   # N_b-weighted per batch
    assert sit["velocity"] == pytest.approx(6 * 1000.0, rel=1e-12)
    assert all(math.isnan(eat[k]) for k in KEYS)
    mean, pooled = out["action_mean"], out["pooled"]
    assert mean["frames"] == 18 and pooled["frames"] == 18
    assert mean["mpjpe"] == pytest.approx((62.5 + 500.0) / 2, rel=1e-12)                    # the empty action is left out
    assert pooled["mpjpe"] == pytest.approx((12 * 62.5 + 6 * 500.0) / 18, rel=1e-12)
    assert mean["velocity"] == pytest.approx(((80 / 12) + 6) / 2 * 1000.0, rel=1e-12)
    assert pooled["velocity"] == pytest.approx((64 + 16 + 36) / 18 * 1000.0, rel=1e-12)
    assert mean["mpjpe"] != pytest.approx(pooled["mpjpe"], rel=1e-3)
    # default names: 0..max id
    out = evaluate.h36m_metrics(_FakeEngine(), pred, pred, lengths, actions, F=F, batch_size=2, mm_per_unit=1.0)
    assert list(out["actions"]) == [0, 1]
    # every action empty: NaN rows, no division error
    out = evaluate.h36m_metrics(_FakeEngine(), pred[:0], pred[:0], [], [], F=F, batch_size=2, mm_per_unit=1.0,
                                action_names=["a"])
    assert out["actions"]["a"]["frames"] == 0 and math.isnan(out["action_mean"]["mpjpe"])
    assert math.isnan(out["pooled"]["velocity"])


class _OracleEngine:
    """Stands in for Engine with d3d_pose_metrics_accumulate's sums computed by the oracle's metric functions on the
    slice it is given: acc += (n J mpjpe, n J n_mpjpe, n J p_mpjpe, n J, n velocity, n)."""
    J = J
    device = torch.device("cpu")

    def pose_metrics_accumulate(self, pred, gt, acc, frame_index=None):
        n = pred.shape[0]
        p, g = pred.unsqueeze(1), gt.unsqueeze(1)
        e = (oracle.mpjpe(p, g).item(), oracle.n_mpjpe(p, g).item(), oracle.p_mpjpe(pred.numpy(), gt.numpy()))
        v = oracle.mean_velocity_error(pred.numpy(), gt.numpy())
        acc += torch.tensor([n * J * e[0], n * J * e[1], n * J * e[2], n * J, n * v, n], dtype=torch.float64)
        return acc


def test_h36m_metrics_runs_equal_the_oracle_loop_on_cpu():
    """The runs of packed frames carry exactly the reference's batches: h36m_metrics over slices of the packed arrays
    equals the oracle's window-by-window loop when both use the same metric functions."""
    F, bs = 27, 3
    lengths, actions = _h36m_shaped(F)
    pred, gt = _poses(sum(lengths), 8)
    out = evaluate.h36m_metrics(_OracleEngine(), torch.from_numpy(pred), torch.from_numpy(gt), lengths, actions, F=F,
                                batch_size=bs, mm_per_unit=1.0)
    ref = h36m_oracle.action_table(pred, gt, lengths, actions, 15, F, bs)
    for a, r in enumerate(ref["actions"]):
        assert out["actions"][a]["frames"] == r["frames"]
        for k in KEYS:
            assert out["actions"][a][k] == pytest.approx(r[k], rel=1e-12, abs=0), (a, k)
    for k in KEYS:
        assert out["action_mean"][k] == pytest.approx(ref["action_mean"][k], rel=1e-12, abs=0)


def test_h36m_metrics_rejects_bad_input():
    pred = torch.zeros(18, J, 3)
    kw = dict(F=4, batch_size=2, mm_per_unit=1.0)
    with pytest.raises(ValueError):
        evaluate.h36m_metrics(_FakeEngine(), pred, pred, [4, 8, 6], [0, 0, 2], action_names=["a", "b"], **kw)
    with pytest.raises(ValueError):
        evaluate.h36m_metrics(_FakeEngine(), pred, pred, [4, 8, 6], [0, -1, 1], **kw)
    with pytest.raises(ValueError):
        evaluate.h36m_metrics(_FakeEngine(), pred[:17], pred[:17], [4, 8, 6], [0, 0, 1], **kw)
    with pytest.raises(ValueError):
        evaluate.h36m_metrics(_FakeEngine(), pred, pred, [4, 8, 6], [0, 1, 0], **kw)
    with pytest.raises(ValueError):
        evaluate.h36m_metrics(_FakeEngine(), pred, pred, [4, 8, 6], [0, 0, 1], F=4, batch_size=2, mm_per_unit=0.0)


def test_gather_packed_without_a_process_group_is_the_identity():
    x = torch.randn(5, J, 3)
    assert evaluate.gather_packed(x) is x


_GATHER_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from diff3dhpe_b200 import evaluate
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["MASTER_PORT"], rank=rank, world_size=world)
# frames per rank: unequal, a rank with none (first and last), none at all
for counts in ([5, 3], [2, 9], [0, 7], [4, 0], [0, 0]):
    full = torch.arange(sum(counts) * 17 * 3, dtype=torch.float32).view(-1, 17, 3) * 0.5 - 7.0
    start = sum(counts[:rank])
    got = evaluate.gather_packed(full[start:start + counts[rank]].clone())
    assert got.shape == full.shape and got.dtype == full.dtype, (counts, got.shape)
    assert torch.equal(got, full), counts
dist.barrier(); dist.destroy_process_group()
print("OK", rank)
'''


def test_gather_packed_gloo_world2(tmp_path):
    script = tmp_path / "gather_worker.py"
    script.write_text(_GATHER_WORKER)
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


# ---------------------------------------------------------------------------------------------------------------- GPU
def _assert_rows_match_oracle(out, ref, names):
    """The bounds of test_pose_metrics_golden (d3d_pose_metrics_accumulate against the reference's common/loss.py):
    2e-7 for the three errors, 1e-6 for the velocity error accumulated over several calls."""
    def check(row, r):
        assert row["frames"] == r["frames"]
        for k in ("mpjpe", "p_mpjpe", "n_mpjpe"):
            assert abs(row[k] - r[k]) < 2e-7, (k, row[k], r[k])
        assert abs(row["velocity"] - r["velocity"]) < 1e-6, (row["velocity"], r["velocity"])

    for name, r in zip(names, ref["actions"]):
        check(out["actions"][name], r)
    check(out["action_mean"], ref["action_mean"])
    # pooled = the frame-weighted mean of the per-action rows (every sum carries the N_b weighting)
    n = sum(r["frames"] for r in ref["actions"])
    pooled = {k: sum(r[k] * r["frames"] for r in ref["actions"] if r["frames"]) / n for k in KEYS}
    check(out["pooled"], dict(pooled, frames=n))


@pytest.mark.gpu
def test_h36m_table_matches_oracle_loop():
    """15 actions of 2-3 sequences at F = 27, batches of 3 windows (several per action, some straddling sequences);
    seeded poses; every per-action value and the action mean against the oracle's per-action loop; one
    d3d_pose_metrics_accumulate call per run."""
    from diff3dhpe_b200.engine import Engine
    F, bs = 27, 3
    lengths, actions = _h36m_shaped(F)
    pred, gt = _poses(sum(lengths), 8)
    names = [f"action{a:02d}" for a in range(15)]
    eng = Engine(F, max_clips=1)
    run_start, _ = evaluate.loader_batch_runs(lengths, actions, F, bs)
    n0 = eng.launch_count()
    out = evaluate.h36m_metrics(eng, torch.from_numpy(pred).cuda(), torch.from_numpy(gt), lengths, actions, F=F,
                                batch_size=bs, mm_per_unit=1.0, action_names=names)
    assert eng.launch_count() - n0 == run_start.numel() - 1
    ref = h36m_oracle.action_table(pred, gt, lengths, actions, 15, F, bs)
    _assert_rows_match_oracle(out, ref, names)
    assert out["action_mean"]["mpjpe"] != out["pooled"]["mpjpe"]
    # metres -> mm: the same table times 1000
    mm = evaluate.h36m_metrics(eng, torch.from_numpy(pred).cuda(), torch.from_numpy(gt), lengths, actions, F=F,
                               batch_size=bs, mm_per_unit=1000.0, action_names=names)
    eng.close()
    for k in KEYS:
        assert mm["action_mean"][k] == pytest.approx(1000.0 * out["action_mean"][k], rel=1e-12)


@pytest.mark.gpu
def test_h36m_table_end_to_end_and_sharding():
    """evaluate_sequences -> h36m_metrics with the F = 27 model: the whole table against the oracle loop on the same
    predictions.  Two evaluate_sequences shards (the second with its window_offset) give bit-identical packed
    predictions, and the same table to 1e-12 relative (the kernel's fp64 atomics add in no fixed order)."""
    F, bs, S = 27, 3, 7
    lengths = [61, 27, 100, 45, 80, 54, 33, 120, 29, 70]
    actions = [0, 0, 1, 1, 2, 2, 2, 3, 4, 4]
    names = ["Directions", "Eating", "Phoning", "Sitting", "Walking"]
    torch.manual_seed(0)
    model = synthetic.make_model(F).cuda()
    diff = synthetic.make_diffusion(model, sampling_timesteps=S).cuda().eval()
    sampler = evaluate.DeviceSampler(diff)
    g = torch.Generator().manual_seed(31)
    N = sum(lengths)
    seq2d = (0.3 * torch.randn(N, J, 2, generator=g)).clamp_(-1, 1)
    n_win = evaluate.plan_windows(lengths, F)[0].numel()
    noise = torch.randn(2, n_win, F, J, 3, generator=g).cuda()      # keyed by the global window id

    def noise_fn(ids, flip):
        return noise[int(flip)][ids.cuda()].contiguous(), None

    one = evaluate.evaluate_sequences(sampler, seq2d, None, lengths, noise_fn, device="cuda", F=F, batch_clips=4)
    parts, off = [], 0
    for r in range(2):
        s, c = evaluate.shard_range(len(lengths), r, 2)
        frames = slice(sum(lengths[:s]), sum(lengths[:s + c]))
        res = evaluate.evaluate_sequences(sampler, seq2d[frames], None, lengths[s:s + c], noise_fn, device="cuda", F=F,
                                          batch_clips=4, window_offset=off)
        off += res["n_windows"]
        parts.append(res["pred"])
    sharded = torch.cat(parts)
    assert off == n_win and torch.equal(sharded, one["pred"])

    # ground truth near the predictions, at the scale of tests/golden/metrics.npz, where the bounds of
    # test_pose_metrics_golden hold for the fp32 numpy metrics of the reference
    gt = one["pred"].cpu() + 0.05 * torch.randn(N, J, 3, generator=g)
    eng = model.engine(1)
    kw = dict(F=F, batch_size=bs, mm_per_unit=1.0, action_names=names)
    out = evaluate.h36m_metrics(eng, one["pred"], gt, lengths, actions, **kw)
    ref = h36m_oracle.action_table(one["pred"].cpu().numpy(), gt.numpy(), lengths, actions, len(names), F, bs)
    _assert_rows_match_oracle(out, ref, names)
    again = evaluate.h36m_metrics(eng, sharded, gt, lengths, actions, **kw)
    for a, b in [(out["actions"][n], again["actions"][n]) for n in names] + [(out["action_mean"], again["action_mean"]),
                                                                             (out["pooled"], again["pooled"])]:
        assert a["frames"] == b["frames"]
        for k in KEYS:
            assert b[k] == pytest.approx(a[k], rel=1e-12, abs=0)
    assert 0.0 < out["pooled"]["mpjpe"] < 10.0 and out["pooled"]["frames"] == N
