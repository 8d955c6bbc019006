"""MPI-INF-3DHP PCK / AUC: d3d_pck_accumulate (grouped per-joint error histogram), Engine.pck_table and
evaluate.mpi3dhp_metrics against the numpy oracle.  The CPU tests check the oracle on planted distances and the table
arithmetic; the GPU tests (-m gpu) check the kernel's counts bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from diff3dhpe_b200 import _lib, evaluate, synthetic
from diff3dhpe_b200.engine import Engine
from oracle import mpi3dhp_oracle as ora

J = 17
THR_MM = evaluate.mpi3dhp_thresholds(1.0)
# 64 non-uniform thresholds (mm): dense near 0, coarse above, ending past the 300 mm the errors reach
THR_64 = [float(v) for v in np.unique(np.round(np.concatenate([np.geomspace(0.5, 60, 40), np.linspace(70, 320, 24)]), 3))]
assert len(THR_64) == 64
F32_150_DOWN = float(np.nextafter(np.float32(150), np.float32(0)))
F32_150_UP = float(np.nextafter(np.float32(150), np.float32(1000)))


def _planted_pose_pair():
    """One frame, 17 joints: joint errors 0, 5 (3-4-0), 150 (90-120-0), the fp32 neighbours of 150 below and above
    (as (x, 0, 0)), and 1000 mm for the other 12 joints.  Every one is exact in fp32."""
    gt = np.zeros((1, J, 3), np.float32)
    gt[0, :, :] = [10.0, -20.0, 30.0]
    pred = gt.copy()
    pred[0, 1] += [3.0, 4.0, 0.0]
    pred[0, 2] += [90.0, 120.0, 0.0]
    pred[0, 3] = [F32_150_DOWN, 0.0, 0.0]
    gt[0, 3] = 0.0
    pred[0, 4] = [F32_150_UP, 0.0, 0.0]
    gt[0, 4] = 0.0
    pred[0, 5:] += [1000.0, 0.0, 0.0]
    return pred, gt


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_planted_distances_and_strict_threshold():
    pred, gt = _planted_pose_pair()
    err = ora.joint_errors_fp32(pred, gt)
    assert err.dtype == np.float32
    assert err[0, :5].tolist() == [0.0, 5.0, 150.0, F32_150_DOWN, F32_150_UP]
    counts, err_sum, frames = ora.pck_counts(err, THR_MM)
    # d < 5k: d = 0 -> k = 1..30 (not 0: 0 < 0 is false); d = 5 -> k = 2..30; d = 150 and its upper neighbour -> none;
    # its lower neighbour -> only k = 30
    assert counts[0, :5].sum(axis=1).tolist() == [30, 29, 0, 1, 0]
    assert counts[0, 0, 0] == 0 and counts[0, 0, 1] == 1 and counts[0, 1, 1] == 0 and counts[0, 1, 2] == 1
    assert counts[0, 3, 29] == 0 and counts[0, 3, 30] == 1
    assert counts[0, 5:].sum() == 0 and frames.tolist() == [1]
    assert err_sum[0, 2] == 150.0
    # over joints 0..4: PCK@150 = 3 of 5; AUC = (30 + 29 + 0 + 1 + 0) joint-threshold hits over 31 x 5
    pck, auc, mpjpe = ora.pck_auc(err, THR_MM, range(5), 150.0)
    assert pck == 60.0 and auc == pytest.approx(100.0 * 60 / 155, rel=1e-15)
    assert mpjpe == pytest.approx((0 + 5 + 150 + F32_150_DOWN + F32_150_UP) / 5, rel=1e-15)
    row = Engine.pck_table(counts, err_sum, frames, THR_MM, range(5), 150.0)["all"]
    assert row["pck"] == 60.0 and row["auc"] == pytest.approx(100.0 * 60 / 155, rel=1e-15)
    assert row["mpjpe"] == pytest.approx(mpjpe, rel=1e-15) and row["frames"] == 1


def _synthetic_counts(G=3, n_thr=31, seed=5):
    """Consistent accumulator contents: per (group, joint) non-decreasing counts bounded by the group's frames."""
    rng = np.random.default_rng(seed)
    frames = rng.integers(5, 400, G).astype(np.int64)
    frames[1] = 7                                           # unequal groups: pooled != mean of the groups
    inc = rng.integers(0, 3, (G, J, n_thr))
    counts = np.minimum(np.cumsum(inc, axis=2), frames[:, None, None]).astype(np.int64)
    err_sum = rng.uniform(0.0, 100.0, (G, J)) * frames[:, None]
    return counts, err_sum, frames


def test_pck_table_pooled_and_per_group():
    counts, err_sum, frames = _synthetic_counts()
    joints = evaluate.MPI3DHP_PCK_JOINTS
    tab = Engine.pck_table(torch.from_numpy(counts), torch.from_numpy(err_sum), torch.from_numpy(frames), THR_MM, joints,
                           150.0)
    nj = len(joints)
    for g, row in enumerate(tab["groups"]):
        c = counts[g, list(joints)].sum(axis=0)
        assert row["frames"] == frames[g]
        assert row["pck"] == 100.0 * c[30] / (frames[g] * nj)
        assert row["auc"] == pytest.approx(np.mean(100.0 * c / (frames[g] * nj)), rel=1e-14)
        assert row["mpjpe"] == pytest.approx(err_sum[g, list(joints)].sum() / (frames[g] * nj), rel=1e-14)
    c = counts[:, list(joints)].sum(axis=(0, 1))
    n = frames.sum() * nj
    assert tab["all"]["pck"] == 100.0 * c[30] / n and tab["all"]["frames"] == frames.sum()
    assert tab["all"]["auc"] == pytest.approx(np.mean(100.0 * c / n), rel=1e-14)
    assert tab["all"]["mpjpe"] == pytest.approx(err_sum[:, list(joints)].sum() / n, rel=1e-14)
    # pooling sums counts first: not the mean of the group rows
    assert tab["all"]["pck"] != pytest.approx(np.mean([r["pck"] for r in tab["groups"]]), rel=1e-6)
    # PCK at another threshold, per joint; a threshold that is not in the list is refused
    one = Engine.pck_table(counts, err_sum, frames, THR_MM, [4], 50.0)
    assert one["all"]["pck"] == 100.0 * counts[:, 4, 10].sum() / frames.sum()
    with pytest.raises(ValueError):
        Engine.pck_table(counts, err_sum, frames, THR_MM, joints, 149.0)
    empty = Engine.pck_table(counts, err_sum, np.zeros(3, np.int64), THR_MM, joints, 150.0)["all"]
    assert np.isnan(empty["pck"]) and np.isnan(empty["auc"]) and np.isnan(empty["mpjpe"])


class _FakeEngine:
    """Stands in for Engine in mpi3dhp_metrics: 'accumulates' fixed counts, records the thresholds it was given."""
    J = 17
    device = torch.device("cpu")

    def __init__(self, counts, err_sum, frames):
        self.arrays = counts, err_sum, frames

    def pck_accumulate(self, pred, gt, counts, err_sum, frames, thresholds, frame_index=None, frame_group=None):
        self.thresholds = list(thresholds)
        self.frame_group = frame_group
        for dst, src in zip((counts, err_sum, frames), self.arrays):
            dst += torch.from_numpy(src)


def test_mpi3dhp_metrics_table():
    counts, err_sum, frames = _synthetic_counts()
    eng = _FakeEngine(counts, err_sum, frames)
    pred = torch.zeros(10, J, 3)
    out = evaluate.mpi3dhp_metrics(eng, pred, pred, mm_per_unit=1000.0, frame_group=torch.zeros(10, dtype=torch.int64),
                                   n_groups=3, group_names=["TS1", "TS2", "TS3"])
    assert eng.thresholds == evaluate.mpi3dhp_thresholds(1000.0) and eng.frame_group.dtype == torch.int32
    ref = Engine.pck_table(counts, err_sum, frames, eng.thresholds, evaluate.MPI3DHP_PCK_JOINTS, 0.15)
    every = Engine.pck_table(counts, err_sum, frames, eng.thresholds, range(J), 0.15)
    assert out["overall"]["pck"] == ref["all"]["pck"] and out["overall"]["auc"] == ref["all"]["auc"]
    assert out["overall"]["mpjpe"] == ref["all"]["mpjpe"] * 1000.0
    assert out["overall"]["mpjpe_all_joints"] == every["all"]["mpjpe"] * 1000.0
    assert list(out["groups"]) == ["TS1", "TS2", "TS3"]
    for name, r, a in zip(out["groups"], ref["groups"], every["groups"]):
        assert out["groups"][name] == dict(r, mpjpe=r["mpjpe"] * 1000.0, mpjpe_all_joints=a["mpjpe"] * 1000.0)
    assert list(out["joint_groups"]) == ["Head", "Neck", "Shoulder", "Elbow", "Wrist", "Hip", "Knee", "Ankle"]
    sh = out["joint_groups"]["Shoulder"]
    c = counts[:, [2, 5], 30].sum()
    assert sh["pck"] == 100.0 * c / (frames.sum() * 2) and sh["frames"] == frames.sum()
    assert sh["mpjpe"] == pytest.approx(err_sum[:, [2, 5]].sum() / (frames.sum() * 2) * 1000.0, rel=1e-14)
    # the joint groups partition the 14 evaluated joints
    assert sorted(j for js in evaluate.MPI3DHP_JOINT_GROUPS.values() for j in js) == list(evaluate.MPI3DHP_PCK_JOINTS)
    with pytest.raises(ValueError):
        evaluate.mpi3dhp_metrics(eng, pred, pred, mm_per_unit=1.0, n_groups=3, group_names=["a"])


def test_mpi3dhp_thresholds_units():
    mm = evaluate.mpi3dhp_thresholds(1.0)
    assert mm == [5.0 * k for k in range(31)] and mm[-1] == 150.0
    m = evaluate.mpi3dhp_thresholds(1000.0)
    assert len(m) == 31 and m[0] == 0.0 and m[-1] == 0.15 and m[1] == 0.005
    assert np.all(np.diff(np.asarray(m, np.float32)) > 0)          # still strictly ascending after rounding to fp32
    for k in range(31):
        assert m[k] == pytest.approx(mm[k] / 1000.0, rel=1e-15)
    for bad in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            evaluate.mpi3dhp_thresholds(bad)
    with pytest.raises(TypeError):
        evaluate.mpi3dhp_thresholds()                                # the unit is never assumed
    with pytest.raises(TypeError):
        evaluate.mpi3dhp_metrics(None, None, None)


# ---------------------------------------------------------------------------------------------------------------- GPU
N_FRAMES = 100_000
N_SEQ = 7


def _poses(n=N_FRAMES, seed=11):
    """gt ~ N(0, 300 mm); pred = gt + a random direction times an error uniform in [0, 300] mm; the first frames carry
    planted distances exact in fp32: 0, 5, 150 and its fp32 neighbours, and every 64-threshold value and its
    neighbours, as (x, 0, 0) against a zero ground truth."""
    rng = np.random.default_rng(seed)
    gt = (300.0 * rng.standard_normal((n, J, 3))).astype(np.float32)
    d = rng.standard_normal((n, J, 3))
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    pred = (gt + d * rng.uniform(0.0, 300.0, (n, J, 1))).astype(np.float32)
    plant = [0.0, 5.0, 150.0, F32_150_DOWN, F32_150_UP]
    for t in THR_64:
        t32 = np.float32(t)
        plant += [float(t32), float(np.nextafter(t32, np.float32(0))), float(np.nextafter(t32, np.float32(1e9)))]
    plant = np.asarray(plant, np.float32)
    rows = (plant.size + J - 1) // J
    flat = np.zeros(rows * J, np.float32)
    flat[:plant.size] = plant
    gt[:rows] = 0.0
    pred[:rows] = 0.0
    pred[:rows, :, 0] = flat.reshape(rows, J)
    return pred, gt


def _seq_groups(n=N_FRAMES, n_seq=N_SEQ):
    """Per-sequence group ids of n frames packed as n_seq sequences of unequal length."""
    cuts = np.sort(np.random.default_rng(3).choice(np.arange(1, n), n_seq - 1, replace=False))
    return np.repeat(np.arange(n_seq), np.diff(np.concatenate([[0], cuts, [n]]))).astype(np.int32)


@pytest.fixture(scope="module")
def eng():
    e = Engine(27, max_clips=1)
    yield e
    e.close()


@pytest.fixture(scope="module")
def data():
    pred, gt = _poses()
    return pred, gt, ora.joint_errors_fp32(pred, gt), torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda()


def _run(eng, pred_d, gt_d, thr, G, frame_index=None, frame_group=None, calls=1):
    counts = torch.zeros((G, J, len(thr)), dtype=torch.int64, device="cuda")
    err_sum = torch.zeros((G, J), dtype=torch.float64, device="cuda")
    frames = torch.zeros(G, dtype=torch.int64, device="cuda")
    fi = None if frame_index is None else torch.as_tensor(frame_index, dtype=torch.int64).cuda()
    fg = None if frame_group is None else torch.as_tensor(frame_group, dtype=torch.int32).cuda()
    for _ in range(calls):
        eng.pck_accumulate(pred_d, gt_d, counts, err_sum, frames, thr, fi, fg)
    return counts.cpu().numpy(), err_sum.cpu().numpy(), frames.cpu().numpy()


def _assert_matches(got, ref):
    (c, e, f), (rc, re_, rf) = got, ref
    assert np.array_equal(f, rf)
    assert np.array_equal(c, rc)
    nz = rf > 0
    np.testing.assert_allclose(e[nz], re_[nz], rtol=1e-12, atol=0)
    assert np.all(e[~nz] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("thr_name", ["protocol31", "nonuniform64"])
@pytest.mark.parametrize("G", [1, 7, 4096])
def test_counts_match_oracle(eng, data, thr_name, G):
    """Counts and frames bit-exact, err_sum to 1e-12, for both histogram paths: G = 1 and 7 fit the 32 KB of shared
    memory, G = 4096 does not and is counted with global atomics."""
    pred, gt, err, pred_d, gt_d = data
    thr = THR_MM if thr_name == "protocol31" else THR_64
    bin_bytes = G * J * len(thr) * 4
    assert (bin_bytes <= 32 * 1024) == (G < 4096)
    grp = None if G == 1 else (_seq_groups() if G == 7 else (np.arange(N_FRAMES) % G).astype(np.int32))
    got = _run(eng, pred_d, gt_d, thr, G, frame_group=grp)
    _assert_matches(got, ora.pck_counts(err, thr, frame_group=grp, n_groups=G))
    assert got[0].sum() > 0 and got[0][:, :, 0].sum() < got[0][:, :, -1].sum()


@pytest.mark.gpu
@pytest.mark.parametrize("index", ["none", "permuted", "repeats"])
@pytest.mark.parametrize("groups", ["none", "per_sequence", "out_of_range"])
def test_frame_index_and_groups(eng, data, index, groups):
    pred, gt, err, pred_d, gt_d = data
    rng = np.random.default_rng(17)
    fi = {"none": None, "permuted": rng.permutation(N_FRAMES),
          "repeats": np.concatenate([rng.integers(0, N_FRAMES, 30_000), np.arange(0, 2000), np.arange(0, 2000)])}[index]
    fg = {"none": None, "per_sequence": _seq_groups()}.get(groups)
    if groups == "out_of_range":                  # ids -1 and 7..9 are skipped with all their joints
        fg = _seq_groups()
        fg[rng.integers(0, N_FRAMES, 5000)] = -1
        fg[rng.integers(0, N_FRAMES, 5000)] = rng.integers(N_SEQ, N_SEQ + 3, 5000)
    G = 1 if fg is None else N_SEQ
    got = _run(eng, pred_d, gt_d, THR_MM, G, frame_index=fi, frame_group=fg)
    ref = ora.pck_counts(err, THR_MM, frame_index=fi, frame_group=fg, n_groups=G)
    _assert_matches(got, ref)
    n_listed = N_FRAMES if fi is None else len(fi)
    assert (got[2].sum() < n_listed) == (groups == "out_of_range")


@pytest.mark.gpu
@pytest.mark.parametrize("G", [7, 4096])
def test_two_halves_equal_one_call_and_empty_call(eng, data, G):
    pred, gt, err, pred_d, gt_d = data
    grp = (np.arange(N_FRAMES) % G).astype(np.int32)
    whole = _run(eng, pred_d, gt_d, THR_64, G, frame_group=grp)
    counts = torch.zeros((G, J, 64), dtype=torch.int64, device="cuda")
    err_sum = torch.zeros((G, J), dtype=torch.float64, device="cuda")
    frames = torch.zeros(G, dtype=torch.int64, device="cuda")
    fg = torch.from_numpy(grp).cuda()
    idx = torch.arange(N_FRAMES, device="cuda")
    for part in (idx[: N_FRAMES // 2], idx[N_FRAMES // 2:]):
        eng.pck_accumulate(pred_d, gt_d, counts, err_sum, frames, THR_64, part.contiguous(), fg)
    assert np.array_equal(counts.cpu().numpy(), whole[0]) and np.array_equal(frames.cpu().numpy(), whole[2])
    np.testing.assert_allclose(err_sum.cpu().numpy(), whole[1], rtol=1e-12, atol=0)
    before = [t.clone() for t in (counts, err_sum, frames)]
    n0 = eng.launch_count()
    eng.pck_accumulate(pred_d, gt_d, counts, err_sum, frames, THR_64, idx[:0].contiguous(), fg)
    torch.cuda.synchronize()
    assert eng.launch_count() == n0
    assert all(torch.equal(a, b) for a, b in zip(before, (counts, err_sum, frames)))


@pytest.mark.gpu
def test_nan_error_counts_nowhere(eng):
    pred, gt = _planted_pose_pair()
    pred = np.repeat(pred, 3, axis=0)
    gt = np.repeat(gt, 3, axis=0)
    pred[1, 1, 1] = np.nan                          # joint 1 (error 5 mm) of frame 1
    got = _run(eng, torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), THR_MM, 1)
    ref = ora.pck_counts(ora.joint_errors_fp32(pred, gt), THR_MM)
    assert np.array_equal(got[0], ref[0]) and got[0][0, 1].sum() == 2 * 29 and got[0][0, 0].sum() == 3 * 30
    assert np.isnan(got[1][0, 1]) and np.isfinite(np.delete(got[1][0], 1)).all()
    assert got[2].tolist() == [3]


@pytest.mark.gpu
def test_invalid_arguments_write_nothing(eng, data):
    _, _, _, pred_d, gt_d = data
    lib, h = eng.lib, eng.h
    counts = torch.full((1, J, 64), 7, dtype=torch.int64, device="cuda")
    err_sum = torch.full((1, J), 7.0, dtype=torch.float64, device="cuda")
    frames = torch.full((1,), 7, dtype=torch.int64, device="cuda")
    before = [t.clone() for t in (counts, err_sum, frames)]
    p = lambda t: C.c_void_p(t.data_ptr())                                   # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(thr, n_thr=None, n_groups=1, outs=(counts, err_sum, frames), pred=pred_d):
        arr = (C.c_float * max(len(thr), 1))(*thr)
        o = [None if t is None else p(t) for t in outs]
        return lib.d3d_pck_accumulate(h, None if pred is None else p(pred), p(gt_d), None, None, 1000, arr,
                                      len(thr) if n_thr is None else n_thr, n_groups, o[0], o[1], o[2], stream)

    good = THR_64
    cases = [(-2, dict(thr=[], n_thr=0)), (-2, dict(thr=good + [400.0], n_thr=65)),
             (-2, dict(thr=good[:10] + [float("nan")] + good[11:])), (-2, dict(thr=good[:10] + [good[8]] + good[11:])),
             (-2, dict(thr=[1.0, 2.0, 2.0])), (-2, dict(thr=[1.0, float("inf")])), (-2, dict(thr=good, n_groups=0)),
             (-2, dict(thr=good, n_groups=65537)), (-1, dict(thr=good, outs=(None, err_sum, frames))),
             (-1, dict(thr=good, outs=(counts, None, frames))), (-1, dict(thr=good, outs=(counts, err_sum, None))),
             (-1, dict(thr=good, pred=None))]
    n0 = eng.launch_count()
    for code, kw in cases:
        assert call(**kw) == code, kw
        assert _lib.last_error(h)
    assert lib.d3d_pck_accumulate(None, p(pred_d), p(gt_d), None, None, 1, (C.c_float * 1)(1.0), 1, 1, p(counts),
                                  p(err_sum), p(frames), stream) == -1
    torch.cuda.synchronize()
    assert eng.launch_count() == n0
    assert all(torch.equal(a, b) for a, b in zip(before, (counts, err_sum, frames)))
    with pytest.raises(RuntimeError, match="code -2"):
        eng.pck_accumulate(pred_d, gt_d, counts[:, :, :3].contiguous(), err_sum, frames, [1.0, 3.0, 2.0])


@pytest.mark.gpu
def test_graph_capture_replays(eng, data):
    """The call enqueues one kernel with the thresholds by value: captured once, replayed twice = twice the counts."""
    pred, gt, err, pred_d, gt_d = data
    grp = torch.from_numpy(_seq_groups()).cuda()
    counts = torch.zeros((N_SEQ, J, 31), dtype=torch.int64, device="cuda")
    err_sum = torch.zeros((N_SEQ, J), dtype=torch.float64, device="cuda")
    frames = torch.zeros(N_SEQ, dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                     # warm-up outside the capture (module loading)
        eng.pck_accumulate(pred_d, gt_d, counts, err_sum, frames, THR_MM, None, grp)
    torch.cuda.current_stream().wait_stream(s)
    for t in (counts, err_sum, frames):
        t.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        eng.pck_accumulate(pred_d, gt_d, counts, err_sum, frames, THR_MM, None, grp)
    torch.cuda.synchronize()
    assert counts.sum().item() == 0                 # capture only records
    g.replay()
    g.replay()
    torch.cuda.synchronize()
    rc, re_, rf = ora.pck_counts(err, THR_MM, frame_group=grp.cpu().numpy(), n_groups=N_SEQ)
    assert np.array_equal(counts.cpu().numpy(), 2 * rc) and np.array_equal(frames.cpu().numpy(), 2 * rf)
    np.testing.assert_allclose(err_sum.cpu().numpy(), 2 * re_, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_histogram_path_selection(eng, data):
    """Which kernel runs: the shared-memory histogram up to 32 KB of bins, global atomics above."""
    _, _, _, pred_d, gt_d = data
    from torch.profiler import ProfilerActivity, profile
    names = {}
    for G in (7, 4096):
        grp = (np.arange(N_FRAMES) % G).astype(np.int32)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _run(eng, pred_d, gt_d, THR_MM, G, frame_group=grp)
            torch.cuda.synchronize()
        names[G] = [e.name for e in prof.events() if "pck_hist_kernel" in e.name]
    assert names[7] and all("pck_hist_kernel<true>" in n for n in names[7]), names[7]
    assert names[4096] and all("pck_hist_kernel<false>" in n for n in names[4096]), names[4096]


@pytest.mark.gpu
def test_mpi3dhp_metrics_end_to_end_3dhp_shape():
    """The 3dhp_gt shape (F = 27, no time embedding, MPI-INF-3DHP flip lists): evaluate_sequences over four sequences of
    unequal length, then mpi3dhp_metrics with per-sequence groups built from plan_windows; the whole table equals the
    oracle on the same predictions, and its 17-joint MPJPE equals d3d_mpjpe_accumulate's."""
    F, lengths, mm_per_unit = 27, [61, 27, 100, 45], 300.0
    torch.manual_seed(0)
    model = synthetic.make_model(F, with_time_emb=False).cuda()
    diff = synthetic.make_diffusion(model, sampling_timesteps=7).cuda().eval()
    sampler = evaluate.DeviceSampler(diff)
    g = torch.Generator().manual_seed(21)
    N = sum(lengths)
    seq2d = (0.3 * torch.randn(N, J, 2, generator=g)).clamp_(-1, 1)
    gt = 0.3 * torch.randn(N, J, 3, generator=g)
    gt = gt - gt[:, 14:15]                                     # root-relative to the MPI pelvis

    def noise_fn(ids, flip):
        return diff.draw_noise([len(ids), F, J, 3], "cuda")

    res = evaluate.evaluate_sequences(sampler, seq2d, gt, lengths, noise_fn, device="cuda", F=F, batch_clips=4,
                                      left=synthetic.MPI3DHP_JOINTS_LEFT, right=synthetic.MPI3DHP_JOINTS_RIGHT)
    _, fv, sid = evaluate.plan_windows(lengths, F)
    groups = sid.repeat_interleave((F - fv).long())            # frames each window writes back, in packed order
    assert torch.equal(groups, torch.repeat_interleave(torch.arange(4, dtype=torch.int32), torch.tensor(lengths)))
    names = ["TS1", "TS2", "TS3", "TS4"]
    out = evaluate.mpi3dhp_metrics(model.engine(1), res["pred"], gt, mm_per_unit=mm_per_unit, frame_group=groups,
                                   n_groups=4, group_names=names)

    err = ora.joint_errors_fp32(res["pred"].cpu().numpy(), gt.numpy())
    thr = evaluate.mpi3dhp_thresholds(mm_per_unit)
    bounds = np.cumsum([0] + lengths)

    def check(row, e, joints, all_joints=True):
        pck, auc, mp = ora.pck_auc(e, thr, joints, thr[-1])
        assert row["frames"] == e.shape[0]
        assert row["pck"] == pck and row["auc"] == pytest.approx(auc, rel=1e-12, abs=0)
        assert row["mpjpe"] == pytest.approx(mp * mm_per_unit, rel=1e-12, abs=0)
        if all_joints:
            assert row["mpjpe_all_joints"] == pytest.approx(e.astype(np.float64).mean() * mm_per_unit, rel=1e-12, abs=0)

    check(out["overall"], err, evaluate.MPI3DHP_PCK_JOINTS)
    for k, name in enumerate(names):
        check(out["groups"][name], err[bounds[k]:bounds[k + 1]], evaluate.MPI3DHP_PCK_JOINTS)
    for name, joints in evaluate.MPI3DHP_JOINT_GROUPS.items():
        check(out["joint_groups"][name], err, joints, all_joints=False)
    assert 1.0 < out["overall"]["pck"] < 99.0                  # the synthetic errors straddle 150 mm
    # d3d_mpjpe_accumulate (evaluate_sequences' 'acc') over the same frames: its joint errors may differ from the fp32
    # expression above by one rounding (it lets the compiler fuse the multiply-adds), so the sums agree to ~2^-23
    acc = res["acc"].cpu()
    assert acc[1].item() == N * J
    assert out["overall"]["mpjpe_all_joints"] == pytest.approx(acc[0].item() / acc[1].item() * mm_per_unit, rel=2 ** -22)
