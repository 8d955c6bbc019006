"""The drop-in modules under nn.DataParallel (RUN:216-218, RUN3:182-184): one persistent engine per device, shared by
the master module and every per-call replica, and a C library whose distinct handles may be driven from several threads.

CPU part: torch's `replicate` is emulated step by step (`_replicate_for_data_parallel` on every sub-module, then the
parameter copies set as plain attributes), with a fake `Engine` that records what it is asked to do.
GPU part, one device: two threads with their own handles on cuda:0.  GPU part, >= 2 devices: nn.DataParallel itself,
bit for bit against single-device calls fed each device's own noise draws."""
import copy
import pickle
import threading
from collections import OrderedDict

import pytest
import torch
from torch import nn

from diff3dhpe_b200 import _lib, synthetic
from diff3dhpe_b200 import model as model_mod
from diff3dhpe_b200.diffusion import GaussianDiffusion
from diff3dhpe_b200.engine import Engine
from oracle import diff3d_oracle as oracle

MAXABS_BAR, MPJPE_BAR, MARGIN_F4C = 1e-2, 1e-4, 3.0      # as in test_gpu_sampler.py


# ============================================================================================== CPU: registry
class FakeEngine:
    """Stands in for `Engine`: records creation, weight uploads and schedules; the sampler returns its y_T."""
    log = []

    def __init__(self, num_frame, num_joints, embed_dim, depth, num_heads, mlp_hidden, with_time_emb, max_clips, device,
                 gemm_mode, attn_mode, use_graph):
        self.max_clips, self.rec_device, self.device, self.h = max_clips, device, torch.device("cpu"), object()
        self.F, self.J, self.S = num_frame, num_joints, 0
        self.weights = None
        self.busy = False
        FakeEngine.log.append(("create", device, max_clips))

    def close(self):
        FakeEngine.log.append(("close", self.rec_device))
        self.h = None

    def load_state_dict(self, sd):
        self.weights = {k: v.detach().clone() for k, v in sd.items()}
        FakeEngine.log.append(("load", self.rec_device, len(sd)))

    def set_schedule(self, times, ac, s1m, eta, clip):
        self.S = len(times) - 1
        FakeEngine.log.append(("schedule", self.rec_device, self.S))

    def _enter(self):
        assert not self.busy, "a handle was used by two threads at once"
        self.busy = True

    def forward_denoise(self, x5, t):
        self._enter()
        threading.Event().wait(0.002)
        self.busy = False
        return torch.zeros(x5.shape[:3] + (3,))

    def ddim_sample(self, x2d, y_T, step_noise, trace=False):
        self._enter()
        threading.Event().wait(0.002)
        self.busy = False
        if trace:
            return y_T.clone(), y_T.unsqueeze(-1).repeat(1, 1, 1, 1, self.S), y_T.unsqueeze(-1).repeat(1, 1, 1, 1, self.S)
        return y_T.clone()


def _count(kind, device=None):
    return sum(1 for e in FakeEngine.log if e[0] == kind and (device is None or e[1] == device))


def _replicate(network, n):
    """`torch.nn.parallel.replicate` without the broadcast: every call builds new replica objects whose parameters and
    buffers are new tensors (clones stand in for the per-device copies).  Replica j runs on fake device cuda:j."""
    modules = list(network.modules())
    index = {m: i for i, m in enumerate(modules)}
    copies = [[m._replicate_for_data_parallel() for m in modules] for _ in range(n)]
    for j in range(n):
        for r in copies[j]:
            r._former_parameters = OrderedDict()
        for i, m in enumerate(modules):
            r = copies[j][i]
            for key, child in m._modules.items():
                if child is None:
                    r._modules[key] = None
                else:
                    setattr(r, key, copies[j][index[child]])
            for key, p in m._parameters.items():
                c = p.detach().clone()
                setattr(r, key, c)
                r._former_parameters[key] = c
            for key, b in m._buffers.items():
                setattr(r, key, b.clone())
        for r in copies[j]:
            r._test_device = torch.device("cuda", j)
    return [c[0] for c in copies]


@pytest.fixture
def fake(monkeypatch):
    FakeEngine.log = []
    monkeypatch.setattr(model_mod, "Engine", FakeEngine)

    def device(self):
        root = getattr(self, "_test_device", None)
        return root if root is not None else torch.device("cuda", 0)
    monkeypatch.setattr(model_mod.ConditionalDiffusionMixSTES2SGRANDLinLift, "_engine_device", device)
    return FakeEngine


def _small_diffusion(S=3):
    torch.manual_seed(0)
    m = model_mod.ConditionalDiffusionMixSTES2SGRANDLinLift(num_frame=3, num_joints=17, embed_dim=16, depth=1,
                                                              num_heads=2)
    return GaussianDiffusion(m, timesteps=100, sampling_timesteps=S, clip_denoised=True).eval()


def _dp_call(diff, n_dev, B=4, F=3, **kw):
    """One emulated DataParallel forward: scatter along the batch, one replica per chunk, concurrently."""
    gt, x2d = torch.randn(B, F, 17, 3), torch.randn(B, F, 17, 2)
    chunks = list(zip(gt.chunk(n_dev), x2d.chunk(n_dev)))
    replicas = _replicate(diff, len(chunks))
    outs, errs = [None] * len(chunks), []

    def run(j):
        try:
            outs[j] = replicas[j](chunks[j][0], chunks[j][1], **kw)
        except BaseException as e:      # noqa: BLE001 -- re-raised in the calling thread
            errs.append(e)
    threads = [threading.Thread(target=run, args=(j,)) for j in range(len(chunks))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errs:
        raise errs[0]
    return outs


def test_registry_one_engine_per_device_across_calls(fake):
    diff = _small_diffusion()
    n_params = len(diff.model.state_dict())
    for _ in range(3):
        outs = _dp_call(diff, 4, output_loss=False)
        assert all(o[0] is None and o[1].shape == (1, 3, 17, 3) for o in outs)
    for j in range(4):
        dev = torch.device("cuda", j)
        assert _count("create", dev) == 1 and _count("load", dev) == 1 and _count("schedule", dev) == 1
        rec = diff.model._shared.peek(dev)
        assert rec is not None and rec.engine is not None
        # the upload came from the master's parameters: every tensor, with the master's values
        assert [e for e in FakeEngine.log if e[0] == "load" and e[1] == dev][0][2] == n_params
        for k, v in diff.model.state_dict().items():
            assert torch.equal(rec.engine.weights[k], v)
    assert _count("close") == 0


def test_registry_reuploads_after_master_weight_changes(fake):
    diff = _small_diffusion()
    _dp_call(diff, 2, output_loss=False)
    assert _count("load") == 2
    sd = {k: v + 0.5 for k, v in diff.model.state_dict().items()}
    diff.model.load_state_dict(sd)
    _dp_call(diff, 2, output_loss=False)
    assert _count("load") == 4 and _count("create") == 2
    for j in range(2):
        w = diff.model._shared.peek(torch.device("cuda", j)).engine.weights
        assert all(torch.equal(w[k], v) for k, v in sd.items())
    _dp_call(diff, 2, output_loss=False)
    assert _count("load") == 4
    diff.model.invalidate_weights()
    _dp_call(diff, 2, output_loss=False)
    assert _count("load") == 6
    with torch.no_grad():
        diff.model.fusion_layer.weight.mul_(2.0)          # in-place update of a master parameter
    _dp_call(diff, 2, output_loss=False)
    assert _count("load") == 8 and _count("create") == 2 and _count("schedule") == 2


def test_registry_schedule_once_per_engine_and_other_forward_modes(fake):
    diff = _small_diffusion(S=3)
    _dp_call(diff, 2, output_loss=True)
    _dp_call(diff, 2, output_loss=False, repeat_n=2)        # 2x the clips: both engines grow
    assert _count("create") == 4 and _count("close") == 2 and _count("schedule") == 4
    outs = _dp_call(diff, 2, output_loss=False, output_reverse_diffusion_3d=True)
    assert len(outs[0]) == 4 and outs[0][2].shape == (2, 3, 17, 3, 3)
    assert _count("schedule") == 4 and _count("create") == 4
    loss, pred = _dp_call(diff, 2, output_loss=True)[1]
    assert loss.shape == pred.shape == (2, 3, 17, 3)
    assert _count("schedule") == 4
    diff.sampling_timesteps = 5                             # a changed schedule on the master reaches every device
    _dp_call(diff, 2, output_loss=False)
    assert _count("schedule") == 6 and _count("create") == 4


def test_single_device_path_unchanged(fake):
    diff = _small_diffusion()
    gt, x2d = torch.randn(2, 3, 17, 3), torch.randn(2, 3, 17, 2)
    for _ in range(3):
        diff(gt, x2d, output_loss=True)
    assert (_count("create"), _count("load"), _count("schedule")) == (1, 1, 1)
    assert diff.model._engine is diff.model.engine(2)
    diff.model._engine.close()                              # bench.py closes the engine through this attribute
    diff(gt, x2d, output_loss=False)
    assert _count("create") == 2 and _count("load") == 2 and _count("schedule") == 2


def test_deepcopy_and_pickle_get_an_independent_registry(fake):
    diff = _small_diffusion()
    _dp_call(diff, 2, output_loss=False)
    ema = copy.deepcopy(diff)
    assert ema.model._shared is not diff.model._shared and ema._shared is not diff._shared
    assert ema.model._shared.master(ema.model) is ema.model and ema._shared.master(ema) is ema
    assert ema.model._shared.peek(torch.device("cuda", 0)) is None
    _dp_call(ema, 2, output_loss=False)
    assert _count("create") == 4 and _count("close") == 0
    for j in range(2):
        dev = torch.device("cuda", j)
        assert ema.model._shared.peek(dev).engine is not diff.model._shared.peek(dev).engine
    _dp_call(ema, 2, output_loss=False, repeat_n=2)        # the copy's engines grow; the original's stay open
    assert _count("create") == 6 and _count("close") == 2
    assert all(diff.model._shared.peek(torch.device("cuda", j)).engine.h is not None for j in range(2))
    back = pickle.loads(pickle.dumps(diff))
    assert back.model._shared.master(back.model) is back.model and back.model._shared.peek(torch.device("cuda", 0)) is None
    assert "_shared" not in diff.model.state_dict() and len(back.model.state_dict()) == len(diff.model.state_dict())


def test_library_loads_once_from_concurrent_threads(monkeypatch):
    import ctypes
    monkeypatch.setattr(_lib, "_lib", None)
    opened = []
    real = ctypes.CDLL

    def cdll(path, *a, **kw):
        opened.append(path)
        threading.Event().wait(0.05)        # widen the window in which a second thread could load again
        return real(path, *a, **kw)
    monkeypatch.setattr(_lib.C, "CDLL", cdll)
    got = [None] * 8
    threads = [threading.Thread(target=lambda i=i: got.__setitem__(i, _lib.load())) for i in range(8)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert len(opened) == 1 and all(g is got[0] and g is not None for g in got)


# ============================================================================================== GPU helpers
def _diffusion(F, S, max_clips, with_time_emb=True, device=0, seed=0):
    m = synthetic.make_model(F, with_time_emb=with_time_emb, seed=seed).cuda(device)
    m.max_clips_hint = max_clips
    return synthetic.make_diffusion(m, sampling_timesteps=S).cuda(device).eval()


def _draws(seed, device, shape, S, loss_shape=None, num_timesteps=1000):
    """Reference DataParallel consumption on one device after torch.cuda.manual_seed_all(seed): p_losses' randint and
    randn_like of a `loss_shape` pose batch (output_loss=True), y_T, then S - 1 randn_like (DIFF:275, 293)."""
    torch.cuda.manual_seed_all(seed)
    if loss_shape is not None:
        torch.randint(0, num_timesteps, (loss_shape[0],), device=device)
        torch.randn(loss_shape, device=device)
    y_T = torch.randn(shape, device=device)
    steps = [torch.randn_like(y_T) for _ in range(S - 1)]
    return y_T, (torch.stack(steps) if steps else torch.zeros((0,) + tuple(shape), device=device))


# ============================================================================================== GPU, one device
@pytest.mark.gpu
def test_two_threads_two_handles_on_one_device_are_bit_equal_to_sequential():
    """Distinct handles on cuda:0 created, loaded and used by two threads at once give the same bits as the same calls
    made one after the other.  The threads meet at a barrier between the setup (create, weights, schedule: each ends in
    a device-wide synchronise) and the sampling, so that one thread's setup never runs during the other's graph
    capture on the same device; nn.DataParallel drives one device per thread."""
    F, S, B = 27, 3, 3
    x2d, _ = synthetic.make_inputs(2 * B, F)
    y_T, _ = synthetic.make_noise(2 * B, F, S)
    xs = [x2d[:B].cuda(), x2d[B:].cuda()]
    ns = [y_T[:B].cuda(), y_T[B:].cuda()]
    seq = []
    for i in range(2):
        d = _diffusion(F, S, B)
        seq.append(d.ddim_sample_loop(xs[i], [B, F, 17, 3], noise=(ns[i], None)))
    torch.cuda.synchronize()
    diffs = [_diffusion(F, S, B) for _ in range(2)]
    barrier = threading.Barrier(2)
    outs, errs = [None, None], []

    def run(i):
        try:
            torch.cuda.set_device(0)
            with torch.cuda.stream(torch.cuda.Stream()):
                diffs[i]._engine(B)
                torch.cuda.synchronize()
                barrier.wait()
                outs[i] = [diffs[i].ddim_sample_loop(xs[i], [B, F, 17, 3], noise=(ns[i], None)) for _ in range(3)]
                torch.cuda.synchronize()
        except BaseException as e:      # noqa: BLE001
            errs.append(e)
            barrier.abort()
    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errs, errs
    handles = [d.model._engine.h.value for d in diffs]
    assert handles[0] != handles[1]
    for i in range(2):
        for o in outs[i]:
            assert torch.equal(o, seq[i])


@pytest.mark.gpu
def test_dataparallel_over_one_device_calls_the_module_itself():
    """nn.DataParallel with one device runs the master module directly: same engine, same outputs as without it."""
    F, S, B = 27, 3, 2
    diff = _diffusion(F, S, B)
    x2d, gt = synthetic.make_inputs(B, F)
    torch.cuda.manual_seed_all(5)
    _, direct = diff(gt.cuda(), x2d.cuda(), output_loss=False)
    eng = diff.model._engine
    torch.cuda.manual_seed_all(5)
    _, wrapped = nn.DataParallel(diff, device_ids=[0])(gt.cuda(), x2d.cuda(), output_loss=False)
    assert torch.equal(direct, wrapped) and diff.model._engine is eng


# ============================================================================================== GPU, >= 2 devices
N_DEV = min(torch.cuda.device_count(), 8) if torch.cuda.is_available() else 0
multi_gpu = pytest.mark.skipif(N_DEV < 2, reason="needs at least two visible GPUs")


class Spy:
    """Counts Engine creations, weight uploads and schedule changes (made from DataParallel's worker threads)."""

    def __init__(self, monkeypatch):
        self.n = {"create": 0, "load": 0, "schedule": 0}
        lock = threading.Lock()
        for name, kind in (("__init__", "create"), ("load_state_dict", "load"), ("set_schedule", "schedule")):
            real = getattr(Engine, name)

            def wrapped(*a, _real=real, _kind=kind, **kw):
                with lock:
                    self.n[_kind] += 1
                return _real(*a, **kw)
            monkeypatch.setattr(Engine, name, wrapped)


def _expected(ref, seed, gt, x2d, S, **kw):
    """Per scatter chunk j: the single-device drop-in `ref` (cuda:0) fed the draws device j's generator yields."""
    rep = kw.get("repeat_n", 1)
    out = []
    for j, (g, x) in enumerate(zip(gt.chunk(N_DEV), x2d.chunk(N_DEV))):
        shape = (rep * x.shape[0],) + tuple(x.shape[1:3]) + (3,)
        y_T, _ = _draws(seed, j, shape, S, tuple(g.shape) if kw.get("output_loss", True) else None, ref.num_timesteps)
        ref.draw_noise = lambda target_shape, dev, y=y_T: (y.to(dev), None)
        out.append(ref(g.cuda(0), x.cuda(0), **kw))
        del ref.draw_noise
    return out


@multi_gpu
@pytest.mark.gpu
def test_dataparallel_bit_equal_rng_parity_and_nothing_rebuilt(monkeypatch):
    """(a) bit-equal to per-chunk single-device calls, (b) every device's generator advanced exactly as the
    reference's replicas advance it, (c) the second and third calls create, upload and schedule nothing, (d) weights
    loaded into the master reach every device."""
    F, S, B, seed = 27, 3, 2 * N_DEV + 1, 11
    diff, ref = _diffusion(F, S, B), _diffusion(F, S, B)
    dp = nn.DataParallel(diff, device_ids=list(range(N_DEV)))
    x2d, gt = synthetic.make_inputs(B, F)
    n_chunks = len(x2d.chunk(N_DEV))

    def call():
        torch.cuda.manual_seed_all(seed)
        loss, pred = dp(gt.cuda(), x2d.cuda(), output_loss=False)
        assert loss is None
        return pred, [torch.cuda.get_rng_state(i) for i in range(N_DEV)]

    pred, states = call()
    want = torch.cat([p for _, p in _expected(ref, seed, gt, x2d, S, output_loss=False)])
    assert torch.equal(pred, want)                                                            # (a)
    chunks = x2d.chunk(N_DEV)
    for j, st in enumerate(states):                                                           # (b)
        torch.cuda.manual_seed_all(seed)
        if j < n_chunks:
            _draws(seed, j, (chunks[j].shape[0], F, 17, 3), S)
        assert torch.equal(st, torch.cuda.get_rng_state(j))
    spy = Spy(monkeypatch)
    engines = [diff.model._shared.peek(torch.device("cuda", j)).engine for j in range(n_chunks)]
    ws = [e.workspace_bytes() for e in engines]
    for _ in range(2):                                                                        # (c)
        again, _ = call()
        assert torch.equal(again, pred)
    assert spy.n == {"create": 0, "load": 0, "schedule": 0}
    assert [diff.model._shared.peek(torch.device("cuda", j)).engine for j in range(n_chunks)] == engines
    assert [e.workspace_bytes() for e in engines] == ws
    g = torch.Generator().manual_seed(3)                                                      # (d)
    sd = {k: v + 0.02 * torch.randn(v.shape, generator=g).to(v.device) for k, v in diff.model.state_dict().items()}
    diff.model.load_state_dict(sd)
    ref.model.load_state_dict(sd)
    new, _ = call()
    assert spy.n == {"create": 0, "load": n_chunks, "schedule": 0}
    want = torch.cat([p for _, p in _expected(ref, seed, gt, x2d, S, output_loss=False)])
    assert torch.equal(new, want)
    for x_old, x_new in zip(pred.split([len(c) for c in x2d.chunk(N_DEV)]), new.split([len(c) for c in x2d.chunk(N_DEV)])):
        assert not torch.equal(x_old, x_new)


@multi_gpu
@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(output_loss=True), dict(output_loss=False, repeat_n=2),
                                dict(output_loss=False, output_reverse_diffusion_3d=True)],
                         ids=["loss", "repeat2", "reverse"])
def test_dataparallel_other_forward_modes(kw):
    """(e) output_loss=True (the 3DHP default, RUN3:517-520), repeat_n and the reverse-diffusion outputs per replica."""
    F, S, B, seed = 27, 3, N_DEV + 2, 12
    rep = kw.get("repeat_n", 1)
    diff, ref = _diffusion(F, S, rep * B), _diffusion(F, S, rep * B)
    dp = nn.DataParallel(diff, device_ids=list(range(N_DEV)))
    x2d, gt = synthetic.make_inputs(B, F)
    torch.cuda.manual_seed_all(seed)
    got = dp(gt.cuda(), x2d.cuda(), **kw)
    want = _expected(ref, seed, gt, x2d, S, **kw)
    assert len(got) == len(want[0])
    if kw.get("output_loss"):
        assert got[0].shape == (B, F, 17, 3) and torch.isfinite(got[0]).all()
    else:
        assert got[0] is None
    for i in range(1, len(got)):
        assert torch.equal(got[i], torch.cat([w[i] for w in want]))


@multi_gpu
@pytest.mark.gpu
def test_dataparallel_batch_smaller_than_device_count():
    """(f) DataParallel uses as many replicas as there are clips."""
    F, S, B, seed = 27, 3, N_DEV - 1, 13
    diff, ref = _diffusion(F, S, 1), _diffusion(F, S, 1)
    dp = nn.DataParallel(diff, device_ids=list(range(N_DEV)))
    x2d, gt = synthetic.make_inputs(B, F)
    torch.cuda.manual_seed_all(seed)
    _, pred = dp(gt.cuda(), x2d.cuda(), output_loss=False)
    want = torch.cat([p for _, p in _expected(ref, seed, gt, x2d, S, output_loss=False)])
    assert torch.equal(pred, want)
    assert diff.model._shared.peek(torch.device("cuda", N_DEV - 1)) is None


@multi_gpu
@pytest.mark.gpu
def test_dataparallel_flip_tta_against_oracle():
    """(g) evaluate()'s two forward calls + un-flip/average under DataParallel vs the oracle on the per-device noise,
    within the bounds of test_forward_api_flip_tta_against_oracle."""
    F, B, S = 27, 4, 9
    diff = _diffusion(F, S, B)
    dp = nn.DataParallel(diff, device_ids=list(range(N_DEV)))
    x2d, gt = synthetic.make_inputs(B, F)
    xf = synthetic.flip_2d(x2d)
    preds, noise = [], []
    for seed, x in ((21, x2d), (22, xf)):
        torch.cuda.manual_seed_all(seed)
        preds.append(dp(gt.cuda(), x.cuda(), output_loss=False)[1])
        per = [_draws(seed, j, (c.shape[0], F, 17, 3), S) for j, c in enumerate(x.chunk(N_DEV))]
        noise.append((torch.cat([p[0].cpu() for p in per]), torch.cat([p[1].cpu() for p in per], dim=1)))
    merged = diff.model.engine(B).tta_merge(preds[0], preds[1], synthetic.H36M_JOINTS_LEFT,
                                            synthetic.H36M_JOINTS_RIGHT, 1.0).cpu()
    sd = {k: v.detach().cpu() for k, v in diff.model.state_dict().items()}
    with torch.no_grad():
        ref = oracle.sample_tta(sd, x2d, noise[0], noise[1], sampling_timesteps=S)
    assert (merged - ref).abs().max().item() < MAXABS_BAR / MARGIN_F4C
    assert abs(oracle.mpjpe(merged, gt).item() - oracle.mpjpe(ref, gt).item()) < MPJPE_BAR / MARGIN_F4C
