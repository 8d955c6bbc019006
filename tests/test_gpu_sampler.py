"""GPU (-m gpu): the hot path (forward_denoise, DDIM loop, flip-TTA) through the drop-in modules / C ABI against
the golden vectors of the imported reference and the CPU oracle run live on the same seeded inputs.

Tolerances (north star): per-joint max-abs error <= 1e-2 (pose scale 1) and MPJPE delta <= 0.1 mm = 1e-4.  The
shipped default is GEMM_TC_F4C: fp16 main product + block-scaled e2m1 (mxfp4) correction products in the linears,
single-pass fp16 attention with an exact "- V" term; it is asserted against a 3x tighter bound (measured worst case over
the goldens 2.8e-3 / 1.6e-5, profiles/r02d_parity_report.log).  GEMM_TC_F8C (e5m2 corrections; worst case 9.7e-4 / 7.7e-6)
and the 3-pass split-fp16 mode are asserted against a 4x tighter bound."""
import numpy as np
import pytest
import torch

from diff3dhpe_b200 import _lib, synthetic
from oracle import diff3d_oracle as oracle

pytestmark = pytest.mark.gpu

MAXABS_BAR, MPJPE_BAR = 1e-2, 1e-4
MARGIN = 4.0
MARGIN_F4C = 3.0     # measured worst case over the goldens: 2.8e-3 / 1.6e-5 (tools/parity_report.py, profiles/r02d_parity_report.log)


def _diffusion(F, S, eta=0.0, clip=True, with_time_emb=True, gemm_mode=_lib.GEMM_DEFAULT, attn_mode=_lib.ATTN_DEFAULT,
               use_graph=True, max_clips=1):
    m = synthetic.make_model(F, with_time_emb=with_time_emb).cuda()
    m.gemm_mode, m.attn_mode, m.use_graph, m.max_clips_hint = gemm_mode, attn_mode, use_graph, max_clips
    return synthetic.make_diffusion(m, sampling_timesteps=S, eta=eta, clip_denoised=clip).cuda().eval()


def _mpjpe_delta(a, b, gt):
    return abs(oracle.mpjpe(a, gt).item() - oracle.mpjpe(b, gt).item())


@pytest.mark.parametrize("name", ["denoise_f27_b3", "denoise_f27_b2_notime"])
@pytest.mark.parametrize("gemm_mode", [_lib.GEMM_SIMT_FP32, _lib.GEMM_TC_SPLIT3, _lib.GEMM_TC_F8C, _lib.GEMM_TC_F4C])
def test_forward_denoise_golden(golden, name, gemm_mode):
    g = golden(name)
    F, B = int(g["F"]), int(g["B"])
    diff = _diffusion(F, 1, with_time_emb="notime" not in name, gemm_mode=gemm_mode)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, 1)
    out = diff.model.forward_denoise(torch.cat([x2d, y_T], -1).cuda(), torch.tensor(g["t"]).cuda()).cpu().numpy()
    assert np.abs(out - g["out"]).max() < MAXABS_BAR / MARGIN


@pytest.mark.parametrize("name", ["sampler_f27_b2_s3_clip", "sampler_f27_b2_s3_eta", "sampler_f27_b2_s2_notime",
                                  "sampler_f81_b1_s2_noclip", "sampler_f243_b1_s1_clip", "sampler_f9_b2_s9_clip",
                                  # the BASELINE configurations' frame counts at the full 9 DDIM steps (DIFF:263-300):
                                  # cfg2 (F = 81), cfg3 / cfg5 (F = 243), cfg4 (F = 27, no time embedding)
                                  "sampler_f81_b1_s9_clip", "sampler_f243_b1_s9_clip", "sampler_f27_b2_s9_notime"])
@pytest.mark.parametrize("use_graph,gemm_mode", [(False, _lib.GEMM_TC_F8C), (True, _lib.GEMM_TC_F8C),
                                                 (True, _lib.GEMM_TC_SPLIT3), (True, _lib.GEMM_TC_F4C)])
def test_sampler_golden(golden, name, use_graph, gemm_mode):
    g = golden(name)
    F, B, S, eta = int(g["F"]), int(g["B"]), int(g["S"]), float(g["eta"])
    diff = _diffusion(F, S, eta, bool(g["clip"]), bool(g["with_time_emb"]), gemm_mode=gemm_mode, use_graph=use_graph,
                      max_clips=B)
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, steps = synthetic.make_noise(B, F, S)
    noise = (y_T.cuda(), steps.cuda() if eta != 0 else None)
    trace = "rev" in g
    if trace:
        pred, rev, x0s = diff.ddim_sample_loop_ouput_reverse_diffusion(x2d.cuda(), [B, F, 17, 3], noise=noise)
        tm = MARGIN_F4C if gemm_mode == _lib.GEMM_TC_F4C else MARGIN
        assert np.abs(rev.cpu().numpy() - g["rev"]).max() < MAXABS_BAR / tm
        assert np.abs(x0s.cpu().numpy() - g["x0s"]).max() < MAXABS_BAR / tm
    else:
        pred = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=noise)
        pred2 = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=noise)      # graph replay / determinism
        assert torch.equal(pred, pred2)
    pred = pred.cpu()
    ref = torch.from_numpy(g["pred"])
    # F4C (block-scaled e2m1 corrections): the CPU emulation (tools/precision_probe.py f4c) predicts up to 2.9e-3 /
    # 2.1e-5 at F = 243, S = 9; measured 1.7e-3 / 9e-6 there and 2.8e-3 / 1.5e-5 at F = 27 -- a 3x margin instead of 4x
    margin = MARGIN_F4C if gemm_mode == _lib.GEMM_TC_F4C else MARGIN
    assert (pred - ref).abs().max().item() < MAXABS_BAR / margin
    assert _mpjpe_delta(pred, ref, gt) < MPJPE_BAR / margin


@pytest.mark.parametrize("env", [{"D3D_GEMM_RED": "0"}, {"D3D_LN_ROWS": "1"}, {"D3D_ATTN_WG2": "1"}, {"D3D_ATTN_SLOTS": "3"},
                                 {"D3D_ATTN_SLOTS": "2"}])
@pytest.mark.parametrize("name", ["sampler_f27_b2_s3_clip", "sampler_f243_b1_s9_clip", "sampler_f27_b2_s9_notime"])
def test_sampler_golden_alternative_epilogues(golden, monkeypatch, name, env):
    """Measured-and-kept alternatives of the F4C path, through the whole sampler against the reference goldens:
    D3D_GEMM_RED=0 (residual update by load-add-store instead of the TMA reduction; read when the launch sequence is
    built).  RED on / off must not change a single bit, and neither must the one-row-per-warp LayerNorm kernels
    (D3D_LN_ROWS=1; shipped: two rows per warp sharing every parameter load).  D3D_ATTN_WG2=1 is the
    two-warpgroups-per-slot temporal attention kernel (same arithmetic per element, different summation split of the row;
    measured slower, ships off)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = golden(name)
    F, B, S = int(g["F"]), int(g["B"]), int(g["S"])
    diff = _diffusion(F, S, 0.0, bool(g["clip"]), bool(g["with_time_emb"]), gemm_mode=_lib.GEMM_TC_F4C, max_clips=B)
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, S)
    pred = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T.cuda(), None)).cpu()
    ref = torch.from_numpy(g["pred"])
    assert (pred - ref).abs().max().item() < MAXABS_BAR / MARGIN_F4C
    assert _mpjpe_delta(pred, ref, gt) < MPJPE_BAR / MARGIN_F4C
    if "D3D_ATTN_WG2" not in env and "D3D_ATTN_SLOTS" not in env:
        for k in env:
            monkeypatch.delenv(k)
        diff2 = _diffusion(F, S, 0.0, bool(g["clip"]), bool(g["with_time_emb"]), gemm_mode=_lib.GEMM_TC_F4C, max_clips=B)
        pred2 = diff2.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T.cuda(), None)).cpu()
        assert torch.equal(pred, pred2)


def test_workspace_bytes_and_no_hot_path_allocation():
    """d3d_workspace_bytes (SURVEY.md 8b): the handle's device footprint is fixed after create / set_schedule -- 16 KB per
    token of the largest batch plus the packed weights -- and a sampler call allocates nothing (graph replay needs that)."""
    F, B, S = 27, 3, 2
    diff = _diffusion(F, S, max_clips=B)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, S)
    diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T.cuda(), None))
    eng = diff.model.engine(B)
    before = eng.workspace_bytes()
    tokens = (B * F * 17 + 511) // 512 * 512
    assert before >= tokens * 14 * 1024 and before < tokens * 17 * 1024 + 400 * 2 ** 20
    diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T.cuda(), None))
    diff.ddim_sample_loop(x2d[:2].cuda(), [2, F, 17, 3], noise=(y_T[:2].cuda(), None))
    assert eng.workspace_bytes() == before


def test_fp16_fast_mode_is_within_maxabs_bar(golden):
    g = golden("sampler_f27_b2_s3_clip")
    diff = _diffusion(27, 3, gemm_mode=_lib.GEMM_TC_FP16, max_clips=2)
    x2d, _ = synthetic.make_inputs(2, 27)
    y_T, _ = synthetic.make_noise(2, 27, 3)
    pred = diff.ddim_sample_loop(x2d.cuda(), [2, 27, 17, 3], noise=(y_T.cuda(), None)).cpu().numpy()
    assert np.abs(pred - g["pred"]).max() < 3e-2      # documented fast mode: looser than the parity bar


def test_forward_api_flip_tta_against_oracle():
    """evaluate()'s two GaussianDiffusion.forward calls + un-flip/average (RUN:577-588) vs the oracle, S=9."""
    F, B, S = 27, 2, 9
    diff = _diffusion(F, S, max_clips=B)
    x2d, gt = synthetic.make_inputs(B, F)
    xf = synthetic.flip_2d(x2d)
    n1, n2 = synthetic.make_noise(B, F, S, seed=1), synthetic.make_noise(B, F, S, seed=2)
    y = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(n1[0].cuda(), None))
    yf = diff.ddim_sample_loop(xf.cuda(), [B, F, 17, 3], noise=(n2[0].cuda(), None))
    merged = diff.model.engine(B).tta_merge(y, yf, synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT, 1.0).cpu()
    sd = {k: v.detach().cpu() for k, v in diff.model.state_dict().items()}
    with torch.no_grad():
        ref = oracle.sample_tta(sd, x2d, n1, n2, sampling_timesteps=S)
    assert (merged - ref).abs().max().item() < MAXABS_BAR / MARGIN_F4C      # default mode = F4C
    assert _mpjpe_delta(merged, ref, gt) < MPJPE_BAR / MARGIN_F4C
    # forward(): same signature / return convention as DIFF:421-449, and it consumes S normal draws in order
    torch.manual_seed(77)
    loss, pred = diff(clean_3d_pose=gt.cuda(), noisy_2d_pose=x2d.cuda(), output_loss=False)
    torch.manual_seed(77)
    y_T = torch.randn(B, F, 17, 3, device="cuda")
    for _ in range(S - 1):
        torch.randn_like(y_T)
    after = torch.randn(3, device="cuda")
    pred2 = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T, None))
    assert loss is None and torch.equal(pred, pred2)
    torch.manual_seed(77)
    diff(clean_3d_pose=gt.cuda(), noisy_2d_pose=x2d.cuda(), output_loss=False)
    assert torch.equal(after, torch.randn(3, device="cuda"))
    loss, _ = diff(clean_3d_pose=gt.cuda(), noisy_2d_pose=x2d.cuda(), output_loss=True)     # N1 row: p_losses
    assert loss.shape == (B, F, 17, 3) and torch.isfinite(loss).all()


@pytest.mark.parametrize("name", ["forward_f27_b3_s2_loss", "forward_f9_b2_s2_rep2_l1"])
def test_forward_output_loss_and_repeat_n_golden(golden, monkeypatch, name):
    """N1 + repeat_n: GaussianDiffusion.forward in eval mode with the default output_loss=True (what the 3DHP evaluate()
    calls, RUN3:517-520) against the imported reference with every draw pinned (tools/make_golden.py forward_case): the
    loss tensor of p_losses (DIFF:392-419: randint t, q_sample, one per-sample-t denoiser call, weighted l1 / l2) and the
    prediction averaged over repeat_n tiled copies of the 2D input (DIFF:434,448).  Draw order inside forward():
    randint, randn_like (skipped when `noise=` is given), then the sampler's S draws."""
    g = golden(name)
    F, B, S, rep = int(g["F"]), int(g["B"]), int(g["S"]), int(g["repeat_n"])
    m = synthetic.make_model(F).cuda()
    m.max_clips_hint = rep * B
    from diff3dhpe_b200.diffusion import GaussianDiffusion
    diff = GaussianDiffusion(m, timesteps=1000, sampling_timesteps=S, loss_type=str(g["loss_type"]), clip_denoised=True,
                             beta_schedule='cosine', ddim_sampling_eta=0.0, clipLoss=bool(g["clip_loss"])).cuda().eval()
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(rep * B, F, S)
    loss_noise = torch.randn(B, F, 17, 3, generator=torch.Generator().manual_seed(777))
    t_fixed = torch.tensor(g["t"], dtype=torch.long)
    calls = []
    real_randint = torch.randint

    def fake_randint(low, high, size, **kw):
        calls.append((low, high, tuple(size)))
        return t_fixed.to(kw.get("device", "cpu"))
    monkeypatch.setattr(torch, "randint", fake_randint)
    monkeypatch.setattr(diff, "draw_noise", lambda shape, dev: (y_T.to(dev), None))
    loss, pred = diff(clean_3d_pose=gt.cuda(), noisy_2d_pose=x2d.cuda(), noise=loss_noise.cuda(), repeat_n=rep)
    monkeypatch.setattr(torch, "randint", real_randint)
    assert calls == [(0, 1000, (B,))]
    loss, pred = loss.cpu(), pred.cpu()
    ref_loss, ref_pred = torch.from_numpy(g["loss"]), torch.from_numpy(g["pred"])
    assert pred.shape == ref_pred.shape == (B, F, 17, 3)
    assert (pred - ref_pred).abs().max().item() < MAXABS_BAR / MARGIN_F4C   # default mode = F4C
    assert _mpjpe_delta(pred, ref_pred, gt) < MPJPE_BAR / MARGIN_F4C
    # loss: <= 1e-3 relative on the mean (the quantity evaluate() logs) and element-wise against the loss scale
    assert abs(loss.mean().item() - ref_loss.mean().item()) <= 1e-3 * ref_loss.mean().item()
    assert (loss - ref_loss).abs().max().item() <= 2e-3 * ref_loss.abs().max().item()


def test_forward_denoise_is_asynchronous_per_sample_t():
    """d3d_forward_denoise keeps the per-sample timesteps on the device (no host round trip), so the call can be captured
    into a CUDA graph by the caller -- which a cudaStreamSynchronize inside it would make illegal -- and replayed with new
    timesteps written into the same tensor."""
    F, B = 9, 3
    m = synthetic.make_model(F).cuda()
    m.max_clips_hint = B
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, 1)
    x5 = torch.cat([x2d, y_T], -1).cuda()
    t = torch.tensor([999, 500, 3], device="cuda")
    eager = m.forward_denoise(x5, t)
    eng = m.engine(B)
    out = torch.empty_like(eager)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            out.copy_(eng.forward_denoise(x5, t))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)
    t.copy_(torch.tensor([10, 20, 30], device="cuda"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, m.forward_denoise(x5, t)) and not torch.equal(out, eager)


def test_cfg3_size_batch_is_bit_equal_to_single_clips():
    """The bench's own batch (cfg3: 512 clips x 243 frames = 2.1 M tokens, 34 GB of workspace, byte offsets beyond 2^32,
    more GEMM tiles than two waves of CTA pairs): its first, middle and last clips must equal the same clips sampled
    alone, bit for bit (clips are independent, RUN:577-588; split-invariance is what makes rank-sharding exact).  Two DDIM
    steps so that the head / DDIM update feeds a second denoiser call at that size as well."""
    F, B, S = 243, 512, 2
    diff = _diffusion(F, S, max_clips=B)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, S)
    xd, nd = x2d.cuda(), y_T.cuda()
    full = diff.ddim_sample_loop(xd, [B, F, 17, 3], noise=(nd, None))
    assert torch.isfinite(full).all()
    for i in (0, 255, 256, 511):
        one = diff.ddim_sample_loop(xd[i:i + 1].contiguous(), [1, F, 17, 3], noise=(nd[i:i + 1].contiguous(), None))
        assert torch.equal(one[0], full[i]), f"clip {i} of the 512-clip batch differs from the clip sampled alone"
    # and a ragged middle slice that starts inside a 256-row GEMM tile and a 7-frame spatial-attention group
    part = diff.ddim_sample_loop(xd[300:333].contiguous(), [33, F, 17, 3], noise=(nd[300:333].contiguous(), None))
    assert torch.equal(part, full[300:333])


def test_checkpoint_keys_with_dataparallel_prefix_through_the_abi():
    """RUN:220-235: a checkpoint saved under nn.DataParallel carries 'module.model.' prefixes and the schedule buffers;
    d3d_load_weights strips the prefixes itself (raw key strings cross the ABI) and the result is bit-identical to the
    un-prefixed load."""
    from diff3dhpe_b200.engine import Engine
    F, B = 9, 2
    model = synthetic.make_model(F)
    diff = synthetic.make_diffusion(model, sampling_timesteps=2)
    ckpt = {"module." + k: v.clone() for k, v in diff.state_dict().items() if "alphas" not in k}
    assert any(k.startswith("module.model.STEblocks.0.attn.qkv.weight") for k in ckpt)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, 1)
    x5 = torch.cat([x2d, y_T], -1).cuda()
    t = torch.tensor([400, 30], device="cuda")
    outs = []
    for raw in (False, True):
        eng = Engine(F, max_clips=B)
        eng.load_state_dict({k: v.cuda() for k, v in ckpt.items()} if raw else model.state_dict(), raw_names=raw)
        outs.append(eng.forward_denoise(x5, t).clone())
        eng.close()
    assert torch.equal(outs[0], outs[1])


def test_load_time_range_guard():
    """A linear weight beyond the fp16 operand range, or a non-finite one, is rejected at load time with an error code
    instead of turning into Inf inside every GEMM (SURVEY.md 7.3-1)."""
    from diff3dhpe_b200.engine import Engine
    sd = {k: v.clone() for k, v in synthetic.make_model(9).state_dict().items()}
    eng = Engine(9, max_clips=1)
    eng.load_state_dict(sd)                                            # in range: fine
    bad = dict(sd)
    bad["TTEblocks.3.mlp.fc2.weight"] = sd["TTEblocks.3.mlp.fc2.weight"].clone()
    bad["TTEblocks.3.mlp.fc2.weight"][7, 11] = 7.0e4
    with pytest.raises(RuntimeError, match="code -12.*TTEblocks.3.mlp.fc2.weight.*fp16"):
        eng.load_state_dict(bad)
    bad["TTEblocks.3.mlp.fc2.weight"][7, 11] = float("nan")
    with pytest.raises(RuntimeError, match="code -12.*NaN"):
        eng.load_state_dict(bad)
    eng.close()


@pytest.mark.parametrize("w_scale,g_scale", [(1.5, 1.0), (1.0, 2.0), (2.0, 1.0)])
def test_trained_checkpoint_ranges_stress(w_scale, g_scale):
    """Random-init weights are O(0.04) with LayerNorm gains of exactly 1 and shifts of exactly 0 -- which every golden
    vector shares; trained checkpoints (README.md:66, not available offline) do not.  Scale every linear weight and every
    LayerNorm gain, perturb the gains per channel (+- 0.1) and all biases / shifts (+- 0.05), and compare with the oracle
    run live on the same state dict.  The scales are bounded by the REFERENCE's own conditioning, measured on the CPU
    oracle (fp32) with a 1e-6 relative perturbation of the 2D input: output change 3e-6 at (1, 1), 8e-6 at (1.5, 1),
    4e-6 at (1, 2), 9e-5 at (2, 1) -- and 2.5 (chaotic: a random-weight residual network with gains above ~2) at (2, 2),
    (4, 1), (1, 8), where no two fp32 implementations agree and a parity test is meaningless.  The bar scales with the
    un-clipped output range and, for (2, 1), with the 30x larger sensitivity."""
    F, B, S = 27, 1, 3
    m = synthetic.make_model(F)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if k.endswith(("qkv.weight", "proj.weight", "fc1.weight", "fc2.weight")):
                p.mul_(w_scale)
            elif "norm" in k and k.endswith(".weight"):
                p.mul_(g_scale).add_(0.1 * torch.randn(p.shape, generator=g))
            elif k.endswith(".bias"):
                p.add_(0.05 * torch.randn(p.shape, generator=g))
    m = m.cuda()
    m.max_clips_hint = B
    diff = synthetic.make_diffusion(m, sampling_timesteps=S, clip_denoised=False).cuda().eval()
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, steps = synthetic.make_noise(B, F, S)
    pred = diff.ddim_sample_loop(x2d.cuda(), [B, F, 17, 3], noise=(y_T.cuda(), None)).cpu()
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    with torch.no_grad():
        ref = oracle.ddim_sample_loop(sd, x2d, y_T, steps, sampling_timesteps=S, clip_denoised=False)
    scale = max(1.0, ref.abs().max().item())                  # un-clipped outputs grow with the weights
    assert torch.isfinite(pred).all()
    bar = MAXABS_BAR / 2 * scale * (4.0 if w_scale >= 2.0 else 1.0)
    assert (pred - ref).abs().max().item() < bar


@pytest.mark.parametrize("spatial", [True, False])
def test_attention_with_trained_range_logits(spatial):
    """Attention cores at logits of a trained model (|q.k| / 8 up to ~30: near one-hot softmax rows) instead of the
    random-init +- 1: the max-subtracted softmax, the fp16 P and the exact "- V" term of the tcgen05 kernels against the
    oracle on the same fp16-rounded q, k."""
    from diff3dhpe_b200.engine import Engine
    F, B, J, C = 81, 2, 17, 512
    eng = Engine(F, max_clips=B)
    g = torch.Generator().manual_seed(11)
    qkv = torch.randn(B * F * J, 3 * C, generator=g) * 3.0
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    x = qkv.view(B, F, J, 3 * C)
    seqs = x.reshape(B * F, J, 3 * C) if spatial else x.permute(0, 2, 1, 3).reshape(B * J, F, 3 * C)
    ref = oracle.attention_core(seqs, 8)
    ref = ref.reshape(B, F, J, C) if spatial else ref.reshape(B, J, F, C).permute(0, 2, 1, 3)
    out = eng.op_attention(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT).cpu().view(B, F, J, C)
    eng.close()
    assert torch.isfinite(out).all()
    assert (out - ref).abs().max().item() < 4e-3 * 3.0
