"""GPU (-m gpu): the 256-wide denoiser (embed_dim 256, 8 heads of 32, mlp hidden 512) on the sm_100a kernels.

Op level against fp64 / the oracle: the four GEMMs at their C = 256 shapes, the attention kernel (spatial, temporal and
packed modes at head_dim 32) against oracle.attention_core, its proj operand and the row-wise kernels' operands, and the
time table.  Path level against the oracle-generated fixtures tests/golden/w256_*.npz (tools/make_golden_width256.py):
the DDIM sampler, forward_denoise with per-sample t, graphed == un-graphed and batch-split == single-clip bit for bit.
Path tolerances are the north-star bar (per-joint max-abs 1e-2, |dMPJPE| 1e-4) with the 3x margin the 512-wide F4C
path keeps."""
import numpy as np
import pytest
import torch

from diff3dhpe_b200 import _lib, synthetic
from diff3dhpe_b200.engine import Engine
from oracle import diff3d_oracle as oracle
from test_gpu_rowwise import _E2M1_VAL, e2m1_codes, ue8m0_bytes

pytestmark = pytest.mark.gpu

C, J, HIDDEN = 256, 17, 512
MAXABS_BAR, MPJPE_BAR, MARGIN_F4C = 1e-2, 1e-4, 3.0


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def _engine(F, B=1, **kw):
    return Engine(F, embed_dim=C, mlp_hidden=HIDDEN, max_clips=B, gemm_mode=_lib.GEMM_TC_F4C, **kw)


def _diffusion(F, S, eta=0.0, clip=True, with_time_emb=True, use_graph=True, max_clips=1):
    m = synthetic.make_model(F, with_time_emb=with_time_emb, embed_dim=C).cuda()
    m.use_graph, m.max_clips_hint = use_graph, max_clips
    return synthetic.make_diffusion(m, sampling_timesteps=S, eta=eta, clip_denoised=clip).cuda().eval()


# ------------------------------------------------------------------------------------------------------------ GEMMs
@pytest.mark.parametrize("M", [4131, 1000, 1])
@pytest.mark.parametrize("N,K,act,res", [(3 * C, C, 0, False), (C, C, 0, True), (HIDDEN, C, 1, False), (C, HIDDEN, 0, True)])
def test_linear_f4c_width256_shapes(M, N, K, act, res):
    """qkv (768 x 256), proj (256 x 256, in-place residual), fc1 (512 x 256, GELU -> operand) and fc2 (256 x 512,
    residual) on the F4C tcgen05 kernel against fp64; ragged M (4131 = one F = 243 clip) and a single row."""
    eng = _engine(27)
    a, w, b = _rand((M, K), 1), _rand((N, K), 2, 0.05), _rand((N,), 3, 0.1)
    r = _rand((M, N), 4) if res else None
    ref = a.double() @ w.double().T + b.double()
    if act:
        ref = torch.nn.functional.gelu(ref)
    elif res:
        ref = ref + r.double()
    out = eng.op_linear(a.cuda(), w.cuda(), b.cuda(), residual=None if r is None else r.cuda(), act=act,
                        gemm_mode=_lib.GEMM_TC_F4C).cpu().double()
    eng.close()
    scale = (a.double().abs() @ w.double().abs().T).max().item()
    err = (out - ref).abs().max().item() / scale
    assert err < 4e-4, f"relative error {err:.3e}"


# -------------------------------------------------------------------------------------------------------- attention
def _qkv(B, F, seed):
    qkv = _rand((B * F * J, 3 * C), seed, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()      # the kernels read q, k as fp16 (v as an exact hi / lo pair)
    return qkv


def _attn_ref(qkv, B, F, spatial):
    x = qkv.view(B, F, J, 3 * C).double()
    seqs = x.reshape(B * F, J, 3 * C) if spatial else x.permute(0, 2, 1, 3).reshape(B * J, F, 3 * C)
    ref = oracle.attention_core(seqs, 8)
    ref = ref.reshape(B, F, J, C) if spatial else ref.reshape(B, J, F, C).permute(0, 2, 1, 3)
    return ref.reshape(B * F * J, C)


@pytest.mark.parametrize("F", [1, 9, 27, 64, 81, 243, 256])
@pytest.mark.parametrize("spatial", [True, False])
def test_attention_core_width256(F, spatial):
    """head_dim 32 (SWIZZLE_64B boxes, 2 k-steps of QK^T, P.V with N = 32, scale 32^-0.5 on the fp32 scores) against
    oracle.attention_core in fp64.  The result passes through the proj operand (hi + Q), so per element the bound is
    the fp16 rounding of P and of the V operand of P.V (|out| <= ~4 here) plus the operand's own resolution."""
    B = 2
    eng = _engine(F, B)
    qkv = _qkv(B, F, 20 + F)
    ref = _attn_ref(qkv, B, F, spatial)
    out = eng.op_attention(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT).cpu().double()
    eng.close()
    err = (out - ref).abs()
    assert torch.isfinite(out).all()
    assert (err <= 4e-3 + 1e-3 * ref.abs()).all(), f"max err {err.max().item():.3e}"
    assert err.mean().item() < 5e-4


def _decode_f4c(second, T):
    flat = second.reshape(-1).cpu().numpy()
    c4, sf = flat[:T * C].reshape(T, C), flat[T * C:T * C + T * (C // 16)].reshape(T, C // 16)
    nib = np.stack([c4 & 15, c4 >> 4], axis=-1).reshape(T, 2 * C)
    val = _E2M1_VAL[nib] * np.repeat(np.exp2(sf.astype(np.float64) - 127.0), 32, axis=1)
    return nib, val[:, :C], val[:, C:], sf


@pytest.mark.parametrize("F,B,spatial", [(243, 2, False), (81, 3, False), (27, 5, False), (64, 3, False), (9, 4, True),
                                         (27, 3, True), (1, 2, True), (256, 1, False)])
def test_attention_operand_width256(F, B, spatial):
    """The proj operand the kernel writes (FMT_F4C, one scale block per head and part at head_dim 32: k-blocks h and
    8 + h): hi = fp16(ref) to the kernel's accuracy; every P scale byte the smallest power of two that keeps the block
    maximum of x = hi + Q <= 6; every P value x on its block's e2m1 grid to one step; every Q nibble re-encoded exactly
    by the CPU encoder from its decoded value; |Q| within half an fp16 ulp of hi."""
    eng = _engine(F, B)
    qkv = _qkv(B, F, 70 + F)
    T = B * F * J
    ref = _attn_ref(qkv, B, F, spatial).numpy()
    hi, second = eng.debug_attention_operand(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT)
    eng.close()
    hi = hi.float().cpu().numpy().astype(np.float64)
    nib, P, Q, sf = _decode_f4c(second, T)
    assert np.isfinite(hi).all()
    assert np.abs(hi - ref).max() < 4e-3 + 2 ** -10 * np.abs(ref).max()
    # scale bytes of part P: the smallest power of two keeping the block maximum of x <= 6, with x = hi + Q ~ ref
    x = hi + Q
    blk = np.abs(x).reshape(T, C // 32, 32).max(-1)
    ratio = blk / np.exp2(sf[:, :C // 32].astype(np.float64) - 127.0)
    assert ((ratio <= 6.0 * (1 + 2 ** -9)) & ((ratio > 3.0 * (1 - 2 ** -9)) | (blk < 1e-6))).all()
    # P: x on the e2m1 grid of its block scale, to one step
    step = np.repeat(np.exp2(sf[:, :C // 32].astype(np.float64) - 127.0), 32, axis=1)
    assert (np.abs(P - x) <= step * 1.0 + 1e-6).all()
    # Q re-encoded by the CPU encoder from its own decoded value: identical nibbles (the block scale of x - hi is the
    # kernel's own byte, so the re-encoding of an on-grid value is exact)
    sq = np.repeat(np.exp2(127.0 - sf[:, C // 32:].astype(np.float64)), 32, axis=1)
    q_codes = e2m1_codes((Q * sq).astype(np.float32))
    assert np.array_equal(q_codes & 7, nib[:, C:] & 7)
    # Q's scale byte is that of the block maximum of |x - hi| <= half an fp16 ulp of x
    assert (np.abs(Q) <= 2 ** -11 * np.abs(hi) * 1.35 + 1e-7).all()


# -------------------------------------------------------------------------------------------------------- row-wise
def _encode_f4c(y):
    y = np.ascontiguousarray(y, dtype=np.float32)
    R = y.shape[0]
    h = y.astype(np.float16)
    lo = y - h.astype(np.float32)
    bp = ue8m0_bytes(np.abs(y).reshape(R, C // 32, 32).max(-1))
    bq = ue8m0_bytes(np.abs(lo).reshape(R, C // 32, 32).max(-1))
    p = e2m1_codes(y * np.repeat(np.exp2(127.0 - bp), 32, axis=1).astype(np.float32))
    q = e2m1_codes(lo * np.repeat(np.exp2(127.0 - bq), 32, axis=1).astype(np.float32))
    nib = np.concatenate([p, q], axis=1)
    return h.view(np.uint16), (nib[:, 0::2] | (nib[:, 1::2] << 4)).astype(np.uint8), np.concatenate([bp, bq], axis=1)


def _parts(hi, second, T):
    flat = second.reshape(-1)
    return (hi.view(torch.int16).cpu().numpy().view(np.uint16), flat[:T * C].view(T, C).cpu().numpy(),
            flat[T * C:T * C + T * (C // 16)].view(T, C // 16).cpu().numpy())


@pytest.mark.parametrize("F,B", [(27, 3), (243, 1), (9, 5)])
@pytest.mark.parametrize("rows", ["1", "2"])
def test_rowwise_operands_width256(monkeypatch, F, B, rows):
    """lift + norm1, post-norm + add + norm1 and norm2 at C = 256 (one- and two-rows-per-warp forms): the fp32 residual
    stream against fp64, and every byte of the GEMM operand they write against the CPU encoder of the kernel's own fp32
    LayerNorm (d3d_op_layernorm runs the same per-row arithmetic); head + DDIM output against fp64."""
    monkeypatch.setenv("D3D_LN_ROWS", rows)
    m = synthetic.make_model(F, embed_dim=C)
    sd = {k: v.detach().cuda() for k, v in m.state_dict().items()}
    eng = _engine(F, B)
    eng.load_state_dict(m.state_dict())
    T = B * F * J
    t = torch.tensor([5 + 97 * i for i in range(B)])

    def check_operand(hi, second, x, ln):
        y = eng.op_layernorm(x.contiguous(), sd[ln + ".weight"], sd[ln + ".bias"], 1e-6)
        want = _encode_f4c(y.cpu().numpy())
        got = _parts(hi, second, T)
        for g, w, what in zip(got, want, ("hi", "c4", "sf")):
            assert np.array_equal(g, w), f"{ln}: {what} bytes differ ({(g != w).sum()} of {g.size})"

    # lift (x5 form, per-clip t) -> X and the norm1 operand of block 0
    x5 = torch.cat([0.3 * _rand((T, 2), 11), _rand((T, 3), 12)], 1).cuda()
    X, hi, second = eng.debug_rowwise(_lib.ROWWISE_LIFT, x5, t=t)
    t_emb = oracle.time_mlp({k: v.cpu() for k, v in sd.items()}, t, C).double()
    tv = torch.nn.functional.linear(torch.nn.functional.silu(t_emb), sd["STEblocks.0.time_mlp.1.weight"].double().cpu(),
                                    sd["STEblocks.0.time_mlp.1.bias"].double().cpu())
    ref = (x5.double().cpu() @ sd["fusion_layer.weight"].double().cpu().T + sd["fusion_layer.bias"].double().cpu()).view(B, F, J, C)
    ref = ref + sd["Spatial_pos_embed"].double().cpu() + tv[:, None, None, :]
    assert (X.cpu().double() - ref.reshape(T, C)).abs().max().item() < 1e-4
    check_operand(hi, second, X, "STEblocks.0.norm1")
    # post-norm of block 0 (Spatial_norm) + Temporal_pos_embed + block 1's time vector -> norm1 of block 1
    xin = _rand((T, C), 13).cuda()
    X2, hi, second = eng.debug_rowwise(_lib.ROWWISE_POSTNORM, xin, t=t, block=1)
    check_operand(hi, second, X2, "TTEblocks.0.norm1")
    # norm2 of block 3
    _, hi, second = eng.debug_rowwise(_lib.ROWWISE_NORM2, xin, block=3)
    check_operand(hi, second, xin, "TTEblocks.1.norm2")
    # head (post-norm + head LayerNorm + Linear(256 -> 3))
    out3, _, _ = eng.debug_rowwise(_lib.ROWWISE_HEAD, xin)
    eng.close()
    xd = xin.double().cpu()
    z = torch.nn.functional.layer_norm(xd, (C,), sd["Temporal_norm.weight"].double().cpu(), sd["Temporal_norm.bias"].double().cpu(), 1e-6)
    z = torch.nn.functional.layer_norm(z, (C,), sd["head.0.weight"].double().cpu(), sd["head.0.bias"].double().cpu(), 1e-5)
    ref3 = z @ sd["head.1.weight"].double().cpu().T + sd["head.1.bias"].double().cpu()
    assert (out3.cpu().double() - ref3).abs().max().item() < 2e-5


def test_time_table_width256(golden):
    g = golden("w256_denoise_f27_b3")
    eng = _engine(27, 3)
    eng.load_state_dict(synthetic.make_model(27, embed_dim=C).state_dict())
    tab = eng.op_time_table([float(t) for t in g["t"]]).cpu().numpy()
    eng.close()
    assert np.abs(tab - g["time_table"]).max() < 2e-5


# -------------------------------------------------------------------------------------------------------- path level
def test_forward_denoise_width256(golden):
    """Per-sample t (the p_losses form) through the drop-in module."""
    g = golden("w256_denoise_f27_b3")
    F, B = int(g["F"]), int(g["B"])
    diff = _diffusion(F, 1, max_clips=B)
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, 1)
    out = diff.model.forward_denoise(torch.cat([x2d, y_T], -1).cuda(), torch.tensor(g["t"]).cuda()).cpu().numpy()
    assert np.abs(out - g["out"]).max() < MAXABS_BAR / MARGIN_F4C


@pytest.mark.parametrize("name", ["w256_sampler_f27_b2_s9_notime", "w256_sampler_f81_b1_s9_clip",
                                  "w256_sampler_f243_b1_s9_clip", "w256_sampler_f27_b2_s3_eta_trace"])
def test_sampler_width256(golden, name):
    g = golden(name)
    F, B, S, eta = int(g["F"]), int(g["B"]), int(g["S"]), float(g["eta"])
    x2d, gt = synthetic.make_inputs(B, F)
    y_T, steps = synthetic.make_noise(B, F, S)
    noise = (y_T.cuda(), steps.cuda() if eta != 0 else None)
    diff = _diffusion(F, S, eta, bool(g["clip"]), bool(g["with_time_emb"]), max_clips=B)
    if "rev" in g:
        pred, rev, x0s = diff.ddim_sample_loop_ouput_reverse_diffusion(x2d.cuda(), [B, F, J, 3], noise=noise)
        assert np.abs(rev.cpu().numpy() - g["rev"]).max() < MAXABS_BAR / MARGIN_F4C
        assert np.abs(x0s.cpu().numpy() - g["x0s"]).max() < MAXABS_BAR / MARGIN_F4C
    else:
        pred = diff.ddim_sample_loop(x2d.cuda(), [B, F, J, 3], noise=noise)
        # graphed (default) against un-graphed: bit for bit
        diff.model.use_graph = False
        pred_eager = diff.ddim_sample_loop(x2d.cuda(), [B, F, J, 3], noise=noise)
        assert torch.equal(pred, pred_eager)
    pred = pred.cpu()
    assert np.abs(pred.numpy() - g["pred"]).max() < MAXABS_BAR / MARGIN_F4C
    d = abs(oracle.mpjpe(pred, gt).item() - oracle.mpjpe(torch.from_numpy(g["pred"]), gt).item())
    assert d < MPJPE_BAR / MARGIN_F4C


@pytest.mark.parametrize("F", [27, 243])
def test_batch_split_equals_single_clips_width256(F):
    """Three clips in one call against each clip alone on the same handle: bit for bit (every kernel's arithmetic on a
    token is independent of the other clips of the batch)."""
    B, S = 3, 2
    diff = _diffusion(F, S, max_clips=B)
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, _ = synthetic.make_noise(B, F, S)
    full = diff.ddim_sample_loop(x2d.cuda(), [B, F, J, 3], noise=(y_T.cuda(), None))
    for b in range(B):
        one = diff.ddim_sample_loop(x2d[b:b + 1].cuda(), [1, F, J, 3], noise=(y_T[b:b + 1].cuda(), None))
        assert torch.equal(one, full[b:b + 1]), f"clip {b}"


def test_forward_eval_and_dataparallel_registry_width256():
    """forward() with output_loss / repeat_n through the drop-in GaussianDiffusion at C = 256, and the engine registry
    the nn.DataParallel replicas share: one engine per device whatever the width."""
    F, B, S = 27, 2, 2
    diff = _diffusion(F, S, max_clips=4)
    x2d, gt = synthetic.make_inputs(B, F)
    with torch.no_grad():
        out = diff(clean_3d_pose=gt.cuda(), noisy_2d_pose=x2d.cuda(), output_loss=True, repeat_n=2,
                   output_reverse_diffusion_3d=True)
    tensors = [o for o in out if torch.is_tensor(o)]
    assert len(tensors) >= 3 and all(torch.isfinite(o).all() for o in tensors)
    assert diff._engine(B).C == C
