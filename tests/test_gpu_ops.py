"""GPU (-m gpu): kernel-level parity through the C ABI against the CPU oracle / fp64 torch on the same inputs."""
import numpy as np
import pytest
import torch

from diff3dhpe_b200 import _lib, synthetic
from diff3dhpe_b200.engine import Engine
from oracle import diff3d_oracle as oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng27():
    e = Engine(27, max_clips=4)
    yield e
    e.close()


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


@pytest.fixture(autouse=True)
def _default_cta_group(monkeypatch):
    monkeypatch.delenv("D3D_GEMM_CG", raising=False)
    monkeypatch.delenv("D3D_GEMM_BN", raising=False)
    monkeypatch.delenv("D3D_GEMM_CS", raising=False)


@pytest.mark.parametrize("mode,tol,cg", [(_lib.GEMM_SIMT_FP32, 3e-6, 2), (_lib.GEMM_TC_SPLIT3, 3e-6, 2),
                                         (_lib.GEMM_TC_SPLIT3, 3e-6, 1), (_lib.GEMM_TC_FP16, 2e-3, 2),
                                         (_lib.GEMM_TC_FP16, 2e-3, 1), (_lib.GEMM_TC_F8C, 2e-4, 2),
                                         (_lib.GEMM_TC_F8C, 2e-4, 1), (_lib.GEMM_SIMT_F8C, 2e-4, 2)])
@pytest.mark.parametrize("M,N,K", [(128, 1536, 512), (200, 512, 512), (1000, 1024, 512), (459, 512, 1024),
                                   (37 * 128 + 5, 256, 64), (1, 512, 512), (74 * 256 * 3 + 77, 512, 512)])
def test_linear_parity(eng27, monkeypatch, mode, tol, cg, M, N, K):
    """cg = tcgen05 cta_group: 2 = CTA-pair 256x256 tiles (the product path), 1 = single-CTA 128xBN tiles."""
    monkeypatch.setenv("D3D_GEMM_CG", str(cg))
    a, w, b = _rand((M, K), 1), _rand((N, K), 2, 0.05), _rand((N,), 3, 0.1)
    res = _rand((M, N), 4)
    ref = (a.double() @ w.double().T + b.double() + res.double())
    out = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), residual=res.cuda(), act=0, gemm_mode=mode).cpu()
    scale = (a.double().abs() @ w.double().abs().T).max().item()       # error bound scales with sum |a||w|
    err = (out.double() - ref).abs().max().item() / scale
    assert err < tol, f"relative error {err:.3e}"


@pytest.mark.parametrize("mode,tol", [(_lib.GEMM_SIMT_FP32, 2e-5), (_lib.GEMM_TC_SPLIT3, 2e-5), (_lib.GEMM_TC_F8C, 1.5e-3),
                                      (_lib.GEMM_SIMT_F8C, 1.5e-3)])
def test_linear_gelu_split_epilogue(eng27, mode, tol):
    """fc1 epilogue: bias + exact-erf GELU, written as the A operand of fc2.  In the F8C format the operand keeps
    hi exactly and the lo term as e5m2 (3 significant bits of a 2^-11 correction); the test reads back hi + lo."""
    M, N, K = 300, 1024, 512
    a, w, b = _rand((M, K), 5), _rand((N, K), 6, 0.05), _rand((N,), 7, 0.1)
    ref = torch.nn.functional.gelu(a.double() @ w.double().T + b.double())
    out = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), act=1, gemm_mode=mode).cpu()
    assert (out.double() - ref).abs().max().item() < tol


@pytest.mark.parametrize("cs", [1, 2])
def test_f8c_tc_matches_simt_elementwise(eng27, monkeypatch, cs):
    """Same hi / e5m2 operands in: the tensor-core F8C kernel and the CUDA-core kernel form the same products, so
    they differ only by fp32 accumulation order."""
    monkeypatch.setenv("D3D_GEMM_CS", str(cs))       # 2 = pair clusters with weight-tile TMA multicast (default)
    M, N, K = 777, 1536, 512
    a, w, b = _rand((M, K), 8).cuda(), _rand((N, K), 9, 0.05).cuda(), _rand((N,), 10).cuda()
    x = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_TC_F8C)
    y = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_SIMT_F8C)
    assert (x - y).abs().max().item() < 2e-5


@pytest.mark.parametrize("ew", [8, 16])
@pytest.mark.parametrize("act", [0, 1])
def test_f8c_epilogue_warp_variants(eng27, monkeypatch, ew, act):
    """8 or 16 epilogue warps per CTA (D3D_GEMM_EW_*; shipped: 16 for the GELU epilogue, 8 for the fp32 one) over more
    row tiles than CTA pairs and a ragged last tile: the fp32 + residual epilogue against the CUDA-core kernel on the
    same operands, the packed-pair GELU epilogue against fp64."""
    monkeypatch.setenv("D3D_GEMM_EW_F32", str(ew))
    monkeypatch.setenv("D3D_GEMM_EW_GELU", str(ew))
    M, K = 74 * 256 + 300, 512
    N = 1024 if act else 512
    a, w, b = _rand((M, K), 41), _rand((N, K), 42, 0.05), _rand((N,), 43, 0.1)
    if act:
        ref = torch.nn.functional.gelu(a.double() @ w.double().T + b.double())
        out = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), act=1, gemm_mode=_lib.GEMM_TC_F8C).cpu()
        assert (out.double() - ref).abs().max().item() < 1.5e-3
    else:
        res = _rand((M, N), 44).cuda()
        x = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), residual=res, gemm_mode=_lib.GEMM_TC_F8C)
        y = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), residual=res, gemm_mode=_lib.GEMM_SIMT_F8C)
        # same operands and products, different fp32 accumulation order (measured: 2.0e-5 over 19 244 x 512 outputs)
        assert (x - y).abs().max().item() < 1e-4


F4C_SHAPES = [(128, 1536, 512), (200, 512, 512), (1000, 1024, 512), (459, 512, 1024), (1, 512, 512), (300, 256, 128),
              (74 * 256 * 3 + 77, 512, 512)]


@pytest.mark.parametrize("mode,red", [(_lib.GEMM_TC_F4C, 1), (_lib.GEMM_TC_F4C, 0), (_lib.GEMM_SIMT_F4C, 0)])
@pytest.mark.parametrize("M,N,K", F4C_SHAPES)
def test_linear_parity_f4c(eng27, monkeypatch, mode, red, M, N, K):
    """red = 1 (shipped): the residual sits in the output and the epilogue reduce-adds acc + bias into it through the TMA
    unit (EPI_F32_RED, cp.reduce.async.bulk.tensor .add.f32: the L2 performs the add); red = 0: the load-add-store epilogue.
    FMT_F4C (fp16 main product + block-scaled e2m1 correction products, kind::mxf4.block_scale) against fp64: the
    tensor-core kernel and its CUDA-core twin.  The corrections carry ~2 significant bits of a 2^-11 term, so the bound
    is looser than F8C's 2e-4 and far below single-pass fp16's 2e-3.  Shapes: one tile, ragged M, K = 1024 (8 e2m1
    stages), a single row, the minimum K (one e2m1 stage), and more tiles than CTA pairs (persistent loop: the scale
    factors of tile q live in the accumulator of tile q - 1)."""
    monkeypatch.setenv("D3D_GEMM_RED", str(red))
    a, w, b = _rand((M, K), 1), _rand((N, K), 2, 0.05), _rand((N,), 3, 0.1)
    res = _rand((M, N), 4)
    ref = (a.double() @ w.double().T + b.double() + res.double())
    out = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), residual=res.cuda(), act=0, gemm_mode=mode).cpu()
    scale = (a.double().abs() @ w.double().abs().T).max().item()
    err = (out.double() - ref).abs().max().item() / scale
    assert err < 4e-4, f"relative error {err:.3e}"


def test_reduction_epilogue_is_bit_equal_to_load_add_store(eng27, monkeypatch):
    """(acc + bias) + x rounded once in fp32, whether the SM adds the residual it loaded or the L2 adds the chunk the TMA
    unit hands it: the two epilogues must agree bit for bit (more row tiles than CTA pairs, ragged last tile)."""
    M, N, K = 74 * 256 + 300, 512, 512
    a, w, b = _rand((M, K), 61).cuda(), _rand((N, K), 62, 0.05).cuda(), _rand((N,), 63, 0.1).cuda()
    res = _rand((M, N), 64, 2.0).cuda()
    outs = []
    for red in (1, 0):
        monkeypatch.setenv("D3D_GEMM_RED", str(red))
        outs.append(eng27.op_linear(a, w, b, residual=res, act=0, gemm_mode=_lib.GEMM_TC_F4C))
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("M,N,K", F4C_SHAPES)
def test_f4c_tc_matches_simt_elementwise(eng27, M, N, K):
    """Same hi / e2m1 / scale-factor bytes in: the tcgen05 kernel (TMA-staged scale-factor atoms -> tcgen05.cp -> TMEM,
    kind::mxf4.block_scale MMAs) and the CUDA-core kernel that decodes nibble x 2^(scale - 127) in fp32 form the same
    products, so they differ only by fp32 accumulation order.  This is the bit-level check of the scale-factor layout,
    the SF ids and the TMEM column assignment."""
    a, w, b = _rand((M, K), 8).cuda(), _rand((N, K), 9, 0.05).cuda(), _rand((N,), 10).cuda()
    x = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_TC_F4C)
    y = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_SIMT_F4C)
    assert (x - y).abs().max().item() < 3e-5


@pytest.mark.parametrize("mode", [_lib.GEMM_TC_F4C, _lib.GEMM_SIMT_F4C])
@pytest.mark.parametrize("ew", [8, 16])
def test_linear_gelu_f4c_epilogue(eng27, monkeypatch, mode, ew):
    """fc1 epilogue in the F4C format: bias + exact-erf GELU written as hi fp16 + block-scaled e2m1 images of x and of
    x - hi + their ue8m0 scale bytes; the test reads back hi + q4(x - hi) * scale.  8 and 16 epilogue warps (one word /
    one half-word of scale bytes per row and tile), more row tiles than CTA pairs, ragged last tile."""
    monkeypatch.setenv("D3D_GEMM_EW_GELU", str(ew))
    M, N, K = 74 * 256 + 300, 1024, 512
    a, w, b = _rand((M, K), 5), _rand((N, K), 6, 0.05), _rand((N,), 7, 0.1)
    ref = torch.nn.functional.gelu(a.double() @ w.double().T + b.double())
    out = eng27.op_linear(a.cuda(), w.cuda(), b.cuda(), act=1, gemm_mode=mode).cpu()
    assert (out.double() - ref).abs().max().item() < 2e-3


@pytest.mark.parametrize("F", [81, 100, 243, 256, 65, 129])
def test_attention_two_warpgroups_per_slot(monkeypatch, F):
    """attn_temporal_tc2_kernel (D3D_ATTN_WG2=1; measured slower, ships off): a row's columns and channels split over two
    warpgroups, P in two TMEM column ranges, row maximum / sum exchanged through shared memory.  Same reference and
    tolerance as test_attention_core; F covers 3 chunks (2 + 1 split), 4, 8, the full 256 and the smallest sizes of the
    one- and two-tile paths."""
    monkeypatch.setenv("D3D_ATTN_WG2", "1")
    B, J, C = 2, 17, 512
    eng = Engine(F, max_clips=B)
    qkv = _rand((B * F * J, 3 * C), 20 + F, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    x = qkv.view(B, F, J, 3 * C)
    ref = oracle.attention_core(x.permute(0, 2, 1, 3).reshape(B * J, F, 3 * C), 8).reshape(B, J, F, C).permute(0, 2, 1, 3)
    out = eng.op_attention(qkv.cuda(), B, False, _lib.ATTN_DEFAULT).cpu().view(B, F, J, C)
    eng.close()
    assert (out - ref).abs().max().item() < 4e-3


@pytest.mark.parametrize("F,spatial", [(27, True), (243, True), (9, True), (100, True), (1, True), (9, False), (27, False),
                                       (33, False), (64, False)])
def test_attention_three_slots(monkeypatch, F, spatial):
    """D3D_ATTN_SLOTS=3: the single-tile modes (spatial; packed temporal, F <= 64) with three 128-column TMEM slots and three
    softmax warpgroups per CTA (512 threads) instead of two 256-column slots.  Same reference and tolerance as
    test_attention_core."""
    monkeypatch.setenv("D3D_ATTN_SLOTS", "3")
    B, J, C = 2, 17, 512
    eng = Engine(F, max_clips=B)
    qkv = _rand((B * F * J, 3 * C), 20 + F, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    x = qkv.view(B, F, J, 3 * C)
    seqs = x.reshape(B * F, J, 3 * C) if spatial else x.permute(0, 2, 1, 3).reshape(B * J, F, 3 * C)
    ref = oracle.attention_core(seqs, 8)
    ref = ref.reshape(B, F, J, C) if spatial else ref.reshape(B, J, F, C).permute(0, 2, 1, 3)
    out = eng.op_attention(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT).cpu().view(B, F, J, C)
    eng.close()
    assert (out - ref).abs().max().item() < 4e-3


def test_tc_matches_simt_elementwise(eng27):
    """Same split operands in, so tensor-core and CUDA-core results differ only by accumulation order and the
    dropped lo*lo term (2^-22 relative)."""
    M, N, K = 777, 1536, 512
    a, w, b = _rand((M, K), 8).cuda(), _rand((N, K), 9, 0.05).cuda(), _rand((N,), 10).cuda()
    x = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_TC_SPLIT3)
    y = eng27.op_linear(a, w, b, gemm_mode=_lib.GEMM_SIMT_FP32)
    assert (x - y).abs().max().item() < 2e-5


@pytest.mark.parametrize("eps", [1e-6, 1e-5])
def test_layernorm(eng27, eps):
    x, g, b = _rand((1000, 512), 11, 3.0) + 0.5, _rand((512,), 12) + 1, _rand((512,), 13)
    ref = torch.nn.functional.layer_norm(x, (512,), g, b, eps)
    out = eng27.op_layernorm(x.cuda(), g.cuda(), b.cuda(), eps).cpu()
    assert (out - ref).abs().max().item() < 5e-6


@pytest.mark.parametrize("F", [27, 81, 243, 9, 100, 1, 256])
@pytest.mark.parametrize("mode,tol", [(_lib.ATTN_DEFAULT, 4e-3), (_lib.ATTN_SIMT, 3e-5), (_lib.ATTN_MMA_SYNC, 4e-3)])
@pytest.mark.parametrize("spatial", [True, False])
def test_attention_core(F, mode, tol, spatial):
    """The kernels read q, k as fp16 and v as an fp16 hi/lo pair (what the qkv GEMM epilogue writes), so the
    reference gets the same fp16-rounded q, k.  SIMT mode (fp32 arithmetic) then matches to rounding; the
    tensor-core mode additionally rounds P and the V operand of P.V to fp16 (single pass), tolerance 4e-3 on
    outputs of magnitude ~4 -- the sampler-level effect is bounded by the golden tests."""
    B, J, C = 2, 17, 512
    eng = Engine(F, max_clips=B)
    qkv = _rand((B * F * J, 3 * C), 20 + F, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    x = qkv.view(B, F, J, 3 * C)
    seqs = x.reshape(B * F, J, 3 * C) if spatial else x.permute(0, 2, 1, 3).reshape(B * J, F, 3 * C)
    ref = oracle.attention_core(seqs, 8)
    ref = ref.reshape(B, F, J, C) if spatial else ref.reshape(B, J, F, C).permute(0, 2, 1, 3)
    out = eng.op_attention(qkv.cuda(), B, spatial, mode).cpu().view(B, F, J, C)
    eng.close()
    assert (out - ref).abs().max().item() < tol


@pytest.mark.parametrize("gemm_mode", [_lib.GEMM_TC_F8C, _lib.GEMM_TC_SPLIT3])
@pytest.mark.parametrize("F,B,spatial", [(243, 5, False), (81, 6, False), (129, 3, False), (128, 3, False), (65, 4, False),
                                         (256, 2, False), (243, 5, True), (27, 40, True), (7, 17, True), (1, 1, True),
                                         # packed temporal mode: 4 (F <= 32) or 2 (F <= 64) joints per 128-row tile
                                         (27, 40, False), (32, 3, False), (33, 5, False), (64, 3, False), (9, 2, False),
                                         (1, 2, False)])
def test_attention_tcgen05_operand(F, B, spatial, gemm_mode):
    """The tcgen05/TMEM/TMA attention kernel (temporal: default for F > 64; spatial: units of 7 frames with a
    block-diagonal mask) against the CUDA-core kernel, on EVERY byte of the operand the proj GEMM consumes (hi fp16 |
    fp16 lo, or hi | e5m2(x 2^-8) | e5m2(lo 2^4)).  The larger cases exceed one wave of 148 CTAs x 2 slots, so the
    persistent loop, its barrier phases, the stage / staging reuse and the ragged last spatial group are exercised."""
    J, C = 17, 512
    eng = Engine(F, max_clips=B, gemm_mode=gemm_mode)
    qkv = _rand((B * F * J, 3 * C), 70 + F, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    ref = eng.op_attention(qkv.cuda(), B, spatial, _lib.ATTN_SIMT).cpu()
    hi, second = eng.debug_attention_operand(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT)
    eng.close()
    hi = hi.float().cpu()
    assert torch.isfinite(hi).all()
    assert (hi - ref).abs().max().item() < 4e-3 + 2 ** -10 * ref.abs().max().item()
    if gemm_mode == _lib.GEMM_TC_SPLIT3:
        lo = second.view(torch.float16).float().cpu()
        assert (hi + lo - ref).abs().max().item() < 4e-3
    else:
        a8 = second[:, :C].view(torch.float8_e5m2).float().cpu() * 256.0
        lo8 = second[:, C:].view(torch.float8_e5m2).float().cpu() / 16.0
        assert (a8 - ref).abs().max().item() < 4e-3 + 0.13 * ref.abs().max().item()
        assert ((a8 - ref).abs() <= 0.126 * ref.abs() + 4e-3).all()
        assert (hi + lo8 - ref).abs().max().item() < 4e-3
        # lo is the residual of THIS kernel's hi: |lo8 - (x - hi)| <= 12.5 % of one fp16 half-ulp of x
        assert (lo8.abs() <= 2 ** -11 * hi.abs() * 1.13 + 1e-7).all()


def _decode_f4c(second, T, C):
    """[T*C] c4 bytes + [T*C/16] row-major scale bytes -> (P, Q) fp32 [T, C]: nibble value x 2^(scale - 127)."""
    c4 = second.reshape(-1)[:T * C].view(T, C).cpu().to(torch.int32)
    sf = second.reshape(-1)[T * C:T * C + T * C // 16].view(T, C // 16).cpu().to(torch.int32)
    lut = torch.tensor([0, .5, 1, 1.5, 2, 3, 4, 6, -0., -.5, -1, -1.5, -2, -3, -4, -6])
    nib = torch.stack([c4 & 15, c4 >> 4], dim=-1).reshape(T, 2 * C)           # element 2i = low nibble of byte i
    val = lut[nib]
    scale = torch.exp2(sf.float() - 127.0).repeat_interleave(32, dim=1)          # [T, 2C]
    return (val * scale)[:, :C], (val * scale)[:, C:], sf


@pytest.mark.parametrize("F,B,spatial", [(243, 5, False), (81, 6, False), (129, 3, False), (65, 4, False), (256, 2, False),
                                         (243, 5, True), (27, 40, True), (7, 17, True), (1, 1, True), (27, 40, False),
                                         (64, 2, False), (9, 3, False)])
def test_attention_operand_f4c(F, B, spatial):
    """The attention kernels' output in the FMT_F4C operand format (block-scaled e2m1 images of x and x - hi + ue8m0
    scale bytes written straight into the scale-factor atoms) against the CUDA-core fp32 kernel: hi, hi + Q, and P to
    the quantisation step of its block scale; every scale byte must be the smallest power of two that keeps the block
    maximum <= 6.  All shapes run the tcgen05 kernel's own epilogue: ragged last spatial group, rows beyond F clipped,
    and the packed temporal mode (F <= 64: the scale bytes of row r = f G + jj go to token (f, j0 + jj))."""
    J, C = 17, 512
    eng = Engine(F, max_clips=B, gemm_mode=_lib.GEMM_TC_F4C)
    qkv = _rand((B * F * J, 3 * C), 70 + F, 1.5)
    qkv[:, :2 * C] = qkv[:, :2 * C].half().float()
    T = B * F * J
    ref = eng.op_attention(qkv.cuda(), B, spatial, _lib.ATTN_SIMT).cpu()
    hi, second = eng.debug_attention_operand(qkv.cuda(), B, spatial, _lib.ATTN_DEFAULT)
    eng.close()
    hi = hi.float().cpu()
    P, Q, sf = _decode_f4c(second, T, C)
    assert torch.isfinite(hi).all()
    assert (hi - ref).abs().max().item() < 4e-3 + 2 ** -10 * ref.abs().max().item()
    assert (hi + Q - ref).abs().max().item() < 4e-3
    # scale bytes: block maximum of the kernel's own x ~ ref (4e-3) must land in (3, 6] (or the block is ~0)
    blk = ref.view(T, C // 32, 32).abs().amax(-1)
    s_p = torch.exp2(sf[:, :C // 32].float() - 127.0)
    ratio = blk / s_p
    ok = (ratio <= 6.0 * 1.02) & ((ratio > 3.0 / 1.02) | (blk < 1e-2))     # the kernel's own x is within 4e-3 of ref
    assert ok.all(), f"{(~ok).sum().item()} scale bytes out of range"
    # P = q4(x): within one quantisation step of the block's grid (<= 1 x scale at the top of the range)
    step = s_p.repeat_interleave(32, dim=1)
    assert ((P - ref).abs() <= 1.0 * step * 1.01 + 4e-3).all()
    assert (P - ref).abs().mean().item() < 0.15 * ref.abs().mean().item() + 1e-3      # measured: 0.117
    # Q = q4(x - hi): |x - hi| <= half an fp16 ulp of x; rounding onto the e2m1 grid moves a value up by at most 4/3
    assert (Q.abs() <= 2 ** -11 * hi.abs() * 1.35 + 1e-7).all()


def test_window_gather_scatter_golden(golden):
    """Device windowing (d3d_window_gather / d3d_window_scatter) against the reference generator's windows, bit for
    bit: 2D slices, flipped copies, and the masked write-back of a prediction tensor into packed frame order."""
    from diff3dhpe_b200 import evaluate
    g = golden("windows_f9")
    F, lens = int(g["F"]), g["lens"].tolist()
    eng = Engine(F, max_clips=2)
    ws, fv, _ = evaluate.plan_windows(lens, F)
    x, xf = eng.window_gather(torch.from_numpy(g["seq2d"]).cuda(), ws.cuda(), synthetic.H36M_JOINTS_LEFT,
                              synthetic.H36M_JOINTS_RIGHT)
    assert np.array_equal(x.cpu().numpy(), g["x2d"]) and np.array_equal(xf.cpu().numpy(), g["x2d_flip"])
    pred = _rand((ws.numel(), F, 17, 3), 90)
    out = torch.full((sum(lens), 17, 3), float("nan"), device="cuda")
    eng.window_scatter(pred.cuda(), ws.cuda(), fv.cuda(), out)
    ref = torch.full((sum(lens), 17, 3), float("nan"))
    for w in range(ws.numel()):
        m = torch.from_numpy(g["mask"][w])
        ref[int(ws[w]):int(ws[w]) + F][m] = pred[w][m]
    eng.close()
    assert not torch.isnan(ref).any() and torch.equal(out.cpu(), ref)


def test_window_gather_scatter_large():
    """240 sequences x 2250 frames (the cfg5 sweep), F = 243: gather equals torch indexing, scatter(gather(x)) is the
    identity on every frame (each frame is owned by exactly one window)."""
    from diff3dhpe_b200 import evaluate
    F, n_seq, n = 243, 24, 2250
    eng = Engine(F, max_clips=1)
    ws, fv, _ = evaluate.plan_windows([n] * n_seq, F)
    seq = _rand((n_seq * n, 17, 2), 91).cuda()
    x, xf = eng.window_gather(seq, ws.cuda(), synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT)
    idx = (ws.cuda()[:, None] + torch.arange(F, device="cuda")[None]).reshape(-1)
    ref = seq[idx].view(-1, F, 17, 2)
    assert torch.equal(x, ref) and torch.equal(xf, synthetic.flip_2d(ref))
    seq3 = _rand((n_seq * n, 17, 3), 92).cuda()
    pred = seq3[idx].view(-1, F, 17, 3).contiguous()
    out = torch.zeros_like(seq3)
    eng.window_scatter(pred, ws.cuda(), fv.cuda(), out)
    eng.close()
    assert torch.equal(out, seq3)


def test_pose_metrics_golden(golden):
    """d3d_pose_metrics_accumulate (MPJPE, N-MPJPE, P-MPJPE with a Jacobi 3x3 SVD, velocity error) against the
    reference's common/loss.py values; then with a frame selection (the masked frames of evaluate()) against the oracle
    on the compacted arrays, and accumulated over two calls."""
    g = golden("metrics")
    eng = Engine(9, max_clips=1)
    pred, gt = torch.from_numpy(g["pred"]).cuda(), torch.from_numpy(g["gt"]).cuda()
    acc = torch.zeros(6, dtype=torch.float64, device="cuda")
    eng.pose_metrics_accumulate(pred, gt, acc)
    e1, e2, e3, ev = Engine.pose_metrics(acc)
    assert abs(e1 - float(g["mpjpe"])) < 2e-7 and abs(e3 - float(g["n_mpjpe"])) < 2e-7
    assert abs(e2 - float(g["p_mpjpe"])) < 2e-7 and abs(ev - float(g["velocity"])) < 2e-7
    assert acc[3].item() == 300 * 17 and acc[5].item() == 300
    sel = torch.tensor([i for i in range(300) if i % 7 != 3], dtype=torch.int64)
    acc2 = torch.zeros(6, dtype=torch.float64, device="cuda")
    eng.pose_metrics_accumulate(pred, gt, acc2, sel[:100].cuda().contiguous())
    eng.pose_metrics_accumulate(pred, gt, acc2, sel[100:].cuda().contiguous())
    eng.close()
    p, t = g["pred"][sel.numpy()], g["gt"][sel.numpy()]
    tp, tg = torch.from_numpy(p).unsqueeze(1), torch.from_numpy(t).unsqueeze(1)
    e1, e2, e3, _ = Engine.pose_metrics(acc2)
    assert abs(e1 - oracle.mpjpe(tp, tg).item()) < 2e-7 and abs(e3 - oracle.n_mpjpe(tp, tg).item()) < 2e-7
    assert abs(e2 - oracle.p_mpjpe(p, t)) < 2e-7
    # velocity: per call (np.diff inside one batch) and weighted by the batch's frame count, as evaluate() does
    # (RUN:610-614: epoch_loss_3d_vel += N_b * mean_velocity_error(batch); divided by sum N_b)
    n_a, n_b = 100, sel.numel() - 100
    v = (oracle.mean_velocity_error(p[:n_a], t[:n_a]) * n_a + oracle.mean_velocity_error(p[n_a:], t[n_a:]) * n_b) / (n_a + n_b)
    assert abs(Engine.pose_metrics(acc2)[3] - v) < 1e-6 and acc2[5].item() == n_a + n_b


def test_time_table_golden(golden):
    g = golden("denoise_f27_b3")
    eng = Engine(27, max_clips=3)
    eng.load_state_dict(synthetic.make_model(27).state_dict())
    tab = eng.op_time_table([float(t) for t in g["t"]]).cpu().numpy()
    eng.close()
    assert np.abs(tab - g["time_table"]).max() < 2e-5


@pytest.mark.parametrize("gemm_mode", [_lib.GEMM_SIMT_FP32, _lib.GEMM_TC_SPLIT3, _lib.GEMM_TC_F8C, _lib.GEMM_SIMT_F8C,
                                       _lib.GEMM_TC_F4C, _lib.GEMM_SIMT_F4C])
def test_residual_stream_after_blocks_golden(golden, gemm_mode):
    """Residual stream after STE block 0 and TTE block 0 (sub-sampled) against the imported reference."""
    g = golden("denoise_f27_b3")
    eng = Engine(27, max_clips=3, gemm_mode=gemm_mode)
    eng.load_state_dict(synthetic.make_model(27).state_dict())
    x2d, _ = synthetic.make_inputs(3, 27)
    y_T, _ = synthetic.make_noise(3, 27, 1)
    x5 = torch.cat([x2d, y_T], -1).cuda()
    t = torch.tensor(g["t"], dtype=torch.long).cuda()
    x1 = eng.debug_forward_blocks(x5, t, 1).cpu().numpy()[::8]
    x2 = eng.debug_forward_blocks(x5, t, 2).cpu().numpy()[::8]
    eng.close()
    # q, k (and P, V inside P.V) are fp16 in the attention kernels: 1e-3-level effect on a stream of magnitude ~5
    assert np.abs(x1 - g["x_after_1"]).max() < 4e-3
    assert np.abs(x2 - g["x_after_2"]).max() < 4e-3


def test_tta_merge_3dhp_joint_lists_golden(eng27, golden):
    """The 3DHP evaluate()'s flip-TTA tail (RUN3:522-529) with the MPI-INF-3DHP joint lists
    (common/mpiinf3dhp_dataset.py:17-18), bit for bit against the reference's own index arithmetic."""
    g = golden("tta_tail_3dhp")
    assert g["left"].tolist() == synthetic.MPI3DHP_JOINTS_LEFT and g["right"].tolist() == synthetic.MPI3DHP_JOINTS_RIGHT
    y, yf = torch.from_numpy(g["y"]).cuda(), torch.from_numpy(g["yf"]).cuda()
    merged = eng27.tta_merge(y, yf, synthetic.MPI3DHP_JOINTS_LEFT, synthetic.MPI3DHP_JOINTS_RIGHT, float(g["scale"]))
    assert np.array_equal(merged.cpu().numpy(), g["merged"])
    # the H36M lists on the same tensors give a different answer (the lists are not interchangeable)
    other = eng27.tta_merge(y, yf, synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT, float(g["scale"]))
    assert not np.array_equal(other.cpu().numpy(), g["merged"])


def test_tta_merge_and_mpjpe_golden(eng27, golden):
    g = golden("tta_tail")
    y, yf, gt = (torch.from_numpy(g[k]).cuda() for k in ("y", "yf", "gt"))
    merged = eng27.tta_merge(y, yf, synthetic.H36M_JOINTS_LEFT, synthetic.H36M_JOINTS_RIGHT, float(g["scale"]))
    assert np.array_equal(merged.cpu().numpy(), g["merged"])           # bit-exact: same fp32 op order
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    eng27.mpjpe_accumulate(merged, gt, acc)
    assert acc[1].item() == 3 * 9 * 17
    assert abs(acc[0].item() / acc[1].item() - float(g["mpjpe"])) < 1e-6
    mask = torch.zeros(27, dtype=torch.uint8, device="cuda")
    mask[::2] = 1
    acc.zero_()
    eng27.mpjpe_accumulate(merged, gt, acc, mask)
    ref = torch.norm(merged - gt, dim=-1).reshape(27, 17)[mask.bool()].double()
    assert acc[1].item() == ref.numel() and abs(acc[0].item() - ref.sum().item()) < 1e-4
