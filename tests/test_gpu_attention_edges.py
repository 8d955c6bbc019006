"""Attention kernels (csrc/attention_tc.cu, attention_mma.cu, attention.cu) against an fp64 reference on inputs built to
expose masking and max-pass faults, with a per-element error bound.

Reference: oracle.attention_core in float64 on the kernels' own inputs -- fp16-rounded q, k and a v that is exactly
v_hi + v_lo (the pair launch_pack_qkv16 writes), so every difference is the kernels' own arithmetic.

Error model.  GRAND attention is O = (P - I) V, a difference, so the bound of element (query n, channel d) scales with
what was summed, not with |O|:

    |O - O_ref| <= c * (sum_k P_k |V_kd| + |V_nd|) + u * sum_k |V_kd| + r

  * tcgen05 (all variants) and mma.sync: P and the V operand of P.V are fp16 (v_hi only; |v_lo| <= 2^-11 |v|), the row
    sum is taken from the unrounded fp32 P, the "- V" term is exact.  Analytic ceiling 2^-10 + 2^-16 (two fp16 roundings
    plus an N-term fp32 accumulation).
  * SIMT: fp32 throughout, expf.  Analytic ceiling 2^-14 >= (2 N + 8) 2^-24 for N <= 256.
  * u: P underflow -- an fp16 P below 2^-14 is subnormal (absolute step 2^-24), so u = 2^-25 for the fp16 kernels and
    2^-149 for SIMT.  It matters only where the whole sum is tiny (an exactly-zero V row next to e^-100 weights).
  * r: the read-back of the operand, per element: SPLIT16 hi + lo: 2^-22 |hi| + 2^-25 (fp16 lo, subnormal floor);
    F8C hi + lo8: 2^-14 |hi| + 2^-21 (2 mantissa bits of e5m2, subnormal floor); F4C hi + Q: the Q quantisation step of
    the element's 32-channel block, 2^(byte - 127) (half the widest e2m1 gap).  The fp32 result of the tcgen05 kernels
    is merged from the F4C operand, so it gets the analytic F4C step, max(2^-11 blockmax|x|, 2^-25) / 3.

c is 3x the worst ratio (|O - O_ref| - r - u sum_k |V_k|) / (sum_k P_k |V_k| + |V_query|) measured on one NVIDIA B200
(1000 W power limit) over every case of this file, or the analytic ceiling where 3x would exceed it:

    class      measured    c          ceiling
    tcgen05    8.0e-4      9.92e-4    9.92e-4     (worst: magnitude family; contam 6.7e-4, peak 4.9e-4, ties 4.7e-4)
    mma.sync   7.3e-4      9.92e-4    9.92e-4     (worst: magnitude family; contam 6.7e-4, peak 4.8e-4, ties 4.7e-4)
    SIMT       3.3e-6      1.0e-5     6.10e-5     (worst: contam family)

The fp16 kernels sit at 0.8 of their ceiling: both of their roundings (P and V_hi) are reached nearly in full.  Every
input is seeded and every kernel sums in a fixed order, so the margin is not a matter of chance.

Input families (make_qkv; test_families_produce_their_logit_gaps checks them on the CPU):
  * contam: 16 of the 64 head dims carry a one-hot label (spatial: frame mod 8 + 8 x clip parity; temporal: joint mod 4
    + 4 x clip parity).  A query scores about -40 against every key it may attend and about +40 against every key that
    shares its 128-row tile but not its sequence; zero-filled keys score 0.  Any leak moves the probability to a wrong key.
  * peak: one key beats its row by 8, 30 or 100 logits, at F - 1, 0, every 32- / 64-key chunk edge and in the second half
    of a 64-key chunk (per sequence and head).  A max pass that misses it lets P overflow fp16.
  * ties: q = 0 (uniform P) in heads 0..3; two identical keys at the top of the row, in different chunks, in heads 4..7.
  * magnitude: V scaled by 2^-8, 1, 2^6 and exactly 0 (heads 0..3: the zero head gives all-zero F4C blocks); q near the
    top of fp16 (60000) in heads 4, 5 and k near it (up to 65344) in heads 6, 7: scaled logits of 10^3 .. 10^4, the row
    maximum at least 24 logits above the rest.  (A near-tie at |logit| ~ 10^4 is ill-conditioned in fp32 arithmetic:
    every logit carries |s| 2^-24 of rounding, which moves P by as much.  The model does not cover it.)

Kernels: tcgen05 (two slots; D3D_ATTN_WG2=1 for F > 64; D3D_ATTN_SLOTS=3 in the F4C single-tile modes), mma.sync
(ATTN_MMA_SYNC, and the default entry with D3D_ATTN_TC=0 / D3D_ATTN_TC_SPATIAL=0, which must give the same bits), SIMT.
Outputs: the fp32 result and the operand in all three formats (SPLIT16, F8C, F4C, the last with its scale bytes).

Runtime on one B200 (1000 W power limit): 53 s for the 44 GPU cases (one skips); the CPU tests take a few seconds."""
import functools
import math

import numpy as np
import pytest
import torch

from diff3dhpe_b200 import _lib
from diff3dhpe_b200.engine import Engine
from oracle import diff3d_oracle as oracle
from test_gpu_rowwise import ue8m0_bytes

C, J, H, HD = 512, 17, 8, 64
FAMILIES = ("contam", "peak", "ties", "magnitude")
FMTS = {"F4C": _lib.GEMM_TC_F4C, "F8C": _lib.GEMM_TC_F8C, "SPLIT16": _lib.GEMM_TC_SPLIT3}

# c per kernel class (module docstring)
BOUND_C = {"tcgen05": 2.0 ** -10 + 2.0 ** -16, "mma.sync": 2.0 ** -10 + 2.0 ** -16, "simt": 1.0e-5}
UNDERFLOW = {"tcgen05": 2.0 ** -25, "mma.sync": 2.0 ** -25, "simt": 2.0 ** -149}

TEMPORAL_PACKED_F = [1, 2, 31, 32, 33, 63, 64]
TEMPORAL_F = [65, 95, 96, 97, 127, 128, 129, 160, 161, 192, 193, 224, 225, 243, 255, 256]
# every residue of F mod 7 (the ragged last 7-frame group) and more units than one wave of 148 CTAs x 2 slots
SPATIAL_FB = [(28, 10), (22, 10), (23, 10), (24, 10), (81, 4), (243, 2), (27, 10)]


def temporal_B(F):
    """Clips per temporal case: more (clip, joint group, head) units than 148 CTAs in both modes."""
    return 4 if F <= 64 else 2


# ---------------------------------------------------------------------------------------------------------------------
# Input families
# ---------------------------------------------------------------------------------------------------------------------
def _fp16(x):
    return x.half().float()


def _exact_pair(v):
    """v -> the fp32 value v_hi + v_lo of its fp16 pair; launch_pack_qkv16 splits the result into the same pair, so the
    kernels see exactly this v."""
    h = _fp16(v)
    return h + _fp16(v - h)


def _peak_amp(delta):
    """The fp16 amplitude A with A^2 / 8 ~ delta logits."""
    return float(np.float16(math.sqrt(8.0 * delta)))


def _peak_positions(N):
    return sorted({p for p in (N - 1, 0, 31, 32, 63, 64, 127, 128, 40, 104, 176, 242) if 0 <= p < N})


def _tie_pairs(N):
    pairs = [(0, N - 1), (31, 32), (5, 69), (40, 200), (3, 11)]
    return [(a, b) for a, b in pairs if b < N and a != b] or [(0, 0)]


@functools.lru_cache(maxsize=4)
def make_qkv(family, B, F, spatial):
    """fp32 [B F J, 3C] rows (q | k | v, channel = head * 64 + d, token = (b F + f) J + j) of one family."""
    g = torch.Generator().manual_seed(1000 + 7 * F + 3 * B + 2 * int(spatial) + 101 * FAMILIES.index(family))
    shape = (B, F, J, H, HD)
    bi = torch.arange(B).view(B, 1, 1)
    fi = torch.arange(F).view(1, F, 1)
    ji = torch.arange(J).view(1, 1, J)
    pos = (ji if spatial else fi).expand(B, F, J)                 # key / query position inside its sequence
    seq = (bi * F + fi if spatial else bi * J + ji).expand(B, F, J)
    N = J if spatial else F
    v = torch.randn(shape, generator=g)
    if family == "contam":
        q = torch.zeros(shape)
        k = torch.zeros(shape)
        q[..., :48] = torch.randn(B, F, J, H, 48, generator=g) * 1.2     # legitimate logits: std 1.25
        k[..., :48] = torch.randn(B, F, J, H, 48, generator=g) * 1.2
        label = ((fi % 8) + 8 * (bi % 2)) if spatial else ((ji % 4) + 4 * (bi % 2))
        onehot = torch.nn.functional.one_hot(label.expand(B, F, J), 16).float()[:, :, :, None, :]
        k[..., 48:] = 18.0 * onehot                                   # +-18 * 18 / 8 = +-40.5 logits
        q[..., 48:] = 18.0 - 36.0 * onehot
    elif family == "peak":
        q = torch.randn(shape, generator=g) * 0.5
        k = torch.randn(shape, generator=g) * 0.5
        q[..., 63] = 0.0
        k[..., 63] = 0.0
        combos = [(p, d) for d in (8.0, 30.0, 100.0) for p in _peak_positions(N)]
        idx = (seq[..., None] * H + torch.arange(H)) % len(combos)          # [B, F, J, H]
        p_at = torch.tensor([c[0] for c in combos])[idx]
        amp = torch.tensor([_peak_amp(c[1]) for c in combos])[idx]
        q[..., 63] = amp
        k[..., 63] = torch.where(p_at == pos[..., None], amp, torch.zeros(()))
    elif family == "ties":
        q = torch.randn(shape, generator=g) * 0.5
        k = torch.randn(shape, generator=g) * 1.5
        q[..., :4, :] = 0.0                                           # heads 0..3: uniform P
        pairs = _tie_pairs(N)
        a = _peak_amp(8.0)
        q[..., 4:, 63] = a
        k[..., 4:, :] = torch.randn(B, F, J, 4, HD, generator=g) * 0.5
        k[..., 4:, 63] = 0.0
        kk = k.clone()
        for s in range(B * (F if spatial else J)):                   # two identical keys at the top of each row
            for hh in range(4, H):
                p1, p2 = pairs[(s * H + hh) % len(pairs)]
                b = s // (F if spatial else J)
                r = s % (F if spatial else J)
                t1 = (b, r, p1) if spatial else (b, p1, r)
                t2 = (b, r, p2) if spatial else (b, p2, r)
                kk[t1 + (hh, 63)] = a
                kk[t2 + (hh,)] = kk[t1 + (hh,)]
        k = kk
    elif family == "magnitude":
        q = torch.randn(shape, generator=g) * 1.5
        k = torch.randn(shape, generator=g) * 1.5
        for hh, s in enumerate((2.0 ** -8, 1.0, 2.0 ** 6, 0.0)):
            v[..., hh, :] *= s
        q[..., 4:, :] = torch.randn(B, F, J, 4, HD, generator=g) * 0.3
        k[..., 4:, :] = torch.randn(B, F, J, 4, HD, generator=g) * 0.3
        perm = torch.randperm(256, generator=g)[pos]                  # distinct per position, shared by every sequence
        sign = torch.where(torch.rand(B, F, J, 2, generator=g) < 0.5, -1.0, 1.0)
        q[..., 4:6, 0] = 60000.0 * sign                               # q near the top of fp16
        k[..., 4:6, 0] = ((perm - 128).float() * 2.0 ** -7)[..., None]   # 58.6 logits apart, |logit| <= 7500
        q[..., 6:8, 0] = sign
        k[..., 6:8, 0] = (16384.0 + 192.0 * perm.float())[..., None]  # k near the top of fp16: |logit| 2048 .. 8168
        v[..., 5, :] *= 2.0 ** 6
        v[..., 6, :] *= 2.0 ** -8
    else:
        raise ValueError(family)
    qkv = torch.cat([_fp16(q).reshape(-1, C), _fp16(k).reshape(-1, C), _exact_pair(v).reshape(-1, C)], dim=1)
    return qkv.contiguous()


def _sequences(x, B, F, spatial):
    x = x.view(B, F, J, -1)
    return x.reshape(B * F, J, -1) if spatial else x.permute(0, 2, 1, 3).reshape(B * J, F, -1)


def _tokens(y, B, F, spatial):
    return (y.reshape(B, F, J, -1) if spatial else y.reshape(B, J, F, -1).permute(0, 2, 1, 3)).reshape(B * F * J, -1)


def logits(qkv, B, F, spatial):
    """fp64 scaled logits [Bn, H, N, N] of every sequence."""
    s = _sequences(qkv.double(), B, F, spatial)
    Bn, N, _ = s.shape
    q = s[..., :C].reshape(Bn, N, H, HD).transpose(1, 2)
    k = s[..., C:2 * C].reshape(Bn, N, H, HD).transpose(1, 2)
    return (q @ k.transpose(-2, -1)) * HD ** -0.5


@functools.lru_cache(maxsize=4)
def reference(family, B, F, spatial):
    """(qkv fp32, O_ref fp64 [T, C], S = sum_k P_k |V_k| + |V_query| and A = sum_k |V_k|, fp64 [T, C])."""
    qkv = make_qkv(family, B, F, spatial)
    seqs = _sequences(qkv.double(), B, F, spatial)
    o = oracle.attention_core(seqs, H)
    Bn, N, _ = seqs.shape
    p = torch.softmax(logits(qkv, B, F, spatial), dim=-1)
    va = seqs[..., 2 * C:].reshape(Bn, N, H, HD).transpose(1, 2).abs()
    s = (p @ va + va).transpose(1, 2).reshape(Bn, N, C)
    a = va.sum(-2, keepdim=True).expand(Bn, H, N, HD).transpose(1, 2).reshape(Bn, N, C)
    return qkv, _tokens(o, B, F, spatial), _tokens(s, B, F, spatial), _tokens(a, B, F, spatial)


# ---------------------------------------------------------------------------------------------------------------------
# Checks
# ---------------------------------------------------------------------------------------------------------------------
def _blockmax(x):
    return x.abs().view(x.shape[0], C // 32, 32).amax(-1)


def _per_block(b):
    return b.repeat_interleave(32, dim=1)


def check_bound(out, ref, scale, vsum, cls, allow, what):
    """Returns a failure message or None; NaN / inf fail."""
    c = BOUND_C[cls]
    allow = allow + UNDERFLOW[cls] * vsum
    err = (out - ref).abs()
    ok = err <= c * scale + allow
    if bool(ok.all()):
        return None
    bad = ~ok
    i = int(torch.nonzero(bad)[0][0]), int(torch.nonzero(bad)[0][1])
    r = ((err - allow) / scale.clamp_min(1e-300))[bad]
    return (f"{what}: {int(bad.sum())} elements out of bound (c = {c:.2e}), worst ratio {r.max().item():.3e}; "
            f"first at {i}: out {out[i].item():.6e} ref {ref[i].item():.6e} S {scale[i].item():.3e}")


def operand_parts(hi, second, T, fmt):
    """(hi fp16 [T,C], second part bytes [T,C] (F4C c4) / [T,2C], scale bytes [T,32] int or None)."""
    if fmt == "F4C":
        flat = second.reshape(-1)
        return hi, flat[:T * C].view(T, C), flat[T * C:T * C + T * (C // 16)].view(T, C // 16)
    return hi, second, None


_LUT = torch.tensor([0, .5, 1, 1.5, 2, 3, 4, 6, -0., -.5, -1, -1.5, -2, -3, -4, -6], dtype=torch.float64)


def readback(hi, sec, sf, fmt):
    """(hi + second part as fp64 [T,C], allowance r [T,C], F4C: (P fp64, P step, Q step) per element)."""
    h = hi.float().cpu().double()
    if fmt == "SPLIT16":
        lo = sec.view(torch.float16).cpu().double()
        return h + lo, 2.0 ** -22 * h.abs() + 2.0 ** -25, None
    if fmt == "F8C":
        lo8 = sec[:, C:].view(torch.float8_e5m2).cpu().double() / 16.0
        return h + lo8, 2.0 ** -14 * h.abs() + 2.0 ** -21, None
    T = h.shape[0]
    c4 = sec.cpu().to(torch.int64)
    nib = torch.stack([c4 & 15, c4 >> 4], dim=-1).reshape(T, 2 * C)
    sfd = sf.cpu().to(torch.int64)
    step = torch.exp2(sfd.double() - 127.0)
    val = _LUT[nib] * _per_block(step)
    p_step, q_step = _per_block(step[:, :C // 32]), _per_block(step[:, C // 32:])
    return h + val[:, C:], q_step, (val[:, :C], p_step, q_step)


def check_f4c_bytes(sf, ref, scale, cls, hi, what):
    """P scale bytes equal the encoder's choice wherever the fp64 block maximum is farther from a scale boundary than
    the error bound; exactly-zero blocks (zero bound) get byte 0 in both parts; Q bytes: the smallest power of two
    s >= blockmax|x - hi| / 6 satisfies s < max(2^-11 blockmax|x|, 2^-25) / 3."""
    errs = []
    sfd = sf.cpu().to(torch.int64)
    bp = sfd[:, :C // 32].numpy()
    bq = sfd[:, C // 32:]
    amax = _blockmax(ref).numpy()
    eb = _blockmax(BOUND_C[cls] * scale).numpy()
    lo_b, hi_b = ue8m0_bytes(np.maximum(amax - eb, 0.0)), ue8m0_bytes(amax + eb)
    decided = lo_b == hi_b
    bad = decided & (bp != lo_b)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        errs.append(f"{what}: {int(bad.sum())} P scale bytes differ from the encoder (of {int(decided.sum())} decided); "
                    f"first at {i}: {bp[i]} != {lo_b[i]} (block max {amax[i]:.6e})")
    zero = (amax == 0) & (eb == 0)
    if (bq[torch.from_numpy(zero)] != 0).any():
        errs.append(f"{what}: all-zero blocks with a non-zero Q scale byte")
    hmax = _blockmax(hi.float().cpu().double())
    cap = torch.clamp(2.0 ** -11 * hmax * (1 + 2.0 ** -10), min=2.0 ** -25) / 3.0
    q_over = torch.exp2(bq.double() - 127.0) > cap
    if q_over.any():
        errs.append(f"{what}: {int(q_over.sum())} Q scale bytes above the half-ulp cap")
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# Kernel configurations
# ---------------------------------------------------------------------------------------------------------------------
def kernels(F, spatial):
    """(name, class, attn_mode, env, fmts it applies to) -- env is set around the call."""
    tc_off = {"D3D_ATTN_TC_SPATIAL" if spatial else "D3D_ATTN_TC": "0"}
    ks = [("tcgen05", "tcgen05", _lib.ATTN_DEFAULT, {}, tuple(FMTS))]
    if not spatial and F > 64:
        ks.append(("tcgen05_wg2", "tcgen05", _lib.ATTN_DEFAULT, {"D3D_ATTN_WG2": "1"}, ("F4C",)))
    if spatial or F <= 64:
        ks.append(("tcgen05_slots3", "tcgen05", _lib.ATTN_DEFAULT, {"D3D_ATTN_SLOTS": "3"}, ("F4C",)))
    ks += [("mma_sync", "mma.sync", _lib.ATTN_MMA_SYNC, {}, tuple(FMTS)),
           ("default_tc_off", "mma.sync", _lib.ATTN_DEFAULT, tc_off, tuple(FMTS)),
           ("simt", "simt", _lib.ATTN_SIMT, {}, tuple(FMTS))]
    return ks


@pytest.fixture(scope="module")
def engine():
    """Engines keyed by (F, gemm mode), shared by the tests of this module."""
    cache = {}

    def get(F, fmt, B):
        key = (F, fmt)
        e = cache.get(key)
        if e is None or e.max_clips < B:
            if e is not None:
                e.close()
            e = cache[key] = Engine(F, max_clips=B, gemm_mode=FMTS[fmt])
        return e

    yield get
    for e in cache.values():
        e.close()


def run_case(engine, monkeypatch, F, B, spatial):
    """Every family x kernel x output of one shape; returns the failure messages."""
    errs = []
    T = B * F * J
    for family in FAMILIES:
        qkv, ref, scale, vsum = reference(family, B, F, spatial)
        qd = qkv.cuda()
        f32 = {}
        for name, cls, mode, env, fmts in kernels(F, spatial):
            tag = f"{family} F={F} B={B} {'spatial' if spatial else 'temporal'} {name}"
            with monkeypatch.context() as m:
                for kk, vv in env.items():
                    m.setenv(kk, vv)
                # fp32 result (engine in the shipped F4C mode: the tcgen05 result is merged from the F4C operand)
                out = engine(F, "F4C", B).op_attention(qd, B, spatial, mode).cpu()
                f32[name] = out
                allow = 0.0
                if cls == "tcgen05":
                    allow = _per_block(torch.clamp(2.0 ** -11 * _blockmax(ref.abs() + BOUND_C[cls] * scale), min=2.0 ** -25)
                                       ) / 3.0 * (1 + 2.0 ** -8)
                msg = check_bound(out.double(), ref, scale, vsum, cls, allow, tag + " fp32")
                if msg:
                    errs.append(msg)
                for fmt in fmts:
                    hi, second = engine(F, fmt, B).debug_attention_operand(qd, B, spatial, mode)
                    hi, sec, sf = operand_parts(hi, second, T, fmt)
                    if not bool(torch.isfinite(hi.float()).all()):
                        errs.append(f"{tag} {fmt}: non-finite hi")
                        continue
                    val, r, f4 = readback(hi, sec, sf, fmt)
                    msg = check_bound(val, ref, scale, vsum, cls, r, f"{tag} {fmt} read-back")
                    if msg:
                        errs.append(msg)
                    if f4 is not None:
                        p, p_step, _ = f4
                        msg = check_bound(p, ref, scale, vsum, cls, p_step, f"{tag} F4C P = q4(x)")
                        if msg:
                            errs.append(msg)
                        errs += check_f4c_bytes(sf, ref, scale, cls, hi, f"{tag} F4C")
        # the default entry with the tcgen05 kernel switched off runs the mma.sync kernel: the same bits
        if not torch.equal(f32["default_tc_off"], f32["mma_sync"]):
            errs.append(f"{family} F={F}: default entry with tcgen05 off differs from ATTN_MMA_SYNC")
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("F", TEMPORAL_PACKED_F + TEMPORAL_F)
def test_temporal_attention_edges(engine, monkeypatch, F):
    """Temporal mode: packed tiles (F <= 64: G = 4 joints per tile up to F = 32, 2 up to 64) and the one- / two-tile
    kernel (F > 64) at every chunk boundary of softmax_row (NCH = 3 / 8 / runtime, ragged last 32-column chunk), the
    two-warpgroup split point c_split and the 64-key chunks of the mma.sync kernel."""
    errs = run_case(engine, monkeypatch, F, temporal_B(F), False)
    assert not errs, "\n".join(errs[:20])


@pytest.mark.gpu
@pytest.mark.parametrize("F,B", SPATIAL_FB)
def test_spatial_attention_edges(engine, monkeypatch, F, B):
    """Spatial mode (7 frames x 17 joints per tile, block-diagonal mask; rows 119..127 are the next group's or the next
    clip's tokens): every residue of F mod 7, more units than one wave."""
    errs = run_case(engine, monkeypatch, F, B, True)
    assert not errs, "\n".join(errs[:20])


SPLIT_CASES = [  # (F, B, spatial, attn_mode, env)
    (23, 6, True, _lib.ATTN_DEFAULT, {}),
    (27, 5, False, _lib.ATTN_DEFAULT, {}),           # packed, G = 4
    (63, 5, False, _lib.ATTN_DEFAULT, {}),           # packed, G = 2
    (243, 3, False, _lib.ATTN_DEFAULT, {}),
    (243, 3, False, _lib.ATTN_DEFAULT, {"D3D_ATTN_WG2": "1"}),
    (97, 3, False, _lib.ATTN_MMA_SYNC, {}),
    (23, 6, True, _lib.ATTN_MMA_SYNC, {}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["F4C", "F8C"])
@pytest.mark.parametrize("F,B,spatial,mode,env", SPLIT_CASES)
def test_batch_split_is_bit_identical(engine, monkeypatch, fmt, F, B, spatial, mode, env):
    """Clip b of a B-clip call equals, bit for bit, the same clip run alone (B = 1): every operand byte (hi, second
    part, scale bytes) and the fp32 result.  nn.DataParallel splits batches arbitrarily and relies on this."""
    if env.get("D3D_ATTN_WG2") and fmt != "F4C":
        pytest.skip("the two-warpgroup kernel writes the F4C operand only")
    for kk, vv in env.items():
        monkeypatch.setenv(kk, vv)
    e = engine(F, fmt, B)
    qd = make_qkv("magnitude", B, F, spatial).cuda()
    T, Tc = B * F * J, F * J
    hi, second = e.debug_attention_operand(qd, B, spatial, mode)
    full = [x.cpu() for x in operand_parts(hi, second, T, fmt) if x is not None]
    out = e.op_attention(qd, B, spatial, mode).cpu()
    for b in range(B):
        qb = qd[b * Tc:(b + 1) * Tc].contiguous()
        hb, sb = e.debug_attention_operand(qb, 1, spatial, mode)
        one = [x.cpu() for x in operand_parts(hb, sb, Tc, fmt) if x is not None]
        for name, a, o in zip(("hi", "second", "scale bytes"), full, one):
            assert torch.equal(a[b * Tc:(b + 1) * Tc].view(torch.uint8), o.view(torch.uint8)), f"clip {b}: {name}"
        ob = e.op_attention(qb, 1, spatial, mode).cpu()
        assert torch.equal(out[b * Tc:(b + 1) * Tc], ob), f"clip {b}: fp32 result"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the families produce their logit gaps
# ---------------------------------------------------------------------------------------------------------------------
def _tile_keys_spatial(B, F):
    """(group start token, number of query rows) of every spatial tile; keys are tokens [start, start + 128)."""
    out = []
    for b in range(B):
        for g in range((F + 6) // 7):
            out.append(((b * F + 7 * g) * J, 17 * min(7, F - 7 * g)))
    return out


@pytest.mark.parametrize("F,B,spatial", [(23, 3, True), (27, 3, True), (27, 2, False), (63, 2, False), (97, 1, False),
                                         (1, 2, False), (256, 1, False)])
def test_families_produce_their_logit_gaps(F, B, spatial):
    N = J if spatial else F
    T = B * F * J
    # contam: legitimate keys at -40 +- spread, keys sharing a tile but not the sequence at +40 +- spread
    qkv = make_qkv("contam", B, F, spatial).double()
    L = logits(qkv, B, F, spatial)
    assert L.max() < -28 and L.min() > -53
    q = qkv[:, :C].view(T, H, HD)
    k = torch.cat([qkv[:, C:2 * C], torch.zeros(128, C, dtype=torch.float64)]).view(T + 128, H, HD)   # zero-fill past T
    if spatial:
        for start, rows in _tile_keys_spatial(B, F):
            s = torch.einsum("rhd,khd->hrk", q[start:start + rows], k[start:start + 128]) / 8
            own = (torch.arange(rows)[:, None] // 17) == (torch.arange(128)[None] // 17)
            zero = (start + torch.arange(128)) >= T
            other = ~own & ~zero[None]
            assert s[:, other].min() > 28, "a key of another sequence in the tile does not score high"
            assert (s[:, own].max() < -28)
    else:
        G = 4 if F <= 32 else (2 if F <= 64 else 1)
        if G > 1:
            for b in range(B):
                for j0 in range(0, J, G):
                    toks = [(b * F + f) * J + j for f in range(F) for j in range(j0, min(j0 + G, J))]
                    jt = torch.tensor([j for f in range(F) for j in range(j0, min(j0 + G, J))])
                    s = torch.einsum("rhd,khd->hrk", q[toks], k[toks]) / 8
                    other = jt[:, None] != jt[None]
                    if other.any():                                  # the last group may hold one joint only
                        assert s[:, other].min() > 28
    # peak: the planted key is the row's unique maximum, delta (8 / 30 / 100) - 3 above everything else
    qkv = make_qkv("peak", B, F, spatial).double()
    L = logits(qkv, B, F, spatial)
    if N > 1:
        top2 = L.topk(2, dim=-1).values
        gap = top2[..., 0] - top2[..., 1]
        assert gap.min() > 5 and (gap > 97).any() and ((gap > 27) & (gap < 33)).any()
        am = L.argmax(-1)
        if N > 128:
            for p in (0, 31, 32, 63, 64, 127, 128, 40, N - 1):
                assert (am == p).any(), f"no row peaks at {p}"
    # ties: q = 0 rows are flat; the other rows have exactly two equal maxima
    qkv = make_qkv("ties", B, F, spatial).double()
    L = logits(qkv, B, F, spatial)
    assert torch.equal(L[:, :4], torch.zeros_like(L[:, :4]))
    if N > 1:
        top = L[:, 4:].max(-1, keepdim=True).values
        assert ((L[:, 4:] == top).sum(-1) == 2).all()
    # magnitude: V scales, an exactly-zero head, logits of 10^3 .. 10^4 with separated maxima in heads 4..7
    qkv = make_qkv("magnitude", B, F, spatial).double()
    v = qkv[:, 2 * C:].view(T, H, HD)
    assert torch.equal(v[:, 3], torch.zeros_like(v[:, 3]))
    assert v[:, 0].abs().max() < 2.0 ** -5 and v[:, 2].abs().max() > 2.0 ** 7
    L = logits(qkv, B, F, spatial)
    assert 3e3 < L[:, 4:].abs().max() < 1.1e4
    if N > 1:
        top2 = L[:, 4:].topk(2, dim=-1).values
        assert (top2[..., 0] - top2[..., 1]).min() > 22
    assert qkv[:, :C].abs().max() == 60000.0 and qkv[:, C:2 * C].abs().max() >= 16384
    assert torch.equal(qkv[:, :2 * C], _fp16(qkv[:, :2 * C].float()).double())


def test_exact_pair_is_what_the_packer_writes():
    """v = v_hi + v_lo exactly after _exact_pair, and splitting it again (fp16 hi, fp16 of the remainder, as
    launch_pack_qkv16 does) gives a pair that sums to it exactly."""
    g = torch.Generator().manual_seed(5)
    v = torch.cat([torch.randn(100000, generator=g) * s for s in (2.0 ** -8, 1.0, 2.0 ** 6)])
    w = _exact_pair(v)
    h = _fp16(w)
    lo = _fp16(w - h)
    assert torch.equal((h.double() + lo.double()), w.double())
    assert ((w - v).abs() <= 2.0 ** -22 * v.abs() + 2.0 ** -25).all()     # fp16 lo: 11 bits, subnormal step 2^-24
