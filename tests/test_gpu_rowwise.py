"""Row-wise kernels of the hot path (csrc/rowwise.cu: lift_ln, postnorm_add_ln, ln_split, head_ddim and their
two-rows-per-warp forms), one launch at a time through d3d_debug_rowwise, on the handle's own workspace and with the
arguments the denoiser call passes:

  - fp32 outputs (X after the lift / post-norm, the head output) against fp64 references built from the state dict;
  - the GEMM A operand they write, byte for byte, against a CPU encoder of the kernel's own fp32 LayerNorm
    (d3d_op_layernorm runs the same per-row arithmetic), and decoded against the fp64 LayerNorm;
  - the one-row and two-row forms against each other, bit for bit;
  - the quantiser's edge cases (scale-byte boundaries, e2m1 ties, -0, empty blocks) planted through zero gains;
  - the DDIM update of head_ddim against the reference's fp32 expression, bit for bit.

Every LayerNorm of the test model gets its own gain and shift and the pos-embeds / time MLP / head are far from zero,
so a kernel that reads the wrong parameter vector, pos-embed row or time vector gives a visibly different result.
The encoder self-test at the bottom runs without a GPU."""
import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from diff3dhpe_b200 import _lib, synthetic
from diff3dhpe_b200.engine import Engine
from oracle import diff3d_oracle as oracle

C = 512
J = 17
FMTS = {"F4C": _lib.GEMM_TC_F4C, "F8C": _lib.GEMM_TC_F8C, "SPLIT16": _lib.GEMM_TC_SPLIT3}

# ---------------------------------------------------------------------------------------------------------------------
# Bit-exact CPU encoder of the activation operand formats (csrc/operand.cuh), written from their definitions
# ---------------------------------------------------------------------------------------------------------------------
_E2M1_MID = np.array([0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0])      # midpoints of the grid 0, .5, 1, 1.5, 2, 3, 4, 6
_E2M1_VAL = np.array([0, .5, 1, 1.5, 2, 3, 4, 6, -0., -.5, -1, -1.5, -2, -3, -4, -6])


def e2m1_codes(v):
    """fp32 values -> e2m1 nibbles: round to nearest, ties to the even code, saturating at 6.  The sign bit is the
    input's, so a negative value that rounds to zero gives -0 (nibble 8)."""
    v = np.asarray(v, dtype=np.float32)
    a = np.abs(v).astype(np.float64)
    code = np.searchsorted(_E2M1_MID, a, side="left")           # midpoints strictly below a
    tie = (code < 7) & (_E2M1_MID[np.minimum(code, 6)] == a)
    code = np.where(tie & (code % 2 == 1), code + 1, code)
    return (code | (np.signbit(v).astype(np.int64) << 3)).astype(np.uint8)


def e5m2_codes(v):
    """fp32 values -> e5m2 bytes: round to nearest even (subnormals down to 2^-16), saturating at 57344, sign kept."""
    v = np.asarray(v, dtype=np.float32)
    a = np.abs(v).astype(np.float64)
    _, ex = np.frexp(a)                                          # a = m 2^ex, m in [0.5, 1)
    step = np.ldexp(1.0, np.maximum(ex - 1, -14) - 2)            # 2 mantissa bits; subnormal step 2^-16
    q = np.minimum(np.rint(a / step) * step, 57344.0)
    _, qx = np.frexp(q)
    e = qx - 1
    normal = q >= 2.0 ** -14
    code = np.where(normal, ((e + 15) << 2) + np.round((q / np.ldexp(1.0, e) - 1.0) * 4.0).astype(np.int64),
                    np.round(q / 2.0 ** -16).astype(np.int64))
    return (code | (np.signbit(v).astype(np.int64) << 7)).astype(np.uint8)


def ue8m0_bytes(amax):
    """Scale byte of a block: the smallest power of two s = 2^(byte - 127) with amax / s <= 6; 0 for an all-zero block.
    (Blocks whose maximum is below 6 * 2^-126 never occur in these tests; the kernels give them byte 1.)"""
    a = np.asarray(amax, dtype=np.float64)
    k = np.ceil(np.log2(np.where(a > 0, a, 1.0) / 6.0))
    k = np.where(a > 6.0 * np.exp2(k), k + 1, k)                 # exact comparisons: settle the log2 rounding
    k = np.where(a <= 3.0 * np.exp2(k), k - 1, k)
    return np.where(a > 0, np.clip(k + 127, 0, 253), 0).astype(np.uint8)


def encode_operand(y, fmt):
    """fp32 LayerNorm rows [R, 512] -> (hi fp16 bits [R,512], second bytes, scale bytes [R,32] or None):
    SPLIT16 second = fp16 lo [R,512] as bytes; F8C second = e5m2(x 2^-8) | e5m2(lo 2^4) [R,1024]; F4C second = the c4
    bytes [R,512] (q4(x) nibbles | q4(lo) nibbles, element 2i in the low nibble) with scale bytes P | Q per 32 columns."""
    y = np.ascontiguousarray(y, dtype=np.float32)
    R = y.shape[0]
    h = y.astype(np.float16)
    lo = y - h.astype(np.float32)                                # exact in fp32
    if fmt == "SPLIT16":
        return h.view(np.uint16), lo.astype(np.float16).view(np.uint8).reshape(R, 2 * C), None
    if fmt == "F8C":
        return h.view(np.uint16), np.concatenate([e5m2_codes(y * np.float32(2.0 ** -8)),
                                                  e5m2_codes(lo * np.float32(16.0))], axis=1), None
    bp = ue8m0_bytes(np.abs(y).reshape(R, C // 32, 32).max(-1))
    bq = ue8m0_bytes(np.abs(lo).reshape(R, C // 32, 32).max(-1))
    # x / scale: a power-of-two scaling, exact in fp32 for every scale these blocks get
    p = e2m1_codes(y * np.repeat(np.exp2(127.0 - bp), 32, axis=1).astype(np.float32))
    q = e2m1_codes(lo * np.repeat(np.exp2(127.0 - bq), 32, axis=1).astype(np.float32))
    nib = np.concatenate([p, q], axis=1)
    return h.view(np.uint16), (nib[:, 0::2] | (nib[:, 1::2] << 4)).astype(np.uint8), np.concatenate([bp, bq], axis=1)


def decode_f4c(c4, sf):
    """c4 bytes [R,512] + scale bytes [R,32] -> (P, Q) fp64 [R,512]: nibble value x 2^(byte - 127)."""
    nib = np.stack([c4 & 15, c4 >> 4], axis=-1).reshape(c4.shape[0], 2 * C)
    val = _E2M1_VAL[nib] * np.repeat(np.exp2(sf.astype(np.float64) - 127.0), 32, axis=1)
    return val[:, :C], val[:, C:]


def operand_parts(hi, second, fmt, rows=None):
    """The raw operand of d3d_debug_rowwise -> (hi bits, second bytes, scale bytes or None) as numpy, optionally only
    `rows` (a device index tensor) of it."""
    T = hi.shape[0]
    if fmt == "F4C":
        flat = second.reshape(-1)
        sec, sf = flat[:T * C].view(T, C), flat[T * C:T * C + T * (C // 16)].view(T, C // 16)
    else:
        sec, sf = second, None
    if rows is not None:
        hi, sec = hi[rows], sec[rows]
        sf = None if sf is None else sf[rows]
    return (hi.view(torch.int16).cpu().numpy().view(np.uint16), sec.cpu().numpy(),
            None if sf is None else sf.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# Planted quantiser edge cases: 32-column blocks (k-block index, beta values, hi values, P codes, Q codes, P byte,
# Q byte) with hand-computed encodings; columns past the listed values are 0.
# ---------------------------------------------------------------------------------------------------------------------
_TIES = [0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0, -0.25, -0.75, -1.25, -1.75, -2.5, -3.5, -5.0]
_TIE_CODES = [0, 2, 2, 4, 4, 6, 6, 8, 10, 10, 12, 12, 14, 14]
_F16 = [float(np.float16(v)) for v in (1.1, -0.3, 2.7, 0.01)]
PLANTED = [
    # amax = 6 * 2^-1 exactly: scale 2^-1, the block maximum maps to 6
    (0, [3.0, -1.5, 0.75, 2.0, -0.25, 1.0, 0.5, -3.0], None, [7, 13, 3, 6, 9, 4, 2, 15], [], 126, 0),
    # amax 2^-20 above 6 * 2^-1 (hi = 3): scale 2^0; lo = 2^-20 gets the scale 2^-22 and maps to 4
    (3, [3.0 + 2.0 ** -20, 1.0, -2.0, 0.5], [3.0, 1.0, -2.0, 0.5], [5, 2, 12, 1], [6], 127, 105),
    # e2m1 ties of the first part at scale 1, and negatives that round to -0
    (5, [6.0] + _TIES, None, [7] + _TIE_CODES, [], 127, 0),
    # e2m1 ties of the second part: x = 1 + u 2^-16, hi = 1, lo = u 2^-16 at scale 2^-16; -0.1 2^-16 rounds to -0
    (6, [1.0 + u * 2.0 ** -16 for u in [6.0] + _TIES + [-0.1]], [1.0] * 16, [6] * 16, [7] + _TIE_CODES + [8], 125, 111),
    # fp16-exact values off the e2m1 grid: the second part is all zero (scale byte 0); 5.398 rounds to 6
    (9, _F16, None, [4, 9, 7, 0], [], 126, 0),
    # an all-zero block
    (10, [], None, [], [], 0, 0),
    # amax = 6 * 2^2 exactly: scale 2^2
    (12, [24.0, -12.0, 1.0, -2.0, 7.0], None, [7, 13, 0, 9, 4], [], 129, 0),
    # amax one fp32 step below 6 * 2^-5: scale 2^-5 (byte 122); lo = -2^-26 gets 2^-28 and maps to -4
    (15, [0.1875 - 2.0 ** -26, 0.09375], [0.1875, 0.09375], [7, 5], [14], 122, 99),
]


def planted_beta():
    """512-vector with the PLANTED blocks (other columns 0) and the mask of their columns."""
    beta, mask = np.zeros(C, np.float32), np.zeros(C, bool)
    for kb, vals, *_ in PLANTED:
        beta[32 * kb:32 * kb + len(vals)] = np.asarray(vals, np.float32)
        mask[32 * kb:32 * kb + 32] = True
    return beta, mask


def check_planted(hi, sec, sf, what):
    """The planted blocks of every row of an F4C operand (numpy parts) against the hand-computed encodings."""
    errs = []
    for kb, vals, his, pc, qc, bp, bq in PLANTED:
        n = len(vals)
        want_hi = np.zeros(32, np.float16)
        want_hi[:n] = np.asarray(his if his is not None else vals, np.float16)
        want_p, want_q = np.zeros(32, np.uint8), np.zeros(32, np.uint8)
        want_p[:len(pc)], want_q[:len(qc)] = pc, qc
        cols = np.arange(32 * kb, 32 * kb + 32)
        got_p = (sec[:, cols // 2] >> (4 * (cols % 2))) & 15
        got_q = (sec[:, C // 2 + cols // 2] >> (4 * (cols % 2))) & 15
        for name, got, want in (("hi", hi[:, 32 * kb:32 * kb + 32], want_hi.view(np.uint16)), ("P nibbles", got_p, want_p),
                                ("Q nibbles", got_q, want_q), ("P scale byte", sf[:, kb], bp),
                                ("Q scale byte", sf[:, 16 + kb], bq)):
            bad = np.argwhere(got != want)
            if bad.size:
                errs.append(f"{what}: block {kb} {name}: {len(bad)} mismatches, first at {tuple(bad[0])}: "
                            f"{np.asarray(got)[tuple(bad[0])]} != {np.broadcast_to(want, got.shape)[tuple(bad[0])]}")
    return errs


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the encoder itself
# ---------------------------------------------------------------------------------------------------------------------
def test_operand_encoder_known_values():
    """Hand-computed encodings: e2m1 ties to even and -0, scale bytes at and just past 6 2^k, empty and fp16-exact
    blocks (PLANTED), e5m2 rounding / subnormals / saturation, fp16 hi / lo."""
    beta, _ = planted_beta()
    hi, sec, sf = encode_operand(np.stack([beta, -beta]), "F4C")
    assert check_planted(hi[:1], sec[:1], sf[:1], "encoder") == []
    # the negated row: same magnitudes, sign bits flipped where the value is non-zero or a negative value rounded to -0
    p_neg = (sec[1, :256, None] >> np.array([0, 4])) & 15
    p_pos = (sec[0, :256, None] >> np.array([0, 4])) & 15
    nz = beta.reshape(256, 2) != 0
    assert np.array_equal(p_neg[nz] & 7, p_pos[nz] & 7) and np.array_equal(p_neg[nz] >> 3, 1 - (p_pos[nz] >> 3))
    assert np.array_equal(sf[0], sf[1])
    assert e2m1_codes([0.0, -0.0, 0.2499, 0.2501, 6.0, 7.0, -100.0]).tolist() == [0, 8, 0, 1, 7, 7, 15]
    # e5m2: 1.25 (exact), 1.125 (tie -> 1.0), 1.375 (tie -> 1.5), 2^-16 (smallest subnormal), 2^-17 (tie -> 0),
    # 3 2^-17 (tie -> 2 2^-16), 57344 and beyond (saturate), -0
    assert e5m2_codes([1.25, 1.125, 1.375, 2.0 ** -16, 2.0 ** -17, 3 * 2.0 ** -17, 57344.0, 1e6, -0.0, -1.0]).tolist() == \
        [0x3D, 0x3C, 0x3E, 0x01, 0x00, 0x02, 0x7B, 0x7B, 0x80, 0xBC]
    assert ue8m0_bytes([0.0, 6.0, np.float32(6.0) * (1 + 2.0 ** -21), 3.0, np.nextafter(np.float32(3.0), np.float32(4)),
                        1e-3]).tolist() == [0, 127, 128, 126, 127, 127 - 12]
    h, lo, _ = encode_operand(np.array([[1.0 + 2.0 ** -12] + [0.0] * 511], np.float32), "SPLIT16")
    assert h[0, 0] == 0x3C00 and lo[0, :2].view(np.float16)[0] == np.float16(2.0 ** -12)


@pytest.mark.parametrize("fmt", list(FMTS))
def test_operand_encoder_round_trip(fmt):
    """encode -> decode (as the GEMM reads the operand) stays within one quantisation step of the input: the scale of
    its block for F4C, 3 significant bits of the 2^-11 correction for F8C, fp16 of it for SPLIT16."""
    g = torch.Generator().manual_seed(5)
    y = (torch.randn(64, C, generator=g) * torch.exp(torch.randn(64, 1, generator=g) * 2)).numpy()
    hi, sec, sf = encode_operand(y, fmt)
    x = y.astype(np.float64)
    h = hi.view(np.float16).astype(np.float64)
    if fmt == "F4C":
        P, Q = decode_f4c(sec, sf)
        sp = np.repeat(np.exp2(sf[:, :16].astype(np.float64) - 127), 32, axis=1)
        sq = np.repeat(np.exp2(sf[:, 16:].astype(np.float64) - 127), 32, axis=1)
        assert (np.abs(P - x) <= sp).all() and (np.abs(h + Q - x) <= sq).all()
        bmax = np.abs(y).reshape(64, 16, 32).max(-1)
        ratio = bmax / np.exp2(sf[:, :16].astype(np.float64) - 127)
        assert ((ratio > 3) & (ratio <= 6)).all()
    elif fmt == "F8C":
        lo8 = _e5m2_value(sec[:, C:]) / 16.0
        assert (np.abs(_e5m2_value(sec[:, :C]) * 256.0 - x) <= 2.0 ** -3 * np.abs(x) + 2.0 ** -9).all()
        assert (np.abs(h + lo8 - x) <= 2.0 ** -14 * np.abs(x) + 2.0 ** -21).all()
    else:
        lo = sec.view(np.float16).astype(np.float64)
        assert (np.abs(h + lo - x) <= 2.0 ** -22 * np.abs(x) + 2.0 ** -25).all()


def _e5m2_value(b):
    b = np.asarray(b).astype(np.int64)
    e, m = (b >> 2) & 31, b & 3
    mag = np.where(e == 0, m * 2.0 ** -16, (1 + m / 4.0) * np.exp2(e.astype(np.float64) - 15))
    return np.where(b & 0x80, -mag, mag)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
LN_NAMES = ["Spatial_norm", "Temporal_norm", "head.0"] + [f"{k}blocks.{i}.{n}" for k in ("STE", "TTE") for i in range(8)
                                                          for n in ("norm1", "norm2")]

# Bounds against fp64, about 3x the worst case measured on B200 over every shape, format and form of the tests below
# (including the cfg3-size batch)
TOL_LIFT = 1.5e-6   # X after the lift, O(1-3) values: measured 4.4e-7
TOL_X = 1.2e-5      # X after the post-norm, O(1-5) values: measured 4.0e-6 (rows of mean 30 sigma and of magnitude 1e3)
TOL_LN = 1.2e-5     # d3d_op_layernorm, the fp32 LayerNorm the operands encode, on those inputs: measured 3.8e-6
TOL_HEAD = 6.5e-6   # head output, O(1-3) values: measured 2.1e-6


def _block(b):
    return f"{'STE' if b % 2 == 0 else 'TTE'}blocks.{b // 2}."


def _state(F, seed=7, planted=False):
    """make_model(F)'s weights with every LayerNorm given its own gain (1 +- 0.3) and shift (+- 0.2), pos-embeds of
    O(0.5), per-block time Linear weights x3 and a head.1 with O(2) outputs.  planted: in addition every LayerNorm gets
    gain 0 and the PLANTED shifts on the planted blocks, so its output there is exactly those values."""
    sd = {k: v.detach().clone() for k, v in synthetic.make_model(F).state_dict().items()}
    g = torch.Generator().manual_seed(seed)
    beta_p, mask = planted_beta()
    for n in LN_NAMES:
        sd[n + ".weight"] = 1.0 + 0.3 * (2 * torch.rand(C, generator=g) - 1)
        sd[n + ".bias"] = 0.2 * (2 * torch.rand(C, generator=g) - 1)
        if planted:
            sd[n + ".weight"][torch.from_numpy(mask)] = 0.0
            sd[n + ".bias"][torch.from_numpy(mask)] = torch.from_numpy(beta_p[mask])
    sd["Spatial_pos_embed"] = 0.5 * torch.randn(sd["Spatial_pos_embed"].shape, generator=g)
    sd["Temporal_pos_embed"] = 0.5 * torch.randn(sd["Temporal_pos_embed"].shape, generator=g)
    for k in sd:
        if "blocks." in k and k.endswith("time_mlp.1.weight"):
            sd[k] = sd[k] * 3.0
    sd["head.1.weight"] = 0.1 * torch.randn(3, C, generator=g)
    sd["head.1.bias"] = 0.5 * torch.randn(3, generator=g)
    return sd


class _Case:
    """One handle (F, B, operand format) with the perturbed weights loaded, its state dict and the time table of the
    clips' timesteps (from d3d_op_time_table, itself pinned against the reference at 2e-5)."""

    def __init__(self, F, B, fmt, planted=False):
        self.F, self.B, self.fmt, self.T = F, B, fmt, B * F * J
        self.eng = Engine(F, max_clips=B, gemm_mode=FMTS[fmt])
        self.sd = _state(F, planted=planted)
        self.eng.load_state_dict(self.sd)
        t8 = [999, 1, 500, 250, 750, 100, 37, 640]
        self.t = torch.tensor([t8[i % 8] for i in range(B)], dtype=torch.int64)
        self.tab = self.eng.op_time_table([float(v) for v in t8]).cpu().double()

    def p(self, name):
        return self.sd[name].double()

    def tvec(self, b, shared, rows):
        """[R,512] time vector of block b for token rows `rows` (numpy int64)."""
        clip = np.zeros_like(rows) if shared else (rows // (self.F * J)) % 8
        return self.tab[torch.from_numpy(clip), b]

    def close(self):
        self.eng.close()


_cache = {}


def _case(F, B, fmt):
    """One live handle at a time (the tests of a (F, B, format) run consecutively)."""
    key = (F, B, fmt)
    if key not in _cache:
        for c in _cache.values():
            c.close()
        _cache.clear()
        _cache[key] = _Case(F, B, fmt)
    return _cache[key]


@pytest.fixture(scope="module", autouse=True)
def _close_cases():
    yield
    for c in _cache.values():
        c.close()
    _cache.clear()


def _ln64(x, case, name, eps):
    return Fn.layer_norm(x, (C,), case.p(name + ".weight"), case.p(name + ".bias"), eps)


def _x_rows(T, seed):
    """Residual-stream rows: random O(1.5) rows with a per-row offset, and every 8 rows one with |mean| / sigma = 30
    (two-pass variance), one constant row (variance 0: the LayerNorm is exactly beta) and one of magnitude ~1e3."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(T, C, generator=g) * 1.5 + 0.3 * torch.randn(T, 1, generator=g)
    kind = torch.arange(T) % 8
    n5, n6, n7 = int((kind == 5).sum()), int((kind == 6).sum()), int((kind == 7).sum())
    sign = torch.where(torch.arange(n5) % 2 == 0, 1.0, -1.0)[:, None]
    x[kind == 5] = sign * 30.0 + torch.randn(n5, C, generator=g)
    x[kind == 6] = torch.randn(n6, 1, generator=g).expand(n6, C)
    x[kind == 7] = 700.0 * torch.randn(n7, C, generator=g)
    return x


def _x5_rows(T, seed):
    g = torch.Generator().manual_seed(seed)
    x5 = torch.cat([(0.3 * torch.randn(T, 2, generator=g)).clamp(-1, 1), torch.randn(T, 3, generator=g)], 1)
    x5[::11] = 0.0
    return x5


def _forms(case, op, inp, block, monkeypatch):
    """(per-sample t: one row per warp), (shared t: two rows per warp), (shared t, D3D_LN_ROWS=1: one row per warp)."""
    monkeypatch.delenv("D3D_LN_ROWS", raising=False)
    per = case.eng.debug_rowwise(op, inp, case.t, False, block)
    two = case.eng.debug_rowwise(op, inp, case.t, True, block)
    monkeypatch.setenv("D3D_LN_ROWS", "1")
    one = case.eng.debug_rowwise(op, inp, case.t, True, block)
    monkeypatch.delenv("D3D_LN_ROWS")
    return {"one-row per-sample t": per, "two-row shared t": two, "one-row shared t": one}


def _maxerr(a, b):
    return (a.double() - b.double()).abs().max().item() if a.numel() else 0.0


def _bytes_diff(name, got, want):
    if got is None and want is None:
        return []
    bad = np.argwhere(got != want)
    if not bad.size:
        return []
    i = tuple(bad[0])
    return [f"{name}: {len(bad)} of {got.size} differ, first at {i}: {got[i]} != {want[i]}"]


def _check_operand(case, hi, second, x_in, ln_name, eps, what, rows=None):
    """The operand the launch wrote (rows `rows` of it, device index, or all) = the CPU encoding of
    d3d_op_layernorm(x_in) bit for bit; decoded, it lies within one quantisation step of the fp64 LayerNorm of x_in.
    x_in: the kernel's own fp32 input rows of that LayerNorm (device, already restricted to `rows`)."""
    errs = []
    ln32 = case.eng.op_layernorm(x_in.contiguous(), case.sd[ln_name + ".weight"].to(x_in.device),
                                 case.sd[ln_name + ".bias"].to(x_in.device), eps).cpu()
    ref = _ln64(x_in.cpu().double(), case, ln_name, eps)
    e_ln = _maxerr(ln32, ref)
    if not e_ln < TOL_LN:
        errs.append(f"{what}: d3d_op_layernorm vs fp64 {e_ln:.3e}")
    got = operand_parts(hi, second, case.fmt, rows)
    want = encode_operand(ln32.numpy(), case.fmt)
    for name, g_, w_ in zip(("hi", "second", "scale bytes"), got, want):
        errs += _bytes_diff(f"{what}: operand {name}", g_, w_)
    # decoded: guards against an encoder error that mirrors a kernel error
    r = ref.numpy()
    h = got[0].view(np.float16).astype(np.float64)
    if case.fmt == "F4C":
        P, Q = decode_f4c(got[1], got[2])
        sp = np.repeat(np.exp2(got[2][:, :16].astype(np.float64) - 127), 32, axis=1)
        sq = np.repeat(np.exp2(got[2][:, 16:].astype(np.float64) - 127), 32, axis=1)
        ok = (np.abs(h + Q - r) <= sq + TOL_LN).all() and (np.abs(P - r) <= sp + TOL_LN).all()
    elif case.fmt == "F8C":
        lo = _e5m2_value(got[1][:, C:]) / 16.0
        ok = (np.abs(h + lo - r) <= 2.0 ** -14 * np.abs(r) + TOL_LN).all()
    else:
        ok = (np.abs(h + got[1].view(np.float16).astype(np.float64) - r) <= 2.0 ** -22 * np.abs(r) + TOL_LN).all()
    if not ok:
        errs.append(f"{what}: decoded operand outside one quantisation step of the fp64 LayerNorm")
    return errs


def _check_forms_equal(runs, fmt, what):
    """The two-row kernel and the one-row kernel on the same (shared) time vector: every output bit equal."""
    (out2, hi2, sec2), (out1, hi1, sec1) = runs["two-row shared t"], runs["one-row shared t"]
    errs = []
    if out2 is not None and not torch.equal(out2.view(torch.int32), out1.view(torch.int32)):
        errs.append(f"{what}: two-row != one-row (fp32 output)")
    if hi2 is not None:
        for name, a, b in zip(("hi", "second", "scale bytes"), operand_parts(hi2, sec2, fmt), operand_parts(hi1, sec1, fmt)):
            errs += _bytes_diff(f"{what}: two-row vs one-row operand {name}", a, b)
    return errs


SHAPES = [(1, 7), (27, 1), (81, 3), (243, 5), (256, 4)]     # T = 119 (< 128), 459 (odd), 4131 (ragged last tile), 20655
#                                                            (161 tiles, odd), 17408 (136 tiles)
OPS = ["lift", "postnorm", "norm2", "head"]


@pytest.mark.gpu
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("F,B", SHAPES)
def test_rowwise_kernel(monkeypatch, F, B, fmt, op):
    """One row-wise kernel in all its forms on one handle:
      lift     X = fusion_layer(x5) + Spatial_pos_embed[t mod J] + time vector (clip t / (J F)) ; A = norm1_0(X)
      postnorm into blocks 1 (Spatial_norm + Temporal_pos_embed[(t / J) mod F]), 2 (Temporal_norm), 15 (Spatial_norm):
               X = post(X) (+ tpos) + time vector of the block ; A = norm1 of the block (X)
      norm2    of blocks 0 and 9: A = norm2(X)
      head     out = head.1(head.0 (eps 1e-5) of Temporal_norm (eps 1e-6) of X)
    fp32 outputs against fp64 (TOL_LIFT / TOL_X / TOL_HEAD), the operand byte for byte against the CPU encoder of the
    kernel's own LayerNorm and decoded against fp64, and the two-row form against the one-row form bit for bit."""
    case = _case(F, B, fmt)
    T = case.T
    dev = case.eng.device
    rows = np.arange(T)
    errs = []
    if op == "lift":
        x5 = _x5_rows(T, 11 + F)
        runs = _forms(case, _lib.ROWWISE_LIFT, x5.to(dev), 0, monkeypatch)
        base = x5.double() @ case.p("fusion_layer.weight").T + case.p("fusion_layer.bias") + \
            case.p("Spatial_pos_embed")[0][torch.from_numpy(rows % J)]
        for form in ("one-row per-sample t", "two-row shared t"):
            out, hi, second = runs[form]
            ref = base + case.tvec(0, "shared" in form, rows)
            e = _maxerr(out.cpu(), ref)
            if not e < TOL_LIFT:
                errs.append(f"lift {form}: X vs fp64 {e:.3e}")
            errs += _check_operand(case, hi, second, out, "STEblocks.0.norm1", 1e-6, f"lift {form}")
        errs += _check_forms_equal(runs, fmt, "lift")
    elif op == "postnorm":
        x = _x_rows(T, 21 + F)
        for b in (1, 2, 15):
            runs = _forms(case, _lib.ROWWISE_POSTNORM, x.to(dev), b, monkeypatch)
            post = "Spatial_norm" if (b - 1) % 2 == 0 else "Temporal_norm"
            base = _ln64(x.double(), case, post, 1e-6)
            if b == 1:
                base = base + case.p("Temporal_pos_embed")[0][torch.from_numpy((rows // J) % F)]
            for form in ("one-row per-sample t", "two-row shared t"):
                out, hi, second = runs[form]
                ref = base + case.tvec(b, "shared" in form, rows)
                e = _maxerr(out.cpu(), ref)
                if not e < TOL_X:
                    errs.append(f"postnorm into {b} {form}: X vs fp64 {e:.3e}")
                errs += _check_operand(case, hi, second, out, _block(b) + "norm1", 1e-6, f"postnorm into {b} {form}")
            errs += _check_forms_equal(runs, fmt, f"postnorm into {b}")
    elif op == "norm2":
        x = _x_rows(T, 31 + F)
        xd = x.to(dev)
        for b in (0, 9):
            runs = _forms(case, _lib.ROWWISE_NORM2, xd, b, monkeypatch)
            for form in ("one-row per-sample t", "two-row shared t"):
                _, hi, second = runs[form]
                errs += _check_operand(case, hi, second, xd, _block(b) + "norm2", 1e-6, f"norm2 of {b} {form}")
            errs += _check_forms_equal(runs, fmt, f"norm2 of {b}")
    else:
        x = _x_rows(T, 41 + F)
        runs = _forms(case, _lib.ROWWISE_HEAD, x.to(dev), 0, monkeypatch)
        h = _ln64(_ln64(x.double(), case, "Temporal_norm", 1e-6), case, "head.0", 1e-5)
        ref = h @ case.p("head.1.weight").T + case.p("head.1.bias")
        for form in ("one-row per-sample t", "two-row shared t"):
            e = _maxerr(runs[form][0].cpu(), ref)
            if not e < TOL_HEAD:
                errs.append(f"head {form}: out vs fp64 {e:.3e}")
        errs += _check_forms_equal(runs, fmt, "head")
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", list(FMTS))
def test_rowwise_quantiser_edge_cases(monkeypatch, fmt):
    """Every LayerNorm has gain 0 on the PLANTED 32-column blocks, so its output there is exactly the planted shift:
    scale-byte boundaries (block maximum exactly 6 2^k and one fp32 step above / below), e2m1 ties of both parts, values
    that round to -0, an fp16-exact block (second-part scale byte 0) and an all-zero block.  Through lift, post-norm and
    norm2 in every form: the F4C operand against the hand-computed encodings, every format against the CPU encoder.
    F = 27, B = 1: 459 rows (odd: the two-row tail), 4 row tiles."""
    F, B = 27, 1
    case = _Case(F, B, fmt, planted=True)
    dev = case.eng.device
    T = case.T
    errs = []
    try:
        for op, name, inp, block, ln in ((_lib.ROWWISE_LIFT, "lift", _x5_rows(T, 3), 0, "STEblocks.0.norm1"),
                                         (_lib.ROWWISE_POSTNORM, "postnorm into 2", _x_rows(T, 4), 2, "STEblocks.1.norm1"),
                                         (_lib.ROWWISE_NORM2, "norm2 of 0", _x_rows(T, 5), 0, "STEblocks.0.norm2")):
            inp = inp.to(dev)
            runs = _forms(case, op, inp, block, monkeypatch)
            for form, (out, hi, second) in runs.items():
                what = f"{name} {form}"
                errs += _check_operand(case, hi, second, inp if op == _lib.ROWWISE_NORM2 else out, ln, 1e-6, what)
                if fmt == "F4C":
                    errs += check_planted(*operand_parts(hi, second, fmt), what)
            errs += _check_forms_equal(runs, fmt, name)
    finally:
        case.close()
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
def test_rowwise_cfg3_size():
    """The bench's batch (F = 243, B = 512: T = 2 115 072 rows, X offsets past 2^32 bytes) in the production form (F4C,
    one time vector for every clip: two rows per warp): lift -> post-norm into block 2 -> norm2 of block 3 and the head
    on that stream.  Checked on the first and last 512 rows and the 512 rows around rows 2^20 / 2^21 (X byte offsets 2^31
    / 2^32, operand byte offsets 2^30 / 2^31)."""
    F, B = 243, 512
    case = _Case(F, B, "F4C")
    dev = case.eng.device
    T = case.T
    assert T == 2115072
    rows = np.concatenate([np.arange(0, 512), np.arange(2 ** 20 - 256, 2 ** 20 + 256), np.arange(2 ** 21 - 256, 2 ** 21 + 256),
                           np.arange(T - 512, T)])
    rd = torch.from_numpy(rows).to(dev)
    errs = []
    try:
        g = torch.Generator(device=dev).manual_seed(9)
        x5 = torch.randn(T, 5, device=dev, generator=g)
        x5[:, :2] = (0.3 * x5[:, :2]).clamp(-1, 1)
        x1, hi, second = case.eng.debug_rowwise(_lib.ROWWISE_LIFT, x5, case.t, True, 0)
        ref = x5[rd].cpu().double() @ case.p("fusion_layer.weight").T + case.p("fusion_layer.bias") + \
            case.p("Spatial_pos_embed")[0][torch.from_numpy(rows % J)] + case.tvec(0, True, rows)
        e = _maxerr(x1[rd].cpu(), ref)
        if not e < TOL_LIFT:
            errs.append(f"lift: X vs fp64 {e:.3e}")
        errs += _check_operand(case, hi, second, x1[rd], "STEblocks.0.norm1", 1e-6, "cfg3 lift", rd)
        del x5, hi, second
        x2, hi, second = case.eng.debug_rowwise(_lib.ROWWISE_POSTNORM, x1, case.t, True, 2)
        ref = _ln64(x1[rd].cpu().double(), case, "Temporal_norm", 1e-6) + case.tvec(2, True, rows)
        e = _maxerr(x2[rd].cpu(), ref)
        if not e < TOL_X:
            errs.append(f"postnorm into 2: X vs fp64 {e:.3e}")
        errs += _check_operand(case, hi, second, x2[rd], "STEblocks.1.norm1", 1e-6, "cfg3 postnorm into 2", rd)
        del x1, hi, second
        _, hi, second = case.eng.debug_rowwise(_lib.ROWWISE_NORM2, x2, case.t, True, 3)
        errs += _check_operand(case, hi, second, x2[rd], "TTEblocks.1.norm2", 1e-6, "cfg3 norm2 of 3", rd)
        del hi, second
        out, _, _ = case.eng.debug_rowwise(_lib.ROWWISE_HEAD, x2, case.t, True, 0)
        h = _ln64(_ln64(x2[rd].cpu().double(), case, "Temporal_norm", 1e-6), case, "head.0", 1e-5)
        e = _maxerr(out[rd].cpu(), h @ case.p("head.1.weight").T + case.p("head.1.bias"))
        if not e < TOL_HEAD:
            errs.append(f"head: out vs fp64 {e:.3e}")
        del out, x2
    finally:
        case.close()
        torch.cuda.empty_cache()
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
@pytest.mark.parametrize("B,eta,clip", [(2, 0.0, True), (2, 0.5, False), (1, 0.5, True)])
def test_ddim_update_is_bit_exact(B, eta, clip):
    """head_ddim's update (literal DIFF:295-297, one rounding per torch op) with the step scalars of d3d_set_schedule
    (DIFF:287-292 in fp32): every step of the S = 9 trace equals the reference's fp32 expression evaluated by torch on
    the kernel's own x0 and previous y, bit for bit; the last step returns x0; clipping keeps x0 in [-1, 1].  B = 1 gives
    an odd row count (the two-row head's tail)."""
    F, S = 27, 9
    m = synthetic.make_model(F).cuda()
    m.max_clips_hint = B
    diff = synthetic.make_diffusion(m, sampling_timesteps=S, eta=eta, clip_denoised=clip).cuda().eval()
    x2d, _ = synthetic.make_inputs(B, F)
    y_T, steps = synthetic.make_noise(B, F, S)
    _, rev, x0s = diff.ddim_sample_loop_ouput_reverse_diffusion(
        x2d.cuda(), [B, F, J, 3], noise=(y_T.cuda(), steps.cuda() if eta != 0 else None))
    rev, x0s = rev.cpu(), x0s.cpu()
    bufs = {k: getattr(diff, k).detach().cpu() for k in ("alphas_cumprod", "sqrt_one_minus_alphas_cumprod")}
    coefs = oracle.ddim_coefficients(bufs, diff.ddim_times(), eta)
    assert len(coefs) == S and coefs[-1] is None and all(co is not None for co in coefs[:-1])
    y = y_T
    for s, co in enumerate(coefs):
        x0 = x0s[..., s]
        if co is None:
            want = x0
        else:
            noise = steps[s] if eta != 0 else torch.zeros_like(y)
            want = x0 * co["sqrt_alpha_next"] + co["c"] * ((y - co["alpha"] * x0) / co["sqrt_one_minus"]) + co["sigma"] * noise
        got = rev[..., s]
        assert torch.equal(got, want), f"step {s}: {(got - want).abs().max().item():.3e} max difference"
        y = got
    if clip:
        assert x0s.abs().max().item() <= 1.0
