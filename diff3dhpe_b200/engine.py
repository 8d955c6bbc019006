"""`Engine`: a thin Python owner of one d3d_handle.  PyTorch is used here only for device memory and
streams; every computation is a call through the C ABI (include/diff3d_b200.h)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _lib


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_dev(t: torch.Tensor, device: torch.device, shape=None, dtype=torch.float32, name="tensor"):
    if not t.is_cuda or t.device != device:
        raise ValueError(f"{name} must live on {device}, got {t.device}")
    if t.dtype != dtype:
        raise ValueError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name} must have shape {tuple(shape)}, got {tuple(t.shape)}")


class Engine:
    """One handle = one device, one (F, J, depth, with_time_emb) model, workspace for `max_clips` clips."""

    def __init__(self, num_frame: int, num_joints: int = 17, embed_dim: int = 512, depth: int = 8, num_heads: int = 8,
                 mlp_hidden: int = 1024, with_time_emb: bool = True, max_clips: int = 1, device=None,
                 gemm_mode: int = _lib.GEMM_DEFAULT, attn_mode: int = _lib.ATTN_DEFAULT, use_graph: bool = True):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("diff3dhpe_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.F, self.J, self.C, self.depth = num_frame, num_joints, embed_dim, depth
        self.with_time_emb = bool(with_time_emb)
        self.max_clips = max_clips
        self.S = 0
        cfg = _lib.Config(num_frame, num_joints, embed_dim, depth, num_heads, mlp_hidden, int(with_time_emb), max_clips,
                          gemm_mode, attn_mode, self.device.index, int(use_graph))
        h = C.c_void_p()
        torch.cuda.init()
        with torch.cuda.device(self.device):
            rc = self.lib.d3d_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise RuntimeError(f"d3d_create failed (code {rc}): {_lib.last_error(None)}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.d3d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ weights / schedule
    def load_state_dict(self, sd: Dict[str, torch.Tensor], raw_names: bool = False):
        """Accepts the reference's keys, with or without 'module.' / 'model.' prefixes; schedule buffers
        (top-level keys such as 'alphas_cumprod') are skipped as RUN:226-235 does.  `raw_names=True` hands the
        checkpoint's own key strings ('module.model.STEblocks.0...') across the ABI and lets d3d_load_weights strip the
        prefixes itself.  Raises RuntimeError (code -12) when a linear weight is non-finite or outside the fp16
        operand range."""
        keep, descs = [], []
        for k, v in sd.items():
            name = k
            if name.startswith("module."):
                name = name[7:]
            if name.startswith("model."):
                name = name[6:]
            elif "." not in name and name not in ("Spatial_pos_embed", "Temporal_pos_embed"):
                continue                      # GaussianDiffusion buffers
            t = v.detach().to(dtype=torch.float32).contiguous()
            keep.append(((k if raw_names else name).encode(), t))
        arr = (_lib.TensorDesc * len(keep))()
        for i, (name, t) in enumerate(keep):
            arr[i].name = name
            arr[i].data = t.data_ptr()
            arr[i].numel = t.numel()
            arr[i].on_device = 1 if (t.is_cuda and t.device == self.device) else 0
            if t.is_cuda and t.device != self.device:
                keep[i] = (name, t.cpu())
                arr[i].data = keep[i][1].data_ptr()
        if any(t.is_cuda for _, t in keep):
            torch.cuda.synchronize(self.device)
        _lib.check(self.lib.d3d_load_weights(self.h, arr, len(keep)), self.h, "d3d_load_weights")

    def set_schedule(self, times: Sequence[int], alphas_cumprod: torch.Tensor, sqrt_one_minus: torch.Tensor,
                     eta: float, clip_denoised: bool):
        S = len(times) - 1
        ac = alphas_cumprod.detach().to("cpu", torch.float32).contiguous()
        s1m = sqrt_one_minus.detach().to("cpu", torch.float32).contiguous()
        tarr = (C.c_int32 * (S + 1))(*[int(t) for t in times])
        _lib.check(self.lib.d3d_set_schedule(self.h, S, tarr, C.cast(ac.data_ptr(), C.POINTER(C.c_float)),
                                             C.cast(s1m.data_ptr(), C.POINTER(C.c_float)), ac.numel(), float(eta),
                                             int(bool(clip_denoised))), self.h, "d3d_set_schedule")
        self.S = S

    # ------------------------------------------------------------------ hot path
    def forward_denoise(self, x5: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        B = x5.shape[0]
        _check_dev(x5, self.device, (B, self.F, self.J, 5), name="x")
        t = t.to(device=self.device, dtype=torch.int64).contiguous()
        if t.numel() != B:
            raise ValueError("time must have one entry per clip")
        out = torch.empty((B, self.F, self.J, 3), device=self.device, dtype=torch.float32)
        _lib.check(self.lib.d3d_forward_denoise(self.h, _ptr(x5), _ptr(t), _ptr(out), B, self._stream()), self.h,
                   "d3d_forward_denoise")
        return out

    def ddim_sample(self, x2d: torch.Tensor, noise0: torch.Tensor, step_noise: Optional[torch.Tensor] = None,
                    trace: bool = False):
        B = x2d.shape[0]
        _check_dev(x2d, self.device, (B, self.F, self.J, 2), name="x2d")
        _check_dev(noise0, self.device, (B, self.F, self.J, 3), name="noise0")
        if step_noise is not None:
            _check_dev(step_noise, self.device, (self.S - 1, B, self.F, self.J, 3), name="step_noise")
        y0 = torch.empty_like(noise0)
        ty = tx = None
        if trace:
            ty = torch.empty((B, self.F, self.J, 3, self.S), device=self.device, dtype=torch.float32)
            tx = torch.empty_like(ty)
        _lib.check(self.lib.d3d_ddim_sample(self.h, _ptr(x2d), _ptr(noise0), _ptr(step_noise), _ptr(y0), _ptr(ty),
                                            _ptr(tx), B, self._stream()), self.h, "d3d_ddim_sample")
        return (y0, ty, tx) if trace else y0

    def ddim_sample_host(self, x2d: torch.Tensor, noise0: torch.Tensor, step_noise: Optional[torch.Tensor],
                         y0: torch.Tensor):
        """Host (pinned) buffers in, host buffer out; synchronises the stream.  The e2e entry point."""
        B = x2d.shape[0]
        for name, t in (("x2d", x2d), ("noise0", noise0), ("y0", y0)):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous fp32 host tensor")
        _lib.check(self.lib.d3d_ddim_sample_host(self.h, _ptr(x2d), _ptr(noise0), _ptr(step_noise), _ptr(y0), B,
                                                 self._stream()), self.h, "d3d_ddim_sample_host")
        return y0

    def tta_merge(self, y: torch.Tensor, y_flip: torch.Tensor, joints_left, joints_right, scale: float = 1.0):
        _check_dev(y, self.device, name="y")
        _check_dev(y_flip, self.device, tuple(y.shape), name="y_flip")
        n = len(joints_left)
        la = (C.c_int32 * n)(*joints_left)
        ra = (C.c_int32 * n)(*joints_right)
        out = torch.empty_like(y)
        _lib.check(self.lib.d3d_tta_merge(self.h, _ptr(y), _ptr(y_flip), la, ra, n, float(scale), _ptr(out),
                                          y.shape[0] * y.shape[1], self._stream()), self.h, "d3d_tta_merge")
        return out

    def window_gather(self, seq2d: torch.Tensor, win_start: torch.Tensor, joints_left=None, joints_right=None,
                      flip: bool = True):
        """Packed sequences [N, J, 2] + first packed frame of every window -> (x2d [n_win, F, J, 2], flipped copy or
        None), the two inputs of the reference's evaluate() (nosiy_generators.py:264-276), built on the device."""
        _check_dev(seq2d, self.device, name="seq2d")
        _check_dev(win_start, self.device, dtype=torch.int64, name="win_start")
        n_win = win_start.numel()
        if n_win and int(win_start.max()) + self.F > seq2d.shape[0]:
            raise ValueError("a window reaches past the end of the packed sequences")
        x = torch.empty((n_win, self.F, self.J, 2), device=self.device, dtype=torch.float32)
        xf = torch.empty_like(x) if flip else None
        n = len(joints_left) if (flip and joints_left is not None) else 0
        la = (C.c_int32 * max(n, 1))(*(joints_left or [0])[:max(n, 1)])
        ra = (C.c_int32 * max(n, 1))(*(joints_right or [0])[:max(n, 1)])
        _lib.check(self.lib.d3d_window_gather(self.h, _ptr(seq2d), _ptr(win_start), n_win, la, ra, n, _ptr(x), _ptr(xf),
                                              self._stream()), self.h, "d3d_window_gather")
        return x, xf

    def window_scatter(self, pred: torch.Tensor, win_start: torch.Tensor, first_valid: torch.Tensor, out: torch.Tensor):
        """pred [n_win, F, J, 3] -> out [N, J, 3] in packed frame order; frames below first_valid[w] are skipped."""
        n_win = win_start.numel()
        _check_dev(pred, self.device, (n_win, self.F, self.J, 3), name="pred")
        _check_dev(win_start, self.device, (n_win,), torch.int64, "win_start")
        _check_dev(first_valid, self.device, (n_win,), torch.int32, "first_valid")
        _check_dev(out, self.device, name="out")
        _lib.check(self.lib.d3d_window_scatter(self.h, _ptr(pred), _ptr(win_start), _ptr(first_valid), n_win, _ptr(out),
                                               self._stream()), self.h, "d3d_window_scatter")
        return out

    def mpjpe_accumulate(self, pred: torch.Tensor, gt: torch.Tensor, acc: torch.Tensor,
                         frame_mask: Optional[torch.Tensor] = None):
        """acc: fp64[2] on the device: (sum of joint errors, joint count)."""
        _check_dev(pred, self.device, name="pred")
        _check_dev(gt, self.device, tuple(pred.shape), name="gt")
        _check_dev(acc, self.device, (2,), torch.float64, "acc")
        n_frames = pred.numel() // (self.J * 3)
        if frame_mask is not None:
            _check_dev(frame_mask, self.device, dtype=torch.uint8, name="frame_mask")
        _lib.check(self.lib.d3d_mpjpe_accumulate(self.h, _ptr(pred), _ptr(gt), _ptr(frame_mask), n_frames, _ptr(acc),
                                                 self._stream()), self.h, "d3d_mpjpe_accumulate")
        return acc

    def pose_metrics_accumulate(self, pred: torch.Tensor, gt: torch.Tensor, acc: torch.Tensor,
                                frame_index: Optional[torch.Tensor] = None):
        """acc: fp64[6] on the device: sums / counts of MPJPE, N-MPJPE, P-MPJPE over the frames listed in frame_index
        (None = all, in order) and the velocity error weighted per call as evaluate() weights its batches
        (RUN:610-614); one call = one batch; see include/diff3d_b200.h."""
        _check_dev(pred, self.device, name="pred")
        _check_dev(gt, self.device, tuple(pred.shape), name="gt")
        _check_dev(acc, self.device, (6,), torch.float64, "acc")
        n = pred.numel() // (self.J * 3)
        if frame_index is not None:
            _check_dev(frame_index, self.device, dtype=torch.int64, name="frame_index")
            n = frame_index.numel()
        _lib.check(self.lib.d3d_pose_metrics_accumulate(self.h, _ptr(pred), _ptr(gt), _ptr(frame_index), n, _ptr(acc),
                                                        self._stream()), self.h, "d3d_pose_metrics_accumulate")
        return acc

    @staticmethod
    def pose_metrics(acc: torch.Tensor):
        """(mpjpe, p_mpjpe, n_mpjpe, velocity) from an accumulated fp64[6], in the reference's order e1, e2, e3, ev."""
        a = acc.tolist()
        n, nv = max(a[3], 1.0), max(a[5], 1.0)
        return a[0] / n, a[2] / n, a[1] / n, a[4] / nv

    def pck_accumulate(self, pred: torch.Tensor, gt: torch.Tensor, counts: torch.Tensor, err_sum: torch.Tensor,
                       frames: torch.Tensor, thresholds: Sequence[float], frame_index: Optional[torch.Tensor] = None,
                       frame_group: Optional[torch.Tensor] = None):
        """Grouped per-joint histogram of joint errors (d3d_pck_accumulate, see include/diff3d_b200.h).  For the frames
        listed in frame_index (int64, None = all rows in order) adds to counts int64 [G, J, n_thr] the joints whose error
        ||pred - gt|| is below thresholds[k] (strict), to err_sum fp64 [G, J] the sum of the errors and to frames int64
        [G] the frames counted.  A frame's group is frame_group[row] (int32 [n_frames], None = group 0); frames of a group
        outside [0, G) are skipped.  thresholds: 1..64 finite, strictly ascending values in the poses' units (rounded to
        fp32).  Asynchronous on the current stream."""
        _check_dev(pred, self.device, name="pred")
        if tuple(pred.shape[-2:]) != (self.J, 3):
            raise ValueError(f"pred must have shape [..., {self.J}, 3], got {tuple(pred.shape)}")
        _check_dev(gt, self.device, tuple(pred.shape), name="gt")
        n_frames = pred.numel() // (self.J * 3)
        thr = [float(t) for t in thresholds]
        G = counts.shape[0] if counts.dim() == 3 else 0
        _check_dev(counts, self.device, (G, self.J, len(thr)), torch.int64, "counts")
        _check_dev(err_sum, self.device, (G, self.J), torch.float64, "err_sum")
        _check_dev(frames, self.device, (G,), torch.int64, "frames")
        n = n_frames
        if frame_index is not None:
            _check_dev(frame_index, self.device, dtype=torch.int64, name="frame_index")
            n = frame_index.numel()
        if frame_group is not None:
            _check_dev(frame_group, self.device, (n_frames,), torch.int32, "frame_group")
        arr = (C.c_float * max(len(thr), 1))(*thr)
        _lib.check(self.lib.d3d_pck_accumulate(self.h, _ptr(pred), _ptr(gt), _ptr(frame_index), _ptr(frame_group), n,
                                               arr, len(thr), G, _ptr(counts), _ptr(err_sum), _ptr(frames),
                                               self._stream()), self.h, "d3d_pck_accumulate")
        return counts, err_sum, frames

    @staticmethod
    def pck_table(counts, err_sum, frames, thresholds: Sequence[float], joints: Sequence[int], pck_threshold: float):
        """Host-side table from pck_accumulate's buffers, over the joints listed in `joints`: for every group and for all
        groups pooled (counts and frames summed, then divided) a row {'pck': 100 * share of joint errors below
        pck_threshold, 'auc': mean of that share (in %) over all thresholds, 'mpjpe': mean joint error in the poses'
        units, 'frames': frames counted}.  pck_threshold must be one of the thresholds (compared in fp32).  A row
        without frames has NaN metrics.  Returns {'all': row, 'groups': [row of group 0, 1, ...]}."""
        def host(x, dtype):
            return np.asarray(x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x, dtype=dtype)

        c, e, f = host(counts, np.int64), host(err_sum, np.float64), host(frames, np.int64)
        thr32 = np.asarray(thresholds, dtype=np.float32)
        if c.ndim != 3 or c.shape[2] != thr32.size or e.shape != c.shape[:2] or f.shape != c.shape[:1]:
            raise ValueError("counts [G, J, n_thr], err_sum [G, J] and frames [G] do not match the thresholds")
        hit = np.flatnonzero(thr32 == np.float32(pck_threshold))
        if hit.size != 1:
            raise ValueError(f"pck_threshold {pck_threshold} is not one of the thresholds")
        joints = list(joints)
        c, e = c[:, joints, :].sum(axis=1), e[:, joints].sum(axis=1)     # [G, n_thr] int64, [G] fp64

        def row(cnt, err, nf):
            n = int(nf) * len(joints)
            if n == 0:
                return {"pck": float("nan"), "auc": float("nan"), "mpjpe": float("nan"), "frames": int(nf)}
            share = 100.0 * cnt.astype(np.float64) / n
            return {"pck": float(share[hit[0]]), "auc": float(share.mean()), "mpjpe": float(err / n), "frames": int(nf)}

        return {"all": row(c.sum(axis=0), e.sum(), f.sum()), "groups": [row(c[g], e[g], f[g]) for g in range(c.shape[0])]}

    def profile_begin(self):
        _lib.check(self.lib.d3d_profile_begin(self.h), self.h, "d3d_profile_begin")

    def profile_end(self):
        """Returns {class: (total_ms, launches)} for the kernels launched since profile_begin()."""
        n = len(_lib.PROF_CLASSES)
        ms, cnt = (C.c_double * n)(), (C.c_int64 * n)()
        _lib.check(self.lib.d3d_profile_end(self.h, ms, cnt), self.h, "d3d_profile_end")
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(_lib.PROF_CLASSES)}

    def launch_count(self) -> int:
        return int(self.lib.d3d_launch_count(self.h))

    def workspace_bytes(self) -> int:
        """Device bytes owned by the handle (weights + workspace + tables; nothing is allocated on the hot path)."""
        return int(self.lib.d3d_workspace_bytes(self.h))

    # ------------------------------------------------------------------ kernel-level entry points (tests / bench)
    def op_linear(self, a, w, bias, residual=None, act=0, gemm_mode=_lib.GEMM_TC_SPLIT3):
        M, K = a.shape
        N = w.shape[0]
        out = torch.empty((M, N), device=self.device, dtype=torch.float32)
        _lib.check(self.lib.d3d_op_linear(self.h, _ptr(a), _ptr(w), _ptr(bias), _ptr(residual), _ptr(out), M, N, K,
                                          act, gemm_mode, self._stream()), self.h, "d3d_op_linear")
        return out

    def op_linear_bench(self, M, N, K, act=0, gemm_mode=_lib.GEMM_TC_SPLIT3, iters=10) -> float:
        ms = C.c_float()
        _lib.check(self.lib.d3d_op_linear_bench(self.h, M, N, K, act, gemm_mode, iters, C.byref(ms)), self.h,
                   "d3d_op_linear_bench")
        return float(ms.value)

    def op_layernorm(self, x, gamma, beta, eps):
        out = torch.empty_like(x)
        _lib.check(self.lib.d3d_op_layernorm(self.h, _ptr(x), _ptr(gamma), _ptr(beta), eps, _ptr(out),
                                             x.numel() // self.C, self._stream()), self.h, "d3d_op_layernorm")
        return out

    def op_attention(self, qkv, B, spatial, attn_mode=_lib.ATTN_DEFAULT):
        out = torch.empty((qkv.shape[0], self.C), device=self.device, dtype=torch.float32)
        _lib.check(self.lib.d3d_op_attention(self.h, _ptr(qkv), _ptr(out), B, int(spatial), attn_mode, self._stream()),
                   self.h, "d3d_op_attention")
        return out

    def debug_attention_operand(self, qkv, B, spatial, attn_mode=_lib.ATTN_DEFAULT):
        """Attention output in the raw A-operand format of the proj GEMM: (hi fp16 [T,C], second uint8 [T,2C])."""
        T = qkv.shape[0]
        hi = torch.empty((T, self.C), device=self.device, dtype=torch.float16)
        second = torch.empty((T, 2 * self.C), device=self.device, dtype=torch.uint8)
        _lib.check(self.lib.d3d_debug_attention_operand(self.h, _ptr(qkv), _ptr(hi), _ptr(second), B, int(spatial),
                                                        attn_mode, self._stream()), self.h,
                   "d3d_debug_attention_operand")
        return hi, second

    def debug_rowwise(self, op, inp, t=None, shared_t=False, block=0):
        """One row-wise kernel launch in isolation (d3d_debug_rowwise; op = _lib.ROWWISE_*).  inp: x5 [T,5] (LIFT) or the
        residual stream X [T,C]; t: [B] timesteps (LIFT / POSTNORM).  Returns (out, hi, second): out = X after the launch
        [T,C] (LIFT / POSTNORM), the head output [T,3] (HEAD) or None (NORM2); hi fp16 [T,C] and second uint8 [T,2C] = the
        A operand written (None for HEAD), in the layout of debug_attention_operand."""
        T = inp.shape[0]
        B = T // (self.F * self.J)
        _check_dev(inp, self.device, (B * self.F * self.J, 5 if op == _lib.ROWWISE_LIFT else self.C), name="inp")
        if t is not None:
            t = t.to(device=self.device, dtype=torch.int64).contiguous()
            if t.numel() != B:
                raise ValueError("t must have one entry per clip")
        out = hi = second = None
        if op != _lib.ROWWISE_NORM2:
            out = torch.empty((T, 3 if op == _lib.ROWWISE_HEAD else self.C), device=self.device, dtype=torch.float32)
        if op != _lib.ROWWISE_HEAD:
            hi = torch.empty((T, self.C), device=self.device, dtype=torch.float16)
            second = torch.empty((T, 2 * self.C), device=self.device, dtype=torch.uint8)
        _lib.check(self.lib.d3d_debug_rowwise(self.h, op, block, _ptr(inp), _ptr(t), int(bool(shared_t)), B, _ptr(out),
                                              _ptr(hi), _ptr(second), self._stream()), self.h, "d3d_debug_rowwise")
        return out, hi, second

    def op_time_table(self, t_host: Sequence[float]):
        R = len(t_host)
        arr = (C.c_float * R)(*[float(v) for v in t_host])
        out = torch.empty((R, 2 * self.depth, self.C), device=self.device, dtype=torch.float32)
        _lib.check(self.lib.d3d_op_time_table(self.h, arr, R, _ptr(out), self._stream()), self.h, "d3d_op_time_table")
        return out

    def debug_forward_blocks(self, x5, t, n_blocks):
        B = x5.shape[0]
        t = t.to(device=self.device, dtype=torch.int64).contiguous()
        out = torch.empty((B * self.F * self.J, self.C), device=self.device, dtype=torch.float32)
        _lib.check(self.lib.d3d_debug_forward_blocks(self.h, _ptr(x5), _ptr(t), B, n_blocks, _ptr(out), self._stream()),
                   self.h, "d3d_debug_forward_blocks")
        return out
