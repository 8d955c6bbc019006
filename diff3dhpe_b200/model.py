"""Drop-in for the reference's MixSTE seq2seq denoiser module.

Same constructor signature, attribute names and state-dict keys as
`common/nets/model_conditional_diffusion_mixste_s2s_grand_linLift.py:139-220`, so a reference checkpoint loads
unchanged (`load_state_dict(..., strict=False)` as in RUN:226-235) and `torch.manual_seed(s)` followed by
construction yields the same initial weights (sub-modules are created in the reference's order).  The
sub-modules are parameter containers only: `forward_denoise` (MODEL:249-257) is executed by
libdiff3d_b200.so through `Engine`.  Training is outside the scope of this package.
"""
from __future__ import annotations

import threading
import weakref
from contextlib import contextmanager
from functools import partial
from typing import Optional

import torch
import torch.nn as nn

from . import _lib
from .engine import Engine


class _AttentionParams(nn.Module):
    """Parameter holder with the keys of `Attention` (MODEL:59-71): qkv.{weight,bias}, proj.{weight,bias}."""

    def __init__(self, dim, num_heads, qkv_bias):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)


class _MlpParams(nn.Module):
    """Keys of `Mlp` (MODEL:40-48): fc1, fc2."""

    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _BlockParams(nn.Module):
    """Keys of `Block` (MODEL:92-109): norm1, attn.*, norm2, time_mlp.1.*, mlp.*  (creation order matters for
    seed-for-seed identical initialisation)."""

    def __init__(self, dim, num_heads, mlp_ratio, qkv_bias, norm_layer, time_emb_dim):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.attn = _AttentionParams(dim, num_heads, qkv_bias)
        self.norm2 = norm_layer(dim)
        self.time_mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_emb_dim, dim)) if time_emb_dim is not None else None
        self.mlp = _MlpParams(dim, int(dim * mlp_ratio))


class _MasterRef:
    """Link from a module to its master copy, shared by the master and its nn.DataParallel replicas.

    `nn.parallel.replicate` builds each replica with a shallow copy of the master's `__dict__` on every forward call,
    so an object stored there is shared by the replicas, while anything a replica writes on itself is lost after the
    call.  Replicas also hold their parameters and buffers as plain attributes (copies broadcast for this call) and
    `parameters()` / `state_dict()` of a replica are empty, so whatever must be stable across calls is read from the
    master.  The link is weak: a replica must not keep the master alive, and the master does not point at itself."""

    def __init__(self, owner: nn.Module):
        self._owner = weakref.ref(owner)

    def master(self, caller: nn.Module) -> nn.Module:
        owner = self._owner()
        return caller if owner is None else owner


class _EngineRecord:
    """One device's handle and what it was last loaded with.  `lock` serialises every use of the handle (a handle is
    not thread-safe, include/diff3d_b200.h)."""

    def __init__(self):
        self.lock = threading.RLock()
        self.engine: Optional[Engine] = None
        self.engine_key = None
        self.weights_key = None
        self.schedule_key = None        # written by GaussianDiffusion (diffusion.py)


class _EngineRegistry(_MasterRef):
    """One `_EngineRecord` per device, shared by a module and its nn.DataParallel replicas: each device's handle is
    created once and survives calls, whichever replica object runs on that device."""

    def __init__(self, owner: nn.Module):
        super().__init__(owner)
        self._lock = threading.Lock()
        self._records = {}

    def record(self, device: torch.device) -> _EngineRecord:
        with self._lock:
            rec = self._records.get(device)
            if rec is None:
                rec = self._records[device] = _EngineRecord()
            return rec

    def peek(self, device: torch.device) -> Optional[_EngineRecord]:
        with self._lock:
            return self._records.get(device)


class _SharedWithReplicas:
    """Gives every instance a fresh `_shared` object of type `_shared_type` at construction, deep copy and unpickling:
    a copy (an EMA model, say) never shares or closes the original's handles, and the handles are never pickled."""
    _shared_type = _MasterRef

    def __getstate__(self):
        state = super().__getstate__()
        state.pop("_shared", None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        self._shared = self._shared_type(self)


class ConditionalDiffusionMixSTES2SGRANDLinLift(_SharedWithReplicas, nn.Module):
    _shared_type = _EngineRegistry

    def __init__(self, num_frame=9, num_joints=17, in_chans=2, embed_dim=32, depth=4,
                 num_heads=8, mlp_ratio=2., qkv_bias=True, qk_scale=None,
                 drop_rate=0., attn_drop_rate=0., drop_path_rate=0.2, norm_layer=None, with_time_emb=True, **kwargs):
        super().__init__()
        if qk_scale is not None:
            raise ValueError("qk_scale override is not supported by the B200 kernels (head_dim**-0.5 is baked in)")
        if in_chans != 2:
            raise ValueError("in_chans must be 2 (2D keypoints)")
        self.num_frame, self.num_joints, self.embed_dim = num_frame, num_joints, embed_dim
        self.num_heads, self.mlp_ratio = num_heads, mlp_ratio
        self.block_depth = depth
        self.with_time_emb = bool(with_time_emb)

        if with_time_emb:
            time_dim = embed_dim * 2
            # index 0 of the reference Sequential is the parameter-free SinusoidalPosEmb (MODEL:166-174)
            self.time_mlp = nn.Sequential(nn.Identity(), nn.Linear(embed_dim, time_dim), nn.GELU(),
                                          nn.Linear(time_dim, time_dim))
        else:
            time_dim = None
            self.time_mlp = None
        self.fusion_layer = nn.Linear(3 + in_chans, embed_dim)
        norm_layer = norm_layer or partial(nn.LayerNorm, eps=1e-6)
        self.Spatial_pos_embed = nn.Parameter(torch.zeros(1, num_joints, embed_dim))
        self.STEblocks = nn.ModuleList([
            _BlockParams(embed_dim, num_heads, mlp_ratio, qkv_bias, norm_layer, time_dim) for _ in range(depth)])
        self.Spatial_norm = norm_layer(embed_dim)
        self.Temporal_pos_embed = nn.Parameter(torch.zeros(1, num_frame, embed_dim))
        self.TTEblocks = nn.ModuleList([
            _BlockParams(embed_dim, num_heads, mlp_ratio, qkv_bias, norm_layer, time_dim) for _ in range(depth)])
        self.Temporal_norm = norm_layer(embed_dim)
        self.head = nn.Sequential(nn.LayerNorm(embed_dim), nn.Linear(embed_dim, 3))

        # engine state (not part of the state dict): one handle per device, shared with nn.DataParallel replicas
        self._shared = _EngineRegistry(self)
        self._weights_epoch = 0
        self.gemm_mode = _lib.GEMM_DEFAULT
        self.attn_mode = _lib.ATTN_DEFAULT
        self.use_graph = True
        self.max_clips_hint = 1

    # ------------------------------------------------------------------ engine management
    def _weights_fingerprint(self):
        """From the master's parameters: a replica's broadcast copies are new tensors on every call."""
        master = self._shared.master(self)
        return (master._weights_epoch,) + tuple((p.data_ptr(), p._version) for p in master.parameters())

    def invalidate_weights(self):
        """Forces a re-upload (re-packing) of the weights at the next call.  The engine notices parameter updates through
        `(data_ptr, _version)` of every parameter, which covers optimizer steps, `load_state_dict`, `copy_`, `.to()`
        and in-place ops on the parameter itself -- but NOT writes through `.data` (`p.data.copy_(ema)`, EMA / SWA
        weight swaps), which do not bump `_version`: call this after such a write.  (A content checksum would need a
        device -> host synchronisation on every sampler call, which the hot path must not have.)  Every device's
        engine re-uploads at its next call."""
        self._weights_epoch += 1

    def _load_from_state_dict(self, *args, **kwargs):
        self._weights_epoch += 1
        return super()._load_from_state_dict(*args, **kwargs)

    @property
    def _engine(self) -> Optional[Engine]:
        """The engine of the device the parameters live on (None before the first call)."""
        try:
            rec = self._shared.peek(self._engine_device())
        except RuntimeError:            # not on a GPU: no engine
            return None
        return None if rec is None else rec.engine

    def _engine_device(self) -> torch.device:
        """The device this module (or nn.DataParallel replica) runs on: that of its parameters."""
        dev = self.fusion_layer.weight.device
        if dev.type != "cuda":
            raise RuntimeError("diff3dhpe_b200 runs on CUDA (sm_100a) only: move the module to a B200 with .cuda(); "
                               "there is no CPU fallback")
        return dev

    @contextmanager
    def _engine_record(self, batch: int):
        """Holds the lock of the record of the device this module (or replica) runs on while the caller uses its
        engine, after bringing the engine up to date (see `engine`)."""
        dev = self._engine_device()
        rec = self._shared.record(dev)
        with rec.lock:
            need = max(batch, self.max_clips_hint)
            key = (self.gemm_mode, self.attn_mode, self.use_graph)
            if rec.engine is None or rec.engine.h is None or rec.engine_key != key or rec.engine.max_clips < need:
                if rec.engine is not None:
                    rec.engine.close()
                    rec.engine = None
                mlp_hidden = int(self.embed_dim * self.mlp_ratio)
                rec.engine = Engine(self.num_frame, self.num_joints, self.embed_dim, self.block_depth, self.num_heads,
                                    mlp_hidden, self.with_time_emb, need, dev, self.gemm_mode, self.attn_mode,
                                    self.use_graph)
                rec.engine_key, rec.weights_key, rec.schedule_key = key, None, None
            fp = self._weights_fingerprint()
            if rec.weights_key != fp:
                # Uploaded from the master's parameters, the tensors the fingerprint was taken from; the engine stages
                # those of another device through the host.  A replica's copies hold the same values, but reaching them
                # relies on how torch lays replicas out, and this runs once per change of the weights, not per call.
                rec.engine.load_state_dict(dict(self._shared.master(self).state_dict()))
                rec.weights_key = fp
            yield rec

    def engine(self, batch: int = 1) -> Engine:
        """Returns the Engine for the device the parameters live on, (re)building it when the kernel modes changed, the
        required capacity grew or it was closed, and re-uploading weights when any parameter of the master changed.
        Each device keeps its own engine, shared by the module and its nn.DataParallel replicas, for as long as the
        module lives (a module moved to another device keeps the first device's engine too).  The returned engine is
        not locked: use it from one thread at a time."""
        with self._engine_record(batch) as rec:
            return rec.engine

    # ------------------------------------------------------------------ reference API
    def forward_denoise(self, x, time):
        """MODEL:249-257.  x: [B,F,J,5] fp32, time: [B] -> [B,F,J,3]."""
        if self.training:
            raise NotImplementedError("diff3dhpe_b200 implements the inference path only: call .eval() first "
                                      "(training stays with the reference implementation)")
        assert x.dim() == 4, "shape is equal to 4"
        b, f, n, _ = x.shape
        if f != self.num_frame or n != self.num_joints:
            raise ValueError(f"expected [B,{self.num_frame},{self.num_joints},5], got {tuple(x.shape)}")
        with self._engine_record(b) as rec:
            return rec.engine.forward_denoise(x.detach().to(torch.float32).contiguous(), time)

    def forward(self, x, time):
        return self.forward_denoise(x, time)
