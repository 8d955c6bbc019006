"""Drop-in for the reference's `GaussianDiffusion` wrapper (seq2seq variant).

Same constructor and `forward` signature, same registered buffers (so checkpoints and `evaluate()` in
RUN:535-654 work unchanged) as
`common/conditional_diffusion_ddim_normal_directPredict_variableLoss_both_crossFrames.py:99-183, 421-449`.
The DDIM loop (DIFF:263-300) runs inside libdiff3d_b200.so as one CUDA graph; this wrapper only draws the
noise in the reference's order and hands raw device pointers across the C ABI.
"""
from __future__ import annotations

import math
from contextlib import contextmanager

import torch
import torch.nn.functional as F
from torch import nn

from .model import _MasterRef, _SharedWithReplicas


def _betas(name: str, timesteps: int) -> torch.Tensor:
    """fp64 beta schedules of DIFF:52-81."""
    if name == "linear":
        return torch.linspace(1e-4, 0.02, timesteps, dtype=torch.float64)
    steps = timesteps + 1
    if name == "cosine":
        x = torch.linspace(0, timesteps, steps, dtype=torch.float64)
        arg = x / timesteps
    elif name == "logcosine":
        x = torch.logspace(0, 2, steps, dtype=torch.float64)
        arg = x / 1e-1 / timesteps
    else:
        raise ValueError(f"unknown beta schedule {name}")
    s = 0.008
    ac = torch.cos((arg + s) / (1 + s) * math.pi * 0.5) ** 2
    ac = ac / ac[0]
    return torch.clip(1 - (ac[1:] / ac[:-1]), 0, 0.999)


class GaussianDiffusion(_SharedWithReplicas, nn.Module):
    def __init__(self, model, timesteps=100, sampling_timesteps=20, loss_type='l1', conditional=True,
                 clip_denoised=False, beta_schedule='cosine', p2_loss_weight_gamma=0., p2_loss_weight_k=1,
                 ddim_sampling_eta=0., clipLoss=False):
        super().__init__()
        if not conditional:
            raise ValueError("only the conditional sampler (2D keypoints -> 3D) is implemented")
        self.model = model
        self.conditional = conditional
        self.clip_denoised = clip_denoised
        self.clipLoss = clipLoss
        self.loss_type = loss_type

        betas = _betas(beta_schedule, timesteps)
        alphas = 1. - betas
        ac = torch.cumprod(alphas, dim=0)
        ac_prev = F.pad(ac[:-1], (1, 0), value=1.)
        self.sqrt_alphas_cumprod_prev = torch.sqrt(F.pad(ac, (1, 0), value=1.))
        self.num_timesteps = int(betas.shape[0])
        self.sampling_timesteps = sampling_timesteps if sampling_timesteps is not None else self.num_timesteps
        assert self.sampling_timesteps <= self.num_timesteps
        self.is_ddim_sampling = self.sampling_timesteps < self.num_timesteps
        self.ddim_sampling_eta = ddim_sampling_eta

        post_var = betas * (1. - ac_prev) / (1. - ac)
        bufs = {                                                     # DIFF:151-183, fp64 -> fp32
            'betas': betas, 'alphas_cumprod': ac, 'alphas_cumprod_prev': ac_prev,
            'sqrt_recip_alphas': torch.sqrt(1.0 / alphas),
            'sqrt_alphas_cumprod': torch.sqrt(ac), 'sqrt_one_minus_alphas_cumprod': torch.sqrt(1. - ac),
            'log_one_minus_alphas_cumprod': torch.log(1. - ac), 'sqrt_recip_alphas_cumprod': torch.sqrt(1. / ac),
            'sqrt_recipm1_alphas_cumprod': torch.sqrt(1. / ac - 1),
            'posterior_variance': post_var,
            'posterior_log_variance_clipped': torch.log(post_var.clamp(min=1e-20)),
            'posterior_mean_coef1': betas * torch.sqrt(ac_prev) / (1. - ac),
            'posterior_mean_coef2': (1. - ac_prev) * torch.sqrt(alphas) / (1. - ac),
            'p2_loss_weight': (p2_loss_weight_k + ac / (1 - ac)) ** -p2_loss_weight_gamma,
        }
        for k, v in bufs.items():
            self.register_buffer(k, v.to(torch.float32))
        self._shared = _MasterRef(self)      # nn.DataParallel replicas read the schedule's identity from the master

    # ------------------------------------------------------------------ schedule / engine plumbing
    def ddim_times(self):
        """DIFF:270-272."""
        t = torch.linspace(-1, self.num_timesteps - 1, steps=self.sampling_timesteps + 1)
        return list(reversed(t.int().tolist()))

    @contextmanager
    def _locked_engine(self, batch):
        """The model's engine for this device, locked for the caller, with this sampler's schedule set.  The schedule key
        lives in the engine's record, so it survives nn.DataParallel's per-call replicas, and is built from the master's
        `alphas_cumprod` (a replica's copy is a new tensor on every call): an unchanged schedule is never set again,
        which would drop the engine's captured graphs."""
        with self.model._engine_record(batch) as rec:
            master = self._shared.master(self)
            ac = master.alphas_cumprod
            key = (self._shared, self.sampling_timesteps, float(self.ddim_sampling_eta), bool(self.clip_denoised),
                   ac.data_ptr(), ac._version)
            if rec.schedule_key != key:
                rec.engine.set_schedule(self.ddim_times(), ac, master.sqrt_one_minus_alphas_cumprod,
                                        self.ddim_sampling_eta, self.clip_denoised)
                rec.schedule_key = key
            yield rec.engine

    def _engine(self, batch):
        with self._locked_engine(batch) as eng:
            return eng

    def draw_noise(self, target_shape, device):
        """The reference's RNG consumption for one sampler call: randn for y_T (DIFF:275), then one randn_like
        per non-final step (DIFF:293), drawn even when eta == 0."""
        y_T = torch.randn(tuple(target_shape), device=device)
        steps = [torch.randn_like(y_T) for _ in range(self.sampling_timesteps - 1)]
        return y_T, (torch.stack(steps) if (steps and self.ddim_sampling_eta != 0) else None)

    # ------------------------------------------------------------------ reference API
    @torch.no_grad()
    def ddim_sample(self, x, t, condition_x=None):
        """DIFF:251-258: one denoiser evaluation + clamp."""
        time = torch.full((x.shape[0],), t, device=x.device, dtype=torch.long)
        x_start = self.model.forward_denoise(torch.cat([condition_x, x], dim=-1), time)
        return torch.clamp(x_start, min=-1., max=1.) if self.clip_denoised else x_start

    @torch.no_grad()
    def ddim_sample_loop(self, x_in, target_shape, noise=None):
        """DIFF:263-300.  `noise=(y_T, step_noise)` makes the draws explicit (parity tests)."""
        with self._locked_engine(target_shape[0]) as eng:
            y_T, step_noise = noise if noise is not None else self.draw_noise(target_shape, eng.device)
            x_in = x_in.detach().to(device=eng.device, dtype=torch.float32).contiguous()
            return eng.ddim_sample(x_in, y_T.contiguous(), step_noise)

    @torch.no_grad()
    def ddim_sample_loop_ouput_reverse_diffusion(self, x_in, target_shape, noise=None):
        """DIFF:304-347 (sic): also returns the y_t and x_start stacks, each [B,F,J,3,S]."""
        with self._locked_engine(target_shape[0]) as eng:
            y_T, step_noise = noise if noise is not None else self.draw_noise(target_shape, eng.device)
            x_in = x_in.detach().to(device=eng.device, dtype=torch.float32).contiguous()
            return eng.ddim_sample(x_in, y_T.contiguous(), step_noise, trace=True)

    def forward_estimate_pose(self, x, target_shape, output_reverse_diffusion_3d=False):
        """DIFF:350-357."""
        if output_reverse_diffusion_3d:
            return self.ddim_sample_loop_ouput_reverse_diffusion(x, target_shape)
        return self.ddim_sample_loop(x, target_shape)

    def q_sample(self, x_start, t, noise=None):
        """DIFF:360-366."""
        noise = torch.randn_like(x_start) if noise is None else noise
        shape = (t.shape[0],) + (1,) * (x_start.dim() - 1)
        return (self.sqrt_alphas_cumprod.gather(-1, t).reshape(shape) * x_start +
                self.sqrt_one_minus_alphas_cumprod.gather(-1, t).reshape(shape) * noise)

    @torch.no_grad()
    def p_losses(self, x_start, pose_2d, noise=None):
        """DIFF:392-419 in eval mode (the `output_loss=True` branch of forward): random per-sample t, one
        denoiser call through the C ABI, weighted l1/l2 error (no autograd)."""
        b = x_start.shape[0]
        t = torch.randint(0, self.num_timesteps, (b,), device=x_start.device).long()
        noise = torch.randn_like(x_start) if noise is None else noise
        x_noisy = self.q_sample(x_start=x_start, t=t, noise=noise)
        model_out = self.model.forward_denoise(torch.cat([pose_2d, x_noisy], dim=-1).contiguous(), t)
        coef = 1.0 + self.alphas_cumprod[t].view(-1, 1, 1, 1) / self.sqrt_one_minus_alphas_cumprod[t].view(-1, 1, 1, 1)
        if self.clipLoss:
            coef = torch.clamp(coef, max=3.0)
        if self.loss_type == 'l1':
            err = F.l1_loss(model_out, x_start, reduction='none')
        elif self.loss_type == 'l2':
            err = F.mse_loss(model_out, x_start, reduction='none')
        else:
            raise ValueError(f'invalid loss type {self.loss_type}')
        return err * coef

    def forward(self, clean_3d_pose, noisy_2d_pose, noise=None, output_reverse_diffusion_3d=False, output_loss=True,
                repeat_n=1):
        """DIFF:421-449, eval branch."""
        if self.training:
            raise NotImplementedError("diff3dhpe_b200 implements the inference path only: call .eval() first "
                                      "(training stays with the reference implementation)")
        loss_pose = self.p_losses(clean_3d_pose, noisy_2d_pose, noise) if output_loss else None
        b, f, p, c = clean_3d_pose.shape
        noisy_2d_pose = noisy_2d_pose.repeat(repeat_n, 1, 1, 1)
        target_shape = list(clean_3d_pose.shape)
        target_shape[0] = target_shape[0] * repeat_n
        out = self.forward_estimate_pose(noisy_2d_pose, target_shape, output_reverse_diffusion_3d)
        if output_reverse_diffusion_3d:
            pred, rev, x0s = out
            pred = torch.mean(pred.view(repeat_n, b, f, p, -1), dim=0, keepdim=True).squeeze(0)
            return loss_pose, pred, rev, x0s
        pred = torch.mean(out.view(repeat_n, b, f, p, -1), dim=0, keepdim=True).squeeze(0)
        return loss_pose, pred
