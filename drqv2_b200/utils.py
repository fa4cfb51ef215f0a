"""Host-side helpers mirroring the reference's utils.py API for the agent-update path.

Only what the hot path and its caller contract need: ``schedule`` (utils.py:129-149),
``eval_mode`` (utils.py:18-30), ``to_torch`` (utils.py:48-49), ``weight_init``
(utils.py:52-61), ``soft_update_params`` (utils.py:42-45, as one fused kernel over
flat arenas when available) and ``TruncatedNormal`` (utils.py:105-126).
"""
from __future__ import annotations

import math
import re

import numpy as np
import torch
import torch.nn as nn
from torch import distributions as pyd

from . import _lib


class eval_mode:
    """Context manager switching models to eval and back (needs .training / .train())."""

    def __init__(self, *models):
        self.models = models

    def __enter__(self):
        self.prev_states = [m.training for m in self.models]
        for m in self.models:
            m.train(False)

    def __exit__(self, *args):
        for m, s in zip(self.models, self.prev_states):
            m.train(s)
        return False


def to_torch(xs, device):
    return tuple(torch.as_tensor(x, device=device) for x in xs)


def weight_init(m):
    """Orthogonal init, gain sqrt(2) for convs, zero bias — kept on the host through
    torch so that a seed reproduces the reference's parameters exactly."""
    if isinstance(m, nn.Linear):
        nn.init.orthogonal_(m.weight.data)
        if hasattr(m.bias, "data"):
            m.bias.data.fill_(0.0)
    elif isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
        nn.init.orthogonal_(m.weight.data, nn.init.calculate_gain("relu"))
        if hasattr(m.bias, "data"):
            m.bias.data.fill_(0.0)


_LINEAR = re.compile(r"linear\((.+),(.+),(.+)\)")
_STEP_LINEAR = re.compile(r"step_linear\((.+),(.+),(.+),(.+),(.+)\)")


def schedule(schdl, step):
    """Exploration-stddev schedule: a float, 'linear(init,final,T)' or
    'step_linear(init,final1,T1,final2,T2)', evaluated in float64 on the host."""
    try:
        return float(schdl)
    except ValueError:
        pass
    m = _LINEAR.match(schdl)
    if m:
        init, final, duration = (float(g) for g in m.groups())
        mix = np.clip(step / duration, 0.0, 1.0)
        return (1.0 - mix) * init + mix * final
    m = _STEP_LINEAR.match(schdl)
    if m:
        init, final1, duration1, final2, duration2 = (float(g) for g in m.groups())
        if step <= duration1:
            mix = np.clip(step / duration1, 0.0, 1.0)
            return (1.0 - mix) * init + mix * final1
        mix = np.clip((step - duration1) / duration2, 0.0, 1.0)
        return (1.0 - mix) * final1 + mix * final2
    raise NotImplementedError(schdl)


def soft_update_params(net, target_net, tau):
    """tp = tau*p + (1-tau)*tp for every parameter pair, through drq_soft_update.  On the critic / target pair of a
    DrQV2Agent(differentiable="bf16") at the agent's tau: the agent's one-launch soft update, which refreshes the target's bf16 operand
    copies with it; on other differentiable="bf16" targets the copies are re-derived before their next forward."""
    owner = target_net.__dict__.get("_bf16_owner")
    if (owner is not None and owner[1] == "critic_target" and net is owner[0].critic
            and float(tau) == float(owner[0].critic_target_tau)):
        with torch.cuda.device(owner[0]._dev):
            if owner[0]._bf16_dirty:
                owner[0].refresh()
            owner[0]._bf16.step_target()
        return
    stream = torch.cuda.current_stream().cuda_stream
    for p, tp in zip(net.parameters(), target_net.parameters()):
        if not (p.is_cuda and tp.is_cuda):
            raise RuntimeError("soft_update_params: parameters must live on a CUDA device (no CPU fallback)")
        if p.data_ptr() % 16 or tp.data_ptr() % 16:
            # unaligned views of a flat arena: the agent updates the whole arena in one
            # launch instead; per-tensor calls need 16-byte alignment
            raise RuntimeError("soft_update_params: tensors must be 16-byte aligned")
        _lib.call("drq_soft_update", p.data_ptr(), tp.data_ptr(), p.numel(), float(tau), float(1 - tau), stream)
    if getattr(target_net, "differentiable", False) == "bf16":
        target_net.refresh()


class TruncatedNormal(pyd.Normal):
    """Normal(loc, scale) whose samples are clamped to [low+eps, high-eps] with a
    straight-through gradient; ``sample(clip)`` clips the noise first."""

    def __init__(self, loc, scale, low=-1.0, high=1.0, eps=1e-6):
        super().__init__(loc, scale, validate_args=False)
        self.low, self.high, self.eps = low, high, eps

    def _clamp(self, x):
        clamped = torch.clamp(x, self.low + self.eps, self.high - self.eps)
        return x - x.detach() + clamped.detach()

    def sample(self, clip=None, sample_shape=torch.Size(), noise=None):
        shape = self._extended_shape(sample_shape)
        if noise is None:
            noise = torch.randn(shape, dtype=self.loc.dtype, device=self.loc.device)
        noise = noise * self.scale
        if clip is not None:
            noise = torch.clamp(noise, -clip, clip)
        return self._clamp(self.loc + noise)


def adam_scalars(lr, t, beta1=0.9, beta2=0.999, eps=1e-8):
    """float64 scalar math of torch.optim.Adam's step (bias corrections, step size),
    cast to the fp32 `scalars` array of drq_adam_step."""
    bc1 = 1 - beta1 ** t
    bc2 = 1 - beta2 ** t
    return np.array([1 - beta1, beta2, 1 - beta2, bc2 ** 0.5, eps, -(lr / bc1), 0.0, 0.0], dtype=np.float32)
