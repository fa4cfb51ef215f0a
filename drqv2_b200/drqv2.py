"""DrQ-v2 agent on hand-written sm_100a CUDA kernels (libdrqv2_b200.so).

Mirrors the reference's drqv2.py API surface — ``RandomShiftsAug``, ``Encoder``,
``Actor``, ``Critic``, ``DrQV2Agent.{act, update, update_critic, update_actor, train}``
(reference drqv2.py:14-262) — so that ``cfgs/config.yaml``'s ``agent._target_`` can point
here and the reference's ``train.py`` runs unchanged.  Every tensor op of the update is
a kernel of the C ABI in ``include/drqv2_b200.h``; PyTorch only owns memory, streams
and the CUDA graph.  There is no CPU / eager-PyTorch fallback: on a machine without the
built extension or without a CUDA device these classes raise.
"""
from __future__ import annotations

import contextlib
import ctypes
import functools
import gc
import math

import numpy as np
import torch
import torch.nn as nn

import os

from . import _bf16, _lib, dist as _dist, utils
from ._lib import EPI_MASK, EPI_MASK_WIDE, EPI_NONE, EPI_RELU, PLANE, REPR_DIM, call

F32 = 4
# One slot of per-update host scalars (include/drqv2_b200.h DRQ_SCAL_SLOT): Adam scalars (utils.adam_scalars, 8 floats)
# of critic_opt at [0, 8), stddev(step) at [8], encoder_opt at [16, 24), actor_opt at [24, 32).
SCAL_SLOT = 32
SCAL_OFF = dict(critic=0, stddev=8, encoder=16, actor=24)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _on_device(fn):
    """Run a DrQV2Agent method with the agent's device current: kernels are launched on the current device and
    stream while the tensors live on self._dev (DrQV2Agent(device='cuda:1') must not need a set_device call)."""
    @functools.wraps(fn)
    def wrapped(self, *a, **kw):
        if torch.cuda.current_device() == self._dev.index:
            return fn(self, *a, **kw)
        with torch.cuda.device(self._dev):
            return fn(self, *a, **kw)
    return wrapped


def _need_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: tensor is on {t.device}; drqv2_b200 runs on CUDA only (no CPU fallback)")


def _splitk_for(m_rows, K=REPR_DIM, target_blocks=296):
    """Split-K factor for the skinny trunk GEMM (N <= 128): fill ~2 CTAs/SM of the 148 SMs."""
    mblocks = (m_rows + 63) // 64
    s0 = max(1, min(target_blocks // mblocks, K // 64))
    chunk = -(-K // s0)
    chunk = -(-chunk // 16) * 16
    return -(-K // chunk)


# ----------------------------------------------------------------------------- kernel wrappers
def _gemm(A, sa_m, sa_k, B, sb_k, sb_n, C, ldc, M, N, K, bias=0, mask=0, ldmask=0, epi=EPI_NONE,
          acc=0, batch=1, bs=(0, 0, 0, 0, 0), splitk=1):
    call("drq_gemm_f32", A, sa_m, sa_k, B, sb_k, sb_n, C, ldc, bias or None, mask or None, ldmask, M, N, K,
         epi, acc, batch, bs[0], bs[1], bs[2], bs[3], bs[4], splitk, _stream())


def _linear_fwd(x, ldx, W, b, y, ldy, M, n_out, n_in, relu, batch=1, bs=(0, 0, 0, 0, 0)):
    """y = [relu](x @ W.T + b); W is [n_out, n_in] (nn.Linear layout)."""
    _gemm(x, ldx, 1, W, 1, n_in, y, ldy, M, n_out, n_in, bias=b, epi=EPI_RELU if relu else EPI_NONE,
          batch=batch, bs=bs)


def _linear_dgrad(dy, ld_dy, W, dx, ld_dx, M, n_out, n_in, mask=0, ldmask=0, acc=0, batch=1,
                  bs=(0, 0, 0, 0, 0), w_col0=0, n_cols=None):
    """dx = dy @ W[:, w_col0:w_col0+n_cols] (optionally * (mask > 0))."""
    n_cols = n_in if n_cols is None else n_cols
    _gemm(dy, ld_dy, 1, W + F32 * w_col0, n_in, 1, dx, ld_dx, M, n_cols, n_out, mask=mask, ldmask=ldmask,
          epi=EPI_MASK if mask else EPI_NONE, acc=acc, batch=batch, bs=bs)


def _linear_wgrad(dy, ld_dy, x, ldx, dW, M, n_out, n_in, batch=1, bs=(0, 0, 0, 0, 0)):
    """dW[n_out, n_in] = dy.T @ x."""
    _gemm(dy, 1, ld_dy, x, ldx, 1, dW, n_in, n_out, n_in, M, batch=batch, bs=bs)


def _colsum(X, ld, out, M, N, batch=1, bs_x=0, bs_out=0):
    call("drq_colsum_f32", X, ld, out, M, N, batch, bs_x, bs_out, _stream())


def _trunk_fwd(feat, B, W, b, gamma, beta, Fdim, partial, h_out, ld_h, xhat=0, rstd=0):
    """Linear(39200->F) as split-K GEMM, then the fused reduce + bias + LayerNorm + tanh."""
    S = _splitk_for(B)
    _gemm(feat, REPR_DIM, 1, W, 1, REPR_DIM, partial, Fdim, B, Fdim, REPR_DIM, splitk=S,
          bs=(0, 0, B * Fdim, 0, 0))
    call("drq_ln_tanh_fwd", partial, S, B * Fdim, b, gamma, beta, h_out, ld_h, xhat or None, rstd or None,
         None, 0, B, Fdim, 1e-5, _stream())


def _encoder_fwd(obs_u8, shift, w, b, acts, feat, N, cin, pad=4):
    """conv1 (u8 + shift + normalise fused) -> conv2 -> conv3 -> conv4 (compact features).
    w/b: 4 pointers each; acts: 3 wide-plane buffers."""
    s = _stream()
    call("drq_conv1_fwd_f32", obs_u8, shift or None, w[0], b[0], acts[0], N, cin, pad, s)
    call("drq_conv3x3_fwd_f32", acts[0], w[1], b[1], acts[1], N, 39, 0, s)
    call("drq_conv3x3_fwd_f32", acts[1], w[2], b[2], acts[2], N, 37, 0, s)
    call("drq_conv3x3_fwd_f32", acts[2], w[3], b[3], feat, N, 35, 1, s)


# ----------------------------------------------------------------------------- autograd of the module API
# Encoder / Actor / Critic built with differentiable=True record these Functions, so that the reference's own
# update_critic / update_actor bodies (drqv2.py:177-228: loss.backward(); opt.step()) train through the library's
# fp32 kernels.  The forwards launch exactly the kernels of the plain module forwards (bit-identical outputs) and keep
# what the backward reads; each backward is the chain the fused fp32 update runs (_critic_pass, _actor_pass,
# _encoder_bwd), fed by whatever gradient autograd has summed over every consumer of an output.
def _grad_like(t, need):
    return torch.empty_like(t) if need else None


def _trunk_bwd(dh, B, Fd, feat, h, ld_h, xhat, rstd, gamma, W, need_feat, need_w, need_b, need_gamma, need_beta):
    """Backward of Linear(39200->F) + LayerNorm + tanh from dh [B, F]: (dfeat, dW, db, dgamma, dbeta), None where not
    needed.  The feature gradient dz @ W (39200 columns) runs only when the features need it."""
    s = _stream()
    dev = dh.device
    dz = torch.empty(2 * B * Fd, device=dev)        # [dz | dy], drq_ln_tanh_bwd
    dgamma, dbeta = torch.empty(Fd, device=dev), torch.empty(Fd, device=dev)
    call("drq_ln_tanh_bwd", dh.data_ptr(), Fd, h.data_ptr(), ld_h, xhat.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
         dz.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), None, 0, B, Fd, 1, 0, s)
    dW, db = _grad_like(W, need_w), torch.empty(Fd, device=dev) if need_b else None
    if need_w:
        _linear_wgrad(dz.data_ptr(), Fd, feat.data_ptr(), REPR_DIM, dW.data_ptr(), B, Fd, REPR_DIM)
    if need_b:
        _colsum(dz.data_ptr(), Fd, db.data_ptr(), B, Fd)
    dfeat = None
    if need_feat:
        dfeat = torch.empty(B, REPR_DIM, device=dev)
        _linear_dgrad(dz.data_ptr(), Fd, W.data_ptr(), dfeat.data_ptr(), REPR_DIM, B, Fd, REPR_DIM)
    return dfeat, dW, db, dgamma if need_gamma else None, dbeta if need_beta else None


def _mlp_bwd(dy, B, n_in, H, n_out, x, ldx, h1, h2, ws, need):
    """Backward of the 3-layer ReLU MLP (weights ws = (W1, b1, W2, b2, W3, b3)) from dy [B, n_out]: the six parameter
    gradients (None where need[i] is False) and dh1, the gradient w.r.t. the first layer's pre-ReLU output, from which
    the caller takes the input gradient over the column ranges it needs."""
    dev = dy.device
    W1, _, W2, _, W3, _ = ws
    g = [_grad_like(w, n) for w, n in zip(ws, need)]
    dh2, dh1 = torch.empty(B, H, device=dev), torch.empty(B, H, device=dev)
    dyp, h1p, h2p = dy.data_ptr(), h1.data_ptr(), h2.data_ptr()
    if need[4]:
        _linear_wgrad(dyp, n_out, h2p, H, g[4].data_ptr(), B, n_out, H)
    if need[5]:
        _colsum(dyp, n_out, g[5].data_ptr(), B, n_out)
    _linear_dgrad(dyp, n_out, W3.data_ptr(), dh2.data_ptr(), H, B, n_out, H, mask=h2p, ldmask=H)
    if need[2]:
        _linear_wgrad(dh2.data_ptr(), H, h1p, H, g[2].data_ptr(), B, H, H)
    if need[3]:
        _colsum(dh2.data_ptr(), H, g[3].data_ptr(), B, H)
    _linear_dgrad(dh2.data_ptr(), H, W2.data_ptr(), dh1.data_ptr(), H, B, H, H, mask=h1p, ldmask=H)
    if need[0]:
        _linear_wgrad(dh1.data_ptr(), H, x.data_ptr(), ldx, g[0].data_ptr(), B, H, n_in)
    if need[1]:
        _colsum(dh1.data_ptr(), H, g[1].data_ptr(), B, H)
    return g, dh1


def _encoder_fwd_f32_pixels(x, w, b, acts, feat, n, cin):
    """_encoder_fwd from real-valued (already augmented) fp32 pixels"""
    s = _stream()
    call("drq_conv1_fwd_f32_from_f32", x, w[0], b[0], acts[0], n, cin, s)
    call("drq_conv3x3_fwd_f32", acts[0], w[1], b[1], acts[1], n, 39, 0, s)
    call("drq_conv3x3_fwd_f32", acts[1], w[2], b[2], acts[2], n, 37, 0, s)
    call("drq_conv3x3_fwd_f32", acts[2], w[3], b[3], feat, n, 35, 1, s)


class _EncoderFn(torch.autograd.Function):
    """features = Encoder(pixels) (drqv2.py:63-67) through drq_conv1_fwd_f32 / drq_conv3x3_fwd_f32; backward
    drq_feature_grad_wide_f32 -> drq_conv3x3_{wgrad,dgrad}_f32 for conv4..2 -> drq_conv1_wgrad_f32 (no shift: the pixels
    arrive augmented).  Inputs: the pixels - uint8, or fp32 on the 0..255 scale (Encoder(pixels="float"), the
    *_from_f32 conv1 kernels) - then (weight, bias) of conv1..4.  fp32 pixels that require grad get
    drq_conv1_dgrad_f32's gradient; every weight gradient runs only when its parameter needs it."""

    @staticmethod
    def forward(ctx, px, *params):
        n, cin = px.shape[0], px.shape[1]
        dev = px.device
        # zeroed, not empty: drq_conv3x3_wgrad_f32 reads the whole plane of its input activation, slack included
        acts = [torch.zeros(n * 32 * PLANE, device=dev) for _ in range(3)]
        feat = torch.empty(n, REPR_DIM, device=dev)
        fwd = _encoder_fwd if px.dtype == torch.uint8 else _encoder_fwd_f32_pixels
        args = (px.data_ptr(), 0) if px.dtype == torch.uint8 else (px.data_ptr(),)
        fwd(*args, [p.data_ptr() for p in params[0::2]], [p.data_ptr() for p in params[1::2]],
            [a.data_ptr() for a in acts], feat.data_ptr(), n, cin)
        ctx.save_for_backward(px, *acts, feat, params[0], *params[2::2])
        return feat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dfeat):
        px, a1, a2, a3, feat, w1, w2, w3, w4 = ctx.saved_tensors
        need_all = _bf16.needed(ctx)
        need_x, need = need_all[0], need_all[1:]
        if not (need_x or any(need)):
            return (None,) * 9
        n, cin = px.shape[0], px.shape[1]
        dev, s = feat.device, _stream()
        dfeat = dfeat.float().contiguous()
        acts, ws = (a1, a2, a3), (None, w2, w3, w4)
        # d[l] = gradient w.r.t. conv(l+1)'s pre-ReLU output.  Zeroed: the data gradient leaves rows hout+2.. of its
        # output alone and the next layer's data gradient reads two of them, which must be +0
        d = [torch.zeros(n * 32 * PLANE, device=dev) for _ in range(4)]
        wsp = torch.empty(int(_lib.lib().drq_conv_wgrad_ws_floats(32)), device=dev)    # cin <= 16 < 32
        grads = [torch.empty(shape, device=dev) for shape in [(32, cin, 3, 3), (32,)] + [(32, 32, 3, 3), (32,)] * 3]
        call("drq_feature_grad_wide_f32", dfeat.data_ptr(), feat.data_ptr(), d[3].data_ptr(), n, s)
        for layer, hout in ((3, 35), (2, 37), (1, 39)):
            if need[2 * layer] or need[2 * layer + 1]:
                call("drq_conv3x3_wgrad_f32", acts[layer - 1].data_ptr(), d[layer].data_ptr(), wsp.data_ptr(),
                     grads[2 * layer].data_ptr(), grads[2 * layer + 1].data_ptr(), n, hout, s)
            if need_x or any(need[:2 * layer]):
                call("drq_conv3x3_dgrad_f32", d[layer].data_ptr(), ws[layer].data_ptr(), acts[layer - 1].data_ptr(),
                     d[layer - 1].data_ptr(), n, hout, s)
        if need[0] or need[1]:
            if px.dtype == torch.uint8:
                call("drq_conv1_wgrad_f32", px.data_ptr(), None, d[0].data_ptr(), wsp.data_ptr(), grads[0].data_ptr(),
                     grads[1].data_ptr(), n, cin, 4, s)
            else:
                call("drq_conv1_wgrad_f32_from_f32", px.data_ptr(), d[0].data_ptr(), wsp.data_ptr(),
                     grads[0].data_ptr(), grads[1].data_ptr(), n, cin, s)
        dx = None
        if need_x:
            dx = torch.empty(px.shape, device=dev)
            call("drq_conv1_dgrad_f32", d[0].data_ptr(), w1.data_ptr(), dx.data_ptr(), n, cin, s)
        return (dx,) + tuple(g if nd else None for g, nd in zip(grads, need))


class _ActorFn(torch.autograd.Function):
    """mu = tanh(policy(trunk(features))) (drqv2.py:85-89); backward drq_actor_sample_bwd (tanh'), the policy MLP's
    weight / bias / masked data gradients and the trunk backward.  Inputs: features, trunk (W, b, gamma, beta), policy
    (W1, b1, W2, b2, W3, b3)."""

    @staticmethod
    def forward(ctx, feat, tW, tb, gamma, beta, *pw):
        B, dev = feat.shape[0], feat.device
        Fd, H, A = tW.shape[0], pw[0].shape[0], pw[4].shape[0]
        partial = torch.empty(_splitk_for(B) * B * Fd, device=dev)
        h, xhat, rstd = torch.empty(B, Fd, device=dev), torch.empty(B, Fd, device=dev), torch.empty(B, device=dev)
        _trunk_fwd(feat.data_ptr(), B, tW.data_ptr(), tb.data_ptr(), gamma.data_ptr(), beta.data_ptr(), Fd,
                   partial.data_ptr(), h.data_ptr(), Fd, xhat.data_ptr(), rstd.data_ptr())
        p1, p2, mu_pre = torch.empty(B, H, device=dev), torch.empty(B, H, device=dev), torch.empty(B, A, device=dev)
        _linear_fwd(h.data_ptr(), Fd, pw[0].data_ptr(), pw[1].data_ptr(), p1.data_ptr(), H, B, H, Fd, True)
        _linear_fwd(p1.data_ptr(), H, pw[2].data_ptr(), pw[3].data_ptr(), p2.data_ptr(), H, B, H, H, True)
        _linear_fwd(p2.data_ptr(), H, pw[4].data_ptr(), pw[5].data_ptr(), mu_pre.data_ptr(), A, B, A, H, False)
        mu = torch.empty(B, A, device=dev)
        call("drq_actor_sample", mu_pre.data_ptr(), None, None, 0.0, mu.data_ptr(), A, None, None, B, A, _stream())
        ctx.save_for_backward(feat, h, xhat, rstd, p1, p2, mu, tW, gamma, *pw)
        return mu

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dmu):
        feat, h, xhat, rstd, p1, p2, mu, tW, gamma, *pw = ctx.saved_tensors
        need = ctx.needs_input_grad
        B, Fd, H, A = feat.shape[0], tW.shape[0], pw[0].shape[0], pw[4].shape[0]
        dev = feat.device
        dmu = dmu.float().contiguous()
        dmu_pre = torch.empty(B, A, device=dev)
        call("drq_actor_sample_bwd", dmu.data_ptr(), A, mu.data_ptr(), dmu_pre.data_ptr(), None, 0, B, A, 1, 0, _stream())
        gp, dp1 = _mlp_bwd(dmu_pre, B, Fd, H, A, h, Fd, p1, p2, pw, need[5:])
        gt = (None,) * 5
        if any(need[:5]):
            dh = torch.empty(B, Fd, device=dev)
            _linear_dgrad(dp1.data_ptr(), H, pw[0].data_ptr(), dh.data_ptr(), Fd, B, H, Fd)
            gt = _trunk_bwd(dh, B, Fd, feat, h, Fd, xhat, rstd, gamma, tW, *need[:5])
        return (*gt, *gp)


class _CriticFn(torch.autograd.Function):
    """(Q1, Q2) = Critic(features, action) (drqv2.py:115-121); backward per Q head that received a gradient (a None
    gradient skips its head): weight / bias / masked data gradients, then the gradients w.r.t. h and w.r.t. the action
    from the first layer's two column ranges, then the trunk backward.  Inputs: features, action, trunk (W, b, gamma,
    beta), Q1 (W1, b1, W2, b2, W3, b3), Q2 (the same)."""

    @staticmethod
    def forward(ctx, feat, action, tW, tb, gamma, beta, *qw):
        ctx.set_materialize_grads(False)
        B, dev = feat.shape[0], feat.device
        Fd, H = tW.shape[0], qw[0].shape[0]
        A = qw[0].shape[1] - Fd
        partial = torch.empty(_splitk_for(B) * B * Fd, device=dev)
        x, xhat, rstd = torch.empty(B, Fd + A, device=dev), torch.empty(B, Fd, device=dev), torch.empty(B, device=dev)
        _trunk_fwd(feat.data_ptr(), B, tW.data_ptr(), tb.data_ptr(), gamma.data_ptr(), beta.data_ptr(), Fd,
                   partial.data_ptr(), x.data_ptr(), Fd + A, xhat.data_ptr(), rstd.data_ptr())
        call("drq_copy2d_f32", action.data_ptr(), A, x.data_ptr() + F32 * Fd, Fd + A, B, A, _stream())
        qs, hidden = [], []
        for z in range(2):
            w = qw[6 * z:6 * z + 6]
            q, h1, h2 = torch.empty(B, 1, device=dev), torch.empty(B, H, device=dev), torch.empty(B, H, device=dev)
            _linear_fwd(x.data_ptr(), Fd + A, w[0].data_ptr(), w[1].data_ptr(), h1.data_ptr(), H, B, H, Fd + A, True)
            _linear_fwd(h1.data_ptr(), H, w[2].data_ptr(), w[3].data_ptr(), h2.data_ptr(), H, B, H, H, True)
            _linear_fwd(h2.data_ptr(), H, w[4].data_ptr(), w[5].data_ptr(), q.data_ptr(), 1, B, 1, H, False)
            qs.append(q)
            hidden += [h1, h2]
        ctx.save_for_backward(feat, x, xhat, rstd, *hidden, tW, gamma, *qw)
        return qs[0], qs[1]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dq1, dq2):
        feat, x, xhat, rstd, h1a, h2a, h1b, h2b, tW, gamma, *qw = ctx.saved_tensors
        need = ctx.needs_input_grad
        B, Fd, H = feat.shape[0], tW.shape[0], qw[0].shape[0]
        A = qw[0].shape[1] - Fd
        dev = feat.device
        if dq1 is None and dq2 is None:
            return (None,) * 18
        need_h = any(need[0:1] + need[2:6])
        dh = torch.zeros(B, Fd, device=dev) if need_h else None
        dact = torch.zeros(B, A, device=dev) if need[1] else None
        gq = [None] * 12
        for z, (dq, h1, h2) in enumerate(((dq1, h1a, h2a), (dq2, h1b, h2b))):
            if dq is None:
                continue
            w = qw[6 * z:6 * z + 6]
            dq = dq.float().contiguous()
            gq[6 * z:6 * z + 6], dc1 = _mlp_bwd(dq, B, Fd + A, H, 1, x, Fd + A, h1, h2, w, need[6 + 6 * z:12 + 6 * z])
            # d[h | action] = dc1 @ W1, over the two column ranges separately (each only when needed)
            if need_h:
                _linear_dgrad(dc1.data_ptr(), H, w[0].data_ptr(), dh.data_ptr(), Fd, B, H, Fd + A, n_cols=Fd, acc=1)
            if need[1]:
                _linear_dgrad(dc1.data_ptr(), H, w[0].data_ptr(), dact.data_ptr(), A, B, H, Fd + A, w_col0=Fd,
                              n_cols=A, acc=1)
        gt = (None,) * 5
        if need_h:
            gt = _trunk_bwd(dh, B, Fd, feat, x, Fd + A, xhat, rstd, gamma, tW, need[0], *need[2:6])
        return (gt[0], dact, *gt[1:], *gq)


def _flag(differentiable, what):
    """the differentiable= value as stored: False, True or "bf16" (True and "bf16" stay distinct)"""
    if isinstance(differentiable, str):
        if differentiable != "bf16":
            raise ValueError(f"{what}: differentiable must be False, True or 'bf16', got {differentiable!r}")
        return differentiable
    if differentiable not in (False, True):
        raise ValueError(f"{what}: differentiable must be False, True or 'bf16', got {differentiable!r}")
    return bool(differentiable)


def _pixels_flag(pixels, what):
    if not isinstance(pixels, str) or pixels not in ("u8", "float"):
        raise ValueError(f"{what}: pixels must be 'u8' or 'float', got {pixels!r}")
    return pixels


def _check_bf16_dims(A, H, Fd, dev=None):
    """Refuse at construction the head shapes the tensor-core kernels refuse (csrc/heads.cu), which would otherwise
    fail at the first act(), update() or forward.  dev None: the current device, when there is one (the shared-memory
    bound needs its properties)."""
    if not 1 <= A <= _lib.POLICY_MAX_A:
        raise ValueError(f"action_shape ({A},): mode='bf16' supports 1 <= A <= {_lib.POLICY_MAX_A} action dimensions "
                         "(the policy head kernel); mode='fp32' and differentiable=True have no such limit")
    if H % 8:
        raise ValueError(f"hidden_dim {H}: mode='bf16' needs a multiple of 8 (16-byte rows of the bf16 operands); "
                         "mode='fp32' and differentiable=True have no such limit")
    if not 1 <= Fd <= _lib.LN_MAX_F:
        raise ValueError(f"feature_dim {Fd}: the LayerNorm kernels hold 1 <= F <= {_lib.LN_MAX_F} features "
                         "(differentiable=True as well)")
    if dev is None:
        if not torch.cuda.is_available():
            return
        dev = torch.device("cuda", torch.cuda.current_device())
    groups = -(-A // _lib.POLICY_GROUP)
    slab = 4 * H * -(-A // groups)                 # fp32 weights of one policy-head block's action group
    optin = torch.cuda.get_device_properties(dev).shared_memory_per_block_optin
    if slab + _lib.POLICY_STATIC_SMEM > optin:
        raise ValueError(f"hidden_dim {H} with {A} actions: mode='bf16' stages {slab} bytes of policy-head weights per "
                         f"block, more than the {optin - _lib.POLICY_STATIC_SMEM} bytes of shared memory a block can "
                         "have here; mode='fp32' and differentiable=True have no such limit")


def _refresh_bf16(self):
    """differentiable="bf16": re-derive the bf16 operand copies before the next forward - after a change of the
    parameters their version counters do not show (writes through .data or raw pointers)."""
    _bf16.mark_stale(self)


def _wants_graph(module, *inputs):
    """record a Function: the module was built differentiable, autograd records, and something needs a gradient"""
    return (module.differentiable and torch.is_grad_enabled()
            and any(t.requires_grad for t in (*inputs, *module.parameters())))


# ----------------------------------------------------------------------------- modules
class _ShiftFn(torch.autograd.Function):
    """RandomShiftsAug's integer shift with its transpose as the backward (drq_random_shift_bwd_f32).  Inputs: the fp32
    pixels, the int32 shifts [N, 2], pad."""

    @staticmethod
    def forward(ctx, x, shift, pad):
        n, c, h, w = x.shape
        out = torch.empty_like(x)
        call("drq_random_shift_f32", x.data_ptr(), shift.data_ptr(), out.data_ptr(), n, c, h, w, pad, _stream())
        ctx.save_for_backward(shift)
        ctx.pad = pad
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        shift, = ctx.saved_tensors
        dout = dout.float().contiguous()
        n, c, h, w = dout.shape
        dx = torch.empty_like(dout)
        call("drq_random_shift_bwd_f32", dout.data_ptr(), shift.data_ptr(), dx.data_ptr(), n, c, h, w, ctx.pad,
             _stream())
        return dx, None, None


class RandomShiftsAug(nn.Module):
    """Random translation by up to ±pad pixels after replicate padding, as the exact
    integer shift (the reference's bilinear grid_sample equals it to 3.6e-3 on the 0..255
    scale, SURVEY §8a R3).  The draw is the reference's own ``torch.randint`` call, so
    the same patch injects shifts into either implementation.  When autograd records and
    ``x`` requires grad, the output carries the shift's transpose as its backward (the
    gradient w.r.t. ``x``, drq_random_shift_bwd_f32)."""

    def __init__(self, pad):
        super().__init__()
        self.pad = pad

    def forward(self, x):
        n, c, h, w = x.size()
        assert h == w
        _need_cuda(x, "RandomShiftsAug")
        shift = torch.randint(0, 2 * self.pad + 1, size=(n, 1, 1, 2), device=x.device, dtype=x.dtype)
        shift = shift.view(n, 2).to(torch.int32).contiguous()
        x = x.float().contiguous()
        if torch.is_grad_enabled() and x.requires_grad:
            return _ShiftFn.apply(x, shift, self.pad)
        out = torch.empty_like(x)
        call("drq_random_shift_f32", x.data_ptr(), shift.data_ptr(), out.data_ptr(), n, c, h, w, self.pad,
             _stream())
        return out


def _as_u8_pixels(obs):
    if obs.dtype == torch.uint8:
        return obs.contiguous()
    u8 = obs.to(torch.uint8)
    if not torch.equal(u8.to(obs.dtype), obs):
        raise ValueError("Encoder expects integer-valued pixels in [0, 255] (uint8 frames, optionally "
                         "shifted by RandomShiftsAug); got non-integral values")
    return u8.contiguous()


class Encoder(nn.Module):
    differentiable = False      # class default: instances pickled before the flag existed read it too
    pixels = "u8"               # likewise
    refresh = _refresh_bf16

    def __init__(self, obs_shape, *, differentiable=False, pixels="u8"):
        """differentiable=True: forward records an autograd node (_EncoderFn) whenever autograd records and a parameter
        requires grad, so that a loss on the features trains the convs; off (the default), outputs are plain tensors.
        differentiable="bf16": the same on the tensor-core kernels (bf16 operands, fp32 accumulation; _bf16.EncoderFn),
        under no_grad too; up to 10 input channels.
        pixels="u8" (the default): integer-valued pixels in 0..255, which may not require grad.  pixels="float": any
        real-valued pixels on the 0..255 scale, cast to fp32 - with no integrality and no finiteness check - and, when
        the module is differentiable, autograd records and they require grad, obs.grad = dL/dpixels on that scale."""
        super().__init__()
        assert len(obs_shape) == 3
        self.differentiable = _flag(differentiable, "Encoder")
        self.pixels = _pixels_flag(pixels, "Encoder")
        if self.differentiable == "bf16" and int(obs_shape[0]) * 9 + 1 > 96:
            raise ValueError(f"Encoder(differentiable='bf16'): {int(obs_shape[0])} input channels; the tensor-core conv1 "
                             "takes cin * 9 + 1 <= 96, at most 10 channels (differentiable=True takes up to 16)")
        self.repr_dim = 32 * 35 * 35
        chans = [int(obs_shape[0]), 32, 32, 32]
        mods = []
        for i, cin in enumerate(chans):
            mods += [nn.Conv2d(cin, 32, 3, stride=2 if i == 0 else 1), nn.ReLU()]
        self.convnet = nn.Sequential(*mods)
        self.apply(utils.weight_init)

    def conv_ptrs(self):
        convs = [self.convnet[i] for i in (0, 2, 4, 6)]
        return [c.weight.data_ptr() for c in convs], [c.bias.data_ptr() for c in convs]

    def forward(self, obs):
        """obs: [N, C, 84, 84] pixels on the 0..255 scale (uint8, or integer-valued float as
        produced by RandomShiftsAug; any real values with pixels="float").  Returns features [N, 39200]."""
        _need_cuda(obs, "Encoder")
        _need_cuda(self.convnet[0].weight, "Encoder parameters")
        if self.pixels == "float":
            return self._forward_float(obs)
        if self.differentiable and torch.is_grad_enabled() and obs.requires_grad:
            raise ValueError("Encoder(differentiable=True): the pixels require grad, but the integer-shift encoder has no "
                             "gradient w.r.t. its input pixels; pass them detached")
        u8 = _as_u8_pixels(obs)
        if self.differentiable == "bf16":
            _bf16.check_batch(u8.shape[0], "Encoder")
            ops = _bf16.operands(self, "encoder")
            if _wants_graph(self):
                return _bf16.EncoderFn.apply(ops, u8, *self.parameters())
            return _bf16.encoder_forward(ops, u8, [self.convnet[i].bias.data_ptr() for i in (2, 4, 6)])[0]
        if _wants_graph(self):
            return _EncoderFn.apply(u8, *self.parameters())
        n, cin = u8.shape[0], u8.shape[1]
        acts = [torch.empty(n * 32 * PLANE, device=u8.device) for _ in range(3)]
        feat = torch.empty(n, self.repr_dim, device=u8.device)
        w, b = self.conv_ptrs()
        _encoder_fwd(u8.data_ptr(), 0, w, b, [a.data_ptr() for a in acts], feat.data_ptr(), n, cin)
        return feat

    def _forward_float(self, obs):
        x = obs.float().contiguous()
        cin = self.convnet[0].in_channels
        if obs.dim() != 4 or tuple(x.shape[1:]) != (cin, 84, 84):
            raise ValueError(f"Encoder: pixels of shape {tuple(obs.shape)}, expected [N, {cin}, 84, 84]")
        params = list(self.parameters())
        if torch.is_grad_enabled() and x.requires_grad:
            # non-leaf edges: _bf16.needed can tell which the backward reaches, so that torch.autograd.grad(q, obs) runs
            # no weight-gradient kernel (tests/test_gpu_pixel_grad.py::test_saliency_runs_no_encoder_weight_gradient)
            params = [p.view_as(p) for p in params]
        if self.differentiable == "bf16":
            _bf16.check_batch(x.shape[0], "Encoder")
            ops = _bf16.operands(self, "encoder")
            if _wants_graph(self, x):
                return _bf16.EncoderFn.apply(ops, x, *params)
            return _bf16.encoder_forward(ops, x, [self.convnet[i].bias.data_ptr() for i in (2, 4, 6)])[0]
        if _wants_graph(self, x):
            return _EncoderFn.apply(x, *params)
        n, cin = x.shape[0], x.shape[1]
        acts = [torch.empty(n * 32 * PLANE, device=x.device) for _ in range(3)]
        feat = torch.empty(n, self.repr_dim, device=x.device)
        w, b = self.conv_ptrs()
        _encoder_fwd_f32_pixels(x.data_ptr(), w, b, [a.data_ptr() for a in acts], feat.data_ptr(), n, cin)
        return feat


class _Trunk(nn.Sequential):
    def __init__(self, repr_dim, feature_dim):
        super().__init__(nn.Linear(repr_dim, feature_dim), nn.LayerNorm(feature_dim), nn.Tanh())


def _mlp(n_in, hidden, n_out):
    return nn.Sequential(nn.Linear(n_in, hidden), nn.ReLU(inplace=True), nn.Linear(hidden, hidden),
                         nn.ReLU(inplace=True), nn.Linear(hidden, n_out))


def _lin_ptrs(seq):
    out = []
    for i in (0, 2, 4):
        out += [seq[i].weight.data_ptr(), seq[i].bias.data_ptr()]
    return out


def _mlp_fwd(seq, x, ldx, B, n_in, hidden, n_out, out, dev):
    """3-layer ReLU MLP forward with throw-away hidden buffers (module-level API)."""
    w1, b1, w2, b2, w3, b3 = _lin_ptrs(seq)
    h1 = torch.empty(B, hidden, device=dev)
    h2 = torch.empty(B, hidden, device=dev)
    _linear_fwd(x, ldx, w1, b1, h1.data_ptr(), hidden, B, hidden, n_in, True)
    _linear_fwd(h1.data_ptr(), hidden, w2, b2, h2.data_ptr(), hidden, B, hidden, hidden, True)
    _linear_fwd(h2.data_ptr(), hidden, w3, b3, out, n_out, B, n_out, hidden, False)
    return h1, h2


class Actor(nn.Module):
    differentiable = False      # class default: instances pickled before the flag existed read it too
    refresh = _refresh_bf16

    def __init__(self, repr_dim, action_shape, feature_dim, hidden_dim, *, differentiable=False):
        """differentiable=True: the returned distribution's mean carries an autograd node (_ActorFn) whenever autograd
        records and the features or a parameter require grad.  differentiable="bf16": the same on the tensor-core
        kernels (_bf16.ActorFn), under no_grad too, within the tensor-core mode's head shapes."""
        super().__init__()
        self.differentiable = _flag(differentiable, "Actor")
        if self.differentiable == "bf16":
            _check_bf16_dims(int(action_shape[0]), int(hidden_dim), int(feature_dim))
        self.trunk = _Trunk(repr_dim, feature_dim)
        self.policy = _mlp(feature_dim, hidden_dim, action_shape[0])
        self.apply(utils.weight_init)

    def forward(self, obs, std):
        _need_cuda(obs, "Actor")
        B, dev = obs.shape[0], obs.device
        Fd, H, A = self.trunk[0].out_features, self.policy[0].out_features, self.policy[4].out_features
        obs = obs.float().contiguous()
        if self.differentiable == "bf16":
            _bf16.check_batch(B, "Actor")
            ops = _bf16.operands(self, "actor")
            tw = (*self.trunk[0].parameters(), *self.trunk[1].parameters(), *self.policy.parameters())
            mu = _bf16.ActorFn.apply(ops, obs, *tw) if _wants_graph(self, obs) else _bf16.actor_forward(ops, obs, tw)[0]
            return utils.TruncatedNormal(mu, torch.ones_like(mu) * std)
        if _wants_graph(self, obs):
            mu = _ActorFn.apply(obs, *self.trunk[0].parameters(), *self.trunk[1].parameters(), *self.policy.parameters())
            return utils.TruncatedNormal(mu, torch.ones_like(mu) * std)
        partial = torch.empty(_splitk_for(B) * B * Fd, device=dev)
        h = torch.empty(B, Fd, device=dev)
        t = self.trunk
        _trunk_fwd(obs.data_ptr(), B, t[0].weight.data_ptr(), t[0].bias.data_ptr(), t[1].weight.data_ptr(),
                   t[1].bias.data_ptr(), Fd, partial.data_ptr(), h.data_ptr(), Fd)
        mu_pre = torch.empty(B, A, device=dev)
        keep = _mlp_fwd(self.policy, h.data_ptr(), Fd, B, Fd, H, A, mu_pre.data_ptr(), dev)
        mu = torch.empty(B, A, device=dev)
        call("drq_actor_sample", mu_pre.data_ptr(), None, None, 0.0, mu.data_ptr(), A, None, None, B, A, _stream())
        del keep
        return utils.TruncatedNormal(mu, torch.ones_like(mu) * std)


class Critic(nn.Module):
    differentiable = False      # class default: instances pickled before the flag existed read it too
    refresh = _refresh_bf16

    def __init__(self, repr_dim, action_shape, feature_dim, hidden_dim, *, differentiable=False):
        """differentiable=True: Q1 and Q2 carry an autograd node (_CriticFn) whenever autograd records and the features,
        the action or a parameter require grad.  differentiable="bf16": the same on the tensor-core kernels
        (_bf16.CriticFn), under no_grad too, within the tensor-core mode's head shapes."""
        super().__init__()
        self.differentiable = _flag(differentiable, "Critic")
        if self.differentiable == "bf16":
            _check_bf16_dims(int(action_shape[0]), int(hidden_dim), int(feature_dim))
        self.trunk = _Trunk(repr_dim, feature_dim)
        self.Q1 = _mlp(feature_dim + action_shape[0], hidden_dim, 1)
        self.Q2 = _mlp(feature_dim + action_shape[0], hidden_dim, 1)
        self.apply(utils.weight_init)

    def forward(self, obs, action):
        _need_cuda(obs, "Critic")
        B, dev = obs.shape[0], obs.device
        Fd, H = self.trunk[0].out_features, self.Q1[0].out_features
        A = self.Q1[0].in_features - Fd
        obs = obs.float().contiguous()
        action = action.float().contiguous()
        if self.differentiable == "bf16":
            _bf16.check_batch(B, "Critic")
            ops = _bf16.operands(self, "critic")
            cw = (*self.trunk[0].parameters(), *self.trunk[1].parameters(), *self.Q1.parameters(), *self.Q2.parameters())
            if _wants_graph(self, obs, action):
                return _bf16.CriticFn.apply(ops, obs, action, *cw)
            return _bf16.critic_forward(ops, obs, action, cw)[:2]
        if _wants_graph(self, obs, action):
            return _CriticFn.apply(obs, action, *self.trunk[0].parameters(), *self.trunk[1].parameters(),
                                   *self.Q1.parameters(), *self.Q2.parameters())
        partial = torch.empty(_splitk_for(B) * B * Fd, device=dev)
        x = torch.empty(B, Fd + A, device=dev)
        t = self.trunk
        _trunk_fwd(obs.data_ptr(), B, t[0].weight.data_ptr(), t[0].bias.data_ptr(), t[1].weight.data_ptr(),
                   t[1].bias.data_ptr(), Fd, partial.data_ptr(), x.data_ptr(), Fd + A)
        call("drq_copy2d_f32", action.data_ptr(), A, x.data_ptr() + F32 * Fd, Fd + A, B, A, _stream())
        qs = []
        for head in (self.Q1, self.Q2):
            q = torch.empty(B, 1, device=dev)
            keep = _mlp_fwd(head, x.data_ptr(), Fd + A, B, Fd + A, H, 1, q.data_ptr(), dev)
            del keep
            qs.append(q)
        return qs[0], qs[1]


# ----------------------------------------------------------------------------- flat arenas
@contextlib.contextmanager
def _capture(graph, stream=None):
    """``torch.cuda.graph`` with the cyclic garbage collector held off.  A collection in the middle of a
    capture may run the destructors of dead CUDA objects (other agents' graphs, pinned buffers, events);
    cudaFree / cudaEventDestroy from the capturing thread are illegal then and abort the process."""
    was = gc.isenabled()
    gc.collect()
    gc.disable()
    try:
        # thread_local: NCCL's watchdog thread may touch CUDA while this thread captures
        kw = {} if stream is None else {"stream": stream}
        with torch.cuda.graph(graph, capture_error_mode="thread_local", **kw):
            yield
    finally:
        if was:
            gc.enable()


def _pad4(n):
    return (n + 3) // 4 * 4


class _Arena:
    """Flat fp32 storage for parameters / gradients / Adam moments of
    [encoder | critic | actor] (every tensor starts on a 16-byte boundary; the padding
    carries zero gradients) and for the target critic.  Module parameters become views, so state_dict()/pickle see ordinary tensors
    in the reference's layouts while one kernel can update a whole optimiser's range."""

    def __init__(self, encoder, critic, actor, critic_target, device):
        self.seg = {}
        off = 0
        for name, mod in (("encoder", encoder), ("critic", critic), ("actor", actor)):
            n = sum(_pad4(p.numel()) for p in mod.parameters())
            self.seg[name] = (off, n, n)
            off += n
        self.total = off
        self.params = torch.zeros(off, device=device)
        # data-parallel updates average the 8 metrics with the last gradient all-reduce: they live right behind the
        # actor's gradients (the last segment), see DrQV2Agent._sync_grads
        self._grads_full = torch.zeros(off + 8, device=device)
        self.grads, self.metrics_tail = self._grads_full[:off], self._grads_full[off:]
        self.moments = torch.zeros(2, off, device=device)        # [exp_avg | exp_avg_sq]
        self.exp_avg, self.exp_avg_sq = self.moments[0], self.moments[1]
        n_t = self.seg["critic"][2]
        self.target = torch.zeros(n_t, device=device)
        self.offsets = {}
        for name, mod in (("encoder", encoder), ("critic", critic), ("actor", actor)):
            o = self.seg[name][0]
            self.offsets[name] = self._adopt(mod, self.params, self.grads, o)
        self._adopt(critic_target, self.target, None, 0)

    @staticmethod
    def _adopt(mod, flat, flat_grad, off):
        offs = {}
        with torch.no_grad():
            for pname, p in mod.named_parameters():
                n = p.numel()
                view = flat[off:off + n].view(p.shape)
                view.copy_(p.data)
                p.data = view
                p.requires_grad_(False)
                if flat_grad is not None:
                    p.grad = flat_grad[off:off + n].view(p.shape)
                offs[pname] = off
                off += _pad4(n)
        return offs

    def ptr(self, which, net, pname=None):
        base = getattr(self, which).data_ptr()
        if pname is None:
            return base + F32 * self.seg[net][0]
        return base + F32 * self.offsets[net][pname]


class _Workspace:
    """Static buffers of one update at batch size B (allocated once, graph-capturable)."""

    def __init__(self, B, A, Fd, H, cin, device, fp32_encoder=True):
        z = lambda *s: torch.zeros(*s, device=device)
        self.B = B
        NB = 2 * B
        # inputs
        self.obs = torch.zeros(NB, cin, 84, 84, dtype=torch.uint8, device=device)   # [obs | next_obs]
        self.action, self.reward, self.discount = z(B, A), z(B, 1), z(B, 1)
        self.shift = torch.full((NB, 2), 4, dtype=torch.int32, device=device)       # [obs | next_obs]
        self.eps_c, self.eps_a = z(B, A), z(B, A)
        # encoder
        if fp32_encoder:
            self.acts = [z(NB * 32 * PLANE) for _ in range(3)]
            self.feat = z(NB, REPR_DIM)
            self.dpre = [z(B * 32 * PLANE) for _ in range(4)]    # grads w.r.t. conv1..4 pre-ReLU outputs
            self.wgrad_ws = z(int(_lib.lib().drq_conv_wgrad_ws_floats(32)))
        # heads
        self.partial = z(_splitk_for(B) * B * Fd)
        self.xT = z(B, Fd + A)          # [h_target(next) | next_action]
        self.xC = z(B, Fd + A)          # [h_critic(obs) | action]
        self.xA = z(B, Fd + A)          # [h_critic'(obs) | actor action]
        self.hA = z(B, Fd)              # actor trunk output
        self.xhatC, self.rstdC = z(B, Fd), z(B)
        self.xhatA, self.rstdA = z(B, Fd), z(B)
        self.p1, self.p2 = z(B, H), z(B, H)             # actor hidden
        self.mu_pre, self.mu = z(B, A), z(B, A)
        self.c1, self.c2 = z(2, B, H), z(2, B, H)       # twin-Q hidden (both heads)
        self.q, self.tq = z(2, B), z(2, B)
        self.dq = z(2, B)
        self.dc1, self.dc2 = z(2, B, H), z(2, B, H)
        self.dx = z(B, Fd + A)
        self.dz = z(2 * B * Fd)
        self.dact, self.dmu_pre = z(B, A), z(B, A)
        self.dp1, self.dp2 = z(B, H), z(B, H)
        self.dhA = z(B, Fd)
        self.target_q = z(B)
        self.metrics = z(8)


class _Opt:
    """Stand-in for the reference's three torch.optim.Adam objects (drqv2.py:148-150):
    the update itself is drq_adam_ema_step over the flat arena; this object carries the
    hyper-parameters and the step count for inspection / pickling, and step() for code that
    trains through autograd (DrQV2Agent(differentiable=True))."""

    def __init__(self, agent, net, lr):
        self._agent, self.net = agent, net
        self.defaults = dict(lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False)

    def _flat(self, arena):
        """the net's tensors in parameters() order, without the arena's alignment padding"""
        offs = self._agent._arena.offsets[self.net]
        return torch.cat([arena[offs[k]:offs[k] + p.numel()] for k, p in getattr(self._agent, self.net).named_parameters()])

    def state_dict(self):
        a = self._agent._arena
        return dict(step=self._agent._opt_steps[self.net], exp_avg=self._flat(a.exp_avg), exp_avg_sq=self._flat(a.exp_avg_sq),
                    **self.defaults)

    def zero_grad(self, set_to_none=True):
        off, n, _ = self._agent._arena.seg[self.net]
        self._agent._arena.grads[off:off + n].zero_()

    def step(self, closure=None):
        """One torch.optim.Adam step of this network: drq_adam_step over its arena range, with this optimiser's own
        step count and Adam scalars (fetched through the scalar ring in stream order, as the stage API does; the
        exploration stddev act() reads is left as it was).  Unlike torch.optim.Adam, which skips a parameter whose
        .grad is None, this steps every parameter of the network: the arena's gradients are never None (zero_grad
        zeroes them).  The reference's update_critic / update_actor give every parameter they step a gradient, so
        they see no difference.  In the tensor-core mode the bf16 operand copies are re-derived before the next
        act() / update()."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        ag = self._agent
        with torch.cuda.device(ag._dev):
            ag._host_scalars(None, (self.net,))
            ag._fetch_scalars()
            ag._scalars_enqueued()
            a = ag._arena
            off, n = a.seg[self.net][0], a.seg[self.net][2]
            if ag.differentiable == "bf16":
                # Adam and the refresh of this network's bf16 operand copies in one launch, as update() steps it
                getattr(ag._bf16, f"step_{self.net}")()
            else:
                call("drq_adam_step", a.params.data_ptr() + F32 * off, a.grads.data_ptr() + F32 * off,
                     a.exp_avg.data_ptr() + F32 * off, a.exp_avg_sq.data_ptr() + F32 * off, n, ag._sc(self.net), _stream())
                ag._bf16_dirty = True
            ag._opt_steps[self.net] += 1
        return loss


METRIC_KEYS = ("batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss",
               "actor_loss", "actor_logprob", "actor_ent")


class DrQV2Agent:
    def __init__(self, obs_shape, action_shape, device, lr, feature_dim, hidden_dim, critic_target_tau,
                 num_expl_steps, update_every_steps, stddev_schedule, stddev_clip, use_tb,
                 use_cuda_graph=True, seed=None, mode=None, data_parallel=False, prefetch=False, differentiable=False,
                 pixels="u8"):
        """Reference signature (drqv2.py:125-127) plus three keyword-only extras: use_cuda_graph,
        seed (device RNG key) and mode — "fp32" (parity mode, CUDA-core kernels, <= 1e-4 vs the
        reference on pre-optimiser quantities) or "bf16" (tcgen05 tensor-core kernels, bf16
        operands / fp32 accumulation).  Default: $DRQV2_B200_MODE or "bf16" (the performance mode; its
        parity against the bf16-faithful oracle is pinned in tests/test_gpu_bench_config.py).
        data_parallel=True (torch.distributed initialised, one process per GPU): the batch given to
        update() is this rank's shard; gradients are averaged over ranks before each optimiser step and
        parameters are broadcast from rank 0 at construction (drqv2_b200/dist.py).
        prefetch=True: with a host-side replay iterator, pull the next batch at the end of every update and
        copy it to the device on a side stream while that update still runs (the reference's DataLoader
        workers run ahead in the same way); the default keeps drqv2.py:236's one next() per update.
        differentiable=True: encoder, actor and critic record autograd nodes (Encoder / Actor / Critic above) and their
        parameters require grad, so the reference's own update_critic / update_actor bodies (loss.backward();
        opt.step()) train this agent: gradients land in the arena that encoder_opt / critic_opt / actor_opt.step() read
        (INTEGRATION.md).  The fused update() is unaffected.  Not with data_parallel (those steps do not all-reduce).
        pixels="float": agent.encoder takes real-valued pixels, and gives gradients w.r.t. them (Encoder above); act(),
        update() and the stage API read uint8 frames as before."""
        differentiable = _flag(differentiable, "DrQV2Agent")
        pixels = _pixels_flag(pixels, "DrQV2Agent")
        if differentiable and data_parallel:
            raise ValueError(f"DrQV2Agent: differentiable={differentiable!r} with data_parallel=True is not supported - "
                             "the optimisers' step() does not average gradients over ranks")
        if differentiable == "bf16" and (mode or os.environ.get("DRQV2_B200_MODE", "bf16")) != "bf16":
            raise ValueError("DrQV2Agent: differentiable='bf16' runs the tensor-core kernels and needs mode='bf16'; "
                             "differentiable=True trains through the fp32 kernels in either mode")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"DrQV2Agent(device={device!r}): drqv2_b200 has no CPU path; use a CUDA device")
        if not torch.cuda.is_available():
            raise RuntimeError("DrQV2Agent: no CUDA device available (drqv2_b200 has no CPU fallback)")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        _lib.lib()   # fail loudly if the extension is missing
        self.device = device
        self.critic_target_tau = critic_target_tau
        self.update_every_steps = update_every_steps
        self.use_tb = use_tb
        self.num_expl_steps = num_expl_steps
        self.stddev_schedule = stddev_schedule
        self.stddev_clip = stddev_clip
        self.lr = lr
        self.use_cuda_graph = use_cuda_graph
        self.prefetch = bool(prefetch)
        # bf16 mode: encoder backward + encoder_opt.step() on a second stream beside the actor pass (DRQV2_B200_OVERLAP=0: in line)
        self.overlap_encoder_backward = os.environ.get("DRQV2_B200_OVERLAP", "1") != "0"
        # bf16 mode fed from the HBM ring: conv1 reads the frame stacks from the ring by index (DRQV2_B200_RING_DIRECT=0:
        # gather them into a batch buffer first)
        self.ring_direct = os.environ.get("DRQV2_B200_RING_DIRECT", "1") != "0"
        # the actor pass' GEMMs in their 66 KB variant, co-resident with the encoder backward's conv CTAs.  A loss without
        # stream priorities (1769 vs 1834 updates/s: GEMM CTAs that share the encoder backward's SMs cost it more than their
        # own waiting costs), a gain with them (1940 -> 2000: the chain's CTAs are placed first and no longer queue behind a
        # whole conv kernel; DESIGN.md §6)
        self.small_gemms_beside_encoder = os.environ.get("DRQV2_B200_SMALL_GEMMS", "1") != "0"
        self._side_stream = None
        self._side_stream2 = None
        self._main_stream = None
        # schedule switches of the captured tensor-core update (DESIGN.md section 4); every one leaves the results bit-identical
        self.early_encoder_backward = os.environ.get("DRQV2_B200_EARLY_ENC", "1") != "0"
        self.split_prologue = os.environ.get("DRQV2_B200_SPLIT_PROLOGUE", "1") != "0"
        self.encoder_backward_sms = int(os.environ.get("DRQV2_B200_ENC_BWD_SMS", "140"))
        # priorities of (main, encoder-backward, weight-gradient) streams inside the captured update; 0 = default (lowest)
        self._prio = tuple(int(x) for x in os.environ.get("DRQV2_B200_PRIO", "-2,-1,-1").split(","))
        self.mode = mode or os.environ.get("DRQV2_B200_MODE", "bf16")
        if self.mode not in ("fp32", "bf16"):
            raise ValueError(f"mode must be 'fp32' or 'bf16', got {self.mode!r}")
        self.obs_shape = tuple(int(v) for v in obs_shape)
        # conv1's loaders stage a fixed number of input channels: the fp32 kernel up to 16, the tensor-core im2col
        # (K = 9 cin + 1 <= 96) up to 10 (csrc/encoder_f32.cu, csrc/conv1_tc.cu); frame_stack 3 x RGB is 9
        max_cin = 10 if self.mode == "bf16" else 16
        if len(self.obs_shape) != 3 or self.obs_shape[1:] != (84, 84) or not 1 <= self.obs_shape[0] <= max_cin:
            raise ValueError(f"obs_shape {self.obs_shape}: mode={self.mode!r} supports [C, 84, 84] observations with "
                             f"1 <= C <= {max_cin} stacked channels (drqv2.py:53 fixes 84 x 84)")
        self.action_dim = int(action_shape[0])
        self.feature_dim, self.hidden_dim = int(feature_dim), int(hidden_dim)
        if not 1 <= self.feature_dim <= _lib.LN_MAX_F:
            raise ValueError(f"feature_dim {self.feature_dim}: the LayerNorm kernels hold 1 <= F <= {_lib.LN_MAX_F} "
                             "features (in mode='fp32' as well)")
        if self.mode == "bf16":
            _check_bf16_dims(self.action_dim, self.hidden_dim, self.feature_dim, dev)

        # models: built on the host in the reference's order (so a seed reproduces its init)
        self.differentiable = differentiable
        self.encoder = Encoder(self.obs_shape, differentiable=self.differentiable, pixels=pixels)
        self.actor = Actor(self.encoder.repr_dim, action_shape, feature_dim, hidden_dim, differentiable=self.differentiable)
        self.critic = Critic(self.encoder.repr_dim, action_shape, feature_dim, hidden_dim,
                             differentiable=self.differentiable)
        # differentiable="bf16": the target forwards on the tensor cores too (under no_grad: its parameters never
        # require grad)
        self.critic_target = Critic(self.encoder.repr_dim, action_shape, feature_dim, hidden_dim,
                                    differentiable="bf16" if self.differentiable == "bf16" else False)
        self.critic_target.load_state_dict(self.critic.state_dict())
        self._to_device(dev)
        if self.differentiable == "bf16":
            # the modules read this agent's own operand copies (_bf16.operands)
            for role in ("encoder", "actor", "critic", "critic_target"):
                getattr(self, role).__dict__["_bf16_owner"] = (self, role)
        if self.differentiable:
            # .grad stays the arena view _Arena._adopt set: autograd adds into an existing .grad in place
            for m in (self.encoder, self.actor, self.critic):
                m.requires_grad_(True)

        self.encoder_opt = _Opt(self, "encoder", lr)
        self.actor_opt = _Opt(self, "actor", lr)
        self.critic_opt = _Opt(self, "critic", lr)
        self.aug = RandomShiftsAug(pad=4)
        self._opt_steps = dict(encoder=0, critic=0, actor=0)   # torch.optim.Adam keeps one step count per optimiser
        self._seed = int(seed) if seed is not None else int(torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)
        self.data_parallel = bool(data_parallel) and _dist.world() > 1
        # SMs a data-parallel update leaves to NCCL (bf16 mode overlaps its all-reduces with the encoder backward).  Off:
        # with NCCL_MAX_CTAS=8 to match, the 25 MB all-reduce takes 305 us instead of 110 and the 8-GPU step 1.57 ms
        # instead of 1.25 (profiles/r2_dp_8gpu_*.json); without a cap NCCL's CTA count is not ours to plan for
        self.dp_reserve_sms = int(os.environ.get("DRQV2_B200_DP_RESERVE_SMS", "0")) if self.mode == "bf16" else 0
        if self.data_parallel:
            a = self._arena
            _dist.broadcast_([a.params, a.target, a.exp_avg, a.exp_avg_sq])
            self._seed = _dist.rank_seed(self._seed, torch.distributed.get_rank())
            self._bf16_dirty = True
        self.train()
        self.critic_target.train()

    # ------------------------------------------------------------------ plumbing
    def _to_device(self, dev):
        self._dev = dev
        for m in (self.encoder, self.actor, self.critic, self.critic_target):
            m.to(dev)
        self._arena = _Arena(self.encoder, self.critic, self.actor, self.critic_target, dev)
        self._ws = {}
        self._graphs = {}
        self._act_ws = {}
        self._scal_host = torch.zeros(SCAL_SLOT, dtype=torch.float32).pin_memory()
        self._scal_dev = torch.zeros(SCAL_SLOT, device=dev)   # layout: SCAL_OFF
        self._init_scalar_ring()
        self._counter = torch.zeros(1, dtype=torch.int64, device=dev)
        # drq_policy_head_fwd_bf16's scratch words: block ticket + one partial per block of the largest grid it takes
        self._policy_ticket = torch.zeros(1 + _lib.POLICY_MAX_PARTIALS, dtype=torch.int32, device=dev)
        self._metrics_host = torch.zeros(8, dtype=torch.float32).pin_memory()
        self._injected = None
        self._bf16 = _bf16.Bf16State(self) if self.mode == "bf16" else None
        self._bf16_ws = {}
        self._bf16_dirty = True
        self._prefetch, self._stage = None, {}

    def __getstate__(self):
        st = dict(self.__dict__)
        for k in ("_ws", "_graphs", "_act_ws", "_bf16_ws", "_stage"):
            st[k] = {}
        st["_bf16"] = None
        st["_prefetch"] = None
        st["_scal_events"] = [None, None]
        st["_side_stream"] = None
        st["_side_stream2"] = None
        st["_main_stream"] = None
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        # re-pin host staging buffers (pinning does not survive pickling)
        self._scal_host = self._scal_host.clone().pin_memory()
        self._metrics_host = self._metrics_host.clone().pin_memory()
        self._init_scalar_ring()
        # parameters were pickled as views of the arenas (torch keeps shared storage); make
        # sure .grad views exist again
        a = self._arena
        for name, mod in (("encoder", self.encoder), ("critic", self.critic), ("actor", self.actor)):
            for pname, p in mod.named_parameters():
                off = a.offsets[name][pname]
                p.data = a.params[off:off + p.numel()].view(p.shape)
                p.grad = a.grads[off:off + p.numel()].view(p.shape)
        for pname, p in self.critic_target.named_parameters():
            off = a.offsets["critic"][pname] - a.seg["critic"][0]
            p.data = a.target[off:off + p.numel()].view(p.shape)
        self._bf16 = _bf16.Bf16State(self) if self.mode == "bf16" else None
        self._bf16_dirty = True

    @_on_device
    def refresh(self):
        """Re-derive the bf16 operand copies after parameters were changed from outside
        (load_state_dict, manual edits).  No-op in fp32 mode."""
        if self._bf16 is not None:
            self._bf16.repack_all()
        self._bf16_dirty = False
        if self.differentiable == "bf16":     # the parameter versions the copies now match (_bf16.operands)
            self._bf16_keys = {r: _bf16._param_key(getattr(self, r)) for r in ("encoder", "actor", "critic", "critic_target")}

    # ------------------------------------------------------------------ snapshot interop (train.py:192-204)
    _NETS = ("encoder", "actor", "critic")

    def load_reference_agent(self, ref):
        """Take over the state of a reference ``drqv2.DrQV2Agent`` (e.g. ``torch.load(snapshot)['agent']``,
        train.py:199-204): the four networks' parameters and the three Adam optimisers' moments and step."""
        with torch.no_grad():
            for net in self._NETS + ("critic_target",):
                getattr(self, net).load_state_dict(getattr(ref, net).state_dict())
            a = self._arena
            for net in self._NETS:
                opt = getattr(ref, f"{net}_opt")
                step = 0
                for (pname, _), rp in zip(getattr(self, net).named_parameters(), getattr(ref, net).parameters()):
                    st = opt.state.get(rp, {})
                    off = a.offsets[net][pname]
                    n = rp.numel()
                    if "exp_avg" in st:
                        a.exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
                        a.exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
                        step = max(step, int(st["step"]))
                    else:
                        a.exp_avg[off:off + n].zero_()
                        a.exp_avg_sq[off:off + n].zero_()
                self._opt_steps[net] = step
        self._bf16_dirty = True
        return self

    def export_reference_state(self):
        """State for a reference agent: ``{net: state_dict}`` for the four networks and ``{net}_opt``
        entries in ``torch.optim.Adam.state_dict()`` form (parameter ids in ``parameters()`` order), so that
        ``ref.encoder.load_state_dict(s['encoder']); ref.encoder_opt.load_state_dict(s['encoder_opt'])``
        continues training in the reference."""
        out = {net: {k: v.detach().clone() for k, v in getattr(self, net).state_dict().items()}
               for net in self._NETS + ("critic_target",)}
        a = self._arena
        for net in self._NETS:
            state = {}
            for i, (pname, p) in enumerate(getattr(self, net).named_parameters()):
                off, n = a.offsets[net][pname], p.numel()
                if self._opt_steps[net] > 0:
                    state[i] = dict(step=torch.tensor(float(self._opt_steps[net])),
                                    exp_avg=a.exp_avg[off:off + n].view(p.shape).clone(),
                                    exp_avg_sq=a.exp_avg_sq[off:off + n].view(p.shape).clone())
            group = dict(lr=self.lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False, maximize=False,
                         foreach=None, capturable=False, differentiable=False, fused=None, decoupled_weight_decay=False,
                         params=list(range(len(state) if state else len(list(getattr(self, net).parameters())))))
            out[f"{net}_opt"] = dict(state=state, param_groups=[group])
        return out

    def train(self, training=True):
        self.training = training
        self.encoder.train(training)
        self.actor.train(training)
        self.critic.train(training)

    def workspace(self, B):
        ws = self._ws.get(B)
        if ws is None:
            ws = _Workspace(B, self.action_dim, self.feature_dim, self.hidden_dim, self.obs_shape[0], self._dev,
                            fp32_encoder=self.mode == "fp32")
            if self.data_parallel:
                ws.metrics = self._arena.metrics_tail      # averaged over the ranks with the actor's gradients
            self._ws[B] = ws
        return ws

    def bf16_workspace(self, B):
        bw = self._bf16_ws.get(B)
        if bw is None:
            bw = _bf16.Bf16Workspace(B, self.action_dim, self.feature_dim, self.hidden_dim, self._bf16, self._dev)
            self._bf16_ws[B] = bw
        return bw

    def inject_draws(self, shift_obs, shift_next, eps_critic, eps_actor):
        """Parity mode: use these draws (int [B,2] (x,y) shifts, float [B,A] N(0,1) noise) for
        the next update instead of the device RNG — the four draws of one reference update
        in order (drqv2.py:241-242, utils.py:119 twice)."""
        self._injected = (shift_obs, shift_next, eps_critic, eps_actor)

    def _sync_grads(self, first, last=None, metrics=False):
        """Data-parallel: average the gradient range of nets first..last over the ranks (in stream order, on the
        current stream, inside the graph); metrics=True (with the actor, the arena's last segment) takes the
        update's 8 metrics along in the same all-reduce - they are batch means (drqv2.py:191-196,223-226), so
        the mean over ranks of the shard means is the global-batch value.  No-op for a single process."""
        if not self.data_parallel:
            return
        a = self._arena
        off = a.seg[first][0]
        end = a.seg[last or first][0] + a.seg[last or first][2]
        if metrics:
            assert end == a.total
            end += 8
        _dist.average_(a._grads_full[off:end])

    def _p(self, net, pname):
        return self._arena.ptr("params", net, pname)

    def _g(self, net, pname):
        return self._arena.ptr("grads", net, pname)

    def _t(self, pname):
        return self._arena.target.data_ptr() + F32 * self._arena.offsets["critic"][pname] - F32 * self._arena.seg["critic"][0]

    # ------------------------------------------------------------------ act
    @_on_device
    def act(self, obs, step, eval_mode):
        """drqv2.py:164-175: encoder + actor at batch 1, mean in eval mode, else an
        exploration sample (noise not clipped), uniform before num_expl_steps."""
        A, Fd, H = self.action_dim, self.feature_dim, self.hidden_dim
        obs_t = torch.as_tensor(obs)
        batched = obs_t.dim() == 4
        if not batched:
            obs_t = obs_t.unsqueeze(0)
        n = obs_t.shape[0]
        w = self._act_ws.get(n)
        dev = self._dev
        if w is None:
            w = dict(obs=torch.zeros(n, *self.obs_shape, dtype=torch.uint8, device=dev),
                     acts=[torch.zeros(n * 32 * PLANE, device=dev) for _ in range(3)],
                     feat=torch.zeros(n, REPR_DIM, device=dev),
                     partial=torch.zeros(_splitk_for(n) * n * Fd, device=dev),
                     h=torch.zeros(n, Fd, device=dev), p1=torch.zeros(n, H, device=dev),
                     p2=torch.zeros(n, H, device=dev), mu_pre=torch.zeros(n, A, device=dev),
                     eps=torch.zeros(n, A, device=dev), out=torch.zeros(n, A, device=dev),
                     host_in=torch.zeros(n, *self.obs_shape, dtype=torch.uint8).pin_memory(),
                     host_out=torch.zeros(n, A).pin_memory(), graph={})
            if self.mode == "bf16":
                w.update(_bf16.act_workspace(self, n, dev))
            self._act_ws[n] = w
        if obs_t.is_cuda:
            w["obs"].copy_(obs_t, non_blocking=True)
        else:
            w["host_in"].copy_(obs_t)
            w["obs"].copy_(w["host_in"], non_blocking=True)
        stddev = utils.schedule(self.stddev_schedule, step)
        self._scal_host[8] = stddev
        self._scal_dev[8:9].copy_(self._scal_host[8:9], non_blocking=True)
        if self._bf16_dirty:
            self.refresh()
        sample = not eval_mode
        key = bool(sample)
        g = w["graph"].get(key)
        if g is None:
            # warm-up (also opts kernels in to big smem): its action is this call's, and a capture runs nothing - so
            # the first call draws its noise once, as every later replay does
            self._act_body(w, n, sample)
            if self.use_cuda_graph:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with _capture(g):
                    self._act_body(w, n, sample)
                w["graph"][key] = g
        else:
            g.replay()
        w["host_out"].copy_(w["out"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        action = w["host_out"].numpy().copy()
        if sample and step < self.num_expl_steps:
            # drqv2.py:174 action.uniform_(-1.0, 1.0): torch's global generator, so torch.manual_seed reproduces it
            action = torch.empty(action.shape, dtype=torch.float32).uniform_(-1.0, 1.0).numpy()
        return action if batched else action[0]

    def _act_body(self, w, n, sample):
        A, Fd, H = self.action_dim, self.feature_dim, self.hidden_dim
        if self.mode == "bf16":
            return _bf16.act_body(self, w, n, sample)
        if sample:   # exploration noise draw (utils.py:119)
            call("drq_rng_normal_f32", self._seed, self._counter.data_ptr(), w["eps"].data_ptr(), n * A, _stream())
            call("drq_counter_advance", self._counter.data_ptr(), _stream())
        ew = [self._p("encoder", f"convnet.{i}.weight") for i in (0, 2, 4, 6)]
        eb = [self._p("encoder", f"convnet.{i}.bias") for i in (0, 2, 4, 6)]
        _encoder_fwd(w["obs"].data_ptr(), 0, ew, eb, [a.data_ptr() for a in w["acts"]], w["feat"].data_ptr(),
                     n, self.obs_shape[0])
        pa = lambda k: self._p("actor", k)
        _trunk_fwd(w["feat"].data_ptr(), n, pa("trunk.0.weight"), pa("trunk.0.bias"), pa("trunk.1.weight"),
                   pa("trunk.1.bias"), Fd, w["partial"].data_ptr(), w["h"].data_ptr(), Fd)
        _linear_fwd(w["h"].data_ptr(), Fd, pa("policy.0.weight"), pa("policy.0.bias"), w["p1"].data_ptr(), H, n, H, Fd, True)
        _linear_fwd(w["p1"].data_ptr(), H, pa("policy.2.weight"), pa("policy.2.bias"), w["p2"].data_ptr(), H, n, H, H, True)
        _linear_fwd(w["p2"].data_ptr(), H, pa("policy.4.weight"), pa("policy.4.bias"), w["mu_pre"].data_ptr(), A, n, A, H, False)
        call("drq_actor_sample", w["mu_pre"].data_ptr(), w["eps"].data_ptr() if sample else None,
             self._sc("stddev"), 0.0, w["out"].data_ptr(), A, None, None, n, A, _stream())

    # ------------------------------------------------------------------ update
    def update(self, replay_iter, step):
        """drqv2.py:230-262.  Returns {} (and does not advance the iterator) when
        step % update_every_steps != 0."""
        ws = self.update_async(replay_iter, step)
        if ws is None or not self.use_tb:
            return dict()
        return self.read_metrics(ws)

    @_on_device
    def read_metrics(self, ws):
        """The metrics of the update last enqueued on the current stream (one 32-byte D2H copy and a
        stream synchronise; drqv2.py:191-196,223-226)."""
        self._metrics_host.copy_(ws.metrics, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return dict(zip(METRIC_KEYS, self._metrics_host.tolist()))

    @_on_device
    def update_async(self, replay_iter, step):
        """update() without the metrics read-back: enqueues the whole update on the current stream and
        returns its workspace (None when step % update_every_steps != 0) - no host synchronisation, so
        several agents can be driven from one thread (ensemble.AgentEnsemble)."""
        if step % self.update_every_steps != 0:
            return None
        ring = None
        if hasattr(replay_iter, "next_into"):
            # GPU-resident ring: sample + n-step gather straight into the static buffers - or, in the tensor-core mode,
            # no gather of the frame stacks at all: conv1's loader reads them from the ring by index
            B = replay_iter.batch_size
            ws = self.workspace(B)
            fetch = lambda: replay_iter.next_into(ws.obs[:B], ws.action, ws.reward, ws.discount, ws.obs[B:])
            if self.mode == "bf16" and self.ring_direct and hasattr(replay_iter, "ring_source"):
                ring = replay_iter
        else:
            fetch = None
            pf, self._prefetch = self._prefetch, None
            if pf is not None and pf["it"] is replay_iter:
                # the batch was pulled and its host->device copy started while the previous update ran
                B = pf["B"]
                ws = self.workspace(B)
                torch.cuda.current_stream().wait_event(pf["ready"])
                st = pf["stage"]
                for dst, src in ((ws.obs, st["obs"]), (ws.action, st["action"]), (ws.reward, st["reward"]),
                                 (ws.discount, st["discount"])):
                    dst.copy_(src, non_blocking=True)
                st["free"].record()
            else:
                obs, action, reward, discount, next_obs = next(replay_iter)
                B = obs.shape[0]
                ws = self.workspace(B)
                self._load_batch(ws, obs, action, reward, discount, next_obs)
        self._host_scalars(step)
        if self._bf16_dirty:
            self.refresh()
        inj = self._injected
        if inj is not None:
            self._injected = None
            ws.shift[:B].copy_(torch.as_tensor(inj[0]).to(torch.int32).view(B, 2))
            ws.shift[B:].copy_(torch.as_tensor(inj[1]).to(torch.int32).view(B, 2))
            ws.eps_c.copy_(torch.as_tensor(inj[2]).view(B, -1))
            ws.eps_a.copy_(torch.as_tensor(inj[3]).view(B, -1))
        # a captured graph bakes in the ring iterator's pointers and constants (frames, episode table, sampler
        # counter, n-step, discount): one graph per source, not per batch size alone
        src = getattr(replay_iter, "graph_key", None) if fetch is not None else None
        if fetch is not None and src is None:
            src = id(replay_iter)
        key = (B, src, inj is None, ring is not None)
        if fetch is not None and hasattr(replay_iter, "check_ready"):
            replay_iter.check_ready()              # a replayed graph cannot raise: an empty ring is refused here
        state = self._graphs.get(key) if self.use_cuda_graph else None
        if self.data_parallel and self.dp_reserve_sms:
            # grids of the persistent kernels are fixed at launch / capture: leave SMs to the NCCL CTAs that run beside them
            call("drq_set_sm_limit", _lib.lib().drq_device_sm_count() - self.dp_reserve_sms)
        try:
            if not self.use_cuda_graph:
                self._update_body(ws, fetch, draw=inj is None, ring=ring)
            elif state is None:
                # first call at this shape runs eagerly: it is the warm-up (lazy module loading,
                # shared-memory opt-in) that must not happen inside a capture
                self._update_body(ws, fetch, draw=inj is None, ring=ring)
                self._graphs[key] = "warm"
            else:
                if state == "warm":
                    torch.cuda.synchronize()
                    state = torch.cuda.CUDAGraph()
                    with _capture(state, self._capture_stream()):
                        self._update_body(ws, fetch, draw=inj is None, ring=ring)
                    self._graphs[key] = state
                state.replay()
        except BaseException:
            # the device cursor of the scalar ring may or may not have advanced: put it back in step with the host's
            # count, so that later updates do not read another update's slot
            torch.cuda.synchronize()
            self._scal_cursor.fill_(self._scal_enq)
            raise
        finally:
            if self.data_parallel and self.dp_reserve_sms:
                call("drq_set_sm_limit", 148)
        for net in self._opt_steps:
            self._opt_steps[net] += 1
        self._scalars_enqueued()
        if fetch is None and self.prefetch:
            self._start_prefetch(replay_iter, ws)
        return ws

    def _start_prefetch(self, replay_iter, ws):
        """Pull the next host batch now and copy it to device staging buffers on a side stream, so the
        PCIe transfer (32.5 MB at B=256) overlaps this update's kernels.  The reference's DataLoader
        workers run ahead of the consumer in the same way (replay_buffer.py:181-186)."""
        try:
            batch = next(replay_iter)
        except StopIteration:
            return
        obs, action, reward, discount, next_obs = (torch.as_tensor(t) for t in batch)
        B = obs.shape[0]
        st = self._stage.get(B)
        if st is None:
            w = self.workspace(B)
            st = dict(obs=torch.empty_like(w.obs), action=torch.empty_like(w.action), reward=torch.empty_like(w.reward),
                      discount=torch.empty_like(w.discount), free=torch.cuda.Event(), stream=torch.cuda.Stream())
            st["free"].record()
            self._stage[B] = st
        side = st["stream"]
        side.wait_event(st["free"])                  # the previous consumer of the staging buffers is done
        with torch.cuda.stream(side):
            st["obs"][:B].copy_(obs.view(st["obs"][:B].shape), non_blocking=True)
            st["obs"][B:].copy_(next_obs.view(st["obs"][B:].shape), non_blocking=True)
            st["action"].copy_(action.view(st["action"].shape), non_blocking=True)
            st["reward"].copy_(reward.view(st["reward"].shape), non_blocking=True)
            st["discount"].copy_(discount.view(st["discount"].shape), non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(side)
        self._prefetch = dict(it=replay_iter, B=B, stage=st, ready=ready, hold=batch)

    def _load_batch(self, ws, obs, action, reward, discount, next_obs):
        B = ws.B
        for dst, src in ((ws.obs[:B], obs), (ws.obs[B:], next_obs), (ws.action, action),
                         (ws.reward, reward), (ws.discount, discount)):
            src = torch.as_tensor(src)
            if src.is_cuda and src.data_ptr() == dst.data_ptr():
                continue
            dst.copy_(src.view(dst.shape), non_blocking=True)

    _SCAL_SLOTS = 256

    def _init_scalar_ring(self):
        """Pinned ring of per-update scalars the device reads in stream order (drq_scalars_fetch): the host may
        enqueue up to _SCAL_SLOTS / 2 updates ahead of the device without overwriting a slot still to be read."""
        self._scal_ring = torch.zeros(self._SCAL_SLOTS, SCAL_SLOT, dtype=torch.float32).pin_memory()
        self._scal_cursor = torch.zeros(1, dtype=torch.int64, device=self._dev)
        self._scal_enq = 0
        self._scal_events = [None, None]

    @property
    def _opt_step(self):
        """optimiser steps taken by update() (the three counts differ only when the stage API is driven unevenly)"""
        return self._opt_steps["critic"]

    def _sc(self, net):
        """device pointer of `net`'s Adam scalars (or of 'stddev') for the update being enqueued"""
        return self._scal_dev.data_ptr() + F32 * SCAL_OFF[net]

    def _host_scalars(self, step, stepping=("encoder", "critic", "actor")):
        """Adam scalars of the coming step of the optimisers in `stepping` (each with its own step count, as
        torch.optim.Adam) and stddev(step) into the ring slot the device reads next (step None: the stddev last
        written, unchanged - an optimiser step on its own)."""
        half = self._SCAL_SLOTS // 2
        slot = self._scal_enq % self._SCAL_SLOTS
        if slot % half == 0:                       # entering a half of the ring: its previous readers must be done
            ev = self._scal_events[slot // half]
            if ev is not None:
                ev.synchronize()
        for net in stepping:
            o = SCAL_OFF[net]
            self._scal_host[o:o + 8] = torch.from_numpy(utils.adam_scalars(self.lr, self._opt_steps[net] + 1))
        if step is not None:
            stddev = utils.schedule(self.stddev_schedule, step)
            self._scal_host[SCAL_OFF["stddev"]] = stddev
            self._stddev = stddev
        self._scal_ring[slot].copy_(self._scal_host)

    def _fetch_scalars(self):
        """device side of _host_scalars: one tiny kernel, in stream order (graph-capturable)"""
        call("drq_scalars_fetch", self._scal_ring.data_ptr(), self._SCAL_SLOTS, self._scal_cursor.data_ptr(),
             self._scal_dev.data_ptr(), _stream())

    def _scalars_enqueued(self):
        """host bookkeeping after an update that consumes one ring slot has been enqueued"""
        half = self._SCAL_SLOTS // 2
        slot = self._scal_enq % self._SCAL_SLOTS
        if (slot + 1) % half == 0:
            ev = torch.cuda.Event()
            ev.record()
            self._scal_events[slot // half] = ev
        self._scal_enq += 1

    def _encoder_side_stream(self):
        """Second stream for the encoder backward + encoder_opt.step() of the bf16 update (None: run in line).
        Data-parallel updates use it too: the critic's gradient all-reduce, critic_opt.step() and the actor pass run
        beside the encoder backward; the encoder's own (30 k floats) all-reduce follows the join (_update_body)."""
        if not self.overlap_encoder_backward or self.mode != "bf16":
            return None
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self._dev, priority=self._prio[1])
        return self._side_stream

    def _wgrad_side_stream(self):
        """Third stream: the weight-gradient GEMMs / bias-gradient sums run beside the data-gradient chain."""
        if not self.overlap_encoder_backward or self.mode != "bf16":
            return None
        if self._side_stream2 is None:
            self._side_stream2 = torch.cuda.Stream(device=self._dev, priority=self._prio[2])
        return self._side_stream2

    def _capture_stream(self):
        """Stream the update graph is captured on (None: torch's own capture stream).  Kernel nodes keep the priority of
        the stream they were captured on, so the three streams of the schedule can be ranked: when CTAs of two ready
        kernels compete for SMs, the block scheduler takes the higher priority (lower number) first."""
        if self._prio[0] == 0 or self.mode != "bf16":
            return None
        if self._main_stream is None:
            self._main_stream = torch.cuda.Stream(device=self._dev, priority=self._prio[0])
        return self._main_stream

    def _update_body(self, ws, fetch=None, draw=True, ring=None):
        """Everything of one update that runs on the device, in stream order; no host sync."""
        B = ws.B
        s = _stream()
        # one launch: this update's host scalars (Adam bias corrections, stddev) out of the pinned ring and - unless
        # the draws were injected - the four random draws of drqv2.py:34 (x2) and utils.py:119 (x2), counter += 1
        head = (self._scal_ring.data_ptr(), self._SCAL_SLOTS, self._scal_cursor.data_ptr(),
                self._scal_dev.data_ptr(), self._seed, self._counter.data_ptr(), self.aug.pad,
                ws.shift[:B].data_ptr() if draw else None, ws.shift[B:].data_ptr(), ws.eps_c.data_ptr(), ws.eps_a.data_ptr(),
                B, self.action_dim)
        ws.ring_src = None
        if ring is not None:
            # ... and in the same launch the replay sample (replay_buffer.py:142-160): indices, action, n-step reward and
            # discount.  The frame stacks stay in the ring; conv1 reads them through (ep_start, idx).
            ws.ring_src = ring.ring_source()
            tail = (ctypes.byref(ws.ring_src), ws.action.data_ptr(), ws.reward.data_ptr(), ws.discount.data_ptr())
            side = self._wgrad_side_stream() if self.split_prologue else None
            if side is None:
                call("drq_update_prologue_ring", *head, *tail, s)
            else:
                # conv1 waits for the shifts and the sample only; the scalars (a read of pinned host memory), the noise and
                # the n-step chain run beside it and are joined in front of the first kernel behind the encoder
                call("drq_update_prologue_ring_part", *head, *tail, 1, s)
                main = torch.cuda.current_stream()
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    call("drq_update_prologue_ring_part", *head, *tail, 2, _stream())
        else:
            call("drq_update_prologue", *head, s)
            if fetch is not None:
                fetch()
        if self.mode == "bf16":
            bw = self.bf16_workspace(B)
            _bf16.encode(self, ws, bw)
            if ring is not None and self.split_prologue and self._wgrad_side_stream() is not None:
                torch.cuda.current_stream().wait_stream(self._wgrad_side_stream())
            _bf16.critic_pass(self, ws, bw)
            _bf16.actor_pass(self, ws, bw)
            side = self._encoder_side_stream()
            if side is not None:                    # the encoder backward ran beside the actor pass
                torch.cuda.current_stream().wait_stream(side)
                if self.data_parallel:              # encoder_opt.step() of a data-parallel update: after its all-reduce
                    self._sync_grads("encoder")
                    self._bf16.step_encoder()
            return
        self._encode(ws)
        self._critic_pass(ws, ws.feat[:B], ws.feat[B:], encoder_grad=True)
        self._actor_pass(ws, ws.feat[:B])

    def _encode(self, ws):
        B = ws.B
        ew = [self._p("encoder", f"convnet.{i}.weight") for i in (0, 2, 4, 6)]
        eb = [self._p("encoder", f"convnet.{i}.bias") for i in (0, 2, 4, 6)]
        _encoder_fwd(ws.obs.data_ptr(), ws.shift.data_ptr(), ew, eb, [a.data_ptr() for a in ws.acts],
                     ws.feat.data_ptr(), 2 * B, self.obs_shape[0], self.aug.pad)

    def _q_strides(self):
        co = self._arena.offsets["critic"]
        return co["Q2.0.weight"] - co["Q1.0.weight"]   # floats between Q1.* and Q2.* tensors

    def _twin_q_fwd(self, pfn, x, c1, c2, q, B):
        """Both Q heads in one batched launch per layer (drqv2.py:103-111,118-119)."""
        Fd, A, H = self.feature_dim, self.action_dim, self.hidden_dim
        qs = self._q_strides()
        _linear_fwd(x, Fd + A, pfn("Q1.0.weight"), pfn("Q1.0.bias"), c1, H, B, H, Fd + A, True, batch=2,
                    bs=(0, qs, B * H, qs, 0))
        _linear_fwd(c1, H, pfn("Q1.2.weight"), pfn("Q1.2.bias"), c2, H, B, H, H, True, batch=2,
                    bs=(B * H, qs, B * H, qs, 0))
        _linear_fwd(c2, H, pfn("Q1.4.weight"), pfn("Q1.4.bias"), q, 1, B, 1, H, False, batch=2,
                    bs=(B * H, qs, B, qs, 0))

    def _critic_pass(self, ws, feat, feat_next, encoder_grad):
        """update_critic (drqv2.py:177-204) + critic/encoder Adam, no host sync."""
        B, A, Fd, H = ws.B, self.action_dim, self.feature_dim, self.hidden_dim
        s = _stream()
        pc = lambda k: self._p("critic", k)
        gc = lambda k: self._g("critic", k)
        pa = lambda k: self._p("actor", k)
        std_ptr = self._sc("stddev")
        qs = self._q_strides()
        featp, featn = feat.data_ptr(), feat_next.data_ptr()
        # --- target: online actor on next features -> clipped sample (drqv2.py:181-183)
        _trunk_fwd(featn, B, pa("trunk.0.weight"), pa("trunk.0.bias"), pa("trunk.1.weight"), pa("trunk.1.bias"),
                   Fd, ws.partial.data_ptr(), ws.hA.data_ptr(), Fd)
        _linear_fwd(ws.hA.data_ptr(), Fd, pa("policy.0.weight"), pa("policy.0.bias"), ws.p1.data_ptr(), H, B, H, Fd, True)
        _linear_fwd(ws.p1.data_ptr(), H, pa("policy.2.weight"), pa("policy.2.bias"), ws.p2.data_ptr(), H, B, H, H, True)
        _linear_fwd(ws.p2.data_ptr(), H, pa("policy.4.weight"), pa("policy.4.bias"), ws.mu_pre.data_ptr(), A, B, A, H, False)
        call("drq_actor_sample", ws.mu_pre.data_ptr(), ws.eps_c.data_ptr(), std_ptr, float(self.stddev_clip),
             ws.xT.data_ptr() + F32 * Fd, Fd + A, None, None, B, A, s)
        # --- target critic on (next features, next action) (drqv2.py:184)
        _trunk_fwd(featn, B, self._t("trunk.0.weight"), self._t("trunk.0.bias"), self._t("trunk.1.weight"),
                   self._t("trunk.1.bias"), Fd, ws.partial.data_ptr(), ws.xT.data_ptr(), Fd + A)
        self._twin_q_fwd(self._t, ws.xT.data_ptr(), ws.c1.data_ptr(), ws.c2.data_ptr(), ws.tq.data_ptr(), B)
        # --- online critic on (features, action) (drqv2.py:188)
        _trunk_fwd(featp, B, pc("trunk.0.weight"), pc("trunk.0.bias"), pc("trunk.1.weight"), pc("trunk.1.bias"),
                   Fd, ws.partial.data_ptr(), ws.xC.data_ptr(), Fd + A, ws.xhatC.data_ptr(), ws.rstdC.data_ptr())
        call("drq_copy2d_f32", ws.action.data_ptr(), A, ws.xC.data_ptr() + F32 * Fd, Fd + A, B, A, s)
        self._twin_q_fwd(pc, ws.xC.data_ptr(), ws.c1.data_ptr(), ws.c2.data_ptr(), ws.q.data_ptr(), B)
        # --- TD target, loss, dL/dq (drqv2.py:185-189)
        q1, q2 = ws.q.data_ptr(), ws.q.data_ptr() + F32 * B
        call("drq_critic_loss", q1, q2, ws.tq.data_ptr(), ws.tq.data_ptr() + F32 * B, ws.reward.data_ptr(),
             ws.discount.data_ptr(), ws.dq.data_ptr(), ws.dq.data_ptr() + F32 * B, ws.target_q.data_ptr(),
             ws.metrics.data_ptr(), B, s)
        # --- backward through the twin Q heads (both heads per launch)
        BH = B * H
        c1, c2, dc1, dc2, dq = (t.data_ptr() for t in (ws.c1, ws.c2, ws.dc1, ws.dc2, ws.dq))
        _linear_wgrad(dq, 1, c2, H, gc("Q1.4.weight"), B, 1, H, batch=2, bs=(B, BH, qs, 0, 0))
        _colsum(dq, 1, gc("Q1.4.bias"), B, 1, batch=2, bs_x=B, bs_out=qs)
        _linear_dgrad(dq, 1, pc("Q1.4.weight"), dc2, H, B, 1, H, mask=c2, ldmask=H, batch=2, bs=(B, qs, BH, 0, BH))
        _linear_wgrad(dc2, H, c1, H, gc("Q1.2.weight"), B, H, H, batch=2, bs=(BH, BH, qs, 0, 0))
        _colsum(dc2, H, gc("Q1.2.bias"), B, H, batch=2, bs_x=BH, bs_out=qs)
        _linear_dgrad(dc2, H, pc("Q1.2.weight"), dc1, H, B, H, H, mask=c1, ldmask=H, batch=2, bs=(BH, qs, BH, 0, BH))
        _linear_wgrad(dc1, H, ws.xC.data_ptr(), Fd + A, gc("Q1.0.weight"), B, H, Fd + A, batch=2, bs=(BH, 0, qs, 0, 0))
        _colsum(dc1, H, gc("Q1.0.bias"), B, H, batch=2, bs_x=BH, bs_out=qs)
        # d[h] = dc1[Q1] @ W1[Q1][:, :F] + dc1[Q2] @ W1[Q2][:, :F]
        _linear_dgrad(dc1, H, pc("Q1.0.weight"), ws.dx.data_ptr(), Fd + A, B, H, Fd + A, n_cols=Fd)
        _linear_dgrad(dc1 + F32 * BH, H, pc("Q2.0.weight"), ws.dx.data_ptr(), Fd + A, B, H, Fd + A, n_cols=Fd, acc=1)
        # --- trunk backward: tanh, LayerNorm, Linear
        call("drq_ln_tanh_bwd", ws.dx.data_ptr(), Fd + A, ws.xC.data_ptr(), Fd + A, ws.xhatC.data_ptr(),
             ws.rstdC.data_ptr(), pc("trunk.1.weight"), ws.dz.data_ptr(), gc("trunk.1.weight"),
             gc("trunk.1.bias"), None, 0, B, Fd, 1, 0, s)
        _linear_wgrad(ws.dz.data_ptr(), Fd, featp, REPR_DIM, gc("trunk.0.weight"), B, Fd, REPR_DIM)
        _colsum(ws.dz.data_ptr(), Fd, gc("trunk.0.bias"), B, Fd)
        if encoder_grad:
            self._encoder_bwd(ws, featp)
        # --- critic_opt.step(); encoder_opt.step() (drqv2.py:201-202): [encoder|critic] is one range
        a = self._arena
        ranges = [("critic", a.seg["critic"][0], a.seg["critic"][2])]
        if encoder_grad:
            self._sync_grads("encoder", "critic")
            if self._opt_steps["encoder"] == self._opt_steps["critic"]:   # same Adam scalars: [encoder|critic] is one range
                ranges = [("critic", a.seg["encoder"][0], a.seg["encoder"][2] + a.seg["critic"][2])]
            else:
                ranges.append(("encoder", a.seg["encoder"][0], a.seg["encoder"][2]))
        else:
            self._sync_grads("critic")
        for net, off, n in ranges:
            call("drq_adam_step", a.params.data_ptr() + F32 * off, a.grads.data_ptr() + F32 * off,
                 a.exp_avg.data_ptr() + F32 * off, a.exp_avg_sq.data_ptr() + F32 * off, n, self._sc(net), s)

    def _encoder_bwd(self, ws, featp):
        """Backward of the 4-conv encoder on the obs half of the batch (drqv2.py:200)."""
        B, Fd = ws.B, self.feature_dim
        s = _stream()
        pe = lambda k: self._p("encoder", k)
        ge = lambda k: self._g("encoder", k)
        d = [t.data_ptr() for t in ws.dpre]
        acts = [t.data_ptr() for t in ws.acts]
        wsp = ws.wgrad_ws.data_ptr()
        # d(features) = dz @ W_trunk, masked by ReLU and scattered into the wide plane of conv4's output
        _gemm(ws.dz.data_ptr(), Fd, 1, self._p("critic", "trunk.0.weight"), REPR_DIM, 1, d[3], 32 * PLANE,
              B, REPR_DIM, Fd, mask=featp, ldmask=REPR_DIM, epi=EPI_MASK_WIDE)
        for layer, hout in ((3, 35), (2, 37), (1, 39)):
            k = 2 * layer
            call("drq_conv3x3_wgrad_f32", acts[layer - 1], d[layer], wsp, ge(f"convnet.{k}.weight"),
                 ge(f"convnet.{k}.bias"), B, hout, s)
            call("drq_conv3x3_dgrad_f32", d[layer], pe(f"convnet.{k}.weight"), acts[layer - 1], d[layer - 1],
                 B, hout, s)
        call("drq_conv1_wgrad_f32", ws.obs.data_ptr(), ws.shift.data_ptr(), d[0], wsp, ge("convnet.0.weight"),
             ge("convnet.0.bias"), B, self.obs_shape[0], self.aug.pad, s)

    def _actor_pass(self, ws, feat, soft_update=True):
        """update_actor (drqv2.py:206-228) + actor Adam and, when called from update(), the soft target update
        (drqv2.py:259-260) in the same launch."""
        B, A, Fd, H = ws.B, self.action_dim, self.feature_dim, self.hidden_dim
        s = _stream()
        pc = lambda k: self._p("critic", k)
        pa = lambda k: self._p("actor", k)
        ga = lambda k: self._g("actor", k)
        std_ptr = self._sc("stddev")
        qs = self._q_strides()
        featp = feat.data_ptr()
        BH = B * H
        # actor forward on detached features, sample with clipped noise (drqv2.py:209-211)
        _trunk_fwd(featp, B, pa("trunk.0.weight"), pa("trunk.0.bias"), pa("trunk.1.weight"), pa("trunk.1.bias"),
                   Fd, ws.partial.data_ptr(), ws.hA.data_ptr(), Fd, ws.xhatA.data_ptr(), ws.rstdA.data_ptr())
        _linear_fwd(ws.hA.data_ptr(), Fd, pa("policy.0.weight"), pa("policy.0.bias"), ws.p1.data_ptr(), H, B, H, Fd, True)
        _linear_fwd(ws.p1.data_ptr(), H, pa("policy.2.weight"), pa("policy.2.bias"), ws.p2.data_ptr(), H, B, H, H, True)
        _linear_fwd(ws.p2.data_ptr(), H, pa("policy.4.weight"), pa("policy.4.bias"), ws.mu_pre.data_ptr(), A, B, A, H, False)
        call("drq_actor_sample", ws.mu_pre.data_ptr(), ws.eps_a.data_ptr(), std_ptr, float(self.stddev_clip),
             ws.xA.data_ptr() + F32 * Fd, Fd + A, ws.mu.data_ptr(), ws.metrics.data_ptr() + F32 * 6, B, A, s)
        # the just-updated critic on (features, action) (drqv2.py:213-216)
        _trunk_fwd(featp, B, pc("trunk.0.weight"), pc("trunk.0.bias"), pc("trunk.1.weight"), pc("trunk.1.bias"),
                   Fd, ws.partial.data_ptr(), ws.xA.data_ptr(), Fd + A)
        self._twin_q_fwd(pc, ws.xA.data_ptr(), ws.c1.data_ptr(), ws.c2.data_ptr(), ws.q.data_ptr(), B)
        call("drq_actor_loss", ws.q.data_ptr(), ws.q.data_ptr() + F32 * B, ws.dq.data_ptr(),
             ws.dq.data_ptr() + F32 * B, ws.metrics.data_ptr() + F32 * 5, B, s)
        # backward: Q heads data-gradient only (critic weight grads are discarded by the reference)
        c1, c2, dc1, dc2, dq = (t.data_ptr() for t in (ws.c1, ws.c2, ws.dc1, ws.dc2, ws.dq))
        _linear_dgrad(dq, 1, pc("Q1.4.weight"), dc2, H, B, 1, H, mask=c2, ldmask=H, batch=2, bs=(B, qs, BH, 0, BH))
        _linear_dgrad(dc2, H, pc("Q1.2.weight"), dc1, H, B, H, H, mask=c1, ldmask=H, batch=2, bs=(BH, qs, BH, 0, BH))
        _linear_dgrad(dc1, H, pc("Q1.0.weight"), ws.dact.data_ptr(), A, B, H, Fd + A, w_col0=Fd, n_cols=A)
        _linear_dgrad(dc1 + F32 * BH, H, pc("Q2.0.weight"), ws.dact.data_ptr(), A, B, H, Fd + A, w_col0=Fd, n_cols=A, acc=1)
        call("drq_actor_sample_bwd", ws.dact.data_ptr(), A, ws.mu.data_ptr(), ws.dmu_pre.data_ptr(), None, 0, B, A, 1, 0, s)
        # actor MLP backward
        dmu, p1, p2, dp1, dp2 = (t.data_ptr() for t in (ws.dmu_pre, ws.p1, ws.p2, ws.dp1, ws.dp2))
        _linear_wgrad(dmu, A, p2, H, ga("policy.4.weight"), B, A, H)
        _colsum(dmu, A, ga("policy.4.bias"), B, A)
        _linear_dgrad(dmu, A, pa("policy.4.weight"), dp2, H, B, A, H, mask=p2, ldmask=H)
        _linear_wgrad(dp2, H, p1, H, ga("policy.2.weight"), B, H, H)
        _colsum(dp2, H, ga("policy.2.bias"), B, H)
        _linear_dgrad(dp2, H, pa("policy.2.weight"), dp1, H, B, H, H, mask=p1, ldmask=H)
        _linear_wgrad(dp1, H, ws.hA.data_ptr(), Fd, ga("policy.0.weight"), B, H, Fd)
        _colsum(dp1, H, ga("policy.0.bias"), B, H)
        _linear_dgrad(dp1, H, pa("policy.0.weight"), ws.dhA.data_ptr(), Fd, B, H, Fd)
        call("drq_ln_tanh_bwd", ws.dhA.data_ptr(), Fd, ws.hA.data_ptr(), Fd, ws.xhatA.data_ptr(),
             ws.rstdA.data_ptr(), pa("trunk.1.weight"), ws.dz.data_ptr(), ga("trunk.1.weight"),
             ga("trunk.1.bias"), None, 0, B, Fd, 1, 0, s)
        _linear_wgrad(ws.dz.data_ptr(), Fd, featp, REPR_DIM, ga("trunk.0.weight"), B, Fd, REPR_DIM)
        _colsum(ws.dz.data_ptr(), Fd, ga("trunk.0.bias"), B, Fd)
        self._sync_grads("actor", metrics=True)
        # actor_opt.step(), in update() fused with the soft target update of the (already stepped) critic
        a = self._arena
        off, n = a.seg["actor"][0], a.seg["actor"][2]
        coff, cn = a.seg["critic"][0], a.seg["critic"][2]
        tau = float(self.critic_target_tau)
        if soft_update:
            call("drq_adam_ema_step", a.params.data_ptr() + F32 * off, a.grads.data_ptr() + F32 * off,
                 a.exp_avg.data_ptr() + F32 * off, a.exp_avg_sq.data_ptr() + F32 * off, n, self._sc("actor"),
                 a.params.data_ptr() + F32 * coff, a.target.data_ptr(), cn, tau, float(1 - tau), s)
        else:
            call("drq_adam_step", a.params.data_ptr() + F32 * off, a.grads.data_ptr() + F32 * off,
                 a.exp_avg.data_ptr() + F32 * off, a.exp_avg_sq.data_ptr() + F32 * off, n, self._sc("actor"), s)

    # ------------------------------------------------------------------ public stage API
    def _stage_inputs(self, ws, **named):
        for k, v in named.items():
            dst = getattr(ws, k)
            v = torch.as_tensor(v, device=self._dev)
            if v.data_ptr() != dst.data_ptr():
                dst.copy_(v.view(dst.shape))

    def _stage_features(self, ws, feat, row0):
        """Encoded features [B, 39200] (reference order c*1225 + yx, drqv2.py:66) into the update's buffers: the
        fp32 feature matrix, or in bf16 mode the TB operand in the encoder-output order (one pack kernel)."""
        B = ws.B
        feat = torch.as_tensor(feat, device=self._dev)
        if self.mode == "fp32":
            dst = ws.feat[row0 * B:(row0 + 1) * B]
            if feat.data_ptr() != dst.data_ptr():
                dst.copy_(feat)
            return
        bw = self.bf16_workspace(B)
        feat = feat.float().contiguous()
        call("drq_pack_features_tb", feat.data_ptr(), bw.feat.ptr(row=row0 * bw.RB), B, _stream())

    def _stage_noise(self, dst, which):
        """N(0,1) draw of a stage-API call (utils.py:119): the injected one (inject_draws slot `which`), else the
        device generator."""
        inj = self._injected
        if inj is not None and inj[which] is not None:
            dst.copy_(torch.as_tensor(inj[which]).view(dst.shape))
            inj = list(inj)
            inj[which] = None
            self._injected = inj if any(v is not None for v in inj[2:]) else None
            return
        call("drq_rng_normal_f32", self._seed, self._counter.data_ptr(), dst.data_ptr(), dst.numel(), _stream())
        call("drq_counter_advance", self._counter.data_ptr(), _stream())

    def _stage_scalars(self, step, stepping):
        self._host_scalars(step, stepping)
        self._fetch_scalars()
        self._scalars_enqueued()
        if self._bf16_dirty:
            self.refresh()

    def update_critic(self, obs, action, reward, discount, next_obs, step):
        """drqv2.py:177-204 on encoded features [B, 39200]: critic loss, backward, critic_opt.step().
        fp32 mode: when `obs` is the feature buffer this agent's own encode produced (as inside update()), the
        encoder receives its gradient and steps too, as autograd would; any other tensor is a detached input
        and leaves the encoder untouched (a reference encoder whose gradients are None is skipped by Adam in the
        same way).  bf16 mode: features are always external (the tensor-core encoder keeps its output in its own
        bf16 layout), so only the critic is updated."""
        with torch.cuda.device(self._dev):
            B = obs.shape[0]
            ws = self.workspace(B)
            own = self.mode == "fp32" and obs.data_ptr() == ws.feat.data_ptr()
            self._stage_features(ws, obs, 0)
            self._stage_features(ws, next_obs, 1)
            self._stage_inputs(ws, action=action, reward=reward, discount=discount)
            stepping = ("encoder", "critic") if own else ("critic",)
            self._stage_noise(ws.eps_c, 2)
            self._stage_scalars(step, stepping)
            if self.mode == "fp32":
                self._critic_pass(ws, ws.feat[:B], ws.feat[B:], encoder_grad=own)
            else:
                _bf16.critic_pass(self, ws, self.bf16_workspace(B), encoder_grad=False)
            for net in stepping:
                self._opt_steps[net] += 1
            metrics = dict()
            if self.use_tb:
                m = ws.metrics.tolist()
                metrics = dict(critic_target_q=m[1], critic_q1=m[2], critic_q2=m[3], critic_loss=m[4])
            return metrics

    def update_actor(self, obs, step):
        """drqv2.py:206-228 on (detached) features: actor loss, backward, actor_opt.step().  The target critic is
        not touched (its soft update belongs to update(), drqv2.py:259-260)."""
        with torch.cuda.device(self._dev):
            B = obs.shape[0]
            ws = self.workspace(B)
            self._stage_features(ws, obs, 0)
            self._stage_noise(ws.eps_a, 3)
            self._stage_scalars(step, ("actor",))
            if self.mode == "fp32":
                self._actor_pass(ws, ws.feat[:B], soft_update=False)
            else:
                _bf16.actor_pass(self, ws, self.bf16_workspace(B), soft_update=False, standalone=True)
            self._opt_steps["actor"] += 1
            metrics = dict()
            if self.use_tb:
                m = ws.metrics.tolist()
                metrics = dict(actor_loss=m[5], actor_logprob=m[6], actor_ent=m[7])
            return metrics
