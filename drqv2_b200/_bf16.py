"""bf16 tensor-core mode of the DrQ-v2 update: the same arithmetic as the fp32 path in drqv2.py
(reference drqv2.py:177-262) with every dense contraction on tcgen05 kernels, re-scheduled so
that work sharing an operand shares a launch:

  * one split-K trunk GEMM covers the four trunk forwards that read the batch's features
    (actor(next), critic_target(next), actor(obs), critic(obs); reference drqv2.py:182-184,187,210)
    - the actor's parameters do not change between update_critic and update_actor;
  * the actor MLP runs once on [obs | next] rows;
  * the online and target twin-Q heads run as one 4-head batched launch per layer.

Inside the captured graph the update runs on three streams (DESIGN.md §4): the data-gradient chain on the main
stream, the encoder backward + encoder_opt.step() beside the actor pass, and the weight-gradient GEMMs, bias sums
and the soft target update beside both.

Master parameters, gradients and Adam state stay fp32 in the reference layouts; this module owns
the derived bf16 operand copies (re-packed after every optimiser step) and the bf16 activations:
  * encoder activations / gradients: "WB" layout (include/drqv2_b200.h),
  * everything the heads touch (features, hidden activations, their gradients, Linear weights):
    the tile-blocked "TB" layout X_tb[row/R][f/8][row%R][8] (R = 128 activations, 64 weights) -
    one buffer is both the K-major operand (contraction over features) and the MN-major operand
    (contraction over rows), and every GEMM tile is one contiguous bulk copy.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import (GEMM_KK, GEMM_KMN, GEMM_MNMN, PLB, REPR_DIM, TB_ACT, TB_W, TEPI_F32, TEPI_MASK_BF16,
                   TEPI_RELU_BF16, TEPI_TRUNK_DGRAD, TEPI_TRUNK_WGRAD, WB_SLACK, call)

F32, BF = 4, 2


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ceil(n, m):
    return (n + m - 1) // m * m


def splitk_for(ctas_per_split, K=REPR_DIM, target_blocks=148):
    s0 = max(1, min(target_blocks // max(1, ctas_per_split), K // 128))
    chunk = -(-K // s0)
    chunk = -(-chunk // 128) * 128
    return -(-K // chunk)


class TB:
    """`batch` bf16 matrices [rows][feats] in the tile-blocked layout (zero initialised)."""

    def __init__(self, rows, feats, dev, batch=1, rblk=TB_ACT):
        self.rows, self.feats, self.batch, self.rblk = rows, feats, batch, rblk
        self.units = _ceil(feats, 16) // 8
        self.rpad = _ceil(rows, rblk)
        self.stride = self.units * self.rpad * 8          # elements between batch entries
        self.buf = torch.zeros(batch * self.stride, dtype=torch.bfloat16, device=dev)

    def off(self, z=0, row=0, feat=0):
        assert feat % 8 == 0 and row % self.rblk == 0, "TB pointers are row-block / unit aligned"
        return z * self.stride + ((row // self.rblk) * self.units + feat // 8) * self.rblk * 8

    def ptr(self, z=0, row=0, feat=0):
        return self.buf.data_ptr() + BF * self.off(z, row, feat)

    def view(self, z=0):
        """[rpad][units*8] view (tests / debugging)."""
        x = self.buf[z * self.stride:(z + 1) * self.stride].view(self.rpad // self.rblk, self.units, self.rblk, 8)
        return x.permute(0, 2, 1, 3).reshape(self.rpad, self.units * 8)

    def dense(self, z=0):
        return self.view(z)[:self.rows, :self.feats].float()

    def load(self, x, z=0):
        """fill entry z from a [rows][feats] tensor (tests)."""
        pad = torch.zeros(self.rpad, self.units * 8, dtype=torch.bfloat16, device=self.buf.device)
        pad[:x.shape[0], :x.shape[1]] = x.to(torch.bfloat16)
        self.buf[z * self.stride:(z + 1) * self.stride].view(self.rpad // self.rblk, self.units, self.rblk, 8).copy_(
            pad.view(self.rpad // self.rblk, self.rblk, self.units, 8).permute(0, 2, 1, 3))


def _strides(inner=(0, 0, 0, 0, 0), outer=(0, 0, 0, 0, 0), split=0):
    return (C.c_int64 * 11)(*inner, *outer, split)


def gemm(A, units_a, B, units_b, mode, Cp, ldc, M, N, K, epi, bias=0, mask=0, units_mask=0, acc=0, batch=1,
         batch_inner=None, strides=None, splitk=1, bn=64, n_store=0):
    """batch_inner defaults to batch: the inner strides (strides[0:5]) then index all entries."""
    call("drq_gemm_bf16", A, units_a, B, units_b, mode, Cp, ldc, n_store, bias or None, mask or None, units_mask,
         M, N, K, epi, acc, batch, batch_inner or batch, strides, splitk, bn, _stream())


class LnJob(C.Structure):
    _fields_ = [("partial", C.c_void_p), ("ld_partial", C.c_int64), ("split_stride", C.c_int64), ("S", C.c_int32),
                ("bias", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
                ("h_out", C.c_void_p), ("ld_h", C.c_int64), ("xhat", C.c_void_p), ("rstd", C.c_void_p),
                ("h_bf16", C.c_void_p), ("units_bf16", C.c_int64), ("row0_bf16", C.c_int64),
                ("tail", C.c_void_p), ("ld_tail", C.c_int64), ("n_tail", C.c_int32)]


class PackJob(C.Structure):
    _fields_ = [("kind", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32), ("reserved", C.c_int32),
                ("w", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p), ("out2", C.c_void_p)]


PACK_LINEAR, PACK_TRUNK, PACK_CONV, PACK_CONV1 = 0, 1, 2, 3


def pack_multi(jobs):
    arr = (PackJob * len(jobs))(*jobs)
    call("drq_pack_multi", arr, len(jobs), _stream())


class OptSeg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("ema", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32),
                ("off", C.c_int64), ("n", C.c_int64), ("out", C.c_void_p), ("out2", C.c_void_p)]


OPT_PLAIN, OPT_LINEAR, OPT_TRUNK, OPT_CONV, OPT_CONV1 = 0, 1, 2, 3, 4


class WgReduceJob(C.Structure):
    _fields_ = [("partial", C.c_void_p), ("dw", C.c_void_p), ("db", C.c_void_p), ("n_images", C.c_int32),
                ("hout", C.c_int32), ("cin", C.c_int32), ("reserved", C.c_int32)]


class ColsumJob(C.Structure):
    _fields_ = [("X", C.c_void_p), ("ld", C.c_int64), ("out", C.c_void_p), ("M", C.c_int32), ("N", C.c_int32),
                ("tb", C.c_int32), ("reserved", C.c_int32), ("Y", C.c_void_p)]


class PolicySample(C.Structure):
    """drq_policy_sample: one TruncatedNormal sample job of drq_policy_head_fwd_bf16"""
    _fields_ = [("row0", C.c_int32), ("rows", C.c_int32), ("eps", C.c_void_p), ("action_out", C.c_void_p),
                ("ld_a", C.c_int64), ("mu_out", C.c_void_p), ("metrics", C.c_void_p), ("a_bf16", C.c_void_p),
                ("units_a", C.c_int64), ("feat_off", C.c_int32), ("reserved", C.c_int32)]


def colsum_multi(jobs):
    arr = (ColsumJob * len(jobs))(*jobs)
    call("drq_colsum_multi", arr, len(jobs), _stream())


def ln_tanh_multi(jobs, B, Fd):
    arr = (LnJob * len(jobs))(*jobs)
    call("drq_ln_tanh_fwd_multi", arr, len(jobs), B, Fd, 1e-5, _stream())


class Bf16State:
    """Packed bf16 weights of an agent (independent of the batch size)."""
    TARGET, ACTOR, CRITIC = 0, 1, 2          # slots of the merged trunk weight: [target | actor | critic]

    def __init__(self, agent):
        dev = agent._dev
        a = agent._arena
        A, Fd, H = agent.action_dim, agent.feature_dim, agent.hidden_dim
        self.agent = agent
        self.FP = _ceil(Fd, TB_W)                                   # trunk rows per slot
        self.trunk = TB(3 * self.FP, REPR_DIM, dev, rblk=TB_W)      # encoder-output feature order (c/8, yx, c%8)
        self.q0 = TB(H, Fd + A, dev, batch=4, rblk=TB_W)            # [critic Q1, critic Q2, target Q1, target Q2]
        self.q2 = TB(H, H, dev, batch=4, rblk=TB_W)
        self.p0 = TB(H, Fd, dev, rblk=TB_W)
        self.p2 = TB(H, H, dev, rblk=TB_W)
        self.p4 = TB(A, H, dev, rblk=TB_W)
        co, base_c = a.offsets["critic"], a.seg["critic"][0]
        self.c_off = {k: co[k] - base_c for k in ("trunk.0.weight", "Q1.0.weight", "Q1.2.weight")}
        qs = agent._q_strides()
        assert co["Q2.0.weight"] - co["Q1.0.weight"] == qs and co["Q2.2.weight"] - co["Q1.2.weight"] == qs
        # fp32 distance between the online critic's and the target's parameter blocks (bias / w3 strides)
        d = a.target.data_ptr() - a.ptr("params", "critic")
        assert d % F32 == 0
        self.target_minus_critic = d // F32
        # encoder: conv1 packed + (fwd, dgrad) operands of conv2..4
        self.conv1_w = torch.zeros(_lib.lib().drq_conv1_w_packed_elems(), dtype=torch.bfloat16, device=dev)   # fp16 weights + fused bias
        self.conv_wf = [torch.zeros(36 * 32 * 8, dtype=torch.bfloat16, device=dev) for _ in range(3)]
        self.conv_wd = [torch.zeros(36 * 32 * 8, dtype=torch.bfloat16, device=dev) for _ in range(3)]
        self.build_opt_plans()

    def trunk_ptr(self, slot):
        return self.trunk.ptr(row=slot * self.FP)

    # ---- bf16 operand refresh: one launch per optimiser phase
    def _encoder_jobs(self):
        ag = self.agent
        jobs = [PackJob(PACK_CONV1, 0, ag.obs_shape[0], 0, ag._p("encoder", "convnet.0.weight"),
                        ag._p("encoder", "convnet.0.bias"), self.conv1_w.data_ptr(), None)]
        for i, k in enumerate((2, 4, 6)):
            jobs.append(PackJob(PACK_CONV, 0, 0, 0, ag._p("encoder", f"convnet.{k}.weight"), None,
                                self.conv_wf[i].data_ptr(), self.conv_wd[i].data_ptr()))
        return jobs

    def _critic_like_jobs(self, src_ptr, slot, z0):
        ag = self.agent
        A, Fd, H = ag.action_dim, ag.feature_dim, ag.hidden_dim
        qs = ag._q_strides()
        jobs = [PackJob(PACK_TRUNK, Fd, REPR_DIM, 0, src_ptr + F32 * self.c_off["trunk.0.weight"], None, self.trunk_ptr(slot), None)]
        for z in range(2):
            jobs.append(PackJob(PACK_LINEAR, H, Fd + A, 0, src_ptr + F32 * (self.c_off["Q1.0.weight"] + z * qs), None,
                                self.q0.ptr(z0 + z), None))
            jobs.append(PackJob(PACK_LINEAR, H, H, 0, src_ptr + F32 * (self.c_off["Q1.2.weight"] + z * qs), None,
                                self.q2.ptr(z0 + z), None))
        return jobs

    def _actor_jobs(self):
        ag = self.agent
        A, Fd, H = ag.action_dim, ag.feature_dim, ag.hidden_dim
        pa = lambda k: ag._p("actor", k)
        return [PackJob(PACK_TRUNK, Fd, REPR_DIM, 0, pa("trunk.0.weight"), None, self.trunk_ptr(self.ACTOR), None),
                PackJob(PACK_LINEAR, H, Fd, 0, pa("policy.0.weight"), None, self.p0.ptr(), None),
                PackJob(PACK_LINEAR, H, H, 0, pa("policy.2.weight"), None, self.p2.ptr(), None),
                PackJob(PACK_LINEAR, A, H, 0, pa("policy.4.weight"), None, self.p4.ptr(), None)]

    # ---- optimiser step + operand refresh in one launch (drq_adam_pack_step)
    def _segments(self, mod, offs, base, ema, packed):
        """One segment per tensor of `mod` in arena order; tensors without a bf16 copy merge into PLAIN runs.
        packed: pname -> (kind, rows, cols, out, out2)."""
        segs = []
        skip = None
        for pname, prm in mod.named_parameters():
            if pname == skip:
                continue
            off, n = offs[pname] - base, prm.numel()
            if pname in packed:
                kind, rows, cols, out, out2 = packed[pname]
                if kind == OPT_CONV1:                      # weight and bias are one segment
                    skip = pname.replace("weight", "bias")
                    assert offs[skip] - base == off + n
                    n += 32
                segs.append(OptSeg(kind, ema, rows, cols, off, n, out, out2))
            elif segs and segs[-1].kind == OPT_PLAIN and segs[-1].ema == ema and segs[-1].off + segs[-1].n == off:
                segs[-1].n += _ceil(n, 4)                  # arena tensors start on 16-byte boundaries
            else:
                segs.append(OptSeg(OPT_PLAIN, ema, 0, 0, off, _ceil(n, 4), None, None))
        return segs

    def _critic_like_packed(self, slot, z0):
        ag = self.agent
        A, Fd, H = ag.action_dim, ag.feature_dim, ag.hidden_dim
        pk = {"trunk.0.weight": (OPT_TRUNK, Fd, REPR_DIM, self.trunk_ptr(slot), None)}
        for z in range(2):
            pk[f"Q{z + 1}.0.weight"] = (OPT_LINEAR, H, Fd + A, self.q0.ptr(z0 + z), None)
            pk[f"Q{z + 1}.2.weight"] = (OPT_LINEAR, H, H, self.q2.ptr(z0 + z), None)
        return pk

    def build_opt_plans(self):
        ag = self.agent
        a = ag._arena
        A, Fd, H = ag.action_dim, ag.feature_dim, ag.hidden_dim
        enc = {"convnet.0.weight": (OPT_CONV1, ag.obs_shape[0], 0, self.conv1_w.data_ptr(), None)}
        for i, k in enumerate((2, 4, 6)):
            enc[f"convnet.{k}.weight"] = (OPT_CONV, 0, 0, self.conv_wf[i].data_ptr(), self.conv_wd[i].data_ptr())
        segs_e = self._segments(ag.encoder, a.offsets["encoder"], 0, 0, enc)
        segs_c = self._segments(ag.critic, a.offsets["critic"], 0, 0, self._critic_like_packed(self.CRITIC, 0))
        self.plan_encoder = (OptSeg * len(segs_e))(*segs_e)
        self.plan_critic_only = (OptSeg * len(segs_c))(*segs_c)
        segs = segs_e + segs_c
        self.plan_critic = (OptSeg * len(segs))(*segs)
        act = {"trunk.0.weight": (OPT_TRUNK, Fd, REPR_DIM, self.trunk_ptr(self.ACTOR), None),
               "policy.0.weight": (OPT_LINEAR, H, Fd, self.p0.ptr(), None),
               "policy.2.weight": (OPT_LINEAR, H, H, self.p2.ptr(), None),
               "policy.4.weight": (OPT_LINEAR, A, H, self.p4.ptr(), None)}
        segs_a = self._segments(ag.actor, a.offsets["actor"], 0, 0, act)
        segs_t = self._segments(ag.critic, a.offsets["critic"], a.seg["critic"][0], 1, self._critic_like_packed(self.TARGET, 2))
        self.plan_actor_only = (OptSeg * len(segs_a))(*segs_a)
        self.plan_target = (OptSeg * len(segs_t))(*segs_t)
        segs = segs_a + segs_t
        self.plan_actor = (OptSeg * len(segs))(*segs)

    def step_critic_encoder(self):
        """critic_opt.step(); encoder_opt.step() (drqv2.py:201-202) and their bf16 operand copies."""
        ag = self.agent
        a = ag._arena
        if ag._opt_steps["encoder"] != ag._opt_steps["critic"]:     # one launch shares one set of Adam scalars
            self.step_critic()
            self.step_encoder()
            return
        call("drq_adam_pack_step", a.params.data_ptr(), a.grads.data_ptr(), a.exp_avg.data_ptr(), a.exp_avg_sq.data_ptr(),
             ag._sc("critic"), None, None, 0.0, 0.0, self.plan_critic, len(self.plan_critic), _stream())

    def _step(self, plan, net):
        ag = self.agent
        a = ag._arena
        call("drq_adam_pack_step", a.params.data_ptr(), a.grads.data_ptr(), a.exp_avg.data_ptr(), a.exp_avg_sq.data_ptr(),
             ag._sc(net), None, None, 0.0, 0.0, plan, len(plan), _stream())

    def step_critic(self):
        """critic_opt.step() (drqv2.py:201) and the critic's bf16 operand copies."""
        self._step(self.plan_critic_only, "critic")

    def step_encoder(self):
        """encoder_opt.step() (drqv2.py:202) and the encoder's bf16 operand copies."""
        self._step(self.plan_encoder, "encoder")

    def step_actor(self):
        """actor_opt.step() (drqv2.py:221) and the actor's bf16 operand copies."""
        self._step(self.plan_actor_only, "actor")

    def step_target(self):
        """utils.soft_update_params(critic, critic_target, tau) (drqv2.py:259-260) and the target's bf16 operand copies."""
        ag = self.agent
        a = ag._arena
        tau = float(ag.critic_target_tau)
        call("drq_adam_pack_step", None, None, None, None, None, a.ptr("params", "critic"), a.target.data_ptr(), tau,
             float(1 - tau), self.plan_target, len(self.plan_target), _stream())

    def step_actor_target(self):
        """actor_opt.step() and the soft target update (drqv2.py:221,259-260) and their bf16 operand copies."""
        ag = self.agent
        a = ag._arena
        tau = float(ag.critic_target_tau)
        call("drq_adam_pack_step", a.params.data_ptr(), a.grads.data_ptr(), a.exp_avg.data_ptr(), a.exp_avg_sq.data_ptr(),
             ag._sc("actor"), a.ptr("params", "critic"), a.target.data_ptr(), tau, float(1 - tau),
             self.plan_actor, len(self.plan_actor), _stream())

    def repack_critic_encoder(self):
        """after critic_opt.step() / encoder_opt.step() (drqv2.py:201-202)"""
        pack_multi(self._critic_like_jobs(self.agent._arena.ptr("params", "critic"), self.CRITIC, 0) + self._encoder_jobs())

    def repack_actor_target(self):
        """after actor_opt.step() and the soft target update (drqv2.py:221,259-260)"""
        pack_multi(self._actor_jobs() + self._critic_like_jobs(self.agent._arena.target.data_ptr(), self.TARGET, 2))

    def repack_all(self):
        self.repack_critic_encoder()
        self.repack_actor_target()


class Bf16Workspace:
    """Activation buffers of one batch size.  Rows of the two-half buffers: obs at [0, B), next_obs at
    [RB, RB + B) with RB = B rounded up to a 128-row block."""

    def __init__(self, B, A, Fd, H, st, dev):
        L = _lib.lib()
        zb = lambda *s: torch.zeros(*s, dtype=torch.bfloat16, device=dev)
        zf = lambda *s: torch.zeros(*s, device=dev)
        NB = 2 * B
        self.B = B
        self.RB = RB = _ceil(B, TB_ACT)
        self.acts = [zb(L.drq_wb_elems(NB)) for _ in range(3)]      # conv1..3 outputs, [obs | next]
        self.cs_act = NB * PLB + WB_SLACK
        self.feat = TB(2 * RB, REPR_DIM, dev)                        # feature order (c/8)*9800 + yx*8 + c%8
        self.dpre = [zb(L.drq_wb_elems(B)) for _ in range(4)]
        self.cs_d = B * PLB + WB_SLACK
        # per-CTA weight-gradient partials of conv1..conv4, reduced by one launch at the end of the backward
        self.wg_ws = [zf(L.drq_conv1_wgrad_bf16_ws_floats())] + [zf(L.drq_conv_wgrad_bf16_ws_floats()) for _ in range(3)]
        FP = st.FP
        self.NT = 2 * FP                                             # columns of one trunk GEMM half
        ntiles = (RB // TB_ACT) * (self.NT // 128)
        self.S2 = splitk_for(2 * ntiles)                             # merged (2 halves) trunk forward
        self.S1 = splitk_for((RB // TB_ACT) * (FP // 64))            # single trunk forward (actor pass)
        self.partial = zf(max(self.S2 * 2 * B * self.NT, self.S1 * B * FP))
        self.x = TB(B, Fd + A, dev, batch=2)                         # [xC = (h_critic(obs), action) | xT = (h_target(next), next action)]
        self.xA = TB(B, Fd + A, dev)                                 # (h_critic'(obs), actor action)
        self.hA = TB(2 * RB, Fd, dev)                                # actor trunk output, [obs | next]
        self.p1, self.p2 = TB(2 * RB, H, dev), TB(2 * RB, H, dev)
        self.mu_pre = zf(RB + B, A)
        self.hA_next_f32 = zf(B, Fd)
        self.c1, self.c2 = TB(B, H, dev, batch=4), TB(B, H, dev, batch=4)   # [critic Q1, Q2, target Q1, Q2]
        self.q4 = zf(4, B)
        self.dc1, self.dc2 = TB(B, H, dev, batch=2), TB(B, H, dev, batch=2)
        self.dp1, self.dp2 = TB(B, H, dev), TB(B, H, dev)
        self.dz = TB(B, Fd, dev)
        self.dmu = TB(B, A, dev)
        self.SX = 8 if H % 1024 == 0 else 1                          # split-K of the Q heads' first-layer data gradient
        self.dxf = zf(2 * self.SX, B, Fd + A)                        # partial planes [split][head]


def encode(agent, ws, bw):
    """conv1 (u8 + aug + normalise fused) .. conv4 on tensor cores; features TB bf16 (channel-group-major order)."""
    st, B, s = agent._bf16, ws.B, _stream()
    be = lambda i: agent._p("encoder", f"convnet.{i}.bias")
    acts = [a.data_ptr() for a in bw.acts]
    src = getattr(ws, "ring_src", None)
    if src is not None:          # frame stacks by index, straight from the replay ring
        call("drq_conv1_fwd_bf16_ring", C.byref(src), B, ws.shift.data_ptr(), st.conv1_w.data_ptr(), acts[0], 2 * B,
             agent.aug.pad, s)
    else:
        call("drq_conv1_fwd_bf16", ws.obs.data_ptr(), ws.shift.data_ptr(), st.conv1_w.data_ptr(), acts[0],
             2 * B, agent.obs_shape[0], agent.aug.pad, s)
    call("drq_conv3x3_fwd_bf16", acts[0], st.conv_wf[0].data_ptr(), be(2), acts[1], 2 * B, 39, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", acts[1], st.conv_wf[1].data_ptr(), be(4), acts[2], 2 * B, 37, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", acts[2], st.conv_wf[2].data_ptr(), be(6), bw.feat.ptr(), 2 * B, 35, 2, bw.feat.units,
         B, bw.RB, s)


def twin_q_layers(agent, bw, x, z0, nets, B):
    """Layers 1-2 of the 2 x nets Q heads of networks z0 .. z0 + nets - 1 (0 = online critic, 1 = target) on
    x[z0 ..], one launch per layer (drqv2.py:103-111)."""
    st = agent._bf16
    A, Fd, H = agent.action_dim, agent.feature_dim, agent.hidden_dim
    qs_f, tmc = agent._q_strides(), st.target_minus_critic
    pc = lambda k: agent._p("critic", k) + F32 * z0 * tmc
    c1, c2, w0, w2 = bw.c1, bw.c2, st.q0, st.q2
    gemm(x.ptr(z0), x.units, w0.ptr(2 * z0), w0.units, GEMM_KK, c1.ptr(2 * z0), c1.units, B, H, Fd + A, TEPI_RELU_BF16,
         bias=pc("Q1.0.bias"), batch=2 * nets, batch_inner=2,
         strides=_strides((0, w0.stride, c1.stride, qs_f, 0), (x.stride, 2 * w0.stride, 2 * c1.stride, tmc, 0)))
    gemm(c1.ptr(2 * z0), c1.units, w2.ptr(2 * z0), w2.units, GEMM_KK, c2.ptr(2 * z0), c2.units, B, H, H, TEPI_RELU_BF16,
         bias=pc("Q1.2.bias"), batch=2 * nets, batch_inner=2,
         strides=_strides((c1.stride, w2.stride, c2.stride, qs_f, 0), (2 * c1.stride, 2 * w2.stride, 2 * c2.stride, tmc, 0)))


def twin_q_heads(agent, bw, nets, B):
    """the scalar heads Linear(hidden, 1) of 2 x nets Q heads -> q4[0 : 2 * nets] (drqv2.py:106,111)"""
    st = agent._bf16
    H = agent.hidden_dim
    pc = lambda k: agent._p("critic", k)
    c2 = bw.c2
    call("drq_q_head_fwd_bf16", c2.ptr(), c2.units, c2.stride, pc("Q1.4.weight"), pc("Q1.4.bias"), bw.q4.data_ptr(),
         B, H, 2 * nets, agent._q_strides(), 2, st.target_minus_critic, _stream())


def twin_q_fwd(agent, bw, x, nets, B):
    """Layers 1-2 and the scalar head of `nets` x 2 Q heads in one launch per layer.  nets = 2: online
    critic on x[0] and target on x[1] -> q4[0:4]; nets = 1: online critic on x -> q4[0:2]."""
    twin_q_layers(agent, bw, x, 0, nets, B)
    twin_q_heads(agent, bw, nets, B)


def actor_mlp_fwd(agent, hA, p1, p2, mu_pre, M, samples=(), clip=0.0):
    """policy MLP (drqv2.py:77-81) on the first M rows of hA; the Linear(hidden, A) head and the TruncatedNormal
    samples of the row ranges in `samples` (PolicySample jobs, utils.py:112-126) are one launch."""
    st = agent._bf16
    A, Fd, H = agent.action_dim, agent.feature_dim, agent.hidden_dim
    pa = lambda k: agent._p("actor", k)
    w0, w2 = st.p0, st.p2
    gemm(hA.ptr(), hA.units, w0.ptr(), w0.units, GEMM_KK, p1.ptr(), p1.units, M, H, Fd, TEPI_RELU_BF16,
         bias=pa("policy.0.bias"))
    gemm(p1.ptr(), p1.units, w2.ptr(), w2.units, GEMM_KK, p2.ptr(), p2.units, M, H, H, TEPI_RELU_BF16,
         bias=pa("policy.2.bias"))
    jobs = (PolicySample * max(1, len(samples)))(*samples)
    call("drq_policy_head_fwd_bf16", p2.ptr(), p2.units, pa("policy.4.weight"), pa("policy.4.bias"), mu_pre, M, H, A,
         jobs, len(samples), agent._sc("stddev"), float(clip), agent._policy_ticket.data_ptr(), _stream())


class _Beside:
    """Weight-gradient work beside the data-gradient chain: `with beside:` enqueues on the agent's third stream
    after everything enqueued so far on the main stream; `beside.join()` makes the main stream wait for it.
    Without a third stream (data-parallel mode, DRQV2_B200_OVERLAP=0) both are no-ops."""

    def __init__(self, agent):
        self.side = agent._wgrad_side_stream()
        self.main = torch.cuda.current_stream()
        self.ctx = None

    def __enter__(self):
        if self.side is not None:
            self.side.wait_stream(self.main)
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
            self.ctx = None

    def join(self):
        if self.side is not None:
            self.main.wait_stream(self.side)


def critic_pass(agent, ws, bw, encoder_grad=True):
    """update_critic (drqv2.py:177-204) with critic_opt.step() / encoder_opt.step().  encoder_grad=False (stage API on
    detached features): no gradient into the encoder, only the critic steps."""
    st, s = agent._bf16, _stream()
    beside = _Beside(agent)
    B, A, Fd, H = ws.B, agent.action_dim, agent.feature_dim, agent.hidden_dim
    RB, FP, NT = bw.RB, st.FP, bw.NT
    pc = lambda k: agent._p("critic", k)
    gc = lambda k: agent._g("critic", k)
    pa = lambda k: agent._p("actor", k)
    tp = agent._t
    std_ptr = agent._sc("stddev")
    qs_f = agent._q_strides()
    feat, part, S = bw.feat, bw.partial, bw.S2
    # ---- all four trunk forwards on this batch's features: z = 0 obs rows x [actor | critic], z = 1 next rows x
    # [target | actor]  (slots of the merged trunk weight are [target | actor | critic])
    gemm(feat.ptr(), feat.units, st.trunk_ptr(st.ACTOR), st.trunk.units, GEMM_KK, part.data_ptr(), NT, B, NT, REPR_DIM,
         TEPI_F32, batch=2, batch_inner=1, splitk=S, bn=128,
         strides=_strides(outer=(feat.off(row=RB), -st.trunk.off(row=FP), B * NT, 0, 0), split=2 * B * NT))
    pz = lambda z, col: part.data_ptr() + F32 * (z * B * NT + col)
    job = lambda p, net_p, names, h_out, ld_h, xhat, rstd, tb, row0, tail=None: LnJob(
        p, NT, 2 * B * NT, S, net_p(names[0]), net_p(names[1]), net_p(names[2]), h_out, ld_h, xhat, rstd,
        tb.buf.data_ptr(), tb.units, row0, tail, A, A if tail else 0)
    tn = ("trunk.0.bias", "trunk.1.weight", "trunk.1.bias")
    ln_tanh_multi([
        job(pz(0, 0), pa, tn, ws.hA.data_ptr(), Fd, ws.xhatA.data_ptr(), ws.rstdA.data_ptr(), bw.hA, 0),       # actor(obs)
        job(pz(0, FP), pc, tn, ws.xC.data_ptr(), Fd + A, ws.xhatC.data_ptr(), ws.rstdC.data_ptr(), bw.x, 0,
            ws.action.data_ptr()),                                                                         # critic(obs) ++ action
        job(pz(1, 0), tp, tn, ws.xT.data_ptr(), Fd + A, None, None, bw.x, bw.x.rpad),                          # target(next) -> x[1]
        job(pz(1, FP), pa, tn, bw.hA_next_f32.data_ptr(), Fd, None, None, bw.hA, RB),                          # actor(next)
    ], B, Fd)
    split_q = beside.side is not None
    if split_q:                                     # online Q(obs, action) does not wait for the actor: beside the actor MLP
        with beside:
            twin_q_layers(agent, bw, bw.x, 0, 1, B)
    # ---- actor MLP on [obs | next] rows at once (drqv2.py:182 and :210 use the same actor parameters)
    # ... with, in the policy head's launch, the next action - clipped sample (drqv2.py:183) -> xT's action columns - and
    # already the actor pass' own sample on the obs rows (drqv2.py:210-212: same actor, same stddev, its own noise) ->
    # xA's action columns, mu, log-prob / entropy metrics
    xA = bw.xA
    actor_mlp_fwd(agent, bw.hA, bw.p1, bw.p2, bw.mu_pre.data_ptr(), RB + B, clip=agent.stddev_clip, samples=[
        PolicySample(RB, B, ws.eps_c.data_ptr(), ws.xT.data_ptr() + F32 * Fd, Fd + A, None, None, bw.x.ptr(1), bw.x.units, Fd, 0),
        PolicySample(0, B, ws.eps_a.data_ptr(), ws.xA.data_ptr() + F32 * Fd, Fd + A, ws.mu.data_ptr(),
                     ws.metrics.data_ptr() + F32 * 6, xA.ptr(), xA.units, Fd, 0)])
    # ---- target Q on (next, next action) and online Q on (obs, action)
    if split_q:
        twin_q_layers(agent, bw, bw.x, 1, 1, B)
        beside.join()
        twin_q_heads(agent, bw, 2, B)
    else:
        twin_q_fwd(agent, bw, bw.x, 2, B)           # 4 heads per launch
    # ---- TD target + critic loss (drqv2.py:185-189) and the backward through the scalar Q heads, one launch
    q = bw.q4.data_ptr()
    c1, c2, dc1, dc2 = bw.c1, bw.c2, bw.dc1, bw.dc2
    w0, w2, xC = st.q0, st.q2, bw.x
    U, HS = c1.units, c1.stride
    call("drq_q_head_bwd_loss_bf16", 1, q, q + F32 * 2 * B, ws.reward.data_ptr(), ws.discount.data_ptr(),
         ws.target_q.data_ptr(), ws.metrics.data_ptr(), c2.ptr(), U, HS, pc("Q1.4.weight"), dc2.ptr(),
         gc("Q1.4.weight"), gc("Q1.4.bias"), B, H, qs_f, s)
    with beside:
        gemm(dc2.ptr(), U, c1.ptr(), U, GEMM_MNMN, gc("Q1.2.weight"), H, H, H, B, TEPI_F32, batch=2,
             strides=_strides((HS, HS, qs_f, 0, 0)), bn=128)
    gemm(dc2.ptr(), U, w2.ptr(), w2.units, GEMM_KMN, dc1.ptr(), U, B, H, H, TEPI_MASK_BF16, mask=c1.ptr(), units_mask=U,
         batch=2, strides=_strides((HS, w2.stride, HS, 0, HS)))
    with beside:
        gemm(dc1.ptr(), U, xC.ptr(0), xC.units, GEMM_MNMN, gc("Q1.0.weight"), Fd + A, H, Fd + A, B, TEPI_F32, batch=2,
             strides=_strides((HS, 0, qs_f, 0, 0)))
    # d[h] = sum over heads and K chunks of dc1 @ W0[:, :F]: partial planes, summed by the consumer
    PS = B * (Fd + A)
    gemm(dc1.ptr(), U, w0.ptr(), w0.units, GEMM_KMN, bw.dxf.data_ptr(), Fd + A, B, Fd, H, TEPI_F32, batch=2,
         splitk=bw.SX, strides=_strides((HS, w0.stride, PS, 0, 0), split=2 * PS))
    # ---- trunk backward
    call("drq_ln_tanh_bwd", bw.dxf.data_ptr(), Fd + A, ws.xC.data_ptr(), Fd + A, ws.xhatC.data_ptr(),
         ws.rstdC.data_ptr(), pc("trunk.1.weight"), ws.dz.data_ptr(), None, None,
         bw.dz.ptr(), bw.dz.units, B, Fd, 2 * bw.SX, PS, s)
    with beside:
        gemm(bw.dz.ptr(), bw.dz.units, feat.ptr(), feat.units, GEMM_MNMN, gc("trunk.0.weight"), REPR_DIM, Fd, REPR_DIM, B,
             TEPI_TRUNK_WGRAD, bn=128)
        # all bias gradients of the critic backward in one launch
        colsum_multi([ColsumJob(dc2.ptr(0), U, gc("Q1.2.bias"), B, H, 1, 0), ColsumJob(dc2.ptr(1), U, gc("Q2.2.bias"), B, H, 1, 0),
                      ColsumJob(dc1.ptr(0), U, gc("Q1.0.bias"), B, H, 1, 0), ColsumJob(dc1.ptr(1), U, gc("Q2.0.bias"), B, H, 1, 0),
                      ColsumJob(ws.dz.data_ptr(), Fd, gc("trunk.0.bias"), B, Fd, 0, 0),
                      # LayerNorm affine: dgamma = sum_b dy * xhat, dbeta = sum_b dy (dy staged behind dz by drq_ln_tanh_bwd)
                      ColsumJob(ws.dz.data_ptr() + F32 * B * Fd, Fd, gc("trunk.1.weight"), B, Fd, 0, 0, ws.xhatC.data_ptr()),
                      ColsumJob(ws.dz.data_ptr() + F32 * B * Fd, Fd, gc("trunk.1.bias"), B, Fd, 0, 0)])
    # ---- encoder backward
    d = [t.data_ptr() for t in bw.dpre]
    acts = [t.data_ptr() for t in bw.acts]
    ge = lambda k: agent._g("encoder", k)
    if not encoder_grad:
        beside.join()
        agent._sync_grads("critic")
        st.step_critic()
        return
    gemm(bw.dz.ptr(), bw.dz.units, st.trunk_ptr(st.CRITIC), st.trunk.units, GEMM_KMN, d[3], bw.cs_d, B, REPR_DIM, Fd,
         TEPI_TRUNK_DGRAD, mask=feat.ptr(), units_mask=feat.units, bn=128)
    def encoder_backward():
        s2 = _stream()
        jobs = []
        for layer, hout in ((3, 35), (2, 37), (1, 39)):
            k = 2 * layer
            call("drq_conv3x3_wgrad_bf16", acts[layer - 1], 2 * B, d[layer], bw.wg_ws[layer].data_ptr(), None, None, B, hout, s2)
            jobs.append(WgReduceJob(bw.wg_ws[layer].data_ptr(), ge(f"convnet.{k}.weight"), ge(f"convnet.{k}.bias"), B, hout, 0, 0))
            call("drq_conv3x3_dgrad_bf16", d[layer], st.conv_wd[layer - 1].data_ptr(), acts[layer - 1], 2 * B,
                 d[layer - 1], B, hout, s2)
        src = getattr(ws, "ring_src", None)
        if src is not None:
            call("drq_conv1_wgrad_bf16_ring", C.byref(src), B, ws.shift.data_ptr(), d[0], bw.wg_ws[0].data_ptr(), None, None,
                 B, agent.aug.pad, s2)
        else:
            call("drq_conv1_wgrad_bf16", ws.obs.data_ptr(), ws.shift.data_ptr(), d[0], bw.wg_ws[0].data_ptr(), None, None,
                 B, agent.obs_shape[0], agent.aug.pad, s2)
        jobs.append(WgReduceJob(bw.wg_ws[0].data_ptr(), ge("convnet.0.weight"), ge("convnet.0.bias"), B, 0, agent.obs_shape[0], 0))
        arr = (WgReduceJob * len(jobs))(*jobs)
        call("drq_conv_wgrad_reduce_multi", arr, len(jobs), s2)   # all four layers' partials -> dW, db in one launch

    side = agent._encoder_side_stream()
    if side is None:
        beside.join()                               # the critic's weight gradients are complete
        encoder_backward()
        # critic_opt.step(); encoder_opt.step(); refresh their bf16 operand copies
        agent._sync_grads("encoder", "critic")      # data-parallel: mean over ranks (no-op otherwise)
        st.step_critic_encoder()
        return
    # The actor pass needs the stepped critic but nothing of the encoder's backward (it works on this update's
    # features, drqv2.py:256), so the encoder backward and encoder_opt.step() run on a second stream beside
    # critic_opt.step() and the whole actor pass; DrQV2Agent._update_body joins the streams at the end.
    main = torch.cuda.current_stream()
    early = agent.early_encoder_backward and not agent.data_parallel
    if not early:
        beside.join()                               # the critic's weight gradients are complete
    side.wait_stream(main)                          # early: the encoder backward needs the trunk's data gradient only
    with torch.cuda.stream(side):
        prev = _lib.lib().drq_device_sm_count()      # SMs the persistent kernels may use now (a data-parallel reservation lowers it)
        lim = min(agent.encoder_backward_sms, prev)
        if lim:                                     # leave SMs to the small kernels of the actor pass (grids are fixed at capture)
            call("drq_set_sm_limit", lim)
        try:
            encoder_backward()
        finally:
            if lim:
                call("drq_set_sm_limit", prev)
        if not agent.data_parallel:                 # data-parallel: after the join and the encoder's all-reduce (_update_body)
            st.step_encoder()
    if early:
        beside.join()
    agent._sync_grads("critic")                     # data-parallel: beside the encoder backward (no-op otherwise)
    st.step_critic()


def actor_pass(agent, ws, bw, soft_update=True, standalone=False):
    """update_actor; see _actor_pass.  Inside update() this pass runs beside the encoder backward, whose persistent conv
    kernels keep 148 KB of every SM's shared memory: its GEMMs are launched in their small-footprint variant
    (drq_set_gemm_small) so that their CTAs fit next to the conv CTAs instead of waiting for a conv kernel to end."""
    small = agent._encoder_side_stream() is not None and not standalone and agent.small_gemms_beside_encoder
    if small:
        call("drq_set_gemm_small", 1)
    try:
        _actor_pass(agent, ws, bw, soft_update, standalone)
    finally:
        if small:
            call("drq_set_gemm_small", 0)


def _actor_pass(agent, ws, bw, soft_update=True, standalone=False):
    """update_actor (drqv2.py:206-228).  Inside update() the actor's own forward on obs already ran with the critic
    pass (its parameters have not changed since); here: sample, the stepped critic's Q, and the backward.
    standalone=True (stage API): run that forward on the obs rows first.  soft_update=False: leave the target
    critic alone (update() applies drqv2.py:259-260 beside / after this pass)."""
    st, s = agent._bf16, _stream()
    beside = _Beside(agent)
    B, A, Fd, H = ws.B, agent.action_dim, agent.feature_dim, agent.hidden_dim
    FP = st.FP
    pc = lambda k: agent._p("critic", k)
    pa = lambda k: agent._p("actor", k)
    ga = lambda k: agent._g("actor", k)
    std_ptr = agent._sc("stddev")
    feat, xA = bw.feat, bw.xA
    if standalone:
        gemm(feat.ptr(), feat.units, st.trunk_ptr(st.ACTOR), st.trunk.units, GEMM_KK, bw.partial.data_ptr(), FP, B, FP,
             REPR_DIM, TEPI_F32, splitk=bw.S1, strides=_strides(split=B * FP))
        ln_tanh_multi([LnJob(bw.partial.data_ptr(), FP, B * FP, bw.S1, pa("trunk.0.bias"), pa("trunk.1.weight"),
                             pa("trunk.1.bias"), ws.hA.data_ptr(), Fd, ws.xhatA.data_ptr(), ws.rstdA.data_ptr(),
                             bw.hA.buf.data_ptr(), bw.hA.units, 0)], B, Fd)
        actor_mlp_fwd(agent, bw.hA, bw.p1, bw.p2, bw.mu_pre.data_ptr(), B, clip=agent.stddev_clip, samples=[
            PolicySample(0, B, ws.eps_a.data_ptr(), ws.xA.data_ptr() + F32 * Fd, Fd + A, ws.mu.data_ptr(),
                         ws.metrics.data_ptr() + F32 * 6, xA.ptr(), xA.units, Fd, 0)])
    if beside.side is not None and soft_update:
        # the soft target update depends on the stepped critic only (drqv2.py:259-260 runs it after update_actor, on the
        # same critic parameters) and nothing in this pass reads the target: beside the whole pass
        with beside:
            st.step_target()
    # (the sample a = clamp(mu + clip(eps * std)) of drqv2.py:210-211 was drawn with the actor's forward - the policy head's
    # launch in the critic pass, or just above in the stage API)
    # the just-updated critic on (features, action) (drqv2.py:213-216)
    S = bw.S1
    part = bw.partial.data_ptr()
    gemm(feat.ptr(), feat.units, st.trunk_ptr(st.CRITIC), st.trunk.units, GEMM_KK, part, FP, B, FP, REPR_DIM, TEPI_F32,
         splitk=S, strides=_strides(split=B * FP))
    ln_tanh_multi([LnJob(part, FP, B * FP, S, pc("trunk.0.bias"), pc("trunk.1.weight"), pc("trunk.1.bias"),
                         ws.xA.data_ptr(), Fd + A, None, None, xA.ptr(), xA.units, 0)], B, Fd)
    twin_q_fwd(agent, bw, xA, 1, B)
    q = bw.q4.data_ptr()
    c1, c2, dc1, dc2 = bw.c1, bw.c2, bw.dc1, bw.dc2
    w0, w2 = st.q0, st.q2
    U, HS = c1.units, c1.stride
    qs_f = agent._q_strides()
    # actor loss -mean(min(Q1,Q2)) (drqv2.py:213-216) and the backward through the scalar Q heads, one launch
    call("drq_q_head_bwd_loss_bf16", 2, q, None, None, None, None, ws.metrics.data_ptr() + F32 * 5, c2.ptr(), U, HS,
         pc("Q1.4.weight"), dc2.ptr(), None, None, B, H, qs_f, s)
    gemm(dc2.ptr(), U, w2.ptr(), w2.units, GEMM_KMN, dc1.ptr(), U, B, H, H, TEPI_MASK_BF16, mask=c1.ptr(), units_mask=U,
         batch=2, strides=_strides((HS, w2.stride, HS, 0, HS)))
    PS = B * (Fd + A)
    gemm(dc1.ptr(), U, w0.ptr(), w0.units, GEMM_KMN, bw.dxf.data_ptr(), Fd + A, B, Fd + A, H, TEPI_F32, batch=2,
         splitk=bw.SX, strides=_strides((HS, w0.stride, PS, 0, 0), split=2 * PS))
    call("drq_actor_sample_bwd", bw.dxf.data_ptr() + F32 * Fd, Fd + A, ws.mu.data_ptr(), ws.dmu_pre.data_ptr(),
         bw.dmu.ptr(), bw.dmu.units, B, A, 2 * bw.SX, PS, s)
    # actor MLP backward (activations of the obs rows, saved by the forward in the critic pass)
    dmu, hA, p1, p2, dp1, dp2 = bw.dmu, bw.hA, bw.p1, bw.p2, bw.dp1, bw.dp2
    a0, a2, a4 = st.p0, st.p2, st.p4
    with beside:
        gemm(dmu.ptr(), dmu.units, p2.ptr(), U, GEMM_MNMN, ga("policy.4.weight"), H, A, H, B, TEPI_F32, bn=128)
    gemm(dmu.ptr(), dmu.units, a4.ptr(), a4.units, GEMM_KMN, dp2.ptr(), U, B, H, A, TEPI_MASK_BF16, mask=p2.ptr(),
         units_mask=U)
    with beside:
        gemm(dp2.ptr(), U, p1.ptr(), U, GEMM_MNMN, ga("policy.2.weight"), H, H, H, B, TEPI_F32, bn=128)
    gemm(dp2.ptr(), U, a2.ptr(), a2.units, GEMM_KMN, dp1.ptr(), U, B, H, H, TEPI_MASK_BF16, mask=p1.ptr(), units_mask=U)
    with beside:
        gemm(dp1.ptr(), U, hA.ptr(), hA.units, GEMM_MNMN, ga("policy.0.weight"), Fd, H, Fd, B, TEPI_F32)
    gemm(dp1.ptr(), U, a0.ptr(), a0.units, GEMM_KMN, ws.dhA.data_ptr(), Fd, B, Fd, H, TEPI_F32)
    call("drq_ln_tanh_bwd", ws.dhA.data_ptr(), Fd, ws.hA.data_ptr(), Fd, ws.xhatA.data_ptr(), ws.rstdA.data_ptr(),
         pa("trunk.1.weight"), ws.dz.data_ptr(), None, None, bw.dz.ptr(), bw.dz.units,
         B, Fd, 1, 0, s)
    with beside:
        gemm(bw.dz.ptr(), bw.dz.units, feat.ptr(), feat.units, GEMM_MNMN, ga("trunk.0.weight"), REPR_DIM, Fd, REPR_DIM, B,
             TEPI_TRUNK_WGRAD, bn=128)
    colsum_multi([ColsumJob(ws.dmu_pre.data_ptr(), A, ga("policy.4.bias"), B, A, 0, 0),
                  ColsumJob(dp2.ptr(), U, ga("policy.2.bias"), B, H, 1, 0), ColsumJob(dp1.ptr(), U, ga("policy.0.bias"), B, H, 1, 0),
                  ColsumJob(ws.dz.data_ptr(), Fd, ga("trunk.0.bias"), B, Fd, 0, 0),
                  ColsumJob(ws.dz.data_ptr() + F32 * B * Fd, Fd, ga("trunk.1.weight"), B, Fd, 0, 0, ws.xhatA.data_ptr()),
                  ColsumJob(ws.dz.data_ptr() + F32 * B * Fd, Fd, ga("trunk.1.bias"), B, Fd, 0, 0)])
    beside.join()                                   # the actor's weight gradients are complete
    agent._sync_grads("actor", metrics=True)
    if beside.side is not None or not soft_update:
        st.step_actor()                             # the target's soft update already ran beside this pass (or is not wanted)
    else:
        st.step_actor_target()


def act_workspace(agent, n, dev):
    A, Fd, H = agent.action_dim, agent.feature_dim, agent.hidden_dim
    nel = _lib.lib().drq_wb_elems(n)
    zb = lambda *s: torch.zeros(*s, dtype=torch.bfloat16, device=dev)
    FP = agent._bf16.FP
    S = splitk_for((_ceil(n, TB_ACT) // TB_ACT) * (FP // 64))
    return dict(acts_b=[zb(nel) for _ in range(3)], feat_b=TB(n, REPR_DIM, dev), S_b=S,
                partial_b=torch.zeros(S * n * FP, device=dev), h_b=TB(n, Fd, dev), p1_b=TB(n, H, dev),
                p2_b=TB(n, H, dev))


def act_body(agent, w, n, sample):
    """encoder + actor for act() at batch n on the tensor-core path."""
    st, s = agent._bf16, _stream()
    A, Fd = agent.action_dim, agent.feature_dim
    FP = st.FP
    if sample:
        call("drq_rng_normal_f32", agent._seed, agent._counter.data_ptr(), w["eps"].data_ptr(), n * A, s)
        call("drq_counter_advance", agent._counter.data_ptr(), s)
    be = lambda i: agent._p("encoder", f"convnet.{i}.bias")
    acts = [a.data_ptr() for a in w["acts_b"]]
    feat = w["feat_b"]
    call("drq_conv1_fwd_bf16", w["obs"].data_ptr(), None, st.conv1_w.data_ptr(), acts[0], n,
         agent.obs_shape[0], agent.aug.pad, s)
    call("drq_conv3x3_fwd_bf16", acts[0], st.conv_wf[0].data_ptr(), be(2), acts[1], n, 39, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", acts[1], st.conv_wf[1].data_ptr(), be(4), acts[2], n, 37, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", acts[2], st.conv_wf[2].data_ptr(), be(6), feat.ptr(), n, 35, 2, feat.units, 0, 0, s)
    pa = lambda k: agent._p("actor", k)
    S, part = w["S_b"], w["partial_b"].data_ptr()
    gemm(feat.ptr(), feat.units, st.trunk_ptr(st.ACTOR), st.trunk.units, GEMM_KK, part, FP, n, FP, REPR_DIM, TEPI_F32,
         splitk=S, strides=_strides(split=n * FP))
    ln_tanh_multi([LnJob(part, FP, n * FP, S, pa("trunk.0.bias"), pa("trunk.1.weight"), pa("trunk.1.bias"),
                         w["h"].data_ptr(), Fd, None, None, w["h_b"].ptr(), w["h_b"].units, 0)], n, Fd)
    actor_mlp_fwd(agent, w["h_b"], w["p1_b"], w["p2_b"], w["mu_pre"].data_ptr(), n, samples=[
        PolicySample(0, n, w["eps"].data_ptr() if sample else None, w["out"].data_ptr(), A, None, None, None, 0, 0, 0)])


# ----------------------------------------------------------------------------- autograd on the tensor cores
# Encoder / Actor / Critic built with differentiable="bf16" run their forwards on the kernels act() and update() run
# (bf16 operands, fp32 accumulation) and, when autograd records, the tensor-core twins of drqv2.py's _EncoderFn,
# _ActorFn and _CriticFn.  The module boundary carries fp32 tensors in the reference's layouts (features [N, 39200]
# in the order c*1225 + y*35 + x, drqv2.py:66); drq_features_to_ref and drq_pack_features_tb convert at it.  Every
# launch goes to the current stream.

# rows drq_pack_features_tb and drq_features_to_ref take (DRQ_FEATURE_MAX_ROWS): the largest batch of every module
MAX_BATCH = 65408


def check_batch(n, what):
    if not 1 <= n <= MAX_BATCH:
        raise ValueError(f"{what}(differentiable='bf16'): batch {n} outside 1..{MAX_BATCH}, the rows the feature layout "
                         "conversions take; differentiable=True has no such limit")


def _wrap(buf, rows, feats, batch=1, rblk=TB_ACT):
    """a TB around a saved buffer"""
    tb = TB.__new__(TB)
    tb.rows, tb.feats, tb.batch, tb.rblk = rows, feats, batch, rblk
    tb.units = _ceil(feats, 16) // 8
    tb.rpad = _ceil(rows, rblk)
    tb.stride = tb.units * tb.rpad * 8
    tb.buf = buf
    return tb


class Operands:
    """The bf16 operand copies one module's forward and backward read: `conv1`, `wf`, `wd` (encoder), `trunk` /
    `trunk_units` and `p0`, `p2`, `p4` (actor) or `q0`, `q2` with head z at entry z0 + z (critic)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def _param_key(module):
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


def _own_operands(module, kind):
    """Copies owned by a standalone module (drq_pack_multi of its parameters: the pack kinds the agent's copies use),
    re-derived on first use, when a parameter was replaced or changed in place (its version counter moved), or after
    refresh() / utils.soft_update_params marked them stale.
    Once a forward of the module has been captured in a CUDA graph, every forward re-derives them, captured or eager:
    a replay of an optimiser step captured with it (torch.optim.Adam(capturable=True)) changes the parameters without
    moving a version counter, so neither the version counters read at capture time nor those read between replays
    tell whether the copies are current.  Two cases they would get wrong: an eager forward between the warm-up and the
    capture matches the counters, and the captured forwards would then read copies frozen at that eager forward on
    every replay; and inside the graph the actor's and the encoder's last forward runs before their optimiser step
    (the target's before the soft update), so an eager forward after a replay would read copies one step behind."""
    key = _param_key(module)
    ops = module.__dict__.get("_bf16_ops")
    if torch.cuda.is_current_stream_capturing():
        module.__dict__["_bf16_captured"] = True
    elif (ops is not None and ops.key == key and not module.__dict__.get("_bf16_stale", False)
          and not module.__dict__.get("_bf16_captured", False)):
        return ops
    dev = next(module.parameters()).device
    zb = lambda n: torch.zeros(n, dtype=torch.bfloat16, device=dev)
    if ops is None or ops.kind != kind or ops.dev != dev:
        if kind == "encoder":
            ops = Operands(conv1=zb(_lib.lib().drq_conv1_w_packed_elems()), wf=[zb(36 * 32 * 8) for _ in range(3)],
                           wd=[zb(36 * 32 * 8) for _ in range(3)])
        elif kind == "actor":
            Fd, H, A = module.trunk[0].out_features, module.policy[0].out_features, module.policy[4].out_features
            tr = TB(Fd, REPR_DIM, dev, rblk=TB_W)
            ops = Operands(tr=tr, trunk=tr.ptr(), trunk_units=tr.units, p0=TB(H, Fd, dev, rblk=TB_W),
                           p2=TB(H, H, dev, rblk=TB_W), p4=TB(A, H, dev, rblk=TB_W))
        else:
            Fd, H = module.trunk[0].out_features, module.Q1[0].out_features
            A = module.Q1[0].in_features - Fd
            tr = TB(Fd, REPR_DIM, dev, rblk=TB_W)
            ops = Operands(tr=tr, trunk=tr.ptr(), trunk_units=tr.units, q0=TB(H, Fd + A, dev, batch=2, rblk=TB_W),
                           q2=TB(H, H, dev, batch=2, rblk=TB_W), z0=0)
        ops.kind, ops.dev = kind, dev
    if kind == "encoder":
        c = [module.convnet[i] for i in (0, 2, 4, 6)]
        jobs = [PackJob(PACK_CONV1, 0, c[0].in_channels, 0, c[0].weight.data_ptr(), c[0].bias.data_ptr(),
                        ops.conv1.data_ptr(), None)]
        jobs += [PackJob(PACK_CONV, 0, 0, 0, c[i + 1].weight.data_ptr(), None, ops.wf[i].data_ptr(), ops.wd[i].data_ptr())
                 for i in range(3)]
    elif kind == "actor":
        t, p = module.trunk[0], module.policy
        jobs = [PackJob(PACK_TRUNK, t.out_features, REPR_DIM, 0, t.weight.data_ptr(), None, ops.trunk, None)]
        jobs += [PackJob(PACK_LINEAR, p[i].out_features, p[i].in_features, 0, p[i].weight.data_ptr(), None, out.ptr(), None)
                 for i, out in ((0, ops.p0), (2, ops.p2), (4, ops.p4))]
    else:
        t = module.trunk[0]
        jobs = [PackJob(PACK_TRUNK, t.out_features, REPR_DIM, 0, t.weight.data_ptr(), None, ops.trunk, None)]
        for z, q in enumerate((module.Q1, module.Q2)):
            jobs += [PackJob(PACK_LINEAR, q[i].out_features, q[i].in_features, 0, q[i].weight.data_ptr(), None,
                             out.ptr(z), None) for i, out in ((0, ops.q0), (2, ops.q2))]
    pack_multi(jobs)
    ops.key = key
    module.__dict__["_bf16_ops"] = ops
    module.__dict__["_bf16_stale"] = False
    return ops


def _agent_operands(agent, role):
    """An agent's module reads the agent's own copies (Bf16State), which its optimiser steps, update() and the stage API
    keep current; a parameter changed from outside (load_state_dict, an in-place edit) moves a version counter, and any
    other change sets _bf16_dirty: either re-derives every copy first."""
    keys = agent.__dict__.get("_bf16_keys")
    if agent._bf16_dirty or keys is None or any(keys[r] != _param_key(getattr(agent, r)) for r in keys):
        agent.refresh()
    st = agent._bf16
    if role == "encoder":
        return Operands(conv1=st.conv1_w, wf=st.conv_wf, wd=st.conv_wd)
    if role == "actor":
        return Operands(trunk=st.trunk_ptr(st.ACTOR), trunk_units=st.trunk.units, p0=st.p0, p2=st.p2, p4=st.p4)
    slot, z0 = (st.CRITIC, 0) if role == "critic" else (st.TARGET, 2)
    return Operands(trunk=st.trunk_ptr(slot), trunk_units=st.trunk.units, q0=st.q0, q2=st.q2, z0=z0)


def mark_stale(module):
    owner = module.__dict__.get("_bf16_owner")
    if owner is not None:
        owner[0]._bf16_dirty = True
    else:
        module.__dict__["_bf16_stale"] = True


def operands(module, kind):
    owner = module.__dict__.get("_bf16_owner")
    if owner is not None:
        return _agent_operands(*owner)
    return _own_operands(module, kind)


def _zb(n, dev):
    return torch.zeros(n, dtype=torch.bfloat16, device=dev)


# ---- Encoder
def needed(ctx, skip=0):
    """ctx.needs_input_grad narrowed to the inputs this backward pass reaches: under torch.autograd.grad(q, obs) the
    parameters' edges are not executed, and their weight gradients are not computed.  ctx.next_functions lists the
    tensor inputs only (skip = the leading non-tensor inputs).  A leaf under torch.autograd.grad cannot be asked, and
    counts as needed - Encoder(pixels="float") hands its parameters in as views so that it can be asked."""
    need = list(ctx.needs_input_grad)
    ask = getattr(torch._C, "_will_engine_execute_node", None)     # private: absent -> ctx.needs_input_grad as it is
    if ask is None:
        return need
    for i, (node, _) in enumerate(ctx.next_functions):
        if need[skip + i] and node is not None:
            try:
                need[skip + i] = bool(ask(node))
            except Exception:       # a leaf under torch.autograd.grad (RuntimeError), or an API that changed
                pass
    return need


def encoder_forward(ops, px, biases):
    """conv1 (pixels arrive augmented: no shift, as act() runs it) .. conv4 into TB features, then fp32 features in
    the reference order.  px: uint8 pixels, or fp32 ones (Encoder(pixels="float"): drq_conv1_fwd_bf16_from_f32).
    Returns (features, [conv1..3 WB activations])."""
    n, cin = px.shape[0], px.shape[1]
    dev, s = px.device, _stream()
    nel = _lib.lib().drq_wb_elems(n)
    acts = [_zb(nel, dev) for _ in range(3)]     # zeroed: guard rows and the slack are read as zero padding
    ft = TB(n, REPR_DIM, dev)
    a = [t.data_ptr() for t in acts]
    if px.dtype == torch.uint8:
        call("drq_conv1_fwd_bf16", px.data_ptr(), None, ops.conv1.data_ptr(), a[0], n, cin, 4, s)
    else:
        call("drq_conv1_fwd_bf16_from_f32", px.data_ptr(), ops.conv1.data_ptr(), a[0], n, cin, s)
    call("drq_conv3x3_fwd_bf16", a[0], ops.wf[0].data_ptr(), biases[0], a[1], n, 39, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", a[1], ops.wf[1].data_ptr(), biases[1], a[2], n, 37, 0, 0, 0, 0, s)
    call("drq_conv3x3_fwd_bf16", a[2], ops.wf[2].data_ptr(), biases[2], ft.ptr(), n, 35, 2, ft.units, 0, 0, s)
    feat = torch.empty(n, REPR_DIM, device=dev)
    call("drq_features_to_ref", ft.ptr(), 1, feat.data_ptr(), n, s)
    return feat, acts


class EncoderFn(torch.autograd.Function):
    """features = Encoder(pixels) on the tensor cores; backward drq_feature_grad_wide_bf16 -> conv4..2
    drq_conv3x3_{wgrad (partials), dgrad}_bf16 -> drq_conv1_wgrad_bf16 -> one drq_conv_wgrad_reduce_multi.
    Inputs: operand copies, pixels - uint8, or fp32 on the 0..255 scale (Encoder(pixels="float"): the *_from_f32
    conv1 kernels, and drq_conv1_dgrad_bf16 for pixels that require grad) - then (weight, bias) of conv1..4.  Every
    weight gradient runs only when its parameter needs it."""

    @staticmethod
    def forward(ctx, ops, px, *params):
        feat, acts = encoder_forward(ops, px, [p.data_ptr() for p in params[3::2]])
        ctx.ops = ops
        ctx.save_for_backward(px, *acts, feat)
        return feat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dfeat):
        px, a1, a2, a3, feat = ctx.saved_tensors
        need_all = needed(ctx, skip=1)
        need_x, need = need_all[1], need_all[2:]
        if not (need_x or any(need)):
            return (None,) * 10
        n, cin = px.shape[0], px.shape[1]
        dev, s, L = feat.device, _stream(), _lib.lib()
        dfeat = dfeat.float().contiguous()
        nel = L.drq_wb_elems(n)
        acts = [a1.data_ptr(), a2.data_ptr(), a3.data_ptr()]
        # d[l]: gradient w.r.t. conv(l+1)'s pre-ReLU output.  d[3] is written whole by drq_feature_grad_wide_bf16; the
        # data gradients write rows < hout + 2 of each image, the rest must stay zero
        d = [_zb(nel, dev) for _ in range(3)] + [torch.empty(nel, dtype=torch.bfloat16, device=dev)]
        dp = [t.data_ptr() for t in d]
        ws = [torch.zeros(L.drq_conv1_wgrad_bf16_ws_floats(), device=dev)] + \
             [torch.zeros(L.drq_conv_wgrad_bf16_ws_floats(), device=dev) for _ in range(3)]
        grads = [torch.empty(shape, device=dev) for shape in [(32, cin, 3, 3), (32,)] + [(32, 32, 3, 3), (32,)] * 3]
        call("drq_feature_grad_wide_bf16", dfeat.data_ptr(), feat.data_ptr(), dp[3], n, s)
        jobs = []
        for layer, hout in ((3, 35), (2, 37), (1, 39)):
            if need[2 * layer] or need[2 * layer + 1]:
                call("drq_conv3x3_wgrad_bf16", acts[layer - 1], n, dp[layer], ws[layer].data_ptr(), None, None, n, hout, s)
                jobs.append(WgReduceJob(ws[layer].data_ptr(), grads[2 * layer].data_ptr(),
                                        grads[2 * layer + 1].data_ptr(), n, hout, 0, 0))
            if need_x or any(need[:2 * layer]):
                call("drq_conv3x3_dgrad_bf16", dp[layer], ctx.ops.wd[layer - 1].data_ptr(), acts[layer - 1], n,
                     dp[layer - 1], n, hout, s)
        if need[0] or need[1]:
            if px.dtype == torch.uint8:
                call("drq_conv1_wgrad_bf16", px.data_ptr(), None, dp[0], ws[0].data_ptr(), None, None, n, cin, 4, s)
                jobs.append(WgReduceJob(ws[0].data_ptr(), grads[0].data_ptr(), grads[1].data_ptr(), n, 0, cin, 0))
            else:
                call("drq_conv1_wgrad_bf16_from_f32", px.data_ptr(), dp[0], ws[0].data_ptr(), grads[0].data_ptr(),
                     grads[1].data_ptr(), n, cin, s)
        if jobs:
            call("drq_conv_wgrad_reduce_multi", (WgReduceJob * len(jobs))(*jobs), len(jobs), s)
        dx = None
        if need_x:
            dx = torch.empty(px.shape, device=dev)
            call("drq_conv1_dgrad_bf16", dp[0], ctx.ops.conv1.data_ptr(), dx.data_ptr(), n, cin, s)
        return (None, dx) + tuple(g if nd else None for g, nd in zip(grads, need))


# ---- heads: the trunk (Linear(39200 -> F) + LayerNorm + tanh) shared by Actor and Critic
def _trunk_forward(ops, feat, Fd, tb, gamma, beta, h_ld, tail=None, A=0):
    """pack the fp32 features, the split-K trunk GEMM with act()'s split rule, the LayerNorm tail.  Returns
    (feature TB, h fp32 [B, h_ld], xhat, rstd, bf16 h TB of Fd + A features (the action appended when tail))."""
    B, dev, s = feat.shape[0], feat.device, _stream()
    ft = TB(B, REPR_DIM, dev)
    call("drq_pack_features_tb", feat.data_ptr(), ft.ptr(), B, s)
    FP = _ceil(Fd, TB_W)
    S = splitk_for((ft.rpad // TB_ACT) * (FP // 64))
    part = torch.empty(S * B * FP, device=dev)
    gemm(ft.ptr(), ft.units, ops.trunk, ops.trunk_units, GEMM_KK, part.data_ptr(), FP, B, FP, REPR_DIM, TEPI_F32,
         splitk=S, strides=_strides(split=B * FP))
    h, xhat, rstd = torch.empty(B, Fd, device=dev), torch.empty(B, Fd, device=dev), torch.empty(B, device=dev)
    hb = TB(B, Fd + A, dev)
    ln_tanh_multi([LnJob(part.data_ptr(), FP, B * FP, S, tb, gamma, beta, h.data_ptr(), Fd, xhat.data_ptr(),
                         rstd.data_ptr(), hb.buf.data_ptr(), hb.units, 0, tail, A, A if tail else 0)], B, Fd)
    return ft, h, xhat, rstd, hb


def _trunk_backward(ops, dh_planes, ld, n_planes, plane_stride, B, Fd, ft, h, xhat, rstd, gamma, need_feat, jobs, gp):
    """tanh / LayerNorm backward from dh (n_planes summed on the fly), the trunk weight gradient (reference column
    order) and, when need_feat, the feature gradient in the reference order.  gp = (dW, db, dgamma, dbeta): db / dgamma
    / dbeta join the caller's colsum jobs.  Returns dfeat or None."""
    dev, s = h.device, _stream()
    dz = torch.empty(2 * B * Fd, device=dev)        # [dz | dy]
    zt = TB(B, Fd, dev)
    call("drq_ln_tanh_bwd", dh_planes, ld, h.data_ptr(), Fd, xhat.data_ptr(), rstd.data_ptr(), gamma, dz.data_ptr(),
         None, None, zt.ptr(), zt.units, B, Fd, n_planes, plane_stride, s)
    gemm(zt.ptr(), zt.units, ft.ptr(), ft.units, GEMM_MNMN, gp[0].data_ptr(), REPR_DIM, Fd, REPR_DIM, B, TEPI_TRUNK_WGRAD,
         bn=128)
    dy = dz.data_ptr() + F32 * B * Fd
    jobs += [ColsumJob(dz.data_ptr(), Fd, gp[1].data_ptr(), B, Fd, 0, 0),
             ColsumJob(dy, Fd, gp[2].data_ptr(), B, Fd, 0, 0, xhat.data_ptr()),
             ColsumJob(dy, Fd, gp[3].data_ptr(), B, Fd, 0, 0)]
    colsum_multi(jobs)
    if not need_feat:
        return None
    de = torch.empty(B, REPR_DIM, device=dev)       # encoder-output order
    gemm(zt.ptr(), zt.units, ops.trunk, ops.trunk_units, GEMM_KMN, de.data_ptr(), REPR_DIM, B, REPR_DIM, Fd, TEPI_F32)
    dfeat = torch.empty(B, REPR_DIM, device=dev)
    call("drq_features_to_ref", de.data_ptr(), 0, dfeat.data_ptr(), B, s)
    return dfeat


# ---- Actor
def actor_forward(ops, feat, tw):
    """mu = tanh(policy(trunk(features))) (drqv2.py:85-89) as act() computes it in eval mode.  tw: the Actor's
    (trunk.0 W, b, LayerNorm gamma, beta, policy W1, b1, W2, b2, W3, b3) tensors.  Returns (mu, saved)."""
    B, dev, s = feat.shape[0], feat.device, _stream()
    Fd, H, A = tw[0].shape[0], tw[4].shape[0], tw[8].shape[0]
    ft, h, xhat, rstd, hb = _trunk_forward(ops, feat, Fd, tw[1].data_ptr(), tw[2].data_ptr(), tw[3].data_ptr(), Fd)
    p1, p2 = TB(B, H, dev), TB(B, H, dev)
    gemm(hb.ptr(), hb.units, ops.p0.ptr(), ops.p0.units, GEMM_KK, p1.ptr(), p1.units, B, H, Fd, TEPI_RELU_BF16,
         bias=tw[5].data_ptr())
    gemm(p1.ptr(), p1.units, ops.p2.ptr(), ops.p2.units, GEMM_KK, p2.ptr(), p2.units, B, H, H, TEPI_RELU_BF16,
         bias=tw[7].data_ptr())
    mu_pre, mu = torch.empty(B, A, device=dev), torch.empty(B, A, device=dev)
    job = PolicySample(0, B, None, mu.data_ptr(), A, None, None, None, 0, 0, 0)
    call("drq_policy_head_fwd_bf16", p2.ptr(), p2.units, tw[8].data_ptr(), tw[9].data_ptr(), mu_pre.data_ptr(), B, H, A,
         (PolicySample * 1)(job), 1, None, 0.0, None, s)
    return mu, (ft.buf, h, xhat, rstd, hb.buf, p1.buf, p2.buf, mu)


class ActorFn(torch.autograd.Function):
    """mu on the tensor cores; backward drq_actor_sample_bwd, the policy MLP's MNMN (weight) / KMN (data) GEMMs, the
    trunk backward and one drq_colsum_multi for every bias, LayerNorm affine included.  Inputs: operand copies,
    features, trunk (W, b, gamma, beta), policy (W1, b1, W2, b2, W3, b3)."""

    @staticmethod
    def forward(ctx, ops, feat, *tw):
        mu, saved = actor_forward(ops, feat, tw)
        ctx.ops = ops
        ctx.save_for_backward(*saved, tw[2])
        return mu

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dmu):
        ftb, h, xhat, rstd, hbb, p1b, p2b, mu, gamma = ctx.saved_tensors
        need = ctx.needs_input_grad[1:]
        if not any(need):
            return (None,) * 12
        ops, s = ctx.ops, _stream()
        B, A = mu.shape
        Fd, H, dev = h.shape[1], ops.p0.rows, h.device
        ft, hb = _wrap(ftb, B, REPR_DIM), _wrap(hbb, B, Fd)
        p1, p2 = _wrap(p1b, B, H), _wrap(p2b, B, H)
        U = p1.units
        dmu = dmu.float().contiguous()
        dmu_pre, dmt = torch.empty(B, A, device=dev), TB(B, A, dev)
        call("drq_actor_sample_bwd", dmu.data_ptr(), A, mu.data_ptr(), dmu_pre.data_ptr(), dmt.ptr(), dmt.units, B, A, 1,
             0, s)
        g = [torch.empty(shape, device=dev) for shape in ((Fd, REPR_DIM), (Fd,), (Fd,), (Fd,), (H, Fd), (H,), (H, H), (H,),
                                                         (A, H), (A,))]
        dp1, dp2 = TB(B, H, dev), TB(B, H, dev)
        gemm(dmt.ptr(), dmt.units, p2.ptr(), U, GEMM_MNMN, g[8].data_ptr(), H, A, H, B, TEPI_F32, bn=128)
        gemm(dmt.ptr(), dmt.units, ops.p4.ptr(), ops.p4.units, GEMM_KMN, dp2.ptr(), U, B, H, A, TEPI_MASK_BF16,
             mask=p2.ptr(), units_mask=U)
        gemm(dp2.ptr(), U, p1.ptr(), U, GEMM_MNMN, g[6].data_ptr(), H, H, H, B, TEPI_F32, bn=128)
        gemm(dp2.ptr(), U, ops.p2.ptr(), ops.p2.units, GEMM_KMN, dp1.ptr(), U, B, H, H, TEPI_MASK_BF16, mask=p1.ptr(),
             units_mask=U)
        gemm(dp1.ptr(), U, hb.ptr(), hb.units, GEMM_MNMN, g[4].data_ptr(), Fd, H, Fd, B, TEPI_F32)
        dh = torch.empty(B, Fd, device=dev)
        gemm(dp1.ptr(), U, ops.p0.ptr(), ops.p0.units, GEMM_KMN, dh.data_ptr(), Fd, B, Fd, H, TEPI_F32)
        jobs = [ColsumJob(dmu_pre.data_ptr(), A, g[9].data_ptr(), B, A, 0, 0),
                ColsumJob(dp2.ptr(), U, g[7].data_ptr(), B, H, 1, 0), ColsumJob(dp1.ptr(), U, g[5].data_ptr(), B, H, 1, 0)]
        dfeat = _trunk_backward(ops, dh.data_ptr(), Fd, 1, 0, B, Fd, ft, h, xhat, rstd, gamma.data_ptr(), need[0], jobs,
                                g[:4])
        return (None, dfeat) + tuple(t if nd else None for t, nd in zip(g, need[1:]))


# ---- Critic
def critic_forward(ops, feat, action, cw):
    """(Q1, Q2) = Critic(features, action) (drqv2.py:115-121).  cw: trunk (W, b, gamma, beta), Q1 (W1, b1, W2, b2, W3,
    b3), Q2 (the same).  One launch per layer and head.  Returns (q1, q2, saved)."""
    B, dev, s = feat.shape[0], feat.device, _stream()
    Fd, H = cw[0].shape[0], cw[4].shape[0]
    A = cw[4].shape[1] - Fd
    ft, h, xhat, rstd, xb = _trunk_forward(ops, feat, Fd, cw[1].data_ptr(), cw[2].data_ptr(), cw[3].data_ptr(), Fd,
                                           tail=action.data_ptr(), A=A)
    c1, c2 = TB(B, H, dev, batch=2), TB(B, H, dev, batch=2)
    qs = []
    for z in range(2):
        w = cw[4 + 6 * z:10 + 6 * z]
        gemm(xb.ptr(), xb.units, ops.q0.ptr(ops.z0 + z), ops.q0.units, GEMM_KK, c1.ptr(z), c1.units, B, H, Fd + A,
             TEPI_RELU_BF16, bias=w[1].data_ptr())
        gemm(c1.ptr(z), c1.units, ops.q2.ptr(ops.z0 + z), ops.q2.units, GEMM_KK, c2.ptr(z), c2.units, B, H, H,
             TEPI_RELU_BF16, bias=w[3].data_ptr())
        q = torch.empty(B, 1, device=dev)
        call("drq_q_head_fwd_bf16", c2.ptr(z), c2.units, c2.stride, w[4].data_ptr(), w[5].data_ptr(), q.data_ptr(), B, H,
             1, 0, 1, 0, s)
        qs.append(q)
    return qs[0], qs[1], (ft.buf, xb.buf, h, xhat, rstd, c1.buf, c2.buf)


class CriticFn(torch.autograd.Function):
    """(Q1, Q2) on the tensor cores; backward per head that received a gradient (a None gradient skips its head):
    drq_q_head_bwd_bf16, the Q MLP's weight / masked data GEMMs, the first layer's data gradient as split-K planes
    [head][split], drq_plane_sum_f32 over their action columns, and the trunk backward (drq_ln_tanh_bwd sums the
    same planes' h columns).  Inputs: operand copies, features, action, trunk (W, b, gamma, beta), Q1 and Q2 (W1, b1,
    W2, b2, W3, b3 each)."""

    @staticmethod
    def forward(ctx, ops, feat, action, *cw):
        ctx.set_materialize_grads(False)
        q1, q2, saved = critic_forward(ops, feat, action, cw)
        ctx.ops = ops
        ctx.save_for_backward(*saved, cw[2], cw[8], cw[14])
        return q1, q2

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dq1, dq2):
        ftb, xbb, h, xhat, rstd, c1b, c2b, gamma, w3a, w3b = ctx.saved_tensors
        need = ctx.needs_input_grad[1:]
        if (dq1 is None and dq2 is None) or not any(need):
            return (None,) * 19
        ops, s = ctx.ops, _stream()
        B, Fd = h.shape
        H = ops.q2.rows
        A = ops.q0.feats - Fd
        dev = h.device
        ft, xb = _wrap(ftb, B, REPR_DIM), _wrap(xbb, B, Fd + A)
        c1, c2 = _wrap(c1b, B, H, batch=2), _wrap(c2b, B, H, batch=2)
        U, K1 = c1.units, Fd + A
        heads = [z for z, dq in enumerate((dq1, dq2)) if dq is not None]
        SX = 8 if H % 1024 == 0 else 1                 # the fused update's split of this K = H contraction
        PS = B * K1
        dxf = torch.empty(len(heads) * SX, B, K1, device=dev)    # planes [head][split]
        dc1, dc2 = TB(B, H, dev, batch=2), TB(B, H, dev, batch=2)
        gq = [None] * 12
        jobs = []
        for i, z in enumerate(heads):
            dq = (dq1, dq2)[z].float().contiguous()
            g = [torch.empty(shape, device=dev) for shape in ((H, K1), (H,), (H, H), (H,), (1, H), (1,))]
            call("drq_q_head_bwd_bf16", dq.data_ptr(), None, c2.ptr(z), U, c2.stride, (w3a, w3b)[z].data_ptr(), dc2.ptr(z),
                 g[4].data_ptr(), g[5].data_ptr(), B, H, 0, s)
            gemm(dc2.ptr(z), U, c1.ptr(z), U, GEMM_MNMN, g[2].data_ptr(), H, H, H, B, TEPI_F32, bn=128)
            gemm(dc2.ptr(z), U, ops.q2.ptr(ops.z0 + z), ops.q2.units, GEMM_KMN, dc1.ptr(z), U, B, H, H, TEPI_MASK_BF16,
                 mask=c1.ptr(z), units_mask=U)
            gemm(dc1.ptr(z), U, xb.ptr(), xb.units, GEMM_MNMN, g[0].data_ptr(), K1, H, K1, B, TEPI_F32)
            gemm(dc1.ptr(z), U, ops.q0.ptr(ops.z0 + z), ops.q0.units, GEMM_KMN, dxf[i * SX].data_ptr(), K1, B, K1, H,
                 TEPI_F32, splitk=SX, strides=_strides(split=PS))
            jobs += [ColsumJob(dc2.ptr(z), U, g[3].data_ptr(), B, H, 1, 0), ColsumJob(dc1.ptr(z), U, g[1].data_ptr(), B, H, 1, 0)]
            gq[6 * z:6 * z + 6] = g
        planes = len(heads) * SX
        dact = None
        if need[1]:
            dact = torch.empty(B, A, device=dev)
            call("drq_plane_sum_f32", dxf.data_ptr() + F32 * Fd, K1, PS, planes, dact.data_ptr(), A, B, A, s)
        gt = [torch.empty(shape, device=dev) for shape in ((Fd, REPR_DIM), (Fd,), (Fd,), (Fd,))]
        dfeat = _trunk_backward(ops, dxf.data_ptr(), K1, planes, PS, B, Fd, ft, h, xhat, rstd, gamma.data_ptr(), need[0],
                                jobs, gt)
        grads = gt + gq
        return (None, dfeat, dact) + tuple(t if nd else None for t, nd in zip(grads, need[2:]))
