"""Every update of a multi-step run held to the reference at the agent's own state (drqv2.py:230-262).

The other whole-update tests compare gradients and losses with the oracle on the first update only (the bf16 ones at
lr = 0, where the optimiser steps do nothing and every stage reads the same parameters whatever their version).  After
real-lr steps they bound the parameters by |got - want| <= 2.5 lr steps.  Adam moves an element by about lr per step
whatever its gradient is (by exactly lr sign(g) on step 1), so both sides move by at most about lr steps and that bound
holds for any finite gradient: a wrong sign, zero, or the gradient of another tensor.  It catches NaN and blow-ups only.
The schedule tests compare CUDA paths with each other, which a version error shared by every path passes.

Here the oracle is re-seeded from the agent's parameters before every update (teacher forcing), so Adam's sign-like
divergence never builds up and every update of a run is held to single-update bounds.  Per update k, with S_k the
agent's state before it:
  1. optimiser, exact: drq_adam_step on the snapshot's parameters / moments with the update's own gradients and the
     Adam scalars of this test's own step count per net, then drq_soft_update of the snapshot target from the stepped
     critic, equal the agent's arenas bit for bit (padding stays zero).  This checks the plumbing: optimiser plans and
     segments, scalar ring slots, step counts, the order of the soft update;
  2. operands fresh (bf16 mode): every packed bf16 operand equals a fresh repack of its fp32 master, bit for bit;
  3. the critic stage at S_k: the oracle loaded with S_k, on the batch and draws the update actually used (read back
     from the workspace, so device-drawn updates are checked too), against the update's critic metrics and the encoder
     and critic gradients;
  4. the actor stage at the agent's stepped critic (drqv2.py:213 reads the critic after critic_opt.step(), :201);
  5. power: the oracle's actor stage at the pre-step critic, and (k >= 1) its critic stage with S_{k-1}'s critic, are
     each at least POWER x the bound of check 3 / 4 away from the right reference in some metric or gradient tensor -
     so a stale read of either version would fail.  A stale target only moves the numbers by tau * (one critic step), which no tolerance
     sees; check 1 covers the target exactly instead.
LR is the smallest of {3e-4, 1e-3, 3e-3} at which (5) holds at every update of configuration 1;
tests/test_update_chain_power_cpu.py asserts that margin with the oracle alone on any machine."""
import math
from collections import OrderedDict

import numpy as np
import pytest
import torch

from oracle import drq_oracle as O
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"
TAU, CLIP = 0.01, 0.3
LR = 3e-4
CONFIG1 = dict(A=6, F=50, H=256, B=64)         # >= 48 images: the parity-plane conv1 and the four-pixel-column forward
POWER = 3.0
NETS = ("encoder", "critic", "actor")
CRITIC_METRICS = ("batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss")
ACTOR_METRICS = ("actor_loss", "actor_logprob")


class Bounds:
    """Tolerances of checks 3 and 4: metrics |got - want| <= rtol |want| + atol; gradients per tensor
    rel-L2 <= max(floor(net, name), own * the fp32 oracle's own rel-L2 to fp64) and, in bf16 mode, cosine >= cos."""

    def __init__(self, rtol, atol, floor, own, cos):
        self.rtol, self.atol, self.floor, self.own, self.cos = rtol, atol, floor, own, cos

    def metric(self, want):
        return self.rtol * abs(want) + self.atol

    def grad(self, net, name, own):
        return max(self.floor(net, name), self.own * own)


# bf16 mode against the bf16-faithful oracle: the rule of test_gpu_bench_config.test_update_bf16_at_bench_config, except
# that conv1's weight gradient, the end of the backward chain, has a floor of 5e-2.  Activations that the kernels (fp32
# accumulation) and the oracle (fp64) round to neighbouring bf16 values flip ReLU units, and the flips add up along the
# chain; on conv1's gradient that noise is 3.6e-2 at B=256 (test_gpu_bench_config), and on a B200 in this module it
# reached 3.5e-2 (1.75x the fp32 oracle's own distance) at update 5 of configuration 1 and 2.3e-2 (2.7x its own) at
# update 1 of configuration 6, where the batches repeat frames of a 100-slot ring.  Every other tensor keeps 2e-2.
BF16 = Bounds(2e-3, 1e-4, lambda net, name: 5e-2 if (net, name) == ("encoder", "convnet.0.weight") else 2e-2, 1.5, 0.95)
# fp32 mode against the exact-operand oracle: the rule of test_gpu_parity._check_update_against_oracle
FP32 = Bounds(1e-4, 1e-6, lambda net, name: 3e-3 if net == "encoder" else 1e-3, 3.0, None)


# ----------------------------------------------------------------------------- oracle side (also used on the CPU)
def oracle_at(state, dtype, operands="bf16", moments=None, lr=LR, sched=SCHED):
    """An OracleAgent holding `state` ({net: {name: tensor}} of the four nets); `moments` (m, v, t) make its own
    optimiser steps continue the run's Adam state"""
    o = O.OracleAgent(state, lr, TAU, sched, CLIP, dtype=dtype, operands=operands)
    o.stage = {}                                   # update_actor records into it; update_critic starts it
    if moments is not None:
        m, v, t = moments
        for net in NETS:
            o.m[net] = OrderedDict((k, x.to(dtype).clone()) for k, x in m[net].items())
            o.v[net] = OrderedDict((k, x.to(dtype).clone()) for k, x in v[net].items())
        o.t = dict(t)
    return o


def critic_stage(o, b, step):
    """aug + encoder + update_critic (drqv2.py:241-250,177-204) with the encoder attached.  Returns the critic
    metrics, the detached features of obs and next_obs and the gradients {encoder, critic}; `o` is left with the
    stepped encoder and critic."""
    enc = {k: v.requires_grad_(True) for k, v in o.p["encoder"].items()}
    feat = o.encode(b["obs"], b["shift_obs"], enc)
    with torch.no_grad():
        feat_next = o.encode(b["next_obs"], b["shift_next"], enc)
    m = o.update_critic(feat, b["action"], b["reward"], b["discount"], feat_next, step, b["eps_critic"], enc=enc)
    m["batch_reward"] = b["reward"].to(o.dtype).mean().item()
    return m, feat.detach(), feat_next, dict(encoder=o.grads["encoder"], critic=o.grads["critic"])


def critic_stage_with(state, critic, feat, feat_next, b, step, operands="bf16", sched=SCHED):
    """the critic stage's metrics and critic gradients with the online critic replaced by `critic` (the rest from
    `state`) on given features"""
    o = oracle_at(dict(state, critic=critic), torch.float64, operands, sched=sched)
    m = o.update_critic(feat, b["action"], b["reward"], b["discount"], feat_next, step, b["eps_critic"])
    m["batch_reward"] = b["reward"].double().mean().item()
    return m, o.grads["critic"]


def actor_stage(o, feat, step, eps_actor, critic=None):
    """update_actor (drqv2.py:206-228) on detached features, with the online critic replaced by `critic` if given.
    Returns the actor metrics and gradients."""
    if critic is not None:
        o.p["critic"] = OrderedDict((k, v.to(o.dtype).clone()) for k, v in critic.items())
    m = o.update_actor(feat, step, eps_actor)
    return m, o.grads["actor"]


def margin(wrong_m, right_m, keys, wrong_g, ref, bounds):
    """how many of check 3 / 4's bounds a wrong reference (metrics, {net: gradients}) is from the right one: the
    largest distance-to-bound ratio over the metrics `keys` and the gradients of the nets in wrong_g"""
    r = max(abs(wrong_m[k] - right_m[k]) / bounds.metric(right_m[k]) for k in keys)
    for net, g in wrong_g.items():
        for name, x in g.items():
            r = max(r, rel_l2(x.numpy(), ref["grads"][net][name].numpy()) / bounds.grad(net, name, ref["own"][net][name]))
    return r


def references(S, S_prev, b, step, bounds, operands="bf16", sched=SCHED, post_critic=None, moments=None, lr=LR):
    """The oracle's side of checks 3-5 at state S on batch / draws b: the critic stage at S and the actor stage at
    `post_critic` (the agent's stepped critic; None: the oracle's own), in fp64 (the reference) and fp32 (the
    yardstick `own`: its rel-L2 to fp64 per gradient tensor), and the power margins (a) of the actor stage at S's
    pre-step critic and (b) of the critic stage at S_prev's critic (None without S_prev).  `oracle` is the fp64
    oracle after both stages (its parameters stepped from `moments`)."""
    o64 = oracle_at(S, torch.float64, operands, moments, lr, sched)
    o32 = oracle_at(S, torch.float32, operands, moments, lr, sched)
    mc, feat, feat_next, g64 = critic_stage(o64, b, step)
    _, feat32, _, g32 = critic_stage(o32, b, step)
    critic = post_critic if post_critic is not None else o64.p["critic"]
    ma, ga64 = actor_stage(o64, feat, step, b["eps_actor"], critic=post_critic)
    _, ga32 = actor_stage(o32, feat32, step, b["eps_actor"], critic=critic)
    ref = dict(critic=mc, actor=ma, grads=dict(encoder=g64["encoder"], critic=g64["critic"], actor=ga64), oracle=o64)
    g32 = dict(encoder=g32["encoder"], critic=g32["critic"], actor=ga32)
    ref["own"] = {net: {n: rel_l2(g32[net][n].numpy(), x.numpy()) for n, x in g.items()} for net, g in ref["grads"].items()}
    stale_m, stale_g = actor_stage(oracle_at(S, torch.float64, operands, sched=sched), feat, step, b["eps_actor"])
    ref["margin_a"] = margin(stale_m, ma, ACTOR_METRICS, dict(actor=stale_g), ref, bounds)
    ref["margin_b"] = None
    if S_prev is not None:
        stale_m, stale_g = critic_stage_with(S, S_prev["critic"], feat, feat_next, b, step, operands, sched)
        ref["margin_b"] = margin(stale_m, mc, CRITIC_METRICS, dict(critic=stale_g), ref, bounds)
    return ref


def actor_ent(A, step, sched=SCHED):
    """drqv2.py:224 with utils.py:105-126's entropy of a Normal: A (1/2 + ln(2 pi)/2 + ln std(step))"""
    return A * (0.5 + 0.5 * math.log(2 * math.pi) + math.log(O.schedule(sched, step)))


# ----------------------------------------------------------------------------- agent side
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _tensors(agent, flat, net, base=0):
    """{name: view} of net's tensors in a flat arena (base: the arena's offset of the critic for the target arena)"""
    a = agent._arena
    return OrderedDict((k, flat[a.offsets[net][k] - base:a.offsets[net][k] - base + p.numel()].view(p.shape))
                       for k, p in getattr(agent, net).named_parameters())


def _state(agent, params, target):
    """the four nets of flat parameter / target arenas as the oracle's CPU parameter dicts"""
    params, target = params.cpu(), target.cpu()
    out = OrderedDict((net, _tensors(agent, params, net)) for net in NETS)
    out["critic_target"] = _tensors(agent, target, "critic", base=agent._arena.seg["critic"][0])
    return out


def _live(agent):
    """masks of the parameter and target arenas: True on the tensors, False on the alignment padding between them"""
    a = agent._arena
    live = torch.zeros(a.total, dtype=torch.bool, device=a.params.device)
    for net in NETS:
        for k, p in getattr(agent, net).named_parameters():
            live[a.offsets[net][k]:a.offsets[net][k] + p.numel()] = True
    c0, cn = a.seg["critic"][0], a.seg["critic"][2]
    return live, live[c0:c0 + cn]


def _snapshot(agent):
    a = agent._arena
    return dict(params=a.params.clone(), m=a.exp_avg.clone(), v=a.exp_avg_sq.clone(), target=a.target.clone())


def check_optimiser_exact(agent, snap, t, live):
    """check 1: Adam of each net from the snapshot with the update's gradients and this test's step counts, then the
    soft update of the snapshot target from the stepped critic, equal the agent's arenas bit for bit"""
    from drqv2_b200 import utils
    from drqv2_b200._lib import call
    a = agent._arena
    p, m, v, tgt = (snap[k].clone() for k in ("params", "m", "v", "target"))
    scalars = []
    for net in NETS:
        off, n = a.seg[net][0], a.seg[net][2]
        scalars.append(torch.from_numpy(utils.adam_scalars(agent.lr, t[net] + 1)).to(p.device))
        call("drq_adam_step", p[off:].data_ptr(), a.grads[off:].data_ptr(), m[off:].data_ptr(), v[off:].data_ptr(), n,
             scalars[-1].data_ptr(), _stream())
    c0, cn = a.seg["critic"][0], a.seg["critic"][2]
    call("drq_soft_update", a.params[c0:].data_ptr(), tgt.data_ptr(), cn, TAU, 1 - TAU, _stream())
    torch.cuda.synchronize()
    bad = []
    for what, got, want in (("param", a.params, p), ("exp_avg", a.exp_avg, m), ("exp_avg_sq", a.exp_avg_sq, v)):
        for net in NETS:
            for (k, x), y in zip(_tensors(agent, got, net).items(), _tensors(agent, want, net).values()):
                if not torch.equal(x, y):
                    bad.append(f"{what} {net}.{k}: {int((x != y).sum())} of {x.numel()} differ")
    for (k, x), y in zip(_tensors(agent, a.target, "critic", base=c0).items(), _tensors(agent, tgt, "critic", base=c0).values()):
        if not torch.equal(x, y):
            bad.append(f"target {k}: {int((x != y).sum())} of {x.numel()} differ")
    assert not bad, "optimiser state differs from drq_adam_step / drq_soft_update on the snapshot: " + "; ".join(bad)
    live, live_t = live
    for what, x in (("param", a.params), ("grad", a.grads), ("exp_avg", a.exp_avg), ("exp_avg_sq", a.exp_avg_sq)):
        assert not x[~live].any(), f"{what} arena padding is not zero"
    assert not a.target[~live_t].any(), "target arena padding is not zero"


def _packed(st):
    """(name, view) of every bf16 operand copy of the agent's Bf16State; the merged trunk weight by slot, the Q-layer
    copies by head"""
    out = []
    for slot, who in ((st.TARGET, "target"), (st.ACTOR, "actor"), (st.CRITIC, "critic")):
        out.append((f"trunk[{who}]", st.trunk.buf[st.trunk.off(row=slot * st.FP):st.trunk.off(row=(slot + 1) * st.FP)]))
    for name, tb in (("Q.0", st.q0), ("Q.2", st.q2)):
        for z, who in enumerate(("critic.Q1", "critic.Q2", "target.Q1", "target.Q2")):
            out.append((f"{who}{name[1:]}", tb.buf[z * tb.stride:(z + 1) * tb.stride]))
    for name, tb in (("policy.0", st.p0), ("policy.2", st.p2), ("policy.4", st.p4)):
        out.append((name, tb.buf))
    out.append(("conv1", st.conv1_w))
    for i in range(3):
        out += [(f"conv{i + 2}.fwd", st.conv_wf[i]), (f"conv{i + 2}.dgrad", st.conv_wd[i])]
    return out


def check_operands_fresh(agent):
    """check 2: every packed bf16 operand equals a fresh repack of its fp32 master, bit for bit"""
    views = _packed(agent._bf16)
    before = [v.clone() for _, v in views]
    agent._bf16.repack_all()
    torch.cuda.synchronize()
    stale = [name for (name, v), b in zip(views, before) if not torch.equal(v.view(torch.int16), b.view(torch.int16))]
    assert not stale, f"bf16 operand copies that differ from a fresh repack of their fp32 masters: {stale}"


def batch_used(agent, ws, fed, ring):
    """the batch and draws the update actually used, read back from its workspace; in ring-direct mode the frame stacks
    rebuilt from the sampled (episode start, index) by the oracle's gather, which the sampled action / n-step reward /
    discount must equal bit for bit"""
    B = ws.B
    b = dict(shift_obs=ws.shift[:B].cpu(), shift_next=ws.shift[B:].cpu(), eps_critic=ws.eps_c.cpu(),
             eps_actor=ws.eps_a.cpu(), action=ws.action.cpu(), reward=ws.reward.cpu(), discount=ws.discount.cpu())
    if ring is not None:
        loader, frames, action, reward, discount = ring
        es, ix = loader._ep_start.cpu().numpy(), loader._idx.cpu().numpy()
        obs, act, rew, disc, nxt = O.ring_gather(frames, action, reward, discount, es, ix, loader.nstep, loader.discount)
        for k, want in (("action", act), ("reward", rew), ("discount", disc)):
            assert np.array_equal(b[k].numpy(), want), f"ws.{k} is not the sample of (ep_start, idx)"
        b.update(obs=torch.from_numpy(obs), next_obs=torch.from_numpy(nxt))
    else:
        for k in ("obs", "action", "reward", "discount"):
            assert torch.equal(getattr(ws, k)[:B].cpu(), fed[k].view(getattr(ws, k)[:B].shape)), f"ws.{k} is not the batch"
        b.update(obs=fed["obs"], next_obs=fed["next_obs"])
    return b


def check_stage(stage, m_gpu, grads, ref, bounds):
    """check 3 (stage "critic": its metrics, encoder and critic gradients) or 4 ("actor") against references();
    returns the largest error-to-bound ratio"""
    keys, nets = (CRITIC_METRICS, ("encoder", "critic")) if stage == "critic" else (ACTOR_METRICS, ("actor",))
    ratio = 0.0
    for k in keys:
        want = ref[stage][k]
        assert abs(m_gpu[k] - want) <= bounds.metric(want), (k, m_gpu[k], want)
        ratio = max(ratio, abs(m_gpu[k] - want) / bounds.metric(want))
    for net in nets:
        for name, want in ref["grads"][net].items():
            got, want = grads[net][name].double().flatten(), want.flatten()
            err, bound = rel_l2(got.numpy(), want.numpy()), bounds.grad(net, name, ref["own"][net][name])
            assert err <= bound, (f"{net}.{name} gradient rel-L2", err, "own", ref["own"][net][name])
            if bounds.cos is not None:
                cos = float(torch.dot(got, want) / (got.norm() * want.norm() + 1e-300))
                assert cos >= bounds.cos, (f"{net}.{name} gradient cosine", cos)
            ratio = max(ratio, err / bound)
    return ratio


def check_power(ref):
    """check 5: the references a stale read would produce are far outside the bounds checks 3 and 4 apply"""
    assert ref["margin_a"] >= POWER, ("actor stage at the pre-step critic is within reach of the bounds", ref["margin_a"])
    assert ref["margin_b"] is None or ref["margin_b"] >= POWER, \
        ("critic stage at the previous critic is within reach of the bounds", ref["margin_b"])


def _ring_feed(tag, A, B, dev):
    from drqv2_b200 import make_replay_loader
    from tests.test_gpu_ring_direct import _ring_with_wrapping_episodes
    key = f"/test/update_chain/{tag}"
    ring = _ring_with_wrapping_episodes(key, A, dev)
    np.random.seed(9)
    loader = make_replay_loader(key, 100, B, 0, False, 3, 0.99)
    host = tuple(x.cpu().numpy() for x in (ring.frames, ring.action, ring.reward, ring.discount))
    return loader, iter(loader), (loader,) + host


def run_chain(monkeypatch, capsys, tag, mode, A, Fd, H, B, updates, ring=True, inject=False, graph=True, overlap=True,
              sched=SCHED, stage_at=None, power_at=None, odd_steps=False, stage_api_rounds=0):
    """Drive `updates` DrQV2Agent.update() calls and hold each one to checks 1-5 (checks 3-5 at the updates in
    `stage_at`, all when None; check 5 asserted at those of `power_at` among them, all when None, its margins reported
    at every one).  ring: fed from a replay ring whose episodes wrap (ring-direct in bf16 mode), else
    host batches; inject: the draws injected, else drawn on the device.  odd_steps: a step the agent must skip
    (step % update_every_steps != 0) between updates.  stage_api_rounds: update_critic / update_actor rounds first,
    so that the encoder's Adam step count trails the critic's and the actor's."""
    from drqv2_b200 import DrQV2Agent
    for k in ("DRQV2_B200_PRIO", "DRQV2_B200_EARLY_ENC", "DRQV2_B200_SPLIT_PROLOGUE", "DRQV2_B200_SMALL_GEMMS",
              "DRQV2_B200_OVERLAP", "DRQV2_B200_RING_DIRECT"):
        monkeypatch.delenv(k, raising=False)                 # the default schedule
    torch.set_num_threads(max(8, torch.get_num_threads()))
    dev = torch.device("cuda")
    bounds, operands = (BF16, "bf16") if mode == "bf16" else (FP32, "exact")
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", LR, Fd, H, TAU, 2000, 2, sched, CLIP, True, use_cuda_graph=graph,
                       seed=5, mode=mode)
    monkeypatch.setattr(agent, "overlap_encoder_backward", overlap)
    params = O.synthetic_params(9, A, Fd, H, seed=4)
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    agent.refresh()
    t = dict(encoder=0, critic=0, actor=0)               # this test's own count of each optimiser's steps
    step = 0
    for r in range(stage_api_rounds):
        fb = O.synthetic_batch(B, A, seed=200 + r)
        with torch.no_grad():
            o = oracle_at(params, torch.float32, operands)
            feat = o.encode(fb["obs"], fb["shift_obs"]).float().to(dev)
            feat_next = o.encode(fb["next_obs"], fb["shift_next"]).float().to(dev)
        agent.inject_draws(None, None, fb["eps_critic"], fb["eps_actor"])
        agent.update_critic(feat, fb["action"].to(dev), fb["reward"].to(dev), fb["discount"].to(dev), feat_next, step)
        agent.update_actor(feat, step)
        t["critic"] += 1
        t["actor"] += 1
        step += 2
    if ring:
        loader, it, ring_host = _ring_feed(tag, A, B, dev)
        assert mode != "bf16" or agent.ring_direct
    else:
        loader, it, ring_host = None, None, None
    live = _live(agent)
    ws = agent.workspace(B)
    prev = None
    for k in range(updates):
        snap = _snapshot(agent)
        fed = None
        if ring:
            m = agent.update(it, step)
        else:
            fed = O.synthetic_batch(B, A, seed=300 + k)
            if inject:
                agent.inject_draws(fed["shift_obs"], fed["shift_next"], fed["eps_critic"], fed["eps_actor"])
            m = agent.update(iter([(fed["obs"], fed["action"], fed["reward"], fed["discount"], fed["next_obs"])]), step)
        torch.cuda.synchronize()
        b = batch_used(agent, ws, fed, ring_host)
        grads = OrderedDict((net, OrderedDict((n, p.grad.cpu()) for n, p in getattr(agent, net).named_parameters()))
                            for net in NETS)
        failures = []

        def attempt(check, fn, *args):
            """run one check; a failure is collected so that the report names every check this update fails"""
            try:
                return fn(*args)
            except AssertionError as e:
                failures.append(f"check {check}: {e}")

        attempt("1 (optimiser state)", check_optimiser_exact, agent, snap, t, live)
        for net in t:
            t[net] += 1
        if mode == "bf16":
            attempt("2 (bf16 operands)", check_operands_fresh, agent)
        want_ent = actor_ent(A, step, sched)
        ent_ok = abs(m["actor_ent"] - want_ent) <= A * 2.0 ** -21 * (1.5 + abs(want_ent / A))
        if not ent_ok:
            failures.append(f"check 4: actor_ent {m['actor_ent']!r}, want {want_ent!r}")
        line = f"{tag} update {k} (step {step}):"
        if stage_at is None or k in stage_at:
            a = agent._arena
            S = _state(agent, snap["params"], snap["target"])
            S_prev = _state(agent, prev["params"], prev["target"]) if prev is not None else None
            post_critic = _state(agent, a.params, a.target)["critic"]
            ref = references(S, S_prev, b, step, bounds, operands, sched, post_critic=post_critic)
            rc = attempt("3 (critic stage at S_k)", check_stage, "critic", m, grads, ref, bounds)
            ra = attempt("4 (actor stage at the stepped critic)", check_stage, "actor", m, grads, ref, bounds)
            if power_at is None or k in power_at:
                attempt("5 (power)", check_power, ref)
            fmt = lambda x: "-" if x is None else f"{x:.2f}"
            line += (f" error / bound: critic stage {fmt(rc)}, actor stage {fmt(ra)}; power margin (a) "
                     f"{fmt(ref['margin_a'])}, (b) {fmt(ref['margin_b'])};")
        line += " exact checks (optimiser, target" + (", bf16 operands" if mode == "bf16" else "") + ", actor_ent) " + \
            ("FAILED" if any(f.startswith(("check 1", "check 2")) for f in failures) or not ent_ok else "passed")
        with capsys.disabled():
            print("\n" + line, end="")
        assert not failures, f"{tag} update {k} (step {step}): " + " | ".join(failures)
        prev = snap
        if odd_steps and k + 1 < updates:
            counter, params_now, enq = loader._counter.clone(), agent._arena.params.clone(), agent._scal_enq
            assert agent.update(it, step + 1) == {}
            torch.cuda.synchronize()
            assert torch.equal(loader._counter, counter) and agent._scal_enq == enq, "a skipped step consumed a batch"
            assert torch.equal(agent._arena.params, params_now), "a skipped step moved the parameters"
        step += 2
    with capsys.disabled():
        print()
    if graph:
        assert any(isinstance(v, torch.cuda.CUDAGraph) for v in agent._graphs.values())
    return agent


# ----------------------------------------------------------------------------- the configurations
def test_chain_bf16_ring_graph(dev, monkeypatch, capsys):
    """1: ring-direct with device draws on the default three-stream schedule: eager warm-up, capture, four replays,
    with skipped odd steps between them"""
    c = CONFIG1
    run_chain(monkeypatch, capsys, "bf16-ring", "bf16", c["A"], c["F"], c["H"], c["B"], 6, odd_steps=True)


def test_chain_bf16_one_stream(dev, monkeypatch, capsys):
    """2: the encoder backward in line: one drq_adam_pack_step for [encoder | critic] (plan_critic) and one for the actor
    with the soft update (step_actor_target)"""
    c = CONFIG1
    run_chain(monkeypatch, capsys, "bf16-one-stream", "bf16", c["A"], c["F"], c["H"], c["B"], 4, overlap=False)


def test_chain_bf16_uneven_step_counts(dev, monkeypatch, capsys):
    """3: two update_critic / update_actor rounds first, so that update() steps the encoder at t = 1.. and the critic and
    the actor at t = 3..: each net must get its own Adam bias corrections; host batches, injected draws"""
    run_chain(monkeypatch, capsys, "bf16-uneven", "bf16", 21, 100, 128, 32, 3, ring=False, inject=True,
              stage_api_rounds=2)


def test_chain_fp32(dev, monkeypatch, capsys):
    """4: the fp32 parity mode, host batches with device draws, captured"""
    run_chain(monkeypatch, capsys, "fp32", "fp32", 6, 50, 256, 32, 4, ring=False)


def test_chain_bf16_walker_shape(dev, monkeypatch, capsys):
    """5: the walker bench shape"""
    run_chain(monkeypatch, capsys, "bf16-walker", "bf16", 6, 50, 1024, 256, 3)


def test_chain_bf16_past_the_scalar_ring(dev, monkeypatch, capsys):
    """6: 300 updates, past the 256 slots of the pinned ring of per-update scalars, with a stddev of its own per update;
    checks 3 and 4 around the wrap as well.  Check 5 is asserted on the first two updates only: 250 updates in, Adam's
    steps at LR move the critic of this B=8 run so little that a one-step-stale critic is only 1.2-5.7 of check 4's
    bounds away (measured on a B200 at updates 254-258 and 299), outside them but without the POWER headroom; the
    margins are reported.  A wrong slot of the scalar ring fails the exact check 1 (Adam scalars) and the actor_ent check (stddev)."""
    run_chain(monkeypatch, capsys, "bf16-300", "bf16", 6, 50, 64, 8, 300, sched="linear(1.0,0.1,600)",
              stage_at={0, 1, 254, 255, 256, 257, 258, 299}, power_at={0, 1})
