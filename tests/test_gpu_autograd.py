"""Autograd through the module API: Encoder / Actor / Critic built with differentiable=True and the optimisers' step().

Per module, the gradients of the library's fp32 kernels against fp64 torch autograd of the oracle's functions, held to
the fp32 mode's bar (DESIGN §2): per-tensor rel-L2 <= max(1e-4, 3x the fp32 oracle's own distance to fp64).  The
feature-gradient kernel bit for bit against a torch restatement, with NaN sentinels around what it writes.  The
reference's own update body (drqv2.py:230-262: aug -> encoder -> update_critic -> update_actor -> soft update) run on a
differentiable agent against the fused update() of an agent with the same seed and draws.  What the flag switches on
and off, and the tensor-core agent's operand copies after an optimiser step."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import drq_oracle as O
from tests.helpers import assert_sentinel_outside, fill_sentinel, rel_l2

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"
HEAD_SHAPES = [(6, 50, 1024), (38, 50, 1024), (21, 100, 1024), (129, 256, 1020)]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    # the fp32 oracle is the yardstick: no TF32 in its convolutions and matrix products
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev


def _oracle_grads(fn, tensors, dtype, grads_out, dev):
    """torch autograd of the oracle function `fn(*tensors)` (a tuple of outputs) in `dtype` on `dev`: the gradients of
    sum(out * grads_out) w.r.t. every tensor (None where an output's upstream gradient is None)"""
    ts = [t.detach().to(dev, dtype).requires_grad_(True) for t in tensors]
    outs = fn(*ts)
    pairs = [(o, g.to(dev, dtype)) for o, g in zip(outs, grads_out) if g is not None]
    return torch.autograd.grad([o for o, _ in pairs], ts, [g for _, g in pairs], allow_unused=True)


def _check(got, names, g32, g64, what, report=None):
    """the fp32 mode's bar, per tensor"""
    for name, a, b, c in zip(names, got, g32, g64):
        if c is None:
            assert a is None, (what, name)
            continue
        err = rel_l2(a.detach().cpu().numpy(), c.cpu().numpy())
        own = rel_l2(b.cpu().numpy(), c.cpu().numpy())
        if report is not None:
            report[name] = (err, own)
        assert err <= max(1e-4, 3 * own), (what, name, err, own)


def _encoder(cin, params, dev, differentiable=True):
    from drqv2_b200 import Encoder
    enc = Encoder((cin, 84, 84), differentiable=differentiable)
    enc.load_state_dict(params["encoder"])
    return enc.to(dev)


def _heads(A, Fd, H, params, dev, differentiable=True):
    from drqv2_b200 import Actor, Critic
    actor = Actor(39200, (A,), Fd, H, differentiable=differentiable)
    critic = Critic(39200, (A,), Fd, H, differentiable=differentiable)
    actor.load_state_dict(params["actor"])
    critic.load_state_dict(params["critic"])
    return actor.to(dev), critic.to(dev)


def _enc_fn(names):
    return lambda obs, *p: (O.encoder_fwd(dict(zip(names, p)), obs),)


def _critic_fn(names):
    return lambda feat, action, *p: O.critic_q(dict(zip(names, p)), feat, action)


def _actor_fn(names):
    return lambda feat, *p: (O.actor_mu(dict(zip(names, p)), feat),)


def _relu_as(x, w, b, on, flips):
    """relu(x @ w.T + b) with the on / off decision of every unit taken from the kernels' forward (`on`, a bool tensor).
    Where it differs from this precision's own decision, the pre-activation must lie within the fp32 sum's rounding of
    zero, |pre| <= 2 * 2^-24 * (K + 8) * (|x| @ |w|.T + |b|): a unit the fp32 forward puts on the other side of zero
    than fp64 does carries its whole gradient on one side only, which no accumulation bound covers."""
    pre = F.linear(x, w, b)
    with torch.no_grad():
        differ = (pre > 0) != on
        bound = 2 * 2.0 ** -24 * (w.shape[1] + 8) * F.linear(x.abs(), w.abs(), b.abs())
        assert bool((pre.abs() <= bound)[differ].all()), "a ReLU decision differs away from zero"
        flips.append(int(differ.sum()))
    return pre * on.to(pre.dtype)


def _critic_fn_as(names, on, flips):
    """O.critic_q (drqv2.py:115-121) with the hidden units' decisions `on` = [(layer 1, layer 2) of Q1, ... of Q2]"""
    def fn(feat, action, *p):
        p = dict(zip(names, p))
        x = torch.cat([O.trunk_fwd(p, feat), action], dim=-1)
        qs = []
        for q, (on1, on2) in zip(("Q1", "Q2"), on):
            y = _relu_as(x, p[f"{q}.0.weight"], p[f"{q}.0.bias"], on1, flips)
            y = _relu_as(y, p[f"{q}.2.weight"], p[f"{q}.2.bias"], on2, flips)
            qs.append(F.linear(y, p[f"{q}.4.weight"], p[f"{q}.4.bias"]))
        return qs[0], qs[1]
    return fn


def _actor_fn_as(names, on, flips):
    """O.actor_mu (drqv2.py:85-89) with the hidden units' decisions `on` = (layer 1, layer 2)"""
    def fn(feat, *p):
        p = dict(zip(names, p))
        y = _relu_as(O.trunk_fwd(p, feat), p["policy.0.weight"], p["policy.0.bias"], on[0], flips)
        y = _relu_as(y, p["policy.2.weight"], p["policy.2.bias"], on[1], flips)
        return (torch.tanh(F.linear(y, p["policy.4.weight"], p["policy.4.bias"])),)
    return fn


# ----------------------------------------------------------------------------- the new kernel
@pytest.mark.parametrize("N", [1, 7, 256])
def test_feature_grad_wide_kernel(dev, N):
    """drq_feature_grad_wide_f32 bit-equal to its torch restatement on [0, 37*41) of every plane, +0 where the feature
    is 0 (also -0) or negative, and the sentinel everywhere else"""
    from drqv2_b200._lib import PLANE, call
    g = torch.Generator().manual_seed(N)
    feat = torch.relu(torch.randn(N, 39200, generator=g))
    feat[:, ::97] = -0.0
    feat[:, 5::89] = -1.0                                       # not a post-ReLU value: the mask is feat > 0
    dfeat = torch.randn(N, 39200, generator=g)
    dfeat[:, 1::3] = -dfeat[:, 1::3].abs()                      # negative gradients where the mask is off give +0
    feat, dfeat = feat.to(dev), dfeat.to(dev)
    dpre = fill_sentinel(torch.empty(N, 32, PLANE, device=dev))
    call("drq_feature_grad_wide_f32", dfeat.data_ptr(), feat.data_ptr(), dpre.data_ptr(), N,
         torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    want = torch.zeros(N, 32, 37, 41, device=dev)
    want[:, :, :35, :35] = torch.where(feat > 0, dfeat, torch.zeros_like(dfeat)).view(N, 32, 35, 35)
    got = dpre[:, :, :37 * 41].contiguous()
    assert torch.equal(got.view(torch.int32), want.view(N, 32, 37 * 41).view(torch.int32))
    written = torch.zeros(N, 32, PLANE, dtype=torch.bool, device=dev)
    written[:, :, :37 * 41] = True
    assert_sentinel_outside(dpre, written, "drq_feature_grad_wide_f32")
    assert int((got.view(torch.int32) == int(np.float32(-0.0).view(np.int32))).sum()) == int(
        ((feat > 0) & (dfeat.view(torch.int32) == int(np.float32(-0.0).view(np.int32)))).sum())


# ----------------------------------------------------------------------------- per-module gradients
@pytest.mark.parametrize("N", [1, 5, 33, 256])
@pytest.mark.parametrize("cin", [3, 9, 16])
def test_encoder_gradients(dev, N, cin):
    params = O.synthetic_params(cin, 6, 50, 64, seed=cin)
    enc = _encoder(cin, params, dev)
    g = torch.Generator().manual_seed(100 * cin + N)
    obs = torch.randint(0, 256, (N, cin, 84, 84), dtype=torch.uint8, generator=g)
    G = torch.randn(N, 39200, generator=g)
    names = list(params["encoder"])
    feat = enc(obs.to(dev))
    got = torch.autograd.grad(feat, list(enc.parameters()), G.to(dev))
    ins = [obs.double()] + [params["encoder"][k] for k in names]
    g64 = _oracle_grads(_enc_fn(names), ins, torch.float64, [G], dev)[1:]
    g32 = _oracle_grads(_enc_fn(names), ins, torch.float32, [G], dev)[1:]
    _check(got, names, g32, g64, f"encoder N={N} cin={cin}")


@pytest.mark.parametrize("B", [1, 33, 256])
@pytest.mark.parametrize("shape", HEAD_SHAPES, ids=[f"A{a}_F{f}_H{h}" for a, f, h in HEAD_SHAPES])
def test_head_gradients(dev, shape, B, capsys):
    """The fp64 reference takes the ReLU decisions of the kernels' forward (read from the saved tensors), so that a
    hidden unit whose pre-activation lies within fp32 rounding of zero - about one in 10^6 - is on for both or off for
    both: at B = 256 a single such unit moves the feature gradient by 2.5e-4 (rel-L2), 400x the fp32 oracle's own
    distance on that case (Q2's layer-1 unit (167, 316) of A = 6: -3.0e-8 in fp64, +8.6e-8 in the kernel).  Any unit
    decided differently must lie within that rounding (_relu_as)."""
    A, Fd, H = shape
    flips = []
    params = O.synthetic_params(9, A, Fd, H, seed=A + B)
    actor, critic = _heads(A, Fd, H, params, dev)
    g = torch.Generator().manual_seed(7 * A + B)
    feat = torch.relu(torch.randn(B, 39200, generator=g))
    action = torch.rand(B, A, generator=g) * 2 - 1
    Gmu, Gq1, Gq2 = torch.randn(B, A, generator=g), torch.randn(B, 1, generator=g), torch.randn(B, 1, generator=g)
    # actor: mu = the returned distribution's mean
    fd = feat.to(dev).requires_grad_(True)
    mu = actor(fd, 0.3).mean
    saved = mu.grad_fn.saved_tensors                      # feat, h, xhat, rstd, p1, p2, ...
    on = (saved[4] > 0, saved[5] > 0)
    names = ["feat"] + list(params["actor"])
    got = torch.autograd.grad(mu, [fd] + list(actor.parameters()), Gmu.to(dev))
    ins = [feat] + list(params["actor"].values())
    _check(got, names, _oracle_grads(_actor_fn(names[1:]), ins, torch.float32, [Gmu], dev),
           _oracle_grads(_actor_fn_as(names[1:], on, flips), ins, torch.float64, [Gmu], dev), f"actor {shape} B={B}")
    # critic: features, action and every parameter
    fd = feat.to(dev).requires_grad_(True)
    ad = action.to(dev).requires_grad_(True)
    q1, q2 = critic(fd, ad)
    saved = q1.grad_fn.saved_tensors                      # feat, x, xhat, rstd, Q1 (h1, h2), Q2 (h1, h2), ...
    on = ((saved[4] > 0, saved[5] > 0), (saved[6] > 0, saved[7] > 0))
    names = ["feat", "action"] + list(params["critic"])
    got = torch.autograd.grad([q1, q2], [fd, ad] + list(critic.parameters()), [Gq1.to(dev), Gq2.to(dev)])
    ins = [feat, action] + list(params["critic"].values())
    _check(got, names, _oracle_grads(_critic_fn(names[2:]), ins, torch.float32, [Gq1, Gq2], dev),
           _oracle_grads(_critic_fn_as(names[2:], on, flips), ins, torch.float64, [Gq1, Gq2], dev),
           f"critic {shape} B={B}")
    with capsys.disabled():
        print(f" [{shape} B={B}: {sum(flips)} hidden unit(s) decided by the kernels' forward]", end="")


def test_critic_q1_gradient_only(dev):
    """a None gradient for Q2 skips its head: its parameters receive no gradient, the rest is Q1's alone"""
    A, Fd, H, B = 6, 50, 256, 33
    params = O.synthetic_params(9, A, Fd, H, seed=3)
    _, critic = _heads(A, Fd, H, params, dev)
    g = torch.Generator().manual_seed(3)
    feat, action = torch.relu(torch.randn(B, 39200, generator=g)), torch.rand(B, A, generator=g) * 2 - 1
    Gq1 = torch.randn(B, 1, generator=g)
    fd, ad = feat.to(dev).requires_grad_(True), action.to(dev).requires_grad_(True)
    q1, _ = critic(fd, ad)
    names = ["feat", "action"] + list(params["critic"])
    got = torch.autograd.grad(q1, [fd, ad] + list(critic.parameters()), Gq1.to(dev), allow_unused=True)
    ins = [feat, action] + list(params["critic"].values())
    fn = _critic_fn(names[2:])
    g64 = _oracle_grads(fn, ins, torch.float64, [Gq1, None], dev)
    assert all(g64[names.index(k)] is None for k in names if k.startswith("Q2."))
    _check(got, names, _oracle_grads(fn, ins, torch.float32, [Gq1, None], dev), g64, "critic, Q1 only")
    # .backward() leaves Q2's .grad untouched
    for p in critic.parameters():
        p.grad = None
    q1, _ = critic(fd, ad)
    (q1 * Gq1.to(dev)).sum().backward()
    for name, p in critic.named_parameters():
        assert (p.grad is None) == name.startswith("Q2."), name


@pytest.mark.parametrize("twice", [False, True], ids=["chained", "features_twice"])
def test_encoder_to_critic_chain(dev, twice):
    """encoder -> critic through autograd; with twice=True the features also feed an extra loss, so the encoder's
    backward starts from the sum of the two consumers' gradients"""
    A, Fd, H, B, cin = 6, 50, 1024, 33, 9
    params = O.synthetic_params(cin, A, Fd, H, seed=11)
    enc = _encoder(cin, params, dev)
    _, critic = _heads(A, Fd, H, params, dev)
    g = torch.Generator().manual_seed(11)
    obs = torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g)
    action = torch.rand(B, A, generator=g) * 2 - 1
    Gq1, Gq2, Gf = torch.randn(B, 1, generator=g), torch.randn(B, 1, generator=g), torch.randn(B, 39200, generator=g)
    feat = enc(obs.to(dev))
    q1, q2 = critic(feat, action.to(dev))
    loss = (q1 * Gq1.to(dev)).sum() + (q2 * Gq2.to(dev)).sum()
    if twice:
        loss = loss + (feat * Gf.to(dev)).sum()
    en, cn = list(params["encoder"]), list(params["critic"])
    got = torch.autograd.grad(loss, list(enc.parameters()) + list(critic.parameters()))

    def fn(obs, action, *p):
        f = O.encoder_fwd(dict(zip(en, p[:8])), obs)
        qa, qb = O.critic_q(dict(zip(cn, p[8:])), f, action)
        return (qa, qb, f) if twice else (qa, qb)

    ins = [obs.double(), action] + list(params["encoder"].values()) + list(params["critic"].values())
    ups = [Gq1, Gq2, Gf] if twice else [Gq1, Gq2]
    g32 = _oracle_grads(fn, ins, torch.float32, ups, dev)[2:]
    g64 = _oracle_grads(fn, ins, torch.float64, ups, dev)[2:]
    _check(got, [f"encoder.{k}" for k in en] + [f"critic.{k}" for k in cn], g32, g64, "encoder -> critic")


# ----------------------------------------------------------------------------- opt-in semantics
def test_flag_off_and_on(dev):
    """without the flag the outputs are plain tensors, bit-equal to the flagged forward's; under no_grad a flagged
    module records and saves nothing; pixels that require grad and double backward are refused"""
    A, Fd, H, B, cin = 6, 50, 256, 5, 9
    params = O.synthetic_params(cin, A, Fd, H, seed=2)
    enc0, enc1 = _encoder(cin, params, dev, False), _encoder(cin, params, dev, True)
    (actor0, critic0), (actor1, critic1) = _heads(A, Fd, H, params, dev, False), _heads(A, Fd, H, params, dev, True)
    g = torch.Generator().manual_seed(2)
    obs = torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev)
    action = (torch.rand(B, A, generator=g) * 2 - 1).to(dev)
    f0, f1 = enc0(obs), enc1(obs)
    assert f0.grad_fn is None and f1.grad_fn is not None
    assert torch.equal(f0, f1)
    mu0, mu1 = actor0(f0, 0.2).mean, actor1(f1, 0.2).mean
    assert mu0.grad_fn is None and mu1.grad_fn is not None and torch.equal(mu0, mu1)
    q0, q1 = critic0(f0, action), critic1(f1, action)
    assert all(q.grad_fn is None for q in q0) and all(q.grad_fn is not None for q in q1)
    assert all(torch.equal(a, b) for a, b in zip(q0, q1))
    # no_grad: nothing recorded, nothing saved
    packed = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: packed.append(t) or t, lambda t: t):
        with torch.no_grad():
            f2 = enc1(obs)
            mu2 = actor1(f2, 0.2).mean
            q2 = critic1(f2, action)
        assert not packed
        assert f2.grad_fn is None and mu2.grad_fn is None and q2[0].grad_fn is None
        assert torch.equal(f2, f0) and torch.equal(mu2, mu0) and torch.equal(q2[0], q0[0])
        critic1(f1, action)                                 # recording: the Function saves its tensors
        assert packed
    with pytest.raises(ValueError):
        enc1(obs.float().requires_grad_(True))
    # double backward
    v = torch.ones_like(q1[0], requires_grad=True)
    gq = torch.autograd.grad(q1[0], [critic1.Q1[0].weight], v, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gq.sum().backward()


def test_agent_flag(dev):
    from drqv2_b200 import DrQV2Agent
    with pytest.raises(ValueError):
        DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, SCHED, 0.3, False, mode="fp32",
                   data_parallel=True, differentiable=True)
    agent = DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, SCHED, 0.3, False, mode="fp32",
                       differentiable=True, use_cuda_graph=False)
    for net in ("encoder", "actor", "critic"):
        assert getattr(agent, net).differentiable
        for p in getattr(agent, net).parameters():
            assert p.requires_grad and p.grad is not None
    assert not agent.critic_target.differentiable
    assert not any(p.requires_grad for p in agent.critic_target.parameters())
    plain = DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, SCHED, 0.3, False, mode="fp32")
    assert not any(p.requires_grad for p in plain.encoder.parameters())
    # an optimiser step leaves the exploration stddev act() last wrote, and counts its own steps
    obs = np.zeros((9, 84, 84), np.uint8)
    agent.act(obs, 50000, False)
    std = float(agent._scal_dev[8])
    agent.critic_opt.step()
    agent.critic_opt.step()
    agent.actor_opt.step()
    torch.cuda.synchronize()
    assert float(agent._scal_dev[8]) == std
    assert agent._opt_steps == dict(encoder=0, critic=2, actor=1)


# ----------------------------------------------------------------------------- the reference's update body
def _aug(agent, x, shift):
    """agent.aug(x) (drqv2.py:241-242) with its torch.randint draw replaced by the injected shift"""
    orig = torch.randint
    torch.randint = lambda lo, hi, size, device=None, dtype=None: shift.view(-1, 1, 1, 2).to(device=device, dtype=dtype)
    try:
        return agent.aug(x)
    finally:
        torch.randint = orig


def _reference_update(agent, b, step, dev):
    """drqv2.py:230-262 transcribed (update + update_critic + update_actor), the noise draws injected through
    TruncatedNormal.sample(noise=...).  Returns the metrics and the critic's gradients of the critic loss (the actor's
    backward adds into them afterwards, as in the reference)."""
    from drqv2_b200 import utils
    metrics = dict()
    obs, action, reward, discount, next_obs = (b[k].to(dev) for k in ("obs", "action", "reward", "discount", "next_obs"))
    obs = _aug(agent, obs.float(), b["shift_obs"])
    next_obs = _aug(agent, next_obs.float(), b["shift_next"])
    obs = agent.encoder(obs)
    with torch.no_grad():
        next_obs = agent.encoder(next_obs)
    metrics["batch_reward"] = reward.mean().item()
    # update_critic
    with torch.no_grad():
        stddev = utils.schedule(agent.stddev_schedule, step)
        dist = agent.actor(next_obs, stddev)
        next_action = dist.sample(clip=agent.stddev_clip, noise=b["eps_critic"].to(dev))
        target_Q1, target_Q2 = agent.critic_target(next_obs, next_action)
        target_V = torch.min(target_Q1, target_Q2)
        target_Q = reward + (discount * target_V)
    Q1, Q2 = agent.critic(obs, action)
    critic_loss = F.mse_loss(Q1, target_Q) + F.mse_loss(Q2, target_Q)
    metrics.update(critic_target_q=target_Q.mean().item(), critic_q1=Q1.mean().item(), critic_q2=Q2.mean().item(),
                   critic_loss=critic_loss.item())
    agent.encoder_opt.zero_grad(set_to_none=True)
    agent.critic_opt.zero_grad(set_to_none=True)
    critic_loss.backward()
    agent.critic_opt.step()
    agent.encoder_opt.step()
    critic_grads = {k: p.grad.clone() for k, p in agent.critic.named_parameters()}
    # update_actor
    obs = obs.detach()
    dist = agent.actor(obs, stddev)
    action = dist.sample(clip=agent.stddev_clip, noise=b["eps_actor"].to(dev))
    log_prob = dist.log_prob(action).sum(-1, keepdim=True)
    Q1, Q2 = agent.critic(obs, action)
    Q = torch.min(Q1, Q2)
    actor_loss = -Q.mean()
    agent.actor_opt.zero_grad(set_to_none=True)
    actor_loss.backward()
    agent.actor_opt.step()
    metrics.update(actor_loss=actor_loss.item(), actor_logprob=log_prob.mean().item(),
                   actor_ent=dist.entropy().sum(dim=-1).mean().item())
    utils.soft_update_params(agent.critic, agent.critic_target, agent.critic_target_tau)
    return metrics, critic_grads


def _agent(A, Fd, H, lr, params, **kw):
    from drqv2_b200 import DrQV2Agent
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, seed=5, mode="fp32", **kw)
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    return agent


@pytest.mark.parametrize("case", [dict(B=256, A=6, F=50, H=1024), dict(B=33, A=38, F=50, H=1024)],
                         ids=["walker_b256", "a38_b33"])
def test_reference_update_body_matches_fused_update(dev, case, capsys):
    torch.set_num_threads(max(8, torch.get_num_threads()))
    B, A, Fd, H, lr = case["B"], case["A"], case["F"], case["H"], 1e-4
    params = O.synthetic_params(9, A, Fd, H, seed=21)
    X = _agent(A, Fd, H, lr, params, use_cuda_graph=False)
    Y = _agent(A, Fd, H, lr, params, differentiable=True)
    # the bar's yardstick: the fp32 oracle's own distance to fp64 on the first update's gradients
    b0 = O.synthetic_batch(B, A, seed=30)
    args = (b0["obs"], b0["action"], b0["reward"], b0["discount"], b0["next_obs"], 0, b0["shift_obs"], b0["shift_next"],
            b0["eps_critic"], b0["eps_actor"])
    o32, o64 = (O.OracleAgent(params, lr, 0.01, SCHED, 0.3, dtype=dt) for dt in (torch.float32, torch.float64))
    o32.update(*args)
    o64.update(*args)
    own = {(net, k): rel_l2(o32.grads[net][k].numpy(), o64.grads[net][k].numpy())
           for net in ("encoder", "critic", "actor") for k in o64.grads[net]}
    worst = dict(metric=0.0, grad=0.0, param_over_lr=0.0)
    bit_equal = dict(grad=0, grad_total=0, param=0, param_total=0)
    for s in range(3):
        b = O.synthetic_batch(B, A, seed=30 + s)
        step = 2 * s
        X.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
        mx = X.update(iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])]), step)
        my, cg = _reference_update(Y, b, step, dev)
        torch.cuda.synchronize()
        for k, v in mx.items():
            d = abs(my[k] - v)
            worst["metric"] = max(worst["metric"], d / max(abs(v), 1e-12))
            assert d <= 1e-4 * abs(v) + 1e-6, (s, k, my[k], v)
        for net in ("encoder", "critic", "actor"):
            for k, p in getattr(X, net).named_parameters():
                gy = cg[k] if net == "critic" else getattr(Y, net).get_parameter(k).grad
                err = rel_l2(gy.cpu().numpy(), p.grad.cpu().numpy())
                worst["grad"] = max(worst["grad"], err)
                bit_equal["grad"] += int(torch.equal(gy, p.grad))
                bit_equal["grad_total"] += 1
                assert err <= max(1e-4, 3 * own[(net, k)]), (s, net, k, err, own[(net, k)])
        for net in ("encoder", "critic", "actor", "critic_target"):
            for k, p in getattr(X, net).named_parameters():
                q = getattr(Y, net).get_parameter(k)
                d = (q.detach() - p.detach()).abs().max().item()
                worst["param_over_lr"] = max(worst["param_over_lr"], d / lr)
                bit_equal["param"] += int(torch.equal(q, p))
                bit_equal["param_total"] += 1
                assert d <= 2.5 * lr * (s + 1), (s, net, k, d)
    assert X._opt_steps == Y._opt_steps == dict(encoder=3, critic=3, actor=3)
    with capsys.disabled():
        print(f"\nreference body through autograd vs update(), {case}: worst metric rel {worst['metric']:.2e}, "
              f"worst gradient rel-L2 {worst['grad']:.2e} ({bit_equal['grad']}/{bit_equal['grad_total']} bit-equal), "
              f"worst parameter |d| {worst['param_over_lr']:.3f} lr ({bit_equal['param']}/{bit_equal['param_total']} "
              "bit-equal)")


# ----------------------------------------------------------------------------- tensor-core agent
def test_bf16_agent_act_after_module_steps(dev):
    """critic_opt.step() / actor_opt.step() on a bf16 agent mark its operand copies stale: act() afterwards is bit-equal
    to a fresh agent given the same parameters through load_state_dict + refresh()"""
    from drqv2_b200 import DrQV2Agent
    A, Fd, H, B, lr = 6, 50, 1024, 32, 1e-3
    params = O.synthetic_params(9, A, Fd, H, seed=9)

    def make(**kw):
        a = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False, seed=5, mode="bf16", **kw)
        for net in ("encoder", "actor", "critic", "critic_target"):
            getattr(a, net).load_state_dict(params[net])
        return a

    P = make(differentiable=True)
    g = torch.Generator().manual_seed(9)
    obs = torch.randint(0, 256, (1024, 9, 84, 84), dtype=torch.uint8, generator=g)
    before = P.act(obs[:2].numpy(), 0, True)          # warm the act path with the initial operand copies
    b = O.synthetic_batch(B, A, seed=9)
    feat = P.encoder(b["obs"].to(dev))
    q1, q2 = P.critic(feat, b["action"].to(dev))
    P.encoder_opt.zero_grad()
    P.critic_opt.zero_grad()
    ((q1 - 1) ** 2 + (q2 - 1) ** 2).mean().backward()
    P.critic_opt.step()
    P.encoder_opt.step()
    mu = P.actor(feat.detach(), 0.2).mean
    Q1, Q2 = P.critic(feat.detach(), mu)
    P.actor_opt.zero_grad()
    (-torch.min(Q1, Q2).mean()).backward()
    P.actor_opt.step()
    Q = make()
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(Q, net).load_state_dict(getattr(P, net).state_dict())
    Q.refresh()
    assert not np.array_equal(P.act(obs[:2].numpy(), 0, True), before)
    for n in (1, 1024):
        x = obs[0].numpy() if n == 1 else obs.numpy()
        assert np.array_equal(P.act(x, 0, True), Q.act(x, 0, True)), n
