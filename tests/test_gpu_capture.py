"""Training through autograd inside a CUDA graph: DrQV2Agent(capturable=True) and standalone differentiable modules.

drq_adam_scalars_advance against utils.adam_scalars; the reference's update body captured once and replayed, against
the same body run eagerly, bit for bit (parameters, Adam moments, target, step counts, act(), losses); standalone
modules with torch.optim.Adam(capturable=True); a 0-d CUDA tensor as the actor's std; what is refused; and the
device step counts through state_dict(), pickling and the reference-snapshot interop."""
import pickle

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import drq_oracle as O

pytestmark = pytest.mark.gpu

SCHED = "0.2"          # a constant stddev schedule: a captured Python float is a constant of the graph
LR = 1e-4
SENT = 0x7FA5A5A5      # fp32 NaN sentinel bits
KINDS = [("bf16", "bf16"), (True, "bf16"), (True, "fp32")]     # (differentiable, mode)
SHAPES = [(256, 6, 1024), (33, 38, 256)]                       # (B, A, H): the walker shape, and a wide action


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    yield torch.device("cuda")


def _s():
    return torch.cuda.current_stream().cuda_stream


# ----------------------------------------------------------------------------- 1. the scalar kernel
def _advance(counters, lr, dev):
    """one drq_adam_scalars_advance per counter (each its own int64), outputs at a 16-float pitch in a sentinel buffer"""
    from drqv2_b200._lib import call
    n = counters.numel()
    out = torch.full((n, 16), 0, dtype=torch.int32, device=dev).fill_(SENT).view(torch.float32)
    for i in range(n):
        call("drq_adam_scalars_advance", counters.data_ptr() + 8 * i, float(lr), 0.9, 0.999, 1e-8,
             out.data_ptr() + 64 * i, _s())
    return out


def test_adam_scalars_advance_matches_host(dev):
    """every t in 1..4096 and 1000 seeded t up to 10^7, three learning rates: the counter moves by exactly one, nothing
    beyond the 8 outputs is written, and the outputs are utils.adam_scalars bit for bit (both sides compute in fp64
    and round once; on a B200 no t of these differs, although CUDA's fp64 pow and glibc's need not agree in the
    last fp64 place)"""
    from drqv2_b200 import utils
    rng = np.random.default_rng(0)
    ts = np.concatenate([np.arange(1, 4097), rng.integers(4097, 10 ** 7 + 1, 1000)])
    for lr in (1e-4, 3e-4, 1e-3):
        counters = torch.tensor(ts - 1, dtype=torch.int64, device=dev)
        out = _advance(counters, lr, dev)
        assert torch.equal(counters.cpu(), torch.tensor(ts, dtype=torch.int64))
        bits = out.view(torch.int32).cpu()
        assert bool((bits[:, 8:] == SENT).all()), "wrote past the 8 scalars"
        got = bits[:, :8].numpy()
        want = np.stack([utils.adam_scalars(lr, int(t)) for t in ts]).view(np.int32)
        rows, cols = np.nonzero(got != want)
        assert rows.size == 0, [(lr, int(ts[r]), int(c)) for r, c in zip(rows, cols)][:20]
    # two launches on one counter: t and t + 1
    c = torch.tensor([41, 41], dtype=torch.int64, device=dev)
    _advance(c[:1], 3e-4, dev)
    out = _advance(c[:1], 3e-4, dev)
    assert int(c[0]) == 43 and int(c[1]) == 41
    assert np.array_equal(out[0, :8].cpu().numpy().view(np.int32), utils.adam_scalars(3e-4, 43).view(np.int32))


# ----------------------------------------------------------------------------- the reference body
def reference_body(agent, batch, step, std=None):
    """drqv2.py:230-262 with update_critic (177-204) and update_actor (206-228) inlined, the batch already on the
    device.  std None: the reference's utils.schedule(stddev_schedule, step); else a 0-d CUDA tensor the caller
    writes before each replay.  Returns the two losses."""
    from drqv2_b200 import utils
    obs, action, reward, discount, next_obs = batch
    obs = agent.aug(obs.float())
    next_obs = agent.aug(next_obs.float())
    obs = agent.encoder(obs)
    with torch.no_grad():
        next_obs = agent.encoder(next_obs)
    with torch.no_grad():
        stddev = utils.schedule(agent.stddev_schedule, step) if std is None else std
        dist = agent.actor(next_obs, stddev)
        next_action = dist.sample(clip=agent.stddev_clip)
        target_Q1, target_Q2 = agent.critic_target(next_obs, next_action)
        target_V = torch.min(target_Q1, target_Q2)
        target_Q = reward + (discount * target_V)
    Q1, Q2 = agent.critic(obs, action)
    critic_loss = F.mse_loss(Q1, target_Q) + F.mse_loss(Q2, target_Q)
    agent.encoder_opt.zero_grad(set_to_none=True)
    agent.critic_opt.zero_grad(set_to_none=True)
    critic_loss.backward()
    agent.critic_opt.step()
    agent.encoder_opt.step()
    obs = obs.detach()
    dist = agent.actor(obs, stddev)
    action = dist.sample(clip=agent.stddev_clip)
    Q1, Q2 = agent.critic(obs, action)
    actor_loss = -torch.min(Q1, Q2).mean()
    agent.actor_opt.zero_grad(set_to_none=True)
    actor_loss.backward()
    agent.actor_opt.step()
    utils.soft_update_params(agent.critic, agent.critic_target, agent.critic_target_tau)
    return critic_loss.detach(), actor_loss.detach()


def warm_up_and_capture(fn, warmup):
    """the capture recipe of INTEGRATION.md: eager warm-up steps on a side stream, then one captured step"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def _batch(B, A, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    return ((torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g).to(dev),
             (torch.rand(B, A, generator=g) * 2 - 1).to(dev), torch.rand(B, 1, generator=g).to(dev),
             torch.full((B, 1), 0.99 ** 3).to(dev),
             torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g).to(dev)))


def _agent(kind, mode, A, H, capturable=True, pixels="float"):
    from drqv2_b200 import DrQV2Agent
    torch.manual_seed(1)
    return DrQV2Agent((9, 84, 84), (A,), "cuda", LR, 50, H, 0.01, 2000, 2, SCHED, 0.3, False, seed=1, mode=mode,
                      differentiable=kind, pixels=pixels, capturable=capturable)


def _steps(agent):
    return {net: getattr(agent, f"{net}_opt").state_dict()["step"] for net in ("encoder", "critic", "actor")}


def _assert_same_state(x, y, what):
    a, b = x._arena, y._arena
    for name in ("params", "exp_avg", "exp_avg_sq", "target"):
        assert torch.equal(getattr(a, name), getattr(b, name)), (what, name)


def _act(agent, obs):
    """eval-mode actions at batch 1 and at batch 4 (no draw)"""
    return np.concatenate([agent.act(obs[0], 100, True), agent.act(obs, 100, True).ravel()])


# ----------------------------------------------------------------------------- 2, 3, 7. the agent
@pytest.mark.parametrize("B,A,H", SHAPES)
@pytest.mark.parametrize("kind,mode", KINDS)
def test_captured_body_equals_eager(dev, kind, mode, B, A, H):
    """P: 3 eager steps of the reference body, then one captured step replayed 5 times; Q: 8 eager steps.  Bit for
    bit: parameters, Adam moments, target, step counts, act() (which reads the bf16 copies the replays refreshed:
    act() ran before the replays, so nothing on the host re-derives them before the last act()) and the losses of
    the last step.  Every draw comes from torch's generator, whose captured draws continue its eager sequence."""
    batch = _batch(B, A, dev)
    obs = batch[0][:4].cpu().numpy()
    P, Q = _agent(kind, mode, A, H), _agent(kind, mode, A, H)
    torch.manual_seed(2)
    g, (lc, la) = warm_up_and_capture(lambda: reference_body(P, batch, 0), 3)
    assert _steps(P) == dict(encoder=3, critic=3, actor=3)     # the capture ran nothing
    act_p = _act(P, obs)
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    torch.manual_seed(2)
    for i in range(8):
        qc, qa = reference_body(Q, batch, 0)
        if i == 2:
            act_q = _act(Q, obs)
    assert np.array_equal(act_p, act_q)
    _assert_same_state(P, Q, (kind, mode))
    assert _steps(P) == _steps(Q) == dict(encoder=8, critic=8, actor=8)
    assert np.array_equal(_act(P, obs), _act(Q, obs))
    assert torch.equal(lc, qc) and torch.equal(la, qa)
    # 7: the device counts through pickling, export_reference_state() and load_reference_agent()
    R = pickle.loads(pickle.dumps(P))
    assert _steps(R) == dict(encoder=8, critic=8, actor=8) and R.capturable
    _assert_same_state(P, R, "pickle")
    from tests.test_gpu_parity import _reference_standin
    ref = _reference_standin(A, 50, H, LR, O.synthetic_params(9, A, 50, H, seed=3))
    st = P.export_reference_state()
    for net in ("encoder", "actor", "critic"):
        getattr(ref, net).load_state_dict(st[net])
        getattr(ref, f"{net}_opt").load_state_dict(st[f"{net}_opt"])
        assert all(float(s["step"]) == 8 for s in getattr(ref, f"{net}_opt").state.values())
    S = _agent(kind, mode, A, H)
    S.load_reference_agent(ref)
    assert _steps(S) == dict(encoder=8, critic=8, actor=8)
    assert torch.equal(S._arena.exp_avg, P._arena.exp_avg)


@pytest.mark.parametrize("kind,mode", KINDS)
def test_capturable_eager_equals_plain_eager(dev, kind, mode):
    """3 eager steps of the same body: the device-side scalars and, in the tensor-core mode, the one-launch Adam +
    pack of differentiable=True give the host path's bits (parameters, moments, target, act())"""
    B, A, H = 64, 6, 256
    batch = _batch(B, A, dev, seed=1)
    obs = batch[0][:4].cpu().numpy()
    X, Y = _agent(kind, mode, A, H), _agent(kind, mode, A, H, capturable=False)
    for ag in (X, Y):
        torch.manual_seed(3)
        for _ in range(3):
            reference_body(ag, batch, 0)
    torch.cuda.synchronize()
    _assert_same_state(X, Y, (kind, mode))
    assert _steps(X) == _steps(Y) == dict(encoder=3, critic=3, actor=3)
    assert np.array_equal(_act(X, obs), _act(Y, obs))


# ----------------------------------------------------------------------------- 4. standalone modules
def _modules(kind, A, H, dev):
    from types import SimpleNamespace

    from drqv2_b200 import Actor, Critic, Encoder, RandomShiftsAug
    torch.manual_seed(4)
    enc = Encoder((9, 84, 84), differentiable=kind, pixels="float").to(dev)
    actor = Actor(O.REPR_DIM, (A,), 50, H, differentiable=kind).to(dev)
    critic = Critic(O.REPR_DIM, (A,), 50, H, differentiable=kind).to(dev)
    target = Critic(O.REPR_DIM, (A,), 50, H, differentiable=kind).to(dev)
    target.load_state_dict(critic.state_dict())
    target.requires_grad_(False)
    opt = lambda m: torch.optim.Adam(m.parameters(), lr=LR, capturable=True)
    return SimpleNamespace(encoder=enc, actor=actor, critic=critic, critic_target=target, aug=RandomShiftsAug(4),
                           encoder_opt=opt(enc), critic_opt=opt(critic), actor_opt=opt(actor), stddev_schedule=SCHED,
                           stddev_clip=0.3, critic_target_tau=0.01)


def _module_state(m):
    out = []
    for net in ("encoder", "actor", "critic", "critic_target"):
        out += [p.detach() for p in getattr(m, net).parameters()]
    for net in ("encoder", "actor", "critic"):
        for st in getattr(m, f"{net}_opt").state.values():
            out += [st["exp_avg"], st["exp_avg_sq"], st["step"]]
    return out


def _eager_forwards(m, batch):
    """what a training loop runs between updates: eager forwards of every module (no draw)"""
    with torch.no_grad():
        feat = m.encoder(batch[0].float())
        return [feat, m.actor(feat, 0.2).mean, *m.critic(feat, batch[1]), *m.critic_target(feat, batch[1])]


@pytest.mark.parametrize("between", [True, False])
@pytest.mark.parametrize("kind", ["bf16", True])
def test_standalone_modules_captured_equal_eager(dev, kind, between):
    """standalone Encoder / Actor / Critic / target with torch.optim.Adam(capturable=True) and
    utils.soft_update_params.  P: 3 eager steps, eager forwards of every module, one captured step, then 5 replays,
    each followed by eager forwards when `between` (acting between updates), else only the last.  Q: the same with 8
    eager steps.  Bit for bit: every eager forward, the last losses, parameters and Adam state.  For the bf16 copies
    this covers both ways they can go stale: eager forwards between replays reading copies from before the replayed
    optimiser steps (between), and captured forwards reading copies frozen at the eager forward before the capture
    (not between: no later eager forward re-derives them)"""
    B, A, H = 64, 6, 256
    batch = _batch(B, A, dev, seed=2)
    P, Q = _modules(kind, A, H, dev), _modules(kind, A, H, dev)
    torch.manual_seed(5)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            reference_body(P, batch, 0)
    torch.cuda.current_stream().wait_stream(side)
    seen_p = [_eager_forwards(P, batch)]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        lc, la = reference_body(P, batch, 0)
    for i in range(5):
        g.replay()
        if between or i == 4:
            seen_p.append(_eager_forwards(P, batch))
    torch.manual_seed(5)
    seen_q = []
    for i in range(8):
        qc, qa = reference_body(Q, batch, 0)
        if i == 2 or (i > 2 and between) or i == 7:
            seen_q.append(_eager_forwards(Q, batch))
    torch.cuda.synchronize()
    assert len(seen_p) == len(seen_q)
    for i, (fp, fq) in enumerate(zip(seen_p, seen_q)):
        for j, (x, y) in enumerate(zip(fp, fq)):
            assert torch.equal(x, y), (kind, between, "eager forwards, set", i, "output", j)
    for i, (x, y) in enumerate(zip(_module_state(P), _module_state(Q))):
        assert torch.equal(x, y), (kind, i)
    assert torch.equal(lc, qc) and torch.equal(la, qa)


# ----------------------------------------------------------------------------- 5. a tensor std
@pytest.mark.parametrize("kind", [False, True, "bf16"])
def test_tensor_std_rewritten_before_each_replay(dev, kind):
    """Actor.forward(obs, std) with a 0-d CUDA std: a captured forward + sample, std rewritten before each replay,
    gives the eager result at the same Python floats"""
    from drqv2_b200 import Actor
    B, A = 32, 6
    torch.manual_seed(6)
    actor = Actor(O.REPR_DIM, (A,), 50, 256, differentiable=kind).to(dev)
    g0 = torch.Generator().manual_seed(6)
    feat = torch.randn(B, O.REPR_DIM, generator=g0).to(dev)
    noise = torch.randn(B, A, generator=g0).to(dev)
    std = torch.tensor(1.0, device=dev)
    run = lambda s: actor(feat, s).sample(clip=0.3, noise=noise)
    g, out = warm_up_and_capture(lambda: run(std), 1)
    for v in (0.1, 0.37, 1.0, 0.05):
        std.fill_(v)
        g.replay()
        assert torch.equal(out, run(v)), (kind, v)


# ----------------------------------------------------------------------------- 6. what is refused
@pytest.mark.filterwarnings("ignore:The CUDA Graph is empty")      # the refused step captured nothing
@pytest.mark.parametrize("kind", ["bf16", True])
def test_step_under_capture_of_a_plain_agent_raises(dev, kind):
    B, A, H = 16, 6, 256
    batch = _batch(B, A, dev, seed=3)
    ag = _agent(kind, "bf16", A, H, capturable=False)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(ValueError, match="capturable=True"):
        with torch.cuda.graph(g):
            ag.critic_opt.step()
    reference_body(ag, batch, 0)
    assert _steps(ag) == dict(encoder=1, critic=1, actor=1)


@pytest.mark.parametrize("kind", [False, True, "bf16"])
def test_u8_encoder_under_capture(dev, kind):
    """float pixels into a pixels="u8" Encoder under capture raise before any work; uint8 pixels capture"""
    from drqv2_b200 import Encoder
    torch.manual_seed(7)
    enc = Encoder((9, 84, 84), differentiable=kind).to(dev)
    u8 = _batch(8, 6, dev, seed=4)[0]
    with pytest.raises(ValueError, match="pixels='float'"):
        with torch.cuda.graph(torch.cuda.CUDAGraph()):
            enc(u8.float())
    g, out = warm_up_and_capture(lambda: enc(u8), 1)
    g.replay()
    assert torch.equal(out, enc(u8))


def test_capturable_agent_refuses_the_host_scalar_paths(dev):
    ag = _agent("bf16", "bf16", 6, 256)
    B = 8
    batch = _batch(B, 6, dev, seed=5)
    it = iter([tuple(t.cpu() for t in batch)] * 2)
    for call in (lambda: ag.update(it, 0), lambda: ag.update_async(it, 0),
                 lambda: ag.update_critic(torch.zeros(B, O.REPR_DIM, device=dev), batch[1], batch[2], batch[3],
                                          torch.zeros(B, O.REPR_DIM, device=dev), 0),
                 lambda: ag.update_actor(torch.zeros(B, O.REPR_DIM, device=dev), 0)):
        with pytest.raises(ValueError, match="capturable=True"):
            call()
    assert _steps(ag) == dict(encoder=0, critic=0, actor=0)
    assert ag.act(batch[0][0].cpu().numpy(), 0, True).shape == (6,)
