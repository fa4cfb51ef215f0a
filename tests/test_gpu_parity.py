"""GPU parity tests: every stage of the CUDA path, called through the C ABI
(drqv2_b200._lib / the Python mirror on top of it), against the oracle and against the
golden vectors of the reference.  Run on the B200 box: pytest -m gpu."""
import hashlib
import io
import json

import numpy as np
import pytest
import torch

from oracle import drq_oracle as O
from tests.helpers import aug_input, episode_arrays, rel_l2

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def make_agent(A, Fd, H, lr, params, use_graph=False, use_tb=True, B=None):
    from drqv2_b200 import DrQV2Agent
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, use_tb,
                       use_cuda_graph=use_graph, seed=5, mode="fp32")
    agent.encoder.load_state_dict(params["encoder"])
    agent.actor.load_state_dict(params["actor"])
    agent.critic.load_state_dict(params["critic"])
    agent.critic_target.load_state_dict(params["critic_target"])
    return agent


def run_update(agent, b, step):
    agent.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
    it = iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])])
    return agent.update(it, step)


# ----------------------------------------------------------------------------- replay ring
def _build_ring(g, first, dev):
    A = g["A"]
    rows = [T + 1 for T in g["lens"]]
    cap = sum(rows)
    ring_f = np.zeros((cap, 3, 84, 84), np.uint8)
    ring_a = np.zeros((cap, A), np.float32)
    ring_r = np.zeros((cap,), np.float32)
    ring_d = np.zeros((cap,), np.float32)
    starts, pos = [], first
    for e, T in enumerate(g["lens"]):
        f, a, r, d = episode_arrays(e, T, A)
        starts.append(pos % cap)
        for t in range(T + 1):
            s = (pos + t) % cap
            ring_f[s], ring_a[s], ring_r[s], ring_d[s] = f[t], a[t], r[t, 0], d[t, 0]
        pos += T + 1
    return cap, starts, (ring_f, ring_a, ring_r, ring_d)


@pytest.mark.parametrize("nstep", [1, 3])
def test_ring_gather_bit_exact_vs_reference_golden(dev, golden_dir, nstep):
    from drqv2_b200 import _lib
    g = json.loads((golden_dir / "replay_golden.json").read_text())
    cap, starts, host = _build_ring(g, first=7, dev=dev)     # last episode wraps around the ring end
    ring = [torch.from_numpy(x).to(dev) for x in host]
    ss = [s for s in g["samples"] if s["nstep"] == nstep]
    B, A = len(ss), g["A"]
    ep_start = torch.tensor([starts[s["episode"]] for s in ss], dtype=torch.int32, device=dev)
    idx = torch.tensor([s["idx"] for s in ss], dtype=torch.int32, device=dev)
    obs = torch.zeros(B, 9, 84, 84, dtype=torch.uint8, device=dev)
    nxt = torch.zeros_like(obs)
    act, rew, disc = torch.zeros(B, A, device=dev), torch.zeros(B, 1, device=dev), torch.zeros(B, 1, device=dev)
    _lib.call("drq_ring_gather_nstep", ring[0].data_ptr(), ring[1].data_ptr(), ring[2].data_ptr(),
              ring[3].data_ptr(), cap, 3, 3, A, ep_start.data_ptr(), idx.data_ptr(), B, nstep, 0.99,
              obs.data_ptr(), nxt.data_ptr(), act.data_ptr(), rew.data_ptr(), disc.data_ptr(), _stream())
    torch.cuda.synchronize()
    obs, nxt, act, rew, disc = (t.cpu().numpy() for t in (obs, nxt, act, rew, disc))
    # vs the reference's own outputs
    for b, s in enumerate(ss):
        assert sha(obs[b]) == s["obs_sha"] and sha(nxt[b]) == s["next_sha"]
        assert np.float32(rew[b, 0]).tobytes().hex() == s["reward_hex"]
        assert np.float32(disc[b, 0]).tobytes().hex() == s["discount_hex"]
        assert np.array_equal(act[b], np.array(s["action"], np.float32))
    # vs the oracle on the same ring
    o = O.ring_gather(*host, ep_start.cpu().numpy(), idx.cpu().numpy(), nstep, 0.99)
    for got, want in zip((obs, act, rew, disc, nxt), o):
        assert np.array_equal(got, want)


def test_ring_sampler_matches_oracle_philox(dev):
    from drqv2_b200 import _lib
    table = np.array([[0, 500], [501, 500], [1002, 37], [1040, 3]], np.int32)
    t = torch.from_numpy(table).to(dev)
    n = torch.tensor([4], dtype=torch.int32, device=dev)
    B = 4096
    for counter, nstep in ((0, 3), (11, 1)):
        c = torch.tensor([counter], dtype=torch.int64, device=dev)
        es = torch.zeros(B, dtype=torch.int32, device=dev)
        ix = torch.zeros(B, dtype=torch.int32, device=dev)
        _lib.call("drq_ring_sample", t.data_ptr(), n.data_ptr(), nstep, 1234567, c.data_ptr(), es.data_ptr(),
                  ix.data_ptr(), B, _stream())
        torch.cuda.synchronize()
        want_s, want_i = O.sample_indices(table, nstep, 1234567, counter, B)
        assert np.array_equal(es.cpu().numpy(), want_s) and np.array_equal(ix.cpu().numpy(), want_i)
        # range property: 1 <= idx <= len - nstep + 1 (replay_buffer.py:150)
        lens = {int(s): int(l) for s, l in table}
        for s_, i_ in zip(want_s, want_i):
            assert 1 <= i_ <= lens[int(s_)] - nstep + 1


def test_update_draws_match_oracle_philox(dev):
    from drqv2_b200 import _lib
    B, A = 300, 6
    c = torch.tensor([9], dtype=torch.int64, device=dev)
    so = torch.zeros(B, 2, dtype=torch.int32, device=dev)
    sn = torch.zeros_like(so)
    ec, ea = torch.zeros(B, A, device=dev), torch.zeros(B, A, device=dev)
    _lib.call("drq_rng_update_draws", 77, c.data_ptr(), 4, so.data_ptr(), sn.data_ptr(), ec.data_ptr(),
              ea.data_ptr(), B, A, _stream())
    torch.cuda.synchronize()
    want_o, want_n = O.update_shifts(77, 9, 4, B)
    assert np.array_equal(so.cpu().numpy(), want_o) and np.array_equal(sn.cpu().numpy(), want_n)
    assert so.min() >= 0 and so.max() <= 8
    big = torch.zeros(4096 * 16, device=dev)
    _lib.call("drq_rng_normal_f32", 77, c.data_ptr(), big.data_ptr(), big.numel(), _stream())
    assert abs(big.mean().item()) < 0.02 and abs(big.std().item() - 1) < 0.02
    assert abs(ec.mean().item()) < 0.1 and abs(ec.std().item() - 1) < 0.1 and not torch.equal(ec, ea)


# ----------------------------------------------------------------------------- augmentation
def test_random_shift_all_81_shifts_bit_exact(dev):
    from drqv2_b200 import RandomShiftsAug
    shifts = torch.tensor([[sx, sy] for sx in range(9) for sy in range(9)], dtype=torch.int32)
    x = torch.from_numpy(aug_input(81, 2)).float()
    want = O.random_shift_exact(x, shifts)
    orig = torch.randint
    torch.randint = lambda lo, hi, size, device=None, dtype=None: shifts.view(81, 1, 1, 2).to(device=device, dtype=dtype)
    try:
        got = RandomShiftsAug(4)(x.to(dev))
    finally:
        torch.randint = orig
    assert torch.equal(got.cpu(), want)
    # replicate-pad + crop identity at the image borders
    xp = torch.nn.functional.pad(x, (4,) * 4, "replicate")
    assert torch.equal(got[8].cpu(), xp[8, :, 8:92, 0:84])       # (sx=0, sy=8)


def test_aug_vs_reference_golden(dev, golden_dir):
    """Integer shift vs the reference's float grid_sample output (3.6e-3 on the 0..255 scale)."""
    from drqv2_b200 import RandomShiftsAug
    g = np.load(golden_dir / "aug_golden.npz")
    shifts = torch.from_numpy(g["shifts"])
    x = torch.from_numpy(aug_input(3, 2)).float().to(dev)
    orig = torch.randint
    torch.randint = lambda lo, hi, size, device=None, dtype=None: shifts.view(3, 1, 1, 2).to(device=device, dtype=dtype)
    try:
        got = RandomShiftsAug(4)(x)
    finally:
        torch.randint = orig
    assert (got.cpu() - torch.from_numpy(g["out"])).abs().max().item() < 8e-3


# ----------------------------------------------------------------------------- encoder
def test_fused_conv1_and_encoder_forward(dev):
    """conv1 with fused aug + normalise, then the full encoder, vs the oracle (fp32 and fp64)."""
    from drqv2_b200 import Encoder, _lib
    from drqv2_b200._lib import PLANE
    N = 6
    params = O.synthetic_params(9, 6, 50, 64, seed=1)
    b = O.synthetic_batch(N, 6, seed=3)
    enc = Encoder((9, 84, 84))
    enc.load_state_dict(params["encoder"])
    enc.to(dev)
    obs = b["obs"].to(dev)
    shift = b["shift_obs"].to(dev)
    w, bias = enc.conv_ptrs()
    a1 = torch.zeros(N, 32, PLANE, device=dev)
    _lib.call("drq_conv1_fwd_f32", obs.data_ptr(), shift.data_ptr(), w[0], bias[0], a1.data_ptr(), N, 9, 4, _stream())
    x = O.random_shift_exact(b["obs"].double(), b["shift_obs"]) / 255.0 - 0.5
    p64 = {k: v.double() for k, v in params["encoder"].items()}
    want = torch.relu(torch.nn.functional.conv2d(x, p64["convnet.0.weight"], p64["convnet.0.bias"], stride=2))
    got = a1[:, :, :41 * 41].view(N, 32, 41, 41).cpu().double()
    assert (got - want).abs().max().item() < 2e-5
    # full encoder through the module API (no aug) and with an integer-valued float input
    feat = enc(obs)
    want_f = O.encoder_fwd(p64, b["obs"].double())
    assert rel_l2(feat.cpu().numpy(), want_f.numpy()) < 2e-6
    assert (feat.cpu().double() - want_f).abs().max().item() < 1e-4 * want_f.abs().max().item()
    feat2 = enc(obs.float())
    assert torch.equal(feat, feat2)
    with pytest.raises(ValueError):
        enc(obs.float() + 0.25)


def test_module_forwards_actor_critic(dev):
    from drqv2_b200 import Actor, Critic
    A, Fd, H, B = 6, 50, 128, 33
    params = O.synthetic_params(9, A, Fd, H, seed=2)
    g = torch.Generator().manual_seed(0)
    feat = torch.rand(B, 39200, generator=g)
    action = torch.rand(B, A, generator=g) * 2 - 1
    actor, critic = Actor(39200, (A,), Fd, H), Critic(39200, (A,), Fd, H)
    actor.load_state_dict(params["actor"])
    critic.load_state_dict(params["critic"])
    actor.to(dev)
    critic.to(dev)
    dist = actor(feat.to(dev), 0.3)
    p64 = {n: {k: v.double() for k, v in d.items()} for n, d in params.items()}
    mu = O.actor_mu(p64["actor"], feat.double())
    assert (dist.mean.cpu().double() - mu).abs().max().item() < 1e-5
    assert torch.allclose(dist.stddev.cpu(), torch.full((B, A), 0.3))
    q1, q2 = critic(feat.to(dev), action.to(dev))
    w1, w2 = O.critic_q(p64["critic"], feat.double(), action.double())
    assert (q1.cpu().double() - w1).abs().max().item() < 1e-4 * w1.abs().max().item() + 1e-6
    assert (q2.cpu().double() - w2).abs().max().item() < 1e-4 * w2.abs().max().item() + 1e-6


# ----------------------------------------------------------------------------- optimiser
def test_adam_and_ema_kernels(dev):
    from drqv2_b200 import _lib, utils
    n = 100_003
    g = torch.Generator().manual_seed(0)
    p = torch.randn(n, generator=g)
    m = torch.randn(n, generator=g) * 1e-3
    v = torch.rand(n, generator=g) * 1e-6
    grad = torch.randn(n, generator=g) * 1e-2
    grad[::7] = 0.0
    npad = (n + 3) // 4 * 4
    bufs = []
    for t in (p, grad, m, v):
        z = torch.zeros(npad, device=dev)
        z[:n] = t.to(dev)
        bufs.append(z)
    for step in (1, 2, 500):
        pp, mm, vv = p.clone(), m.clone(), v.clone()
        O.adam_step(pp, grad, mm, vv, 1e-4, step)
        d = [b.clone() for b in bufs]
        sc = torch.from_numpy(utils.adam_scalars(1e-4, step)).to(dev)
        _lib.call("drq_adam_step", d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), npad,
                  sc.data_ptr(), _stream())
        torch.cuda.synchronize()
        # elementwise op: identical up to fma contraction in torch's CPU kernels
        assert torch.allclose(d[2][:n].cpu(), mm, rtol=2e-6, atol=1e-12)
        assert torch.allclose(d[3][:n].cpu(), vv, rtol=2e-6, atol=1e-15)
        assert torch.allclose(d[0][:n].cpu(), pp, rtol=3e-7, atol=1e-9)      # <= 1-2 ulp of the parameter
    tp = torch.randn(n, generator=g)
    want = tp.clone()
    O.soft_update(p, want, 0.01)
    dp, dt = bufs[0].clone(), torch.zeros(npad, device=dev)
    dt[:n] = tp.to(dev)
    _lib.call("drq_soft_update", dp.data_ptr(), dt.data_ptr(), npad, 0.01, 1 - 0.01, _stream())
    assert torch.equal(dt[:n].cpu(), want)      # two rounded multiplies and an add: bit-exact


# ----------------------------------------------------------------------------- one full update
def _grad_tol(net, name):
    # SURVEY §8c: fp32 evaluations of the reference itself differ by 2e-4..2.5e-3 on encoder
    # gradients; the CUDA path is held to the same kind of bound against the fp64 oracle.
    return 3e-3 if net == "encoder" else 1e-3


def _check_update_against_oracle(agent, oracle32, oracle64, b, step, lr, m_gpu, m32, m64):
    for k in ("batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss"):
        assert m_gpu[k] == pytest.approx(m64[k], rel=1e-4, abs=1e-6), k      # pre-Adam: <= 1e-4 relative
    assert m_gpu["actor_ent"] == pytest.approx(m64["actor_ent"], rel=1e-5)
    # after the first Adam step everything inherits the sign-like noise floor (SURVEY §8c):
    # compare with the fp32 oracle's own distance to fp64 as the yardstick
    for k in ("actor_loss", "actor_logprob"):
        floor = abs(m32[k] - m64[k])
        assert abs(m_gpu[k] - m64[k]) <= max(5 * floor, 2e-3 * abs(m64[k]) + 1e-5), k
    for net in ("encoder", "critic", "actor"):
        mod = getattr(agent, net)
        for name, p in mod.named_parameters():
            g = p.grad.cpu().numpy()
            g64 = oracle64.grads[net][name].numpy()
            g32 = oracle32.grads[net][name].numpy()
            err, own = rel_l2(g, g64), rel_l2(g32, g64)
            if net == "actor":
                assert err <= max(3 * own, 2e-3), (net, name, err, own)     # downstream of Adam
            else:
                assert err <= max(_grad_tol(net, name), 3 * own), (net, name, err, own)
    for net in ("encoder", "critic", "actor", "critic_target"):
        mod = getattr(agent, net)
        for name, p in mod.named_parameters():
            got, want = p.detach().cpu().double(), oracle64.p[net][name]
            assert (got - want).abs().max().item() <= 2.5 * lr * (step // 2 + 1), (net, name)
            if got.numel() > 64 and want.norm() > 0:
                # the sign-like first Adam steps move entries with |g| ~ 0 by up to 2 lr either way (SURVEY §8c): on
                # tensors of small entries (the 39200-wide trunk rows at lr / |w| ~ 2 %) the fp32 oracle's own distance
                # to fp64 is the yardstick
                own = rel_l2(oracle32.p[net][name].numpy(), want.numpy())
                # ... or, where the oracle's two precisions happen to agree, an rms parameter error of 5 % of lr
                # (0.06 % of the entries on the other side of a sign-like step): measured 2.4 % of lr on the
                # actor's 39200-wide trunk rows at B=256, whose gradients pass through the stepped critic
                floor = 0.05 * lr * (got.numel() ** 0.5) / float(want.norm())
                assert rel_l2(got.numpy(), want.numpy()) < max(2e-4, 3 * own, floor), (net, name, own, floor)


@pytest.mark.parametrize("case", [dict(B=16, A=6, F=50, H=256, lr=1e-4), dict(B=5, A=21, F=100, H=128, lr=8e-5)])
def test_update_matches_oracle(dev, case):
    torch.set_num_threads(8)
    A, Fd, H, B, lr = case["A"], case["F"], case["H"], case["B"], case["lr"]
    params = O.synthetic_params(9, A, Fd, H, seed=4)
    agent = make_agent(A, Fd, H, lr, params)
    o32 = O.OracleAgent(params, lr, 0.01, SCHED, 0.3, dtype=torch.float32)
    o64 = O.OracleAgent(params, lr, 0.01, SCHED, 0.3, dtype=torch.float64)
    for s in range(2):
        b = O.synthetic_batch(B, A, seed=10 + s)
        m_gpu = run_update(agent, b, 2 * s)
        args = (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 2 * s, b["shift_obs"],
                b["shift_next"], b["eps_critic"], b["eps_actor"])
        m32, m64 = o32.update(*args), o64.update(*args)
        assert set(m_gpu) == set(m64)
        if s == 0:
            # stage-wise, before any optimiser noise: features and Q values
            ws = agent.workspace(B)
            assert rel_l2(ws.feat[:B].cpu().numpy(), o64.stage["feat"].numpy()) < 1e-5
            assert rel_l2(ws.feat[B:].cpu().numpy(), o64.stage["feat_next"].numpy()) < 1e-5
            assert rel_l2(ws.target_q.cpu().numpy(), o64.stage["target_q"].numpy().ravel()) < 1e-4
        _check_update_against_oracle(agent, o32, o64, b, 2 * s, lr, m_gpu, m32, m64)


def test_update_matches_reference_golden(dev, golden_dir):
    """The CUDA path against numbers recorded from the reference itself (REF-X variant:
    reference code with the integer shift)."""
    g = json.loads((golden_dir / "update_golden.json").read_text())[0]
    c = g["case"]
    params = O.synthetic_params(9, c["A"], c["F"], c["H"], seed=c["pseed"])
    agent = make_agent(c["A"], c["F"], c["H"], c["lr"], params)
    for s, rec in enumerate(g["variants"]["refx"]["steps"]):
        b = O.synthetic_batch(c["B"], c["A"], seed=c["bseed"] + s)
        m = run_update(agent, b, 2 * s)
        for k in ("batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss"):
            assert m[k] == pytest.approx(rec["metrics"][k], rel=1e-4, abs=1e-6), k
        if s == 0:
            for k in ("actor_loss", "actor_logprob", "actor_ent"):
                assert m[k] == pytest.approx(rec["metrics"][k], rel=5e-3, abs=1e-5), k
        for net in ("critic", "encoder"):
            for name, p in getattr(agent, net).named_parameters():
                summ = rec["grads"][net][name]
                got = p.grad.detach().cpu().double().flatten()
                if s == 0:
                    assert abs(float(got.norm()) - summ["l2"]) <= 3e-3 * summ["l2"] + 1e-9, (net, name)
        for net in ("encoder", "actor", "critic", "critic_target"):
            for name, p in getattr(agent, net).named_parameters():
                summ = rec["params"][net][name]
                t = p.detach().cpu().double().flatten()
                probe = t[torch.tensor(summ["probe_idx"])].numpy()
                assert np.max(np.abs(probe - np.array(summ["probe"]))) <= 2.5 * c["lr"] * (s + 1), (net, name)
    # act(): eval mean vs the reference
    obs1 = O.synthetic_batch(1, c["A"], seed=99)["obs"][0].numpy()
    a_eval = agent.act(obs1, 5000, True)
    assert a_eval.shape == (c["A"],) and a_eval.dtype == np.float32
    assert np.allclose(a_eval, g["variants"]["refx"]["act_eval"], atol=5e-3)


def test_graph_replay_equals_eager_bitwise(dev):
    A, Fd, H, B = 6, 50, 128, 8
    params = O.synthetic_params(9, A, Fd, H, seed=6)
    eager = make_agent(A, Fd, H, 1e-4, params, use_graph=False, use_tb=False)
    graph = make_agent(A, Fd, H, 1e-4, params, use_graph=True, use_tb=False)
    for s in range(5):
        b = O.synthetic_batch(B, A, seed=50 + s)
        run_update(eager, b, 2 * s)
        run_update(graph, b, 2 * s)
    torch.cuda.synchronize()
    assert any(isinstance(v, torch.cuda.CUDAGraph) for v in graph._graphs.values())
    for net in ("encoder", "actor", "critic", "critic_target"):
        for (n1, p1), (n2, p2) in zip(getattr(eager, net).named_parameters(), getattr(graph, net).named_parameters()):
            assert torch.equal(p1, p2), (net, n1)


def test_update_skip_rule_and_metrics_contract(dev):
    A, Fd, H, B = 6, 50, 64, 4
    params = O.synthetic_params(9, A, Fd, H, seed=7)
    agent = make_agent(A, Fd, H, 1e-4, params, use_tb=True)
    b = O.synthetic_batch(B, A, seed=1)
    consumed = []

    def it():
        while True:
            consumed.append(1)
            yield (b["obs"].numpy(), b["action"].numpy(), b["reward"].numpy(), b["discount"].numpy(), b["next_obs"].numpy())

    ri = it()
    assert agent.update(ri, 1) == {} and not consumed          # drqv2.py:233-234
    m = agent.update(ri, 2)
    assert len(consumed) == 1
    assert set(m) == {"batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss",
                      "actor_loss", "actor_logprob", "actor_ent"}
    assert all(isinstance(v, float) and np.isfinite(v) for v in m.values())
    agent.use_tb = False
    assert agent.update(ri, 4) == {}
    assert len(consumed) == 2
    # eval_mode contract (utils.py:18-30)
    from drqv2_b200 import utils
    assert agent.training
    with utils.eval_mode(agent):
        assert not agent.training
    assert agent.training


def test_prefetch_is_transparent(dev):
    """prefetch=True pulls host batches one update ahead (H2D overlapped with the running update) and
    changes nothing else: same parameters bit for bit after the same batches and draws."""
    A, Fd, H, B = 6, 50, 64, 4
    params = O.synthetic_params(9, A, Fd, H, seed=7)
    batches = [O.synthetic_batch(B, A, seed=20 + i) for i in range(4)]
    agents = []
    for pf in (False, True):
        agent = make_agent(A, Fd, H, 1e-4, params, use_tb=True)
        agent.prefetch = pf
        pulled = []

        def it():
            for b in batches:
                pulled.append(1)
                yield (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])

        ri = it()
        for i, b in enumerate(batches[:3]):
            agent.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
            agent.update(ri, 2 * i)
        assert len(pulled) == (4 if pf else 3)
        agents.append(agent)
    torch.cuda.synchronize()
    for net in ("encoder", "actor", "critic", "critic_target"):
        for (n1, p1), (_, p2) in zip(getattr(agents[0], net).named_parameters(), getattr(agents[1], net).named_parameters()):
            assert torch.equal(p1, p2), (net, n1)


def test_act_modes(dev):
    A, Fd, H = 12, 50, 128
    params = O.synthetic_params(9, A, Fd, H, seed=8)
    agent = make_agent(A, Fd, H, 1e-4, params, use_graph=True)
    o64 = O.OracleAgent(params, 1e-4, 0.01, SCHED, 0.3, dtype=torch.float64)
    obs = O.synthetic_batch(3, A, seed=5)["obs"]
    for i in range(3):
        a = agent.act(obs[i].numpy(), 5000, True)
        want = o64.act(obs[i], 5000, True)[0].numpy()
        assert a.shape == (A,) and a.dtype == np.float32
        assert np.abs(a - want).max() < 2e-5
    # training mode: noise with std schedule(step), clamped to +-(1-1e-6), not clipped to 0.3
    acts = np.stack([agent.act(obs[0].numpy(), 5000, False) for _ in range(64)])
    mean = o64.act(obs[0], 5000, True)[0].numpy()
    assert np.abs(acts).max() <= 1.0 - 1e-6 + 1e-7
    assert np.abs(acts - mean).max() > 0.3 * 0.5                # noise beyond the update-path clip occurs
    assert acts.std(axis=0).mean() > 0.3
    # before num_expl_steps: uniform actions
    u = np.stack([agent.act(obs[0].numpy(), 10, False) for _ in range(64)])
    assert np.abs(u).max() <= 1.0 and u.std() > 0.4
    # vectorised rollout: batch of observations
    ab = agent.act(obs.numpy(), 5000, True)
    assert ab.shape == (3, A)
    assert np.abs(ab[1] - o64.act(obs[1], 5000, True)[0].numpy()).max() < 2e-5


def test_ring_storage_loader_update_end_to_end(dev, tmp_path):
    """reference-shaped driver: ReplayBufferStorage.add(time_step) -> make_replay_loader ->
    agent.update(replay_iter, step), gather checked against the oracle on the same indices."""
    from collections import namedtuple
    from drqv2_b200 import ReplayBufferStorage, make_replay_loader
    Spec = namedtuple("Spec", "shape dtype name")
    A = 6
    specs = (Spec((9, 84, 84), np.uint8, "observation"), Spec((A,), np.float32, "action"),
             Spec((1,), np.float32, "reward"), Spec((1,), np.float32, "discount"))

    class TS(dict):
        def last(self):
            return self["_last"]

    np.random.seed(3)
    storage = ReplayBufferStorage(specs, tmp_path / "buffer")
    loader = make_replay_loader(tmp_path / "buffer", 64, 8, 4, False, 3, 0.99)
    lens = [9, 5, 12, 7, 20, 11]      # ring of 64 slots: early episodes get evicted
    eps = {}
    for e, T in enumerate(lens):
        f, a, r, d = episode_arrays(e, T, A)
        eps[e] = (f, a, r, d)
        for t in range(T + 1):
            rows = O.stack_rows(t)
            obs = np.concatenate([f[k] for k in rows], axis=0)
            storage.add(TS(observation=obs, action=a[t], reward=r[t], discount=d[t], _last=(t == T)))
    assert len(storage) == sum(lens)
    it = iter(loader)
    ring = loader.ring()
    resident = {s: rows for s, rows in ring.episodes}
    assert sum(resident.values()) <= 64 and len(resident) < len(lens)
    obs, action, reward, discount, next_obs = next(it)
    torch.cuda.synchronize()
    assert obs.shape == (8, 9, 84, 84) and obs.dtype == torch.uint8 and reward.shape == (8, 1)
    # oracle on the sampled indices
    hostring = (ring.frames.cpu().numpy(), ring.action.cpu().numpy(), ring.reward.cpu().numpy(), ring.discount.cpu().numpy())
    es, ix = loader._ep_start.cpu().numpy(), loader._idx.cpu().numpy()
    want = O.ring_gather(*hostring, es, ix, 3, 0.99)
    for got, w in zip((obs, action, reward, discount, next_obs), want):
        assert np.array_equal(got.cpu().numpy(), w)
    for s_, i_ in zip(es, ix):
        assert int(s_) in resident and 1 <= i_ <= resident[int(s_)] - 1 - 3 + 1
    # and the agent consumes the ring iterator directly (zero-copy path, graph captured on 3rd call)
    params = O.synthetic_params(9, A, 50, 64, seed=9)
    agent = make_agent(A, 50, 64, 1e-4, params, use_graph=True, use_tb=True)
    for s in range(4):
        m = agent.update(it, 2 * s)
        assert np.isfinite(m["critic_loss"])
    # a frame stack that is not consecutive frames is rejected
    bad = ReplayBufferStorage(specs, tmp_path / "bad")
    f, a, r, d = eps[0]
    with pytest.raises(ValueError):
        for t in range(3):
            obs = np.concatenate([f[t], f[t], f[(t + 1) % 3]], axis=0)
            bad.add(TS(observation=obs, action=a[t], reward=r[t], discount=d[t], _last=(t == 2)))


def test_replay_snapshot_files_and_resume(dev, tmp_path):
    """save_snapshot leaves the reference's episode files behind, and a new storage over the same directory
    (or over a directory the reference itself wrote) rebuilds the same ring (replay_buffer.py:63-78)."""
    import collections
    import pathlib
    from drqv2_b200 import replay_buffer as R
    Spec = collections.namedtuple("Spec", "shape dtype name")
    A = 6
    specs = (Spec((9, 84, 84), np.uint8, "observation"), Spec((A,), np.float32, "action"),
             Spec((1,), np.float32, "reward"), Spec((1,), np.float32, "discount"))

    class TS(dict):
        def last(self):
            return self["_last"]

    ref_ep = R.load_episode(pathlib.Path(__file__).parent / "golden" / "ref_episode_1_5.npz")
    d1 = tmp_path / "buffer"
    st = R.ReplayBufferStorage(specs, d1)
    loader = R.make_replay_loader(d1, 1000, 4, 0, True, 3, 0.99)           # save_snapshot=True
    for rep in range(2):
        rows = ref_ep["observation"].shape[0]
        for t in range(rows):
            st.add(TS(observation=ref_ep["observation"][t], action=ref_ep["action"][t], reward=ref_ep["reward"][t],
                      discount=ref_ep["discount"][t], _last=t == rows - 1))
    files = R.episode_files(d1)
    assert len(files) == 2 and all(f.stem.split("_")[1:] == [str(i), "5"] for i, f in enumerate(files))
    back = R.load_episode(files[0])
    assert all(np.array_equal(back[k], ref_ep[k]) for k in ref_ep)
    ring1 = loader.ring()
    # resume: a fresh registry entry over the same files
    R._RINGS.pop(str(d1))
    st2 = R.ReplayBufferStorage(specs, d1)
    assert len(st2) == 10
    R.make_replay_loader(d1, 1000, 4, 0, False, 3, 0.99)
    assert st2.load_existing() == 2
    ring2 = R._RINGS[str(d1)]["ring"]
    torch.cuda.synchronize()
    assert ring2.episodes == ring1.episodes
    n = 2 * 6
    assert torch.equal(ring2.frames[:n], ring1.frames[:n]) and torch.equal(ring2.action[:n], ring1.action[:n])
    assert torch.equal(ring2.reward[:n], ring1.reward[:n]) and torch.equal(ring2.discount[:n], ring1.discount[:n])


def _reference_standin(A, Fd, H, lr, p, m=None, v=None, step=0):
    """What a reference DrQV2Agent carries from one update to the next (drqv2.py:137-153): the four networks
    (reference-shaped modules, the names / shapes of drqv2.py:55-59,74-81,100-111) holding parameters `p`, and
    the three torch.optim.Adam optimisers holding moments `m`, `v` after `step` steps (none when m is None)."""
    from types import SimpleNamespace

    from drqv2_b200 import Actor, Critic, Encoder
    ref = SimpleNamespace(encoder=Encoder((9, 84, 84)), actor=Actor(O.REPR_DIM, (A,), Fd, H),
                          critic=Critic(O.REPR_DIM, (A,), Fd, H), critic_target=Critic(O.REPR_DIM, (A,), Fd, H))
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(ref, net).load_state_dict(p[net])
    for net in ("encoder", "actor", "critic"):
        opt = torch.optim.Adam(getattr(ref, net).parameters(), lr=lr)
        if m is not None:
            for k, q in getattr(ref, net).named_parameters():
                opt.state[q] = dict(step=torch.tensor(float(step)), exp_avg=m[net][k].clone(),
                                    exp_avg_sq=v[net][k].clone())
        setattr(ref, f"{net}_opt", opt)
    return ref


def test_reference_snapshot_interop(dev, golden_dir):
    """SURVEY §8f-3: a reference agent's state (what train.py:192-204 pickles) moves into this agent and back.
    The reference agent is the unmodified reference after the two updates recorded in update_golden.json
    (case walker_small, B=8, H=1024, its own grid_sample aug): the oracle replays those updates, the rebuilt
    parameters are checked against the reference's recorded ones, and act() from the taken-over state is
    compared with the action the reference itself returned."""
    from drqv2_b200 import DrQV2Agent
    g = json.loads((golden_dir / "update_golden.json").read_text())[0]
    c, rec = g["case"], g["variants"]["ref"]
    A, Fd, H, lr = c["A"], c["F"], c["H"], c["lr"]
    oracle = O.OracleAgent(O.synthetic_params(9, A, Fd, H, seed=c["pseed"]), lr, 0.01, SCHED, 0.3, aug="grid")
    for s in range(c["steps"]):
        b = O.synthetic_batch(c["B"], A, seed=c["bseed"] + s)
        oracle.update(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 2 * s, b["shift_obs"],
                      b["shift_next"], b["eps_critic"], b["eps_actor"])
    for net, ps in rec["steps"][-1]["params"].items():      # the tolerances of tests/test_oracle_golden.py
        for k, summ in ps.items():
            t = oracle.p[net][k].double().flatten()
            assert np.max(np.abs(t[summ["probe_idx"]].numpy() - summ["probe"])) <= 2.5 * lr * c["steps"], (net, k)
            assert abs(float(t.norm()) - summ["l2"]) <= 1e-4 * summ["l2"] + 1e-6, (net, k)
    ragent = _reference_standin(A, Fd, H, lr, oracle.p, oracle.m, oracle.v, c["steps"])
    mine = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False, seed=1, mode="fp32")
    mine.load_reference_agent(ragent)
    assert mine._opt_step == c["steps"]
    for net in ("encoder", "actor", "critic", "critic_target"):
        for (n1, p1), p2 in zip(getattr(mine, net).named_parameters(), getattr(ragent, net).parameters()):
            assert torch.equal(p1.cpu(), p2), (net, n1)
    for net in ("encoder", "actor", "critic"):
        opt = getattr(ragent, f"{net}_opt")
        sd = getattr(mine, f"{net}_opt").state_dict()
        ref_m = torch.cat([opt.state[p]["exp_avg"].reshape(-1) for p in getattr(ragent, net).parameters()])
        assert torch.equal(sd["exp_avg"][:ref_m.numel()].cpu(), ref_m)
    # the deterministic action the reference returned from this state (act_eval: the oracle's own state is within
    # 2e-5 of it, tests/test_oracle_golden.py), and the oracle's action from the very state taken over
    obs1 = O.synthetic_batch(1, A, seed=99)["obs"][0].numpy()
    got = mine.act(obs1, 5000, True)
    assert np.abs(got - oracle.act(obs1, 5000, True)[0].numpy()).max() < 2e-5
    assert np.abs(got - np.array(rec["act_eval"])).max() < 4e-5
    # and back: a fresh reference agent continues from the exported state
    r2 = _reference_standin(A, Fd, H, lr, O.synthetic_params(9, A, Fd, H, seed=1))
    st = mine.export_reference_state()
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(r2, net).load_state_dict(st[net])
    for net in ("encoder", "actor", "critic"):
        getattr(r2, f"{net}_opt").load_state_dict(st[f"{net}_opt"])
        o1, o2 = getattr(ragent, f"{net}_opt"), getattr(r2, f"{net}_opt")
        for p1, p2 in zip(getattr(ragent, net).parameters(), getattr(r2, net).parameters()):
            assert torch.equal(p1, p2)
            assert torch.equal(o1.state[p1]["exp_avg_sq"], o2.state[p2]["exp_avg_sq"])
            assert float(o2.state[p2]["step"]) == c["steps"]
    # and the reference's optimisers train on from it: one more Adam step with the same gradients keeps the two equal
    for net in ("encoder", "actor", "critic"):
        for (k, p1), p2 in zip(getattr(ragent, net).named_parameters(), getattr(r2, net).parameters()):
            p1.grad, p2.grad = oracle.grads[net][k].clone(), oracle.grads[net][k].clone()
        getattr(ragent, f"{net}_opt").step()
        getattr(r2, f"{net}_opt").step()
        for p1, p2 in zip(getattr(ragent, net).parameters(), getattr(r2, net).parameters()):
            assert torch.equal(p1, p2), net


def test_agent_pickle_roundtrip(dev):
    """train.py:192-204 snapshots the whole agent with torch.save / torch.load."""
    A, Fd, H, B = 6, 50, 64, 4
    params = O.synthetic_params(9, A, Fd, H, seed=11)
    agent = make_agent(A, Fd, H, 1e-4, params, use_graph=True, use_tb=True)
    b = O.synthetic_batch(B, A, seed=2)
    for s in range(3):
        run_update(agent, b, 2 * s)
    buf = io.BytesIO()
    torch.save({"agent": agent}, buf)
    buf.seek(0)
    clone = torch.load(buf, weights_only=False)["agent"]
    for net in ("encoder", "actor", "critic", "critic_target"):
        for (n1, p1), (n2, p2) in zip(getattr(agent, net).named_parameters(), getattr(clone, net).named_parameters()):
            assert torch.equal(p1, p2)
    m1 = run_update(agent, b, 6)
    m2 = run_update(clone, b, 6)
    assert m1 == m2
    # state_dict interchange with reference-shaped modules (names/layouts, drqv2.py:55-59,74-81,100-111)
    sd = agent.critic.state_dict()
    assert list(sd) == list(O.param_shapes(9, A, Fd, H)["critic"])


def test_async_updates_read_their_own_scalars(dev):
    """Updates enqueued back to back without a host sync (use_tb=False, the host runs ahead of the device) read
    the Adam bias corrections / stddev of their own step: same parameters, bit for bit, as the synchronous loop."""
    A, Fd, H, B = 6, 50, 64, 4
    params = O.synthetic_params(9, A, Fd, H, seed=11)
    batches = [O.synthetic_batch(B, A, seed=40 + i) for i in range(8)]
    finals = []
    for sync in (True, False):
        agent = make_agent(A, Fd, H, 1e-3, params, use_tb=sync, use_graph=True)
        for i, b in enumerate(batches):
            agent.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
            agent.update(iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])]), 2 * i)
        torch.cuda.synchronize()
        finals.append([p.detach().clone() for net in ("encoder", "actor", "critic", "critic_target")
                       for p in getattr(agent, net).parameters()])
    for p1, p2 in zip(*finals):
        assert torch.equal(p1, p2)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_ensemble_members_equal_solo_agents(dev, mode):
    """AgentEnsemble (BASELINE configs[3]): members updated concurrently on their own streams end up with exactly
    the parameters of the same agents updated one after the other; members differ from each other (own seed)."""
    from drqv2_b200 import DrQV2Agent
    from drqv2_b200.ensemble import AgentEnsemble
    A, Fd, H, B, K = 6, 50, 64, 4, 3
    args = ((9, 84, 84), (A,), "cuda", 1e-3, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True)
    batches = [[O.synthetic_batch(B, A, seed=60 + 10 * k + i) for i in range(4)] for k in range(K)]
    as_iter = lambda b: iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])])
    ens = AgentEnsemble(K, *args, base_seed=3, mode=mode)
    for i in range(4):
        ms = ens.update([as_iter(batches[k][i]) for k in range(K)], 2 * i)
        assert len(ms) == K and all(np.isfinite(m["critic_loss"]) for m in ms)
    ens.synchronize()
    for k in range(K):
        torch.manual_seed(3 + k)
        solo = DrQV2Agent(*args, seed=3 + k, mode=mode)
        for i in range(4):
            solo.update(as_iter(batches[k][i]), 2 * i)
        torch.cuda.synchronize()
        for net in ("encoder", "actor", "critic", "critic_target"):
            for (n1, p1), (_, p2) in zip(getattr(ens[k], net).named_parameters(), getattr(solo, net).named_parameters()):
                assert torch.equal(p1, p2), (k, net, n1)
    w0 = ens[0].critic.Q1[0].weight
    assert not torch.equal(w0, ens[1].critic.Q1[0].weight)
