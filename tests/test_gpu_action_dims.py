"""More than 32 action dimensions in the tensor-core mode (DMC dog: 38, CMU humanoid: 56, MyoSuite: 39 / 80): the policy
head's action groups over blockIdx.y and the LayerNorm launch's action tail, each against fp64 / a torch fp32
restatement with stray-store sentinels; then the whole update, the stage API, act and the constructor's limits at those
shapes against the oracle.

Bounds as in tests/test_gpu_head_kernels.py: an fp32 sum of n terms is within 2 * 2^-24 (n + 8) A of its fp64 value, A
the same sum over absolute values; values formed with exactly rounded fp32 steps match a torch fp32 restatement bit for
bit, and every bf16 copy is RN-bf16 of the fp32 value the same launch wrote."""
import ctypes as C
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import drq_oracle as O
from tests import test_gpu_bench_config as bench_cfg
from tests import test_gpu_parity as parity
from tests.helpers import assert_sentinel_outside, bits_equal, episode_arrays, fill_sentinel

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"
SUM_C = 2.0


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


def _s():
    return torch.cuda.current_stream().cuda_stream


def _call(name, *a):
    from drqv2_b200 import _lib
    _lib.call(name, *a)
    torch.cuda.synchronize()


def _check(what, got, want, absref, n):
    """|got - want| <= SUM_C 2^-24 (n + 8) A element-wise (a NaN fails)"""
    got, want = got.double(), want.double()
    bound = SUM_C * 2.0 ** -24 * (n + 8) * absref.double()
    bad = ~((got - want).abs() <= bound)
    if bad.any():
        i = int(bad.reshape(-1).nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements out of bound, first at flat {i}: got "
                             f"{float(got.reshape(-1)[i])!r} want {float(want.reshape(-1)[i])!r}")


def _tb(rows, feats, dev):
    from drqv2_b200._bf16 import TB
    t = TB(rows, feats, dev, batch=2)                   # one spare entry
    fill_sentinel(t.buf)
    return t


def _tb_written(t, row0, rows, col0, cols):
    w = torch.zeros(t.batch, t.rpad, t.units * 8, dtype=torch.bool, device=t.buf.device)
    w[0, row0:row0 + rows, col0:col0 + cols] = True
    nb = t.rpad // t.rblk
    return w.view(t.batch, nb, t.rblk, t.units, 8).permute(0, 1, 3, 2, 4).reshape(-1)


def _f32(x):
    return torch.tensor(x, dtype=torch.float32)


# ---------------------------------------------------------------- policy head: action groups over blockIdx.y
@pytest.mark.parametrize("njobs", [0, 1, 2])
@pytest.mark.parametrize("M", [1, 129, 512, 8192])
@pytest.mark.parametrize("A", [33, 38, 56, 64, 80, 128])
def test_policy_head_action_groups(dev, A, M, njobs):
    from drqv2_b200._bf16 import TB, PolicySample
    H, std, clip = 1024, 0.4, 0.3
    g = torch.Generator(device=dev).manual_seed(A * 100003 + M * 7 + njobs)
    p2 = (torch.rand(M, H, device=dev, generator=g) - 0.3).clamp_min(0)
    w4 = (torch.rand(A, H, device=dev, generator=g) - 0.5) * 0.1
    b4 = (torch.rand(A, device=dev, generator=g) - 0.5) * 0.1
    p2b = TB(M, H, dev)
    p2b.load(p2)
    mu_pre = fill_sentinel(torch.empty(M + 1, A, device=dev))
    stdd = torch.tensor([std], device=dev)
    groups = -(-A // 32)
    nblk = -(-M // 8) * groups
    ticket = torch.zeros(1 + nblk + 4, dtype=torch.int32, device=dev)
    ticket[1 + nblk:] = 0x7FA5A5A5                       # words past the block partials stay untouched
    # one job: all rows; two jobs: as the update issues them, [next rows | obs rows] (overlapping at M = 1); metrics
    # ride on the last job
    n0 = max(1, M // 2)
    ranges = [[], [(0, M)], [(M - max(1, M - n0), max(1, M - n0)), (0, n0)]][njobs]
    jobs, outs = [], []
    for i, (r0, r) in enumerate(ranges):
        metrics = i == len(ranges) - 1
        eps = torch.randn(r, A, device=dev, generator=g) * 1.5
        act = fill_sentinel(torch.empty(r + 1, A + 3, device=dev))       # written at a column offset (ld_a = A + 3)
        mu = fill_sentinel(torch.empty(r * A + 4, device=dev))
        met = fill_sentinel(torch.empty(3, device=dev))
        xb = _tb(r, 16 + A, dev)
        jobs.append(PolicySample(r0, r, eps.data_ptr(), act.data_ptr() + 4 * 3, A + 3, mu.data_ptr(),
                                 met.data_ptr() if metrics else None, xb.ptr(), xb.units, 16, 0))
        outs.append((r0, r, eps, act, mu, met if metrics else None, xb))
    arr = (PolicySample * max(1, len(jobs)))(*jobs)

    def launch():
        _call("drq_policy_head_fwd_bf16", p2b.ptr(), p2b.units, w4.data_ptr(), b4.data_ptr(), mu_pre.data_ptr(), M, H, A,
              arr, len(jobs), stdd.data_ptr(), C.c_float(clip), ticket.data_ptr(), _s())
        assert int(ticket[0]) == 0                        # the ticket resets itself for the next launch
        return [t.clone() for t in [mu_pre] + [x for o in outs for x in (o[3], o[4], o[6].buf)] +
                [o[5] for o in outs if o[5] is not None]]

    first = launch()
    # mu_pre against fp64 on the bf16-rounded operands
    pb, wb = p2.to(torch.bfloat16).double(), w4.to(torch.bfloat16).double()
    want = pb @ wb.T + b4.double()
    absref = pb.abs() @ wb.abs().T + b4.double().abs()
    _check("policy_head mu_pre", mu_pre[:M], want, absref, H)
    wm = torch.zeros(M + 1, A, dtype=torch.bool, device=dev)
    wm[:M] = True
    assert_sentinel_outside(mu_pre, wm, "mu_pre")
    lo = _f32(-1.0) + _f32(1e-6)                          # utils.py:113, as the kernel forms it in fp32
    hi = _f32(1.0) - _f32(1e-6)
    for r0, r, eps, act, mu, met, xb in outs:
        # mu = tanhf(mu_pre) (within tanhf's 2 ulp), then drq_actor_sample's exactly rounded steps on that mu
        got_mu = mu[:r * A].view(r, A).cpu()
        tanh64 = torch.tanh(mu_pre[r0:r0 + r].double()).cpu()
        assert ((got_mu.double() - tanh64).abs() <= 2.0 ** -22 * tanh64.abs().clamp_min(2.0 ** -126)).all(), "mu != tanh(mu_pre)"
        e = torch.minimum(torch.maximum(eps.cpu() * _f32(std), -_f32(clip)), _f32(clip))
        a = torch.minimum(torch.maximum(got_mu + e, lo), hi)
        got_a = act[:r, 3:3 + A].cpu()
        assert torch.equal(got_a, a), f"samples differ from the fp32 restatement at {int((got_a != a).sum())} elements"
        w = torch.zeros(r + 1, A + 3, dtype=torch.bool, device=dev)
        w[:r, 3:3 + A] = True
        assert_sentinel_outside(act, w, "action_out")
        wmu = torch.zeros(r * A + 4, dtype=torch.bool, device=dev)
        wmu[:r * A] = True
        assert_sentinel_outside(mu, wmu, "mu_out")
        assert bits_equal(xb.view(0)[:r, 16:16 + A], act[:r, 3:3 + A].to(torch.bfloat16)), "a_bf16 != RN-bf16(action)"
        assert_sentinel_outside(xb.buf, _tb_written(xb, 0, r, 16, A), "a_bf16")
        if met is not None:
            # log-prob mean: per-thread terms, block trees, the partials of all blocks in order, a last tree
            d = got_a.double() - got_mu.double()
            q = d * d / (2 * std * std)
            lp = (-q - np.log(std) - 0.9189385332046727).sum(1).mean()
            lp_abs = (q + abs(np.log(std)) + 0.9189385332046727).sum(1).mean()    # the kernel subtracts both constants
            _check("policy_head logprob", met[:1].cpu(), lp.view(1), lp_abs.view(1), A + nblk // 256 + 32)
            ent = A * (0.5 + 0.9189385332046727 + np.log(std))
            assert abs(float(met[1]) - ent) <= 1e-6 * abs(ent) + 1e-6
            wmet = torch.zeros(3, dtype=torch.bool, device=dev)
            wmet[:2] = True
            assert_sentinel_outside(met, wmet, "metrics")
    assert (ticket[1 + nblk:] == 0x7FA5A5A5).all(), "scratch written past the block partials"
    # the same launch again is bit-identical: a fixed reduction order
    second = launch()
    for x, y in zip(first, second):
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x.view(torch.int16),
                           y.view(torch.int32) if y.dtype == torch.float32 else y.view(torch.int16))


def test_policy_head_refuses_what_it_cannot_hold(dev):
    from drqv2_b200._bf16 import TB, PolicySample
    from drqv2_b200._lib import DrqError
    H = 256
    p2 = TB(16, H, dev)
    w4 = torch.zeros(129, H, device=dev)
    b4, mu_pre = torch.zeros(129, device=dev), torch.zeros(16, 129, device=dev)
    stdd = torch.tensor([0.4], device=dev)
    with pytest.raises(DrqError, match="A <= 128"):
        _call("drq_policy_head_fwd_bf16", p2.ptr(), p2.units, w4.data_ptr(), b4.data_ptr(), mu_pre.data_ptr(), 16, H, 129,
              None, 0, stdd.data_ptr(), C.c_float(0.3), None, _s())
    # a metrics job whose grid has more blocks than the scratch words hold: ceil(70000 / 8) x 2 > 16384
    eps, act, met = torch.zeros(1, 33, device=dev), torch.zeros(1, 33, device=dev), torch.zeros(2, device=dev)
    jobs = (PolicySample * 1)(PolicySample(0, 1, eps.data_ptr(), act.data_ptr(), 33, None, met.data_ptr(), None, 0, 0, 0))
    ticket = torch.zeros(2, dtype=torch.int32, device=dev)
    with pytest.raises(DrqError, match="block partials"):
        _call("drq_policy_head_fwd_bf16", p2.ptr(), p2.units, w4.data_ptr(), b4.data_ptr(), mu_pre.data_ptr(), 70000, H, 33,
              jobs, 1, stdd.data_ptr(), C.c_float(0.3), ticket.data_ptr(), _s())


# ---------------------------------------------------------------- LayerNorm launch: the action tail of [h | action]
@pytest.mark.parametrize("n_tail", [33, 38, 56, 128])
def test_ln_tanh_action_tail(dev, n_tail):
    from drqv2_b200._bf16 import LnJob
    from drqv2_b200._lib import DrqError
    F, B, S = 50, 129, 4
    g = torch.Generator(device=dev).manual_seed(n_tail)
    part = torch.rand(S, B, F, device=dev, generator=g) - 0.5
    bias, gamma, beta = (torch.rand(F, device=dev, generator=g) - 0.5 for _ in range(3))
    h = fill_sentinel(torch.empty(B + 1, F + n_tail, device=dev))
    tail = torch.randn(B, n_tail + 2, device=dev, generator=g)          # ld_tail = n_tail + 2
    RB = 256
    tb = _tb(2 * RB, F + n_tail, dev)
    row0 = RB                                                           # the second half's row block, as xT's rows
    job = LnJob(part.data_ptr(), F, B * F, S, bias.data_ptr(), gamma.data_ptr(), beta.data_ptr(), h.data_ptr(), F + n_tail,
                None, None, tb.buf.data_ptr(), tb.units, row0, tail.data_ptr(), n_tail + 2, n_tail)
    _call("drq_ln_tanh_fwd_multi", (LnJob * 1)(job), 1, B, F, C.c_float(1e-5), _s())
    v = tb.view(0)
    assert bits_equal(v[row0:row0 + B, F:F + n_tail], tail[:, :n_tail].to(torch.bfloat16)), "TB tail != RN-bf16(tail)"
    assert bits_equal(v[row0:row0 + B, :F], h[:B, :F].to(torch.bfloat16)), "TB copy != RN-bf16(h_out)"
    assert_sentinel_outside(tb.buf, _tb_written(tb, row0, B, 0, F + n_tail), "ln_tanh_fwd TB")
    w = torch.zeros(B + 1, F + n_tail, dtype=torch.bool, device=dev)
    w[:B, :F] = True                                                    # the tail columns of h_out are the caller's
    assert_sentinel_outside(h, w, "h_out")
    # a tail the bf16 row cannot hold is refused
    small = _tb(B, F + 8, dev)
    bad = LnJob(part.data_ptr(), F, B * F, S, bias.data_ptr(), gamma.data_ptr(), beta.data_ptr(), h.data_ptr(), F + n_tail,
                None, None, small.buf.data_ptr(), small.units, 0, tail.data_ptr(), n_tail + 2, n_tail)
    with pytest.raises(DrqError, match="does not fit"):
        _call("drq_ln_tanh_fwd_multi", (LnJob * 1)(bad), 1, B, F, C.c_float(1e-5), _s())


# ---------------------------------------------------------------- whole update, stage API, act, constructor
DOG = dict(B=256, A=38, F=50, H=1024, lr=1e-4)
CMU_HUMANOID = dict(B=256, A=56, F=100, H=1024, lr=8e-5)
# The widest supported action vector at a small size.  64 rows, not 16: at B = 16 the actor's gradients carry the ReLU-flip
# noise of 16 rows (the faithful oracle's own fp32 run is 2.5 % from fp64 on actor.trunk.0.bias, the kernels 4.0 %, just
# past 1.5x), while every gradient of the chain that A shapes (policy.4, the critic's action columns) stays within bounds.
WIDE_SMALL = dict(B=64, A=128, F=50, H=256, lr=1e-4)


@pytest.mark.parametrize("case", [DOG, CMU_HUMANOID, WIDE_SMALL], ids=["dog_A38", "cmu_humanoid_A56", "A128_B64"])
def test_update_bf16_many_actions(dev, case, capsys):
    """lr = 0 eager against the bf16-faithful oracle (metrics, features, every gradient), then three captured-graph
    updates at the real lr - the bench-configuration test at these shapes"""
    bench_cfg.test_update_bf16_at_bench_config(dev, case, capsys)


def test_update_fp32_many_actions(dev):
    """fp32 mode at A = 38: <= 1e-4 relative on the pre-optimiser quantities against the fp64 oracle"""
    parity.test_update_matches_oracle(dev, dict(B=16, A=38, F=50, H=256, lr=1e-4))


def test_stage_api_bf16_many_actions(dev):
    from drqv2_b200 import DrQV2Agent
    torch.set_num_threads(max(8, torch.get_num_threads()))
    A, Fd, H, B, lr, steps = 38, 50, 256, 16, 1e-4, 2
    params = O.synthetic_params(9, A, Fd, H, seed=4)
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, use_cuda_graph=False,
                       seed=5, mode="bf16")
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    agent.refresh()
    o = O.OracleAgent(params, lr, 0.01, SCHED, 0.3, dtype=torch.float64, operands="bf16")
    b = O.synthetic_batch(B, A, seed=30)
    with torch.no_grad():
        feat, feat_next = o.encode(b["obs"], b["shift_obs"]), o.encode(b["next_obs"], b["shift_next"])
    f32 = lambda t: t.float().cuda()
    for s in range(steps):
        g = torch.Generator().manual_seed(100 + s)
        eps_c, eps_a = torch.randn(B, A, generator=g), torch.randn(B, A, generator=g)
        agent.inject_draws(None, None, eps_c, eps_a)
        mc = agent.update_critic(f32(feat), b["action"].cuda(), b["reward"].cuda(), b["discount"].cuda(), f32(feat_next), 2 * s)
        ma = agent.update_actor(f32(feat), 2 * s)
        oc = o.update_critic(feat, b["action"], b["reward"], b["discount"], feat_next, 2 * s, eps_c)
        oa = o.update_actor(feat, 2 * s, eps_a)
        tol = 2e-3 if s == 0 else 2e-2
        for k in oc:
            assert abs(mc[k] - oc[k]) <= tol * abs(oc[k]) + 1e-4, (s, k, mc[k], oc[k])
        for k in ("actor_loss", "actor_logprob", "actor_ent"):
            assert abs(ma[k] - oa[k]) <= max(tol, 5e-3) * abs(oa[k]) + 1e-4, (s, k, ma[k], oa[k])
    torch.cuda.synchronize()
    assert agent._opt_steps == dict(encoder=0, critic=steps, actor=steps)
    for net in ("critic", "actor"):
        for name, p in getattr(agent, net).named_parameters():
            assert (p.detach().cpu().double() - o.p[net][name]).abs().max().item() <= 2.5 * lr * steps, (net, name)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_act_many_actions(dev, mode):
    """act at batch 1024 and batch 1 with 38 actions (the bounds of the quadruped act test)"""
    torch.set_num_threads(max(8, torch.get_num_threads()))
    c = dict(A=38, F=50, H=1024)
    n = 1024
    params = O.synthetic_params(9, c["A"], c["F"], c["H"], seed=8)
    agent = bench_cfg._make_agent(c, 1e-4, params, mode, use_graph=True)
    oracle = O.OracleAgent(params, 1e-4, 0.01, SCHED, 0.3, dtype=torch.float64,
                           operands="bf16" if mode == "bf16" else "exact")
    g = torch.Generator().manual_seed(3)
    obs = torch.randint(0, 256, (n, 9, 84, 84), dtype=torch.uint8, generator=g)
    want = oracle.act(obs, 5000, True).numpy()
    tol = 2e-5 if mode == "fp32" else 2e-3
    for rep in range(2):                              # first call eager + capture, second the replay
        got = agent.act(obs.numpy(), 5000, True)
        assert got.shape == (n, c["A"]) and got.dtype == np.float32
        assert np.abs(got - want).max() < tol, (rep, np.abs(got - want).max())
    a = agent.act(obs.numpy(), 5000, False)
    assert np.abs(a).max() <= 1.0
    assert np.abs((a - want).mean()) < 0.05
    for rep in range(2):
        a1 = agent.act(obs[0].numpy(), 5000, True)
        assert a1.shape == (c["A"],) and np.abs(a1 - want[0]).max() < tol


def test_constructor_refuses_what_bf16_cannot_run(dev):
    from drqv2_b200 import DrQV2Agent
    make = lambda A, F, H: DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, F, H, 0.01, 2000, 2, SCHED, 0.3, True, mode="bf16")
    for A, F, H, what in ((129, 50, 256, "1 <= A <= 128"), (0, 50, 256, "1 <= A <= 128"), (38, 50, 1020, "multiple of 8"),
                          (38, 257, 256, "F <= 256"), (128, 50, 4096, "shared memory")):
        with pytest.raises(ValueError, match=what):
            make(A, F, H)
    agent = make(128, 50, 256)
    assert agent.action_dim == 128
    agent = DrQV2Agent((9, 84, 84), (129,), "cuda", 1e-4, 50, 1020, 0.01, 2000, 2, SCHED, 0.3, True, mode="fp32")
    assert agent.action_dim == 129


def test_dog_shape_acts_and_updates_from_the_ring(dev, tmp_path):
    """the default (bf16, graph-captured, ring-fed) agent at the DMC dog shape: act, then updates straight from a
    make_replay_loader ring"""
    from drqv2_b200 import DrQV2Agent, ReplayBufferStorage, make_replay_loader
    A = 38
    Spec = namedtuple("Spec", "shape dtype name")
    specs = (Spec((9, 84, 84), np.uint8, "observation"), Spec((A,), np.float32, "action"),
             Spec((1,), np.float32, "reward"), Spec((1,), np.float32, "discount"))

    class TS(dict):
        def last(self):
            return self["_last"]

    storage = ReplayBufferStorage(specs, tmp_path / "buffer")
    loader = make_replay_loader(tmp_path / "buffer", 256, 32, 0, False, 3, 0.99)
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, 50, 1024, 0.01, 2000, 2, SCHED, 0.3, True)
    assert agent.mode == "bf16"
    for e, T in enumerate((30, 25, 40)):
        f, a, r, d = episode_arrays(e, T, A)
        for t in range(T + 1):
            obs = np.concatenate([f[k] for k in O.stack_rows(t)], axis=0)
            if t == 0:
                act = agent.act(obs, 5000, False)
                assert act.shape == (A,) and np.abs(act).max() <= 1.0
            storage.add(TS(observation=obs, action=a[t], reward=r[t], discount=d[t], _last=(t == T)))
    it = iter(loader)
    for s in range(4):
        m = agent.update(it, 2 * s)
        assert all(np.isfinite(v) for v in m.values()), m
    torch.cuda.synchronize()
    assert any(isinstance(v, torch.cuda.CUDAGraph) for v in agent._graphs.values())
