"""Autograd on the tensor cores: Encoder / Actor / Critic built with differentiable="bf16" and a DrQV2Agent(mode="bf16",
differentiable="bf16") trained through the reference's own update body.

Bit for bit: the four layout / gradient kernels against torch restatements with NaN sentinels around what they write;
the module forwards against the fused update's feature rows and act(); forwards after every way parameters change
against a module or agent freshly loaded with the same fp32 parameters.  Bounded (DESIGN §2, the bf16 update's bar):
per-module gradients against fp64 torch autograd of the oracle's bf16-faithful functions, per-tensor rel-L2 <=
max(2e-2, 1.5 x that oracle's own fp32-vs-fp64 distance); forwards rel-L2 <= 1e-3 (features), 2e-3 (mu, Q)."""
import pickle

import numpy as np
import pytest
import torch

from oracle import drq_oracle as O
from tests.helpers import assert_sentinel_outside, fill_sentinel, rel_l2

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"
TOL = 2e-2
HEAD_SHAPES = [(6, 50, 1024), (38, 50, 1024), (56, 100, 1024), (128, 256, 1024)]
WORST = {}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    if WORST:
        print("\nlargest ratio to each bound: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(WORST.items())))


def _note(what, ratio):
    WORST[what] = max(WORST.get(what, 0.0), ratio)


def _s():
    return torch.cuda.current_stream().cuda_stream


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


# ----------------------------------------------------------------------------- the four kernels, bit for bit
def _enc_order(ref):
    """[n, 39200] reference order c*1225 + yx -> encoder-output order (c/8)*9800 + yx*8 + c%8"""
    n = ref.shape[0]
    return ref.view(n, 4, 8, 1225).permute(0, 1, 3, 2).reshape(n, 39200)


@pytest.mark.parametrize("N", [1, 7, 129, 256])
def test_features_to_ref_kernel(dev, N):
    from drqv2_b200._bf16 import TB
    from drqv2_b200._lib import call
    g = torch.Generator().manual_seed(N)
    ref = torch.randn(N, 39200, generator=g).to(torch.bfloat16).float().to(dev)    # bf16-representable rows
    # TB source: drq_pack_features_tb's output; kernel 1 composed with it is the identity
    tb = TB(N, 39200, dev)
    call("drq_pack_features_tb", ref.data_ptr(), tb.ptr(), N, _s())
    out = fill_sentinel(torch.empty(N + 1, 39200, device=dev))
    call("drq_features_to_ref", tb.ptr(), 1, out.data_ptr(), N, _s())
    torch.cuda.synchronize()
    assert torch.equal(_bits(out[:N]), _bits(ref))
    written = torch.zeros(N + 1, 39200, dtype=torch.bool, device=dev)
    written[:N] = True
    assert_sentinel_outside(out, written, "drq_features_to_ref (TB)")
    # fp32 source in the encoder-output order: a permutation
    src = torch.randn(N, 39200, generator=g).to(dev)
    out = fill_sentinel(torch.empty(N + 1, 39200, device=dev))
    call("drq_features_to_ref", _enc_order(src).contiguous().data_ptr(), 0, out.data_ptr(), N, _s())
    torch.cuda.synchronize()
    assert torch.equal(_bits(out[:N]), _bits(src))
    assert_sentinel_outside(out, written, "drq_features_to_ref (fp32)")


@pytest.mark.parametrize("N", [1, 7, 129, 256])
def test_feature_grad_wide_bf16_kernel(dev, N):
    from drqv2_b200._lib import GUARD, PLB, WB_SLACK, call, lib
    g = torch.Generator().manual_seed(N)
    feat = torch.relu(torch.randn(N, 39200, generator=g))
    feat[:, ::97] = -0.0
    feat[:, 5::89] = -1.0
    dfeat = torch.randn(N, 39200, generator=g)
    dfeat[:, 1::3] = -dfeat[:, 1::3].abs()
    dfeat[:, 2::101] = -0.0
    feat, dfeat = feat.to(dev), dfeat.to(dev)
    nel = lib().drq_wb_elems(N)
    rows = N * PLB + WB_SLACK
    assert nel == 4 * rows * 8
    out = fill_sentinel(torch.empty(nel + 8, dtype=torch.bfloat16, device=dev))
    call("drq_feature_grad_wide_bf16", dfeat.data_ptr(), feat.data_ptr(), out.data_ptr(), N, _s())
    torch.cuda.synchronize()
    val = torch.where(feat > 0, dfeat, torch.zeros_like(dfeat)).to(torch.bfloat16)       # RN-bf16, +0 off the mask
    want = torch.zeros(4, rows, 8, dtype=torch.bfloat16, device=dev)
    img = torch.zeros(N, 4, 8, 41, 41, dtype=torch.bfloat16, device=dev)
    img[:, :, :, :35, :35] = val.view(N, 4, 8, 35, 35)
    pix = torch.zeros(N, 4, PLB, 8, dtype=torch.bfloat16, device=dev)
    pix[:, :, GUARD:GUARD + 41 * 41] = img.view(N, 4, 8, 41 * 41).permute(0, 1, 3, 2)
    want[:, :N * PLB] = pix.permute(1, 0, 2, 3).reshape(4, N * PLB, 8)
    assert torch.equal(_bits(out[:nel]), _bits(want.view(-1)))
    written = torch.zeros(nel + 8, dtype=torch.bool, device=dev)
    written[:nel] = True
    assert_sentinel_outside(out, written, "drq_feature_grad_wide_bf16")
    neg0 = int(np.float32(-0.0).view(np.int32))
    n_neg = int(((feat > 0) & (_bits(dfeat) == neg0)).sum())
    assert int((_bits(out[:nel]) == -32768).sum()) == n_neg      # -0.0 only where the mask is on and dfeat is -0.0


@pytest.mark.parametrize("B", [1, 7, 129, 256])
def test_q_head_bwd_kernel(dev, B):
    """both gradients: drq_q_head_bwd_loss_bf16's critic-loss outputs when fed the dq its loss mode computes; one
    gradient: the other head's outputs keep their sentinels"""
    from drqv2_b200._bf16 import TB
    from drqv2_b200._lib import call
    H = 1024
    g = torch.Generator().manual_seed(B)
    c2 = TB(B, H, dev, batch=2)
    c2.load(torch.relu(torch.randn(B, H, generator=g)).to(dev), 0)
    c2.load(torch.relu(torch.randn(B, H, generator=g)).to(dev), 1)
    ws = H + 8                                                 # floats between the two heads' w3 / b3
    w3 = torch.randn(2 * ws, generator=g).to(dev)
    q, tq = torch.randn(2, B, generator=g).to(dev), torch.randn(2, B, generator=g).to(dev)
    reward, discount = torch.rand(B, generator=g).to(dev), torch.rand(B, generator=g).to(dev)

    def outs():
        return (fill_sentinel(torch.empty_like(c2.buf)), fill_sentinel(torch.empty(2 * ws + 1, device=dev)),
                fill_sentinel(torch.empty(2 * ws + 1, device=dev)))

    dc_a, dw_a, db_a = outs()
    call("drq_q_head_bwd_loss_bf16", 1, q.data_ptr(), tq.data_ptr(), reward.data_ptr(), discount.data_ptr(), None, None,
         c2.ptr(), c2.units, c2.stride, w3.data_ptr(), dc_a.data_ptr(), dw_a.data_ptr(), db_a.data_ptr(), B, H, ws, _s())
    tq_v = reward + discount * torch.minimum(tq[0], tq[1])
    dq = (2.0 / B) * (q - tq_v)
    dq = [dq[0].contiguous(), dq[1].contiguous()]
    dc_b, dw_b, db_b = outs()
    call("drq_q_head_bwd_bf16", dq[0].data_ptr(), dq[1].data_ptr(), c2.ptr(), c2.units, c2.stride, w3.data_ptr(),
         dc_b.data_ptr(), dw_b.data_ptr(), db_b.data_ptr(), B, H, ws, _s())
    torch.cuda.synchronize()
    for a, b in ((dc_a, dc_b), (dw_a, dw_b), (db_a, db_b)):
        assert torch.equal(_bits(a), _bits(b))
    # the restatement: dc2 = RN-bf16(dq w3 (c2 > 0)) at rows < B, features < H
    dcv = TB(B, H, dev, batch=2)
    dcv.buf = dc_b
    for z in range(2):
        c = c2.dense(z)
        want = torch.where(c > 0, dq[z][:, None] * w3[z * ws:z * ws + H][None, :], torch.zeros_like(c)).to(torch.bfloat16)
        assert torch.equal(_bits(dcv.view(z)[:B, :H]), _bits(want))
    # one gradient: head 2 only
    dc_c, dw_c, db_c = outs()
    call("drq_q_head_bwd_bf16", None, dq[1].data_ptr(), c2.ptr(), c2.units, c2.stride, w3.data_ptr(),
         dc_c.data_ptr(), dw_c.data_ptr(), db_c.data_ptr(), B, H, ws, _s())
    torch.cuda.synchronize()
    head = torch.zeros(2 * c2.stride, dtype=torch.bool, device=dev)
    head[c2.stride:] = True
    assert torch.equal(_bits(dc_c)[head], _bits(dc_b)[head])
    assert_sentinel_outside(dc_c, head, "drq_q_head_bwd_bf16 dc2 (Q2 only)")
    wmask = torch.zeros(2 * ws + 1, dtype=torch.bool, device=dev)
    wmask[ws:ws + H] = True
    assert torch.equal(_bits(dw_c)[wmask], _bits(dw_b)[wmask])
    assert_sentinel_outside(dw_c, wmask, "drq_q_head_bwd_bf16 dw3 (Q2 only)")
    bmask = torch.zeros(2 * ws + 1, dtype=torch.bool, device=dev)
    bmask[ws] = True
    assert torch.equal(_bits(db_c)[bmask], _bits(db_b)[bmask])
    assert_sentinel_outside(db_c, bmask, "drq_q_head_bwd_bf16 db3 (Q2 only)")


@pytest.mark.parametrize("B", [1, 7, 129, 256])
def test_plane_sum_kernel(dev, B):
    from drqv2_b200._lib import call
    Fd, A, P = 50, 38, 16
    g = torch.Generator().manual_seed(B)
    planes = torch.randn(P, B, Fd + A, generator=g).to(dev)
    out = fill_sentinel(torch.empty(B + 1, A, device=dev))
    call("drq_plane_sum_f32", planes.data_ptr() + 4 * Fd, Fd + A, B * (Fd + A), P, out.data_ptr(), A, B, A, _s())
    torch.cuda.synchronize()
    want = torch.zeros(B, A, device=dev)
    for s in range(P):
        want = want + planes[s, :, Fd:]
    assert torch.equal(_bits(out[:B]), _bits(want))
    written = torch.zeros(B + 1, A, dtype=torch.bool, device=dev)
    written[:B] = True
    assert_sentinel_outside(out, written, "drq_plane_sum_f32")


# ----------------------------------------------------------------------------- per-module gradients, bounded
def _grads(fn, tensors, dtype, ups, dev):
    ts = [t.detach().to(dev, dtype).requires_grad_(True) for t in tensors]
    outs = fn(*ts)
    pairs = [(o, g.to(dev, dtype)) for o, g in zip(outs, ups) if g is not None]
    return [o.detach() for o in outs], torch.autograd.grad([o for o, _ in pairs], ts, [g for _, g in pairs],
                                                           allow_unused=True)


def _check(got, names, g32, g64, what):
    for name, a, b, c in zip(names, got, g32, g64):
        if c is None:
            assert a is None, (what, name)
            continue
        err = rel_l2(a.detach().cpu().numpy(), c.cpu().numpy())
        bound = max(TOL, 1.5 * rel_l2(b.cpu().numpy(), c.cpu().numpy()))
        _note(f"grad {what.split()[0]}", err / bound)
        assert err <= bound, (what, name, err, bound)


def _fwd_check(got, want, tol, what):
    err = rel_l2(got.detach().cpu().numpy(), want.cpu().numpy())
    _note(f"forward {what}", err / tol)
    assert err <= tol, (what, err)


@pytest.mark.parametrize("N", [1, 5, 33, 256])
@pytest.mark.parametrize("cin", [3, 9, 10])
def test_encoder_gradients(dev, N, cin):
    from drqv2_b200 import Encoder
    params = O.synthetic_params(cin, 6, 50, 64, seed=cin)
    enc = Encoder((cin, 84, 84), differentiable="bf16")
    enc.load_state_dict(params["encoder"])
    enc = enc.to(dev)
    g = torch.Generator().manual_seed(100 * cin + N)
    obs = torch.randint(0, 256, (N, cin, 84, 84), dtype=torch.uint8, generator=g)
    G = torch.randn(N, 39200, generator=g)
    names = list(params["encoder"])
    feat = enc(obs.to(dev))
    got = torch.autograd.grad(feat, list(enc.parameters()), G.to(dev))
    fn = lambda o, *p: (O.encoder_fwd_bf16(dict(zip(names, p)), o),)
    ins = [obs.double()] + [params["encoder"][k] for k in names]
    (f64,), g64 = _grads(fn, ins, torch.float64, [G], dev)
    _, g32 = _grads(fn, ins, torch.float32, [G], dev)
    _fwd_check(feat, f64, 1e-3, "features")
    _check(got, names, g32[1:], g64[1:], f"encoder N={N} cin={cin}")


@pytest.mark.parametrize("B", [1, 33, 256])
@pytest.mark.parametrize("shape", HEAD_SHAPES, ids=[f"A{a}_F{f}_H{h}" for a, f, h in HEAD_SHAPES])
def test_head_gradients(dev, shape, B):
    from drqv2_b200 import Actor, Critic
    A, Fd, H = shape
    params = O.synthetic_params(9, A, Fd, H, seed=A + B)
    actor, critic = Actor(39200, (A,), Fd, H, differentiable="bf16"), Critic(39200, (A,), Fd, H, differentiable="bf16")
    actor.load_state_dict(params["actor"])
    critic.load_state_dict(params["critic"])
    actor, critic = actor.to(dev), critic.to(dev)
    g = torch.Generator().manual_seed(7 * A + B)
    feat = torch.relu(torch.randn(B, 39200, generator=g)).to(torch.bfloat16).float()   # as the encoder hands them over
    action = torch.rand(B, A, generator=g) * 2 - 1
    Gmu, Gq1, Gq2 = torch.randn(B, A, generator=g), torch.randn(B, 1, generator=g), torch.randn(B, 1, generator=g)
    fd = feat.to(dev).requires_grad_(True)
    mu = actor(fd, 0.3).mean
    names = ["feat"] + list(params["actor"])
    got = torch.autograd.grad(mu, [fd] + list(actor.parameters()), Gmu.to(dev))
    fn = lambda f, *p: (O.actor_mu_bf16(dict(zip(names[1:], p)), f),)
    ins = [feat] + list(params["actor"].values())
    (mu64,), g64 = _grads(fn, ins, torch.float64, [Gmu], dev)
    _fwd_check(mu, mu64, 2e-3, "mu")
    _check(got, names, _grads(fn, ins, torch.float32, [Gmu], dev)[1], g64, f"actor {shape} B={B}")
    fd, ad = feat.to(dev).requires_grad_(True), action.to(dev).requires_grad_(True)
    q1, q2 = critic(fd, ad)
    names = ["feat", "action"] + list(params["critic"])
    got = torch.autograd.grad([q1, q2], [fd, ad] + list(critic.parameters()), [Gq1.to(dev), Gq2.to(dev)])
    fn = lambda f, a, *p: O.critic_q_bf16(dict(zip(names[2:], p)), f, a)
    ins = [feat, action] + list(params["critic"].values())
    (w1, w2), g64 = _grads(fn, ins, torch.float64, [Gq1, Gq2], dev)
    _fwd_check(torch.cat([q1, q2]), torch.cat([w1, w2]), 2e-3, "Q")
    _check(got, names, _grads(fn, ins, torch.float32, [Gq1, Gq2], dev)[1], g64, f"critic {shape} B={B}")


def test_critic_q1_gradient_only_and_extra_feature_loss(dev):
    """a None gradient for Q2 skips its head; encoder -> critic with the features also feeding an extra loss"""
    from drqv2_b200 import Critic, Encoder
    A, Fd, H, B, cin = 6, 50, 1024, 33, 9
    params = O.synthetic_params(cin, A, Fd, H, seed=11)
    enc, critic = Encoder((cin, 84, 84), differentiable="bf16"), Critic(39200, (A,), Fd, H, differentiable="bf16")
    enc.load_state_dict(params["encoder"])
    critic.load_state_dict(params["critic"])
    enc, critic = enc.to(dev), critic.to(dev)
    g = torch.Generator().manual_seed(11)
    obs = torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g)
    action = torch.rand(B, A, generator=g) * 2 - 1
    Gq1, Gf = torch.randn(B, 1, generator=g), torch.randn(B, 39200, generator=g)
    feat = enc(obs.to(dev))
    q1, _ = critic(feat, action.to(dev))
    loss = (q1 * Gq1.to(dev)).sum() + (feat * Gf.to(dev)).sum()
    en, cn = list(params["encoder"]), list(params["critic"])
    got = torch.autograd.grad(loss, list(enc.parameters()) + list(critic.parameters()), allow_unused=True)

    def fn(o, a, *p):
        f = O.encoder_fwd_bf16(dict(zip(en, p[:8])), o)
        return O.critic_q_bf16(dict(zip(cn, p[8:])), f, a)[0], f

    ins = [obs.double(), action] + list(params["encoder"].values()) + list(params["critic"].values())
    _, g32 = _grads(fn, ins, torch.float32, [Gq1, Gf], dev)
    _, g64 = _grads(fn, ins, torch.float64, [Gq1, Gf], dev)
    assert all(g64[2 + 8 + cn.index(k)] is None for k in cn if k.startswith("Q2."))
    _check(got, [f"encoder.{k}" for k in en] + [f"critic.{k}" for k in cn], g32[2:], g64[2:], "chain encoder->critic")


def test_semantics(dev):
    """no_grad: tensor cores, nothing saved; double backward and pixels requiring grad raise"""
    from drqv2_b200 import Actor, Critic, Encoder
    A, Fd, H, B, cin = 6, 50, 256, 5, 9
    params = O.synthetic_params(cin, A, Fd, H, seed=2)
    enc, actor, critic = (Encoder((cin, 84, 84), differentiable="bf16"), Actor(39200, (A,), Fd, H, differentiable="bf16"),
                          Critic(39200, (A,), Fd, H, differentiable="bf16"))
    for m, k in ((enc, "encoder"), (actor, "actor"), (critic, "critic")):
        m.load_state_dict(params[k])
        m.to(dev)
    g = torch.Generator().manual_seed(2)
    obs = torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev)
    action = (torch.rand(B, A, generator=g) * 2 - 1).to(dev)
    f1 = enc(obs)
    mu1, q1 = actor(f1, 0.2).mean, critic(f1, action)
    packed = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: packed.append(t) or t, lambda t: t):
        with torch.no_grad():
            f2 = enc(obs)
            mu2 = actor(f2, 0.2).mean
            q2 = critic(f2, action)
        assert not packed
        assert f2.grad_fn is None and mu2.grad_fn is None and q2[0].grad_fn is None
        assert torch.equal(f2, f1) and torch.equal(mu2, mu1) and torch.equal(q2[0], q1[0]) and torch.equal(q2[1], q1[1])
        critic(f1, action)
        assert packed
    with pytest.raises(ValueError):
        enc(obs.float().requires_grad_(True))
    v = torch.ones_like(q1[0], requires_grad=True)
    gq = torch.autograd.grad(q1[0], [critic.Q1[0].weight], v, create_graph=True)[0]
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gq.sum().backward()
    # standalone copies follow the parameters: an in-place edit (version counter), and refresh() after a .data write
    with torch.no_grad():
        critic.Q1[0].weight.mul_(0.5)
    fresh = Critic(39200, (A,), Fd, H, differentiable="bf16").to(dev)
    fresh.load_state_dict(critic.state_dict())
    with torch.no_grad():
        assert all(torch.equal(a, b) for a, b in zip(critic(f1, action), fresh(f1, action)))
        critic.Q2[2].weight.data.mul_(0.5)
        critic.refresh()
        fresh.load_state_dict(critic.state_dict())
        assert all(torch.equal(a, b) for a, b in zip(critic(f1, action), fresh(f1, action)))


# ----------------------------------------------------------------------------- the agent
def _make(A, Fd, H, params, **kw):
    from drqv2_b200 import DrQV2Agent
    a = DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-3, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, seed=5, mode="bf16", **kw)
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(a, net).load_state_dict(params[net])
    return a


def _same_forwards(P, Q, obs, action, what):
    with torch.no_grad():
        fp, fq = P.encoder(obs), Q.encoder(obs)
        assert torch.equal(fp, fq), what
        assert torch.equal(P.actor(fp, 0.2).mean, Q.actor(fq, 0.2).mean), what
        for net in ("critic", "critic_target"):
            assert all(torch.equal(a, b) for a, b in zip(getattr(P, net)(fp, action), getattr(Q, net)(fq, action))), (what, net)


def test_agent_forwards_match_fused_paths_and_stay_current(dev):
    from drqv2_b200 import utils
    from tests.test_gpu_bench_config import _tb_features_nchw
    A, Fd, H, B = 6, 50, 1024, 256
    params = O.synthetic_params(9, A, Fd, H, seed=9)
    P = _make(A, Fd, H, params, differentiable="bf16", use_cuda_graph=True)
    assert P.differentiable == "bf16" and P.critic_target.differentiable == "bf16"
    assert not any(p.requires_grad for p in P.critic_target.parameters())
    b = O.synthetic_batch(B, A, seed=9)
    obs, nobs, action = b["obs"].to(dev), b["next_obs"].to(dev), b["action"].to(dev)
    # the features: the fused update's rows at the same shifts (lr = 0 would not matter: they are read before any step)
    P.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
    feat_before = []
    with torch.no_grad():
        for x, sh in ((obs, b["shift_obs"]), (nobs, b["shift_next"])):
            from tests.test_gpu_autograd import _aug
            feat_before.append(P.encoder(_aug(P, x.float(), sh)))
    P.update(iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])]), 0)
    bw = P.bf16_workspace(B)
    torch.cuda.synchronize()
    assert torch.equal(feat_before[0], _tb_features_nchw(bw.feat, 0, B))
    assert torch.equal(feat_before[1], _tb_features_nchw(bw.feat, bw.RB, B))
    # actor(encoder(obs)).mean == act(eval) at n = 1 and 256
    for n in (1, 256):
        x = obs[:n]
        want = P.act(x.cpu().numpy(), 0, True)
        with torch.no_grad():
            got = P.actor(P.encoder(x), 0.2).mean
        assert np.array_equal(got.cpu().numpy(), want.reshape(n, A)), n

    def check(what):
        Q = _make(A, Fd, H, {net: getattr(P, net).state_dict() for net in ("encoder", "actor", "critic", "critic_target")},
                  differentiable="bf16")
        _same_forwards(P, Q, obs[:33], action[:33], what)
        if what != "load_state_dict":
            x = obs[:4].cpu().numpy()
            Q.refresh()
            assert np.array_equal(P.act(x, 0, True), Q.act(x, 0, True)), what

    check("update()")
    # module steps through autograd
    feat = P.encoder(obs[:33])
    q1, q2 = P.critic(feat, action[:33])
    P.encoder_opt.zero_grad()
    P.critic_opt.zero_grad()
    ((q1 - 1) ** 2 + (q2 - 1) ** 2).mean().backward()
    P.critic_opt.step()
    check("critic_opt.step()")
    P.encoder_opt.step()
    check("encoder_opt.step()")
    mu = P.actor(feat.detach(), 0.2).mean
    Q1, Q2 = P.critic(feat.detach(), mu)
    P.actor_opt.zero_grad()
    (-torch.min(Q1, Q2).mean()).backward()
    P.actor_opt.step()
    check("actor_opt.step()")
    utils.soft_update_params(P.critic, P.critic_target, P.critic_target_tau)
    check("soft_update_params")
    P.critic.load_state_dict(O.synthetic_params(9, A, Fd, H, seed=10)["critic"])
    check("load_state_dict")
    with torch.no_grad():
        P.update_critic(feat.detach(), action[:33], b["reward"][:33].to(dev), b["discount"][:33].to(dev), feat.detach(), 4)
        P.update_actor(feat.detach(), 4)
    check("update_critic / update_actor")
    P = pickle.loads(pickle.dumps(P))
    check("pickle")
    assert P._opt_steps == dict(encoder=2, critic=3, actor=3)


def _reference_update(agent, b, step, dev):
    from tests.test_gpu_autograd import _reference_update as ref
    return ref(agent, b, step, dev)


@pytest.mark.parametrize("case", [dict(B=256, A=6, F=50, H=1024), dict(B=33, A=38, F=50, H=1024)],
                         ids=["walker_b256", "a38_b33"])
def test_reference_update_body(dev, case):
    """three reference updates through autograd on a differentiable="bf16" agent, each against the bf16-faithful
    oracle seeded from the agent's state before it (metrics, critic-loss gradients of encoder and critic) and, for
    the actor stage, at the agent's stepped critic (its metrics and gradients)"""
    B, A, Fd, H, lr = case["B"], case["A"], case["F"], case["H"], 1e-4
    params = O.synthetic_params(9, A, Fd, H, seed=21)
    Y = _make(A, Fd, H, params, differentiable="bf16")
    Y.lr = lr
    for s in range(3):
        b = O.synthetic_batch(B, A, seed=30 + s)
        state = {net: {k: v.detach().cpu().clone() for k, v in getattr(Y, net).state_dict().items()}
                 for net in ("encoder", "actor", "critic", "critic_target")}
        args = (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 2 * s, b["shift_obs"], b["shift_next"],
                b["eps_critic"], b["eps_actor"])
        o64, o32 = (_oracle_at(Y, state, lr, dt) for dt in (torch.float64, torch.float32))
        want = o64.update(*args)
        o32.update(*args)
        enc_g = {}
        my, cg = _reference_update_with_encoder(Y, b, 2 * s, dev, enc_g)
        # the actor stage reads the critic after critic_opt.step() (drqv2.py:201,213): held at the agent's stepped
        # critic, so that an Adam step's sign on a near-zero critic gradient is not charged to the actor stage
        stepped = dict(state, critic={k: v.detach().cpu().clone() for k, v in Y.critic.state_dict().items()})
        for o in (o64, o32):
            oa = _oracle_at(Y, stepped, lr, o.dtype)
            oa.stage = {}
            m = oa.update_actor(oa.encode(b["obs"], b["shift_obs"]), 2 * s, b["eps_actor"])
            o.grads["actor"] = oa.grads["actor"]
            if o is o64:
                want.update(m)
        for k, v in want.items():
            _note("metric", abs(my[k] - v) / (2e-3 * abs(v) + 1e-4))
            assert abs(my[k] - v) <= 2e-3 * abs(v) + 1e-4, (s, k, my[k], v)
        for net, got in (("encoder", enc_g), ("critic", cg),
                         ("actor", {k: p.grad for k, p in Y.actor.named_parameters()})):
            for k in o64.grads[net]:
                err = rel_l2(got[k].cpu().numpy(), o64.grads[net][k].numpy())
                bound = max(TOL, 1.5 * rel_l2(o32.grads[net][k].numpy(), o64.grads[net][k].numpy()))
                _note("grad reference body", err / bound)
                assert err <= bound, (s, net, k, err, bound)
    assert Y._opt_steps == dict(encoder=3, critic=3, actor=3)


def _oracle_at(agent, state, lr, dtype):
    """the bf16-faithful oracle at the agent's parameters and Adam state (moments and step counts), so that its
    critic_opt.step() lands where the agent's does before the actor stage reads the critic (drqv2.py:201,213)"""
    from collections import OrderedDict
    o = O.OracleAgent(state, lr, 0.01, SCHED, 0.3, dtype=dtype, operands="bf16")
    a = agent._arena
    for net in ("encoder", "critic", "actor"):
        offs = a.offsets[net]
        for buf, dst in ((a.exp_avg, o.m), (a.exp_avg_sq, o.v)):
            dst[net] = OrderedDict((k, buf[offs[k]:offs[k] + p.numel()].view(p.shape).detach().cpu().to(dtype).clone())
                                   for k, p in getattr(agent, net).named_parameters())
    o.t = dict(agent._opt_steps)
    return o


def _reference_update_with_encoder(agent, b, step, dev, enc_g):
    """_reference_update of test_gpu_autograd.py, also keeping the encoder's gradients of the critic loss (read before
    encoder_opt.step(): the arena's gradient buffer is what the step consumes, and the actor backward leaves it alone)"""
    orig = agent.encoder_opt.step

    def step_and_keep(closure=None):
        enc_g.update({k: p.grad.clone() for k, p in agent.encoder.named_parameters()})
        return orig(closure)

    agent.encoder_opt.step = step_and_keep
    try:
        return _reference_update(agent, b, step, dev)
    finally:
        del agent.encoder_opt.step
