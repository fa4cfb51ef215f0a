"""Real-valued pixels and gradients w.r.t. them: Encoder(pixels="float") and RandomShiftsAug through autograd.

The new kernels against fp64 on the exact operands they read - drq_conv1_dgrad_{f32,bf16} and
drq_random_shift_bwd_f32 - with sentinels around every output and NaN past every read extent the header leaves
unread, at every image count and channel count, reduced SM budgets for the tensor-core kernel, and two launches bit
for bit.  The float-source conv1 forward and weight gradient: the u8 path's bits on integer-valued pixels, the
existing bounds on non-integral ones.  Modules end to end (RandomShiftsAug -> Encoder -> Critic / Actor) against fp64
autograd of the oracle, and a saliency call that runs no encoder weight-gradient kernel."""
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import drq_oracle as O
from tests.helpers import GUARD, PLB, WB_SLACK, assert_sentinel_outside, check_sum_bound, fill_sentinel, rel_l2

pytestmark = pytest.mark.gpu

NS = [1, 2, 7, 48, 129, 256, 512]
PLANE = 1696
RATIOS = {}          # kernel -> the largest share of c = 2 measured (DESIGN §2)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield torch.device("cuda")
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
    print("pixel-gradient kernels, largest |got - want| / (2 2^-24 (n + 8) A):", RATIOS)


def _s():
    return torch.cuda.current_stream().cuda_stream


def _call(name, *args):
    from drqv2_b200._lib import call
    call(name, *args)


def _dgrad_want(dy, w):
    """fp64 dx (1/255 included) and the same over absolute values, from dY [N, 32, 41, 41] and W [32, cin, 3, 3]"""
    dy, w = dy.double(), w.double()
    want = F.conv_transpose2d(dy, w, stride=2, output_padding=1) / 255
    absref = F.conv_transpose2d(dy.abs(), w.abs(), stride=2, output_padding=1) / 255
    return want, absref


def _padded_out(n, dev):
    """an fp32 output of n elements inside a sentinel-filled buffer; (buffer, view, written mask)"""
    buf = fill_sentinel(torch.empty(n + 128, device=dev))
    written = torch.zeros(n + 128, dtype=torch.bool, device=dev)
    written[64:64 + n] = True
    return buf, buf[64:64 + n], written


# ----------------------------------------------------------------------------- kernels against fp64
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("cin", [1, 3, 9, 10, 16])
def test_conv1_dgrad_f32_kernel(dev, N, cin):
    g = torch.Generator().manual_seed(1000 * cin + N)
    dy = torch.randn(N, 32, 41, 41, generator=g).to(dev)
    w = (0.1 * torch.randn(32, cin, 3, 3, generator=g)).to(dev)
    planes = torch.full((N, 32, PLANE), float("nan"), device=dev)      # the slack [1681, 1696) is not read
    planes[..., :1681] = dy.reshape(N, 32, 1681)
    buf, dx, written = _padded_out(N * cin * 84 * 84, dev)
    _call("drq_conv1_dgrad_f32", planes.data_ptr(), w.data_ptr(), dx.data_ptr(), N, cin, _s())
    assert_sentinel_outside(buf, written, "drq_conv1_dgrad_f32")
    want, absref = _dgrad_want(dy, w)
    check_sum_bound("drq_conv1_dgrad_f32", dx.view(N, cin, 84, 84), want, absref, 128, RATIOS)
    again = torch.empty_like(dx)
    _call("drq_conv1_dgrad_f32", planes.data_ptr(), w.data_ptr(), again.data_ptr(), N, cin, _s())
    assert torch.equal(again.view(torch.int32), dx.view(torch.int32))


def _bf16_dgrad_inputs(N, cin, dev, seed):
    from drqv2_b200 import _lib
    g = torch.Generator().manual_seed(seed)
    dy = torch.randn(N, 32, 41, 41, generator=g).to(dev).bfloat16().float()
    w = (0.1 * torch.randn(32, cin, 3, 3, generator=g)).to(dev)
    b = torch.randn(32, generator=g).to(dev)
    # WB buffer [4][N*PLB + SLACK][8]: positions [0, 1681) of every image hold dY, every other row NaN
    wb = torch.full((4, N * PLB + WB_SLACK, 8), float("nan"), dtype=torch.bfloat16, device=dev)
    rows = wb[:, :N * PLB].view(4, N, PLB, 8)
    rows[:, :, GUARD:GUARD + 1681] = dy.reshape(N, 4, 8, 1681).permute(1, 0, 3, 2).bfloat16()
    packed = torch.empty(_lib.lib().drq_conv1_w_packed_elems(), dtype=torch.bfloat16, device=dev)
    _call("drq_pack_conv1_w_bf16", w.data_ptr(), b.data_ptr(), packed.data_ptr(), cin, _s())
    wq = packed[:12 * 32 * 8].view(12, 32, 8).permute(1, 0, 2).reshape(32, 96)[:, :cin * 9].float()
    # entries k >= cin*9 and the fused biases behind the weights are not read (or reach unused columns)
    kk = torch.arange(96, device=dev).view(12, 1, 8)
    packed[:12 * 32 * 8].view(12, 32, 8).masked_fill_(kk >= cin * 9, float("nan"))
    packed[12 * 32 * 8:] = float("nan")
    return dy, wb, packed, wq.reshape(32, cin, 3, 3)


def _bf16_dgrad_run(wb, packed, N, cin, dev):
    buf, dx, written = _padded_out(N * cin * 84 * 84, dev)
    _call("drq_conv1_dgrad_bf16", wb.data_ptr(), packed.data_ptr(), dx.data_ptr(), N, cin, _s())
    assert_sentinel_outside(buf, written, "drq_conv1_dgrad_bf16")
    return dx


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("cin", [1, 3, 9, 10])
def test_conv1_dgrad_bf16_kernel(dev, N, cin):
    dy, wb, packed, wq = _bf16_dgrad_inputs(N, cin, dev, 2000 * cin + N)
    dx = _bf16_dgrad_run(wb, packed, N, cin, dev)
    want, absref = _dgrad_want(dy, wq)
    check_sum_bound("drq_conv1_dgrad_bf16", dx.view(N, cin, 84, 84), want, absref, 128, RATIOS)
    again = _bf16_dgrad_run(wb, packed, N, cin, dev)
    assert torch.equal(again.view(torch.int32), dx.view(torch.int32))


@pytest.mark.parametrize("sms", [148, 140, 7, 1])
@pytest.mark.parametrize("N", [7, 129, 512])
def test_conv1_dgrad_bf16_sm_budgets(dev, N, sms):
    from drqv2_b200 import _lib
    dy, wb, packed, wq = _bf16_dgrad_inputs(N, 9, dev, 77 + N)
    ref = _bf16_dgrad_run(wb, packed, N, 9, dev)
    _lib.lib().drq_set_sm_limit(sms)
    try:
        dx = _bf16_dgrad_run(wb, packed, N, 9, dev)
    finally:
        _lib.lib().drq_set_sm_limit(148)
    assert torch.equal(dx.view(torch.int32), ref.view(torch.int32))
    want, absref = _dgrad_want(dy, wq)
    check_sum_bound("drq_conv1_dgrad_bf16", dx.view(N, 9, 84, 84), want, absref, 128, RATIOS)


def _shift_bwd(dout, shift, pad, dev):
    N, C, H, W = dout.shape
    buf, dx, written = _padded_out(N * C * H * W, dev)
    _call("drq_random_shift_bwd_f32", dout.data_ptr(), shift.data_ptr(), dx.data_ptr(), N, C, H, W, pad, _s())
    assert_sentinel_outside(buf, written, "drq_random_shift_bwd_f32")
    return dx.view(N, C, H, W)


def _shift_want(dout, shift, pad, dtype):
    x = torch.zeros(dout.shape, dtype=dtype, requires_grad=True)
    out = O.random_shift_exact(x, shift.cpu(), pad)
    g, = torch.autograd.grad(out, x, dout.cpu().to(dtype))
    ga, = torch.autograd.grad(O.random_shift_exact(x, shift.cpu(), pad), x, dout.cpu().to(dtype).abs())
    return g, ga


@pytest.mark.parametrize("N", NS)
def test_random_shift_bwd_kernel(dev, N):
    g = torch.Generator().manual_seed(N)
    shift = torch.randint(0, 9, (N, 2), generator=g, dtype=torch.int32).to(dev)
    dyadic = (torch.randint(-512, 513, (N, 9, 84, 84), generator=g).float() / 64).to(dev)
    got = _shift_bwd(dyadic, shift, 4, dev)
    want, _ = _shift_want(dyadic, shift, 4, torch.float64)
    assert torch.equal(got.cpu().double(), want), "dyadic gradients: sums are exact"
    dout = torch.randn(N, 9, 84, 84, generator=g).to(dev)
    got = _shift_bwd(dout, shift, 4, dev)
    want, absref = _shift_want(dout, shift, 4, torch.float64)
    check_sum_bound("drq_random_shift_bwd_f32", got.cpu(), want, absref, 128, RATIOS)
    assert torch.equal(_shift_bwd(dout, shift, 4, dev).view(torch.int32), got.view(torch.int32))


@pytest.mark.parametrize("H", [7, 84])
@pytest.mark.parametrize("pad", [0, 1, 2, 3, 4])
def test_random_shift_bwd_every_shift(dev, H, pad):
    sx, sy = torch.meshgrid(torch.arange(2 * pad + 1), torch.arange(2 * pad + 1), indexing="ij")
    shift = torch.stack([sx.reshape(-1), sy.reshape(-1)], 1).to(torch.int32).to(dev)
    n = shift.shape[0]
    g = torch.Generator().manual_seed(H + pad)
    dyadic = (torch.randint(-512, 513, (n, 3, H, H), generator=g).float() / 64).to(dev)
    want, _ = _shift_want(dyadic, shift, pad, torch.float64)
    assert torch.equal(_shift_bwd(dyadic, shift, pad, dev).cpu().double(), want)


# ----------------------------------------------------------------------------- float-source conv1 forward / wgrad
def _encoders(cin, mode, params, dev):
    from drqv2_b200 import Encoder
    out = []
    for pixels in ("u8", "float"):
        enc = Encoder((cin, 84, 84), differentiable=mode, pixels=pixels)
        enc.load_state_dict(params)
        out.append(enc.to(dev))
    return out


@pytest.mark.parametrize("mode", [True, "bf16"])
@pytest.mark.parametrize("N", [1, 33, 256])
def test_float_pixels_integer_valued_are_u8_bits(dev, mode, N):
    from drqv2_b200 import _lib
    params = O.synthetic_params(9, 6, 50, 64, seed=3)["encoder"]
    enc_u8, enc_f = _encoders(9, mode, params, dev)
    g = torch.Generator().manual_seed(N)
    obs = torch.randint(0, 256, (N, 9, 84, 84), dtype=torch.uint8, generator=g).to(dev)
    G = torch.randn(N, 39200, generator=g).to(dev)
    prev = _lib.lib().drq_set_conv1_planes(0)           # the u8 im2col selection
    try:
        f_u8 = enc_u8(obs)
        g_u8 = torch.autograd.grad(f_u8, list(enc_u8.parameters()), G)
    finally:
        _lib.lib().drq_set_conv1_planes(prev)
    f_f = enc_f(obs.float())
    g_f = torch.autograd.grad(f_f, list(enc_f.parameters()), G)
    assert torch.equal(f_f.view(torch.int32), f_u8.view(torch.int32))
    for a, b in zip(g_f, g_u8):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    with torch.no_grad():
        assert torch.equal(enc_f(obs).view(torch.int32), f_u8.view(torch.int32))     # uint8 cast to fp32


def _real_pixels(N, cin, g):
    return torch.rand(N, cin, 84, 84, generator=g, dtype=torch.float64).float() * 255


# ---- the fp32 oracle with the kernels' ReLU decisions (the rule of tests/test_gpu_autograd.py::_relu_as): a unit that
# the fp32 kernels put on the other side of zero than fp64 carries its whole gradient on one side only, which no
# accumulation bound covers; where the decisions differ, the pre-activation must lie within the fp32 sum's rounding of
# zero, |pre| <= 2 * 2^-24 * (K + 8) * (the same sum over absolute values)
def _node(t, name):
    """the autograd node called `name` behind t (breadth first)"""
    todo, seen = [t.grad_fn], set()
    while todo:
        n = todo.pop(0)
        if n is None or id(n) in seen:
            continue
        seen.add(id(n))
        if type(n).__name__ == name:
            return n
        todo += [f for f, _ in n.next_functions]
    raise AssertionError(f"no {name} behind the tensor")


def _encoder_decisions(feat):
    """conv1..conv4's ReLU decisions of an fp32 encoder forward, from what _EncoderFn saved: the wide-plane
    activations of conv1..3 (valid 41, 39, 37) and the features"""
    a1, a2, a3, f = _node(feat, "_EncoderFnBackward").saved_tensors[1:5]
    n = f.shape[0]
    ons = [a.view(n, 32, PLANE)[:, :, :hw * 41].reshape(n, 32, hw, 41)[..., :hw] > 0
           for a, hw in ((a1, 41), (a2, 39), (a3, 37))]
    return ons + [f.view(n, 32, 35, 35) > 0]


def _critic_decisions(q1):
    """[(layer 1, layer 2) of Q1, ... of Q2] from what _CriticFn saved"""
    h1a, h2a, h1b, h2b = _node(q1, "_CriticFnBackward").saved_tensors[4:8]
    return [(h1a > 0, h2a > 0), (h1b > 0, h2b > 0)]


def _actor_decisions(mu):
    p1, p2 = _node(mu, "_ActorFnBackward").saved_tensors[4:6]
    return p1 > 0, p2 > 0


def _conv_relu_as(h, w, b, stride, on, flips):
    pre = F.conv2d(h, w, b, stride=stride)
    with torch.no_grad():
        differ = (pre > 0) != on
        bound = 2 * 2.0 ** -24 * (w.shape[1] * 9 + 8) * F.conv2d(h.abs(), w.abs(), b.abs(), stride=stride)
        assert bool((pre.abs() <= bound)[differ].all()), "a conv ReLU decision differs away from zero"
        flips.append(int(differ.sum()))
    return pre * on.to(pre.dtype)


def _encoder_as(p, x, ons, flips):
    """O.encoder_fwd (drqv2.py:63-67) with the decisions `ons` of conv1..4"""
    h = x / 255.0 - 0.5
    for j, (i, stride) in enumerate(zip((0, 2, 4, 6), (2, 1, 1, 1))):
        h = _conv_relu_as(h, p[f"convnet.{i}.weight"], p[f"convnet.{i}.bias"], stride, ons[j], flips)
    return h.reshape(h.shape[0], -1)


def _critic_as(p, feat, action, on, flips):
    from tests.test_gpu_autograd import _relu_as
    x = torch.cat([O.trunk_fwd(p, feat), action], dim=-1)
    qs = []
    for q, (on1, on2) in zip(("Q1", "Q2"), on):
        y = _relu_as(x, p[f"{q}.0.weight"], p[f"{q}.0.bias"], on1, flips)
        y = _relu_as(y, p[f"{q}.2.weight"], p[f"{q}.2.bias"], on2, flips)
        qs.append(F.linear(y, p[f"{q}.4.weight"], p[f"{q}.4.bias"]))
    return qs[0], qs[1]


def _actor_as(p, feat, on, flips):
    from tests.test_gpu_autograd import _relu_as
    y = _relu_as(O.trunk_fwd(p, feat), p["policy.0.weight"], p["policy.0.bias"], on[0], flips)
    y = _relu_as(y, p["policy.2.weight"], p["policy.2.bias"], on[1], flips)
    return torch.tanh(F.linear(y, p["policy.4.weight"], p["policy.4.bias"]))


def _bf16_pixels(x):
    """the tensor-core path's pixel rounding point: RN-bf16(RN-fp32(x - 128)) + 128"""
    return (x.float() - 128).bfloat16().double() + 128


@pytest.mark.parametrize("mode", [True, "bf16"])
@pytest.mark.parametrize("N", [1, 33, 256])
def test_float_pixels_non_integral_forward_and_wgrad(dev, mode, N):
    params = O.synthetic_params(9, 6, 50, 64, seed=4)["encoder"]
    _, enc = _encoders(9, mode, params, dev)
    g = torch.Generator().manual_seed(5 + N)
    x = _real_pixels(N, 9, g)
    G = torch.randn(N, 39200, generator=g)
    feat = enc(x.to(dev))
    ons = _encoder_decisions(feat) if mode is True else None      # read before the backward frees them
    got = torch.autograd.grad(feat, list(enc.parameters()), G.to(dev))
    names = list(params)
    flips = []
    if mode is True:
        fn, xin, tol = (lambda p, xx: _encoder_as(p, xx, ons, flips)), x, 1e-4
    else:
        fn, xin, tol = O.encoder_fwd_bf16, _bf16_pixels(x), 2e-2
    res = {}
    for dt in (torch.float64, torch.float32):
        ts = [p.detach().to(dev, dt).requires_grad_(True) for p in params.values()]
        f = fn(dict(zip(names, ts)), xin.to(dev, dt))
        res[dt] = (f.detach(), torch.autograd.grad(f, ts, G.to(dev, dt)))
    f64, g64 = res[torch.float64]
    f32, g32 = res[torch.float32]
    assert rel_l2(feat.detach().cpu(), f64.cpu()) <= max(tol, 3 * rel_l2(f32.cpu(), f64.cpu())), "features"
    for name, a, b, c in zip(names, got, g32, g64):
        bound = max(tol, (3 if mode is True else 1.5) * rel_l2(b.cpu(), c.cpu()))
        assert rel_l2(a.cpu(), c.cpu()) <= bound, name


# ----------------------------------------------------------------------------- modules end to end
def _modules(mode, A, params, dev):
    from drqv2_b200 import Actor, Critic, Encoder, RandomShiftsAug
    enc = Encoder((9, 84, 84), differentiable=mode, pixels="float")
    actor = Actor(39200, (A,), 50, 1024, differentiable=mode)
    critic = Critic(39200, (A,), 50, 1024, differentiable=mode)
    enc.load_state_dict(params["encoder"])
    actor.load_state_dict(params["actor"])
    critic.load_state_dict(params["critic"])
    return RandomShiftsAug(4), enc.to(dev), actor.to(dev), critic.to(dev)


def _with_shift(aug, x, shift):
    orig = torch.randint
    torch.randint = lambda lo, hi, size, device=None, dtype=None: shift.view(-1, 1, 1, 2).to(device=device, dtype=dtype)
    try:
        return aug(x)
    finally:
        torch.randint = orig


def _shift_exact(x, shift, pad):
    """oracle.random_shift_exact with its index tensors on x's device"""
    n, c, h, w = x.shape
    ar = torch.arange(h, device=x.device).view(1, h)
    rows = (ar + shift[:, 1].long().view(n, 1) - pad).clamp(0, h - 1)
    cols = (ar + shift[:, 0].long().view(n, 1) - pad).clamp(0, w - 1)
    idx_n = torch.arange(n, device=x.device).view(n, 1, 1, 1)
    idx_c = torch.arange(c, device=x.device).view(1, c, 1, 1)
    return x[idx_n, idx_c, rows.view(n, 1, h, 1), cols.view(n, 1, 1, w)]


@pytest.mark.parametrize("mode", [True, "bf16"])
@pytest.mark.parametrize("A", [6, 38])
@pytest.mark.parametrize("B", [1, 33, 256])
def test_pixel_gradient_through_modules(dev, mode, A, B):
    params = O.synthetic_params(9, A, 50, 1024, seed=A + B)
    aug, enc, actor, critic = _modules(mode, A, params, dev)
    g = torch.Generator().manual_seed(A * 1000 + B)
    x = _real_pixels(B, 9, g)
    shift = torch.randint(0, 9, (B, 2), generator=g)
    action = torch.rand(B, A, generator=g) * 2 - 1
    u = torch.randn(B, 3 + A, generator=g)
    xd = x.to(dev).requires_grad_(True)
    feat = enc(_with_shift(aug, xd, shift.to(dev)))
    q1, q2 = critic(feat, action.to(dev))
    mu = actor(feat, 0.1).mean
    flips = []
    if mode is True:
        on_e, on_c, on_a = _encoder_decisions(feat), _critic_decisions(q1), _actor_decisions(mu)
        enc_fn = lambda p, xx: _encoder_as(p, xx, on_e, flips)          # noqa: E731
        crit_fn = lambda p, f, a: _critic_as(p, f, a, on_c, flips)      # noqa: E731
        act_fn = lambda p, f: _actor_as(p, f, on_a, flips)              # noqa: E731
    else:
        enc_fn, crit_fn, act_fn = O.encoder_fwd_bf16, O.critic_q_bf16, O.actor_mu_bf16
    ud = u.to(dev)
    loss = (q1[:, 0] * ud[:, 0]).sum() + (q2[:, 0] * ud[:, 1]).sum() + (torch.minimum(q1, q2)[:, 0] * ud[:, 2]).sum() \
        + (mu * ud[:, 3:]).sum()
    mods = (enc, critic, actor)
    plist = [p for m in mods for p in m.parameters()]
    got = torch.autograd.grad(loss, [xd] + plist)

    keys = [(k, "encoder") for k in params["encoder"]] + [(k, "critic") for k in params["critic"]] + \
           [(k, "actor") for k in params["actor"]]
    def oracle(dt):
        xo = x.to(dev, dt).requires_grad_(True)
        ps = [params[m][k].to(dev, dt).requires_grad_(True) for k, m in keys]
        pd = {m: {} for m in ("encoder", "critic", "actor")}
        for (k, m), t in zip(keys, ps):
            pd[m][k] = t
        xa = _shift_exact(xo, shift.to(dev), 4)
        if mode == "bf16":
            xa = xa + ((xa.detach().float() - 128).bfloat16().to(dt) + 128 - xa.detach())     # the pixel rounding point
        f = enc_fn(pd["encoder"], xa)
        o1, o2 = crit_fn(pd["critic"], f, action.to(dev, dt))
        m_ = act_fn(pd["actor"], f)
        u_ = u.to(dev, dt)
        lo = (o1[:, 0] * u_[:, 0]).sum() + (o2[:, 0] * u_[:, 1]).sum() + (torch.minimum(o1, o2)[:, 0] * u_[:, 2]).sum() \
            + (m_ * u_[:, 3:]).sum()
        return torch.autograd.grad(lo, [xo] + ps)

    g64, g32 = oracle(torch.float64), oracle(torch.float32)
    names = ["pixels"] + [f"{m}.{k}" for k, m in keys]
    for name, a, b, c in zip(names, got, g32, g64):
        own = rel_l2(b.cpu(), c.cpu())
        bound = max(1e-4, 3 * own) if mode is True else max(2e-2, 1.5 * own)
        err = rel_l2(a.cpu(), c.cpu())
        assert err <= bound, (mode, A, B, name, err, bound)


@pytest.mark.parametrize("mode", [True, "bf16"])
def test_saliency_runs_no_encoder_weight_gradient(dev, mode):
    params = O.synthetic_params(9, 6, 50, 1024, seed=9)
    aug, enc, actor, critic = _modules(mode, 6, params, dev)
    for m in (enc, critic):
        m.requires_grad_(True)
    g = torch.Generator().manual_seed(9)
    obs = _real_pixels(64, 9, g).to(dev).requires_grad_(True)
    a = (torch.rand(64, 6, generator=g) * 2 - 1).to(dev)
    q = torch.min(*critic(enc(obs), a)).sum()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        sal, = torch.autograd.grad(q, obs)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "drq" in e.name]
    assert any("conv1_dgrad" in n for n in names), names
    assert not [n for n in names if re.search(r"conv\w*wgrad|conv1_tc_kernel<true", n)], names
    assert bool(torch.isfinite(sal).all()) and float(sal.abs().sum()) > 0
    for p in enc.parameters():
        assert p.grad is None


# ----------------------------------------------------------------------------- the reference body with a user augmentation
def _oracle_at(agent, state, lr, dtype, operands, overlay):
    """the oracle at the agent's parameters and Adam state (tests/test_gpu_autograd_bf16.py::_oracle_at), its
    augmentation followed by the same overlay - and, for the tensor-core agent, by conv1's pixel rounding point"""
    from collections import OrderedDict
    from tests.test_gpu_autograd_bf16 import SCHED
    o = O.OracleAgent(state, lr, 0.01, SCHED, 0.3, dtype=dtype, operands=operands)
    a = agent._arena
    for net in ("encoder", "critic", "actor"):
        offs = a.offsets[net]
        for buf, dst in ((a.exp_avg, o.m), (a.exp_avg_sq, o.v)):
            dst[net] = OrderedDict((k, buf[offs[k]:offs[k] + p.numel()].view(p.shape).detach().cpu().to(dtype).clone())
                                   for k, p in getattr(agent, net).named_parameters())
    o.t = dict(agent._opt_steps)
    ov = overlay.to(dtype)

    def aug(x, shift):
        y = O.random_shift_exact(x, shift) + ov
        return (y.float() - 128).bfloat16().to(dtype) + 128 if operands == "bf16" else y
    o._aug = aug
    return o


@pytest.mark.parametrize("mode", [True, "bf16"])
def test_reference_body_with_real_valued_overlay(dev, mode):
    """three reference updates (drqv2.py:230-262: aug -> encoder -> update_critic -> update_actor, loss.backward(),
    opt.step()) on a pixels="float" agent whose augmentation adds a fixed real-valued overlay - a user augmentation
    feeding agent.encoder - each against the oracle re-seeded from the agent's state before it, under the bounds of
    the multi-update tests (tests/test_gpu_update_chain.py: FP32 / BF16)"""
    from drqv2_b200 import DrQV2Agent
    from tests.test_gpu_autograd_bf16 import SCHED, _reference_update_with_encoder
    from tests.test_gpu_update_chain import BF16, FP32
    B, A, Fd, H, lr = 256, 6, 50, 1024, 1e-4
    params = O.synthetic_params(9, A, Fd, H, seed=21)
    Y = DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, seed=5,
                   mode="bf16" if mode == "bf16" else "fp32", differentiable=mode, pixels="float")
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(Y, net).load_state_dict(params[net])
    # dyadic steps of 1/64 within +-10: the integer pixel plus the overlay is exact in fp32 and fp64
    overlay = torch.randint(-640, 641, (1, 9, 84, 84), generator=torch.Generator().manual_seed(7)).float() / 64
    shift_aug, ovd = Y.aug, overlay.to(dev)
    Y.aug = lambda x: shift_aug(x) + ovd
    bounds, operands = (BF16, "bf16") if mode == "bf16" else (FP32, "exact")
    for s in range(3):
        b = O.synthetic_batch(B, A, seed=30 + s)
        state = {net: {k: v.detach().cpu().clone() for k, v in getattr(Y, net).state_dict().items()}
                 for net in ("encoder", "actor", "critic", "critic_target")}
        args = (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 2 * s, b["shift_obs"], b["shift_next"],
                b["eps_critic"], b["eps_actor"])
        o64, o32 = (_oracle_at(Y, state, lr, dt, operands, overlay) for dt in (torch.float64, torch.float32))
        want = o64.update(*args)
        o32.update(*args)
        enc_g = {}
        my, cg = _reference_update_with_encoder(Y, b, 2 * s, dev, enc_g)
        # the actor stage reads the critic after critic_opt.step() (drqv2.py:201,213): held at the agent's stepped critic
        stepped = dict(state, critic={k: v.detach().cpu().clone() for k, v in Y.critic.state_dict().items()})
        for o in (o64, o32):
            oa = _oracle_at(Y, stepped, lr, o.dtype, operands, overlay)
            oa.stage = {}
            m = oa.update_actor(oa.encode(b["obs"], b["shift_obs"]), 2 * s, b["eps_actor"])
            o.grads["actor"] = oa.grads["actor"]
            if o is o64:
                want.update(m)
        for k, v in want.items():
            assert abs(my[k] - v) <= bounds.metric(v), (mode, s, k, my[k], v)
        for net, got in (("encoder", enc_g), ("critic", cg),
                         ("actor", {k: p.grad for k, p in Y.actor.named_parameters()})):
            for k in o64.grads[net]:
                err = rel_l2(got[k].cpu().numpy(), o64.grads[net][k].numpy())
                bound = bounds.grad(net, k, rel_l2(o32.grads[net][k].numpy(), o64.grads[net][k].numpy()))
                assert err <= bound, (mode, s, net, k, err, bound)
    assert Y._opt_steps == dict(encoder=3, critic=3, actor=3)
