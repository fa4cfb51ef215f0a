"""The small head kernels of the update (csrc/heads.cu, csrc/multi.cu) against fp64, at their update call shapes and at
the edges of their row tiling and template branches.  The whole-update tests compare these only through per-tensor
rel-L2 of whole updates; a wrong row block, a dropped plane or a wrong tie rule moves one tensor by far less than that.

Bounds: fp32 results that are sums of n terms are checked element-wise as |got - want| <= 2^-24 (n + 8) A, A the same sum
over absolute values (SUM_C = 2 spare); LayerNorm outputs as stated at each test.  Values the kernels form with exactly
rounded fp32 steps (the loss gradients, the TD target) are reproduced in torch fp32 and must match bit for bit, and every
bf16 copy must be RN-bf16 of the fp32 value the same launch wrote.  Every output starts as a NaN sentinel one size too
big; what a launch must not write keeps it."""
import ctypes as C

import pytest
import torch

from tests.helpers import assert_sentinel_outside, bits_equal, check_sum_bound, fill_sentinel

pytestmark = pytest.mark.gpu

SUM_C = 2.0
RATIOS = {}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if RATIOS:
        print("\nlargest |got - want| / bound per kernel:", {k: round(v, 4) for k, v in sorted(RATIOS.items())})


def _s():
    return torch.cuda.current_stream().cuda_stream


def _call(name, *a):
    from drqv2_b200 import _lib
    _lib.call(name, *a)
    torch.cuda.synchronize()


def _ceil(n, m):
    return -(-n // m) * m


def _check(kernel, got, want, absref, n, c=SUM_C):
    """|got - want| <= c 2^-24 (n + 8) A element-wise (tests/helpers.check_sum_bound)"""
    check_sum_bound(kernel, got, want, absref, n, RATIOS, c)


def _tb(rows, feats, dev, batch=1):
    from drqv2_b200._bf16 import TB
    t = TB(rows, feats, dev, batch=batch + 1)           # one spare entry
    fill_sentinel(t.buf)
    return t


def _tb_written(t, entries, rows, cols):
    """bool over t.buf: rows < rows, columns < cols of the given entries"""
    w = torch.zeros(t.batch, t.rpad, t.units * 8, dtype=torch.bool, device=t.buf.device)
    for z in entries:
        w[z, :rows, :cols] = True
    nb = t.rpad // t.rblk
    return w.view(t.batch, nb, t.rblk, t.units, 8).permute(0, 1, 3, 2, 4).reshape(-1)


def _rand(g, *shape, lo=-1.0, hi=1.0):
    return torch.rand(*shape, generator=g, dtype=torch.float64) * (hi - lo) + lo


# ---------------------------------------------------------------- trunk tail: split-K sum + bias + LayerNorm + tanh
def check_ln_tanh_fwd(p, bias, gamma, beta, h, xhat, rstd, B, F, S, ratios):
    """h_out [B + 1][ld_h] (and, when not None, xhat [>= B F] and rstd [B + 1]) of one trunk tail on the split planes
    p [S][B][F] (fp64 of the fp32 partials) against fp64; everything but rows < B, columns < F of h_out (the tail columns
    are the caller's), xhat[:B F] and rstd[:B] keeps the sentinel"""
    dev = h.device
    z = p.sum(0) + bias.double().cpu()
    za = p.abs().sum(0) + bias.double().cpu().abs()
    mean = z.mean(1, keepdim=True)
    var = ((z - mean) ** 2).mean(1, keepdim=True)
    r = 1 / torch.sqrt(var + 1e-5)
    xh = (z - mean) * r
    y = xh * gamma.double().cpu() + beta.double().cpu()
    # z carries the fp32 sum's error (S + 4 terms of za); normalised by the row's spread it moves xhat and y
    dz = 2.0 ** -24 * (S + 8) * za + 2.0 ** -22 * z.abs()
    dx = (dz * r).amax(1, keepdim=True) * (1 + xh.abs()) * 2 + 2.0 ** -21 * (1 + xh.abs())
    if rstd is not None:
        rb = (4 * dz.amax(1) * r[:, 0] + 2.0 ** -20) * r[:, 0]      # std moves by at most max|dz|
        re = (rstd[:B].cpu().double() - r[:, 0]).abs()
        assert (re <= rb).all(), f"rstd error {float((re / rb).max())} x bound"
        wr = torch.zeros(B + 1, dtype=torch.bool, device=dev)
        wr[:B] = True
        assert_sentinel_outside(rstd, wr, "rstd")
    if xhat is not None:
        dxe = (xhat[:B * F].view(B, F).cpu().double() - xh).abs()
        assert (dxe <= dx).all(), f"xhat error {float((dxe / dx).max())} x bound"
        ratios["ln_tanh_fwd xhat"] = max(ratios.get("ln_tanh_fwd xhat", 0), float((dxe / dx).max()))
        wx = torch.zeros(xhat.numel(), dtype=torch.bool, device=dev)
        wx[:B * F] = True
        assert_sentinel_outside(xhat, wx, "xhat")
    hw = torch.tanh(y)
    dh = dx * gamma.double().cpu().abs() * (1 - hw ** 2) + 2.0 ** -21
    hg = h[:B, :F].cpu().double()
    assert ((hg - hw).abs() <= dh).all(), f"h error {float(((hg - hw).abs() / dh).max())} x bound"
    ratios["ln_tanh_fwd h"] = max(ratios.get("ln_tanh_fwd h", 0), float(((hg - hw).abs() / dh).max()))
    w = torch.zeros_like(h, dtype=torch.bool)
    w[:B, :F] = True                                                  # the tail columns of h_out are the caller's
    assert_sentinel_outside(h, w, "h_out")


@pytest.mark.parametrize("S", [1, 35, 64, 65, 130, 145, 273])
@pytest.mark.parametrize("B", [1, 3, 129, 512])
@pytest.mark.parametrize("F", [50, 64, 65, 100, 128, 129, 256])
def test_ln_tanh_fwd_multi(dev, F, B, S):
    """four jobs in one launch as critic_pass issues them: tails of 0 / 6 / 21 / 32 columns, bf16 rows at row 0 and at the
    second half's row block"""
    from drqv2_b200._bf16 import LnJob
    g = torch.Generator().manual_seed(F * 1000 + B * 10 + S)
    RB = _ceil(B, 128)
    tails = [0, 6, 21, 32]
    tbs = [_tb(2 * RB, F + 32, dev), _tb(2 * RB, F + 32, dev)]
    jobs, ref, keep = [], [], []
    for j in range(4):
        ldp = F + 3
        part = fill_sentinel(torch.empty(S + 1, B, ldp, device=dev))
        p = _rand(g, S, B, F) / S ** 0.5
        part[:S, :, :F] = p.float().to(dev)
        bias, gamma, beta = (_rand(g, F).float().to(dev) for _ in range(3))
        nt = tails[j]
        ld_h = F + nt
        h = fill_sentinel(torch.empty(B + 1, ld_h, device=dev))
        xhat = fill_sentinel(torch.empty(B * F + 8, device=dev))
        rstd = fill_sentinel(torch.empty(B + 1, device=dev))
        tail = _rand(g, B, max(nt, 1)).float().to(dev)
        tb, row0 = tbs[j // 2], (j % 2) * RB
        jobs.append(LnJob(part.data_ptr(), ldp, B * ldp, S, bias.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                          h.data_ptr(), ld_h, xhat.data_ptr(), rstd.data_ptr(), tb.buf.data_ptr(), tb.units, row0,
                          tail.data_ptr() if nt else None, max(nt, 1), nt))
        keep.append(part)                                             # the launch reads it through a raw pointer
        ref.append((part[:S, :, :F].double().cpu(), bias, gamma, beta, h, xhat, rstd, tail, nt, tb, row0))
    arr = (LnJob * 4)(*jobs)
    _call("drq_ln_tanh_fwd_multi", arr, 4, B, F, C.c_float(1e-5), _s())
    for tb in tbs:
        written = torch.zeros(tb.buf.numel(), dtype=torch.bool, device=dev)
        for (p, bias, gamma, beta, h, xhat, rstd, tail, nt, t2, row0) in ref:
            if t2 is not tb:
                continue
            w = torch.zeros(tb.batch, tb.rpad, tb.units * 8, dtype=torch.bool, device=dev)
            w[0, row0:row0 + B, :F + nt] = True
            nb = tb.rpad // 128
            written |= w.view(tb.batch, nb, 128, tb.units, 8).permute(0, 1, 3, 2, 4).reshape(-1)
        assert_sentinel_outside(tb.buf, written, "ln_tanh_fwd TB")
    for (p, bias, gamma, beta, h, xhat, rstd, tail, nt, tb, row0) in ref:
        check_ln_tanh_fwd(p, bias, gamma, beta, h, xhat, rstd, B, F, S, RATIOS)
        # the bf16 copy is RN-bf16 of h_out, the tail columns bf16(tail)
        v = tb.view(0)
        assert bits_equal(v[row0:row0 + B, :F], h[:B, :F].to(torch.bfloat16)), "TB copy != RN-bf16(h_out)"
        if nt:
            assert bits_equal(v[row0:row0 + B, F:F + nt], tail[:, :nt].to(torch.bfloat16)), "TB tail != bf16(tail)"


# ---------------------------------------------------------------- LayerNorm + tanh backward
@pytest.mark.parametrize("n_planes", [1, 7, 8, 9, 16])
@pytest.mark.parametrize("B", [1, 3, 5, 256, 513])
def test_ln_tanh_bwd(dev, n_planes, B):
    F = 50 if B % 2 else 100
    g = torch.Generator().manual_seed(B * 31 + n_planes)
    ld = F + 21
    PS = B * ld + 5                                                   # plane stride (floats)
    dh = fill_sentinel(torch.empty(n_planes * PS + 8, device=dev))
    planes = _rand(g, n_planes, B, F) * 1e-2
    for p in range(n_planes):
        dh[p * PS:p * PS + B * ld].view(B, ld)[:, :F] = planes[p].float().to(dev)
    h = _rand(g, B, ld, lo=-0.99, hi=0.99).float().to(dev)
    xhat = _rand(g, B, F, lo=-2, hi=2).float().to(dev)
    rstd = _rand(g, B, lo=0.5, hi=3).float().to(dev)
    gamma = _rand(g, F).float().to(dev)
    dz = fill_sentinel(torch.empty(2 * B * F + 16, device=dev))
    zb = _tb(B, F, dev)
    with_param = B > 256
    dgamma = fill_sentinel(torch.empty(F + 4, device=dev))
    dbeta = fill_sentinel(torch.empty(F + 4, device=dev))
    _call("drq_ln_tanh_bwd", dh.data_ptr(), ld, h.data_ptr(), ld, xhat.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
          dz.data_ptr(), dgamma.data_ptr() if with_param else None, dbeta.data_ptr() if with_param else None,
          zb.buf.data_ptr(), zb.units, B, F, n_planes, PS, _s())
    P = planes.sum(0)
    Pa = planes.abs().sum(0)
    hh, xx, rr, gg = (t.double().cpu() for t in (h[:, :F], xhat, rstd, gamma))
    dy = P * (1 - hh ** 2)
    dya = Pa * (1 - hh ** 2).abs()
    _check("ln_tanh_bwd dy", dz[B * F:2 * B * F].view(B, F).cpu(), dy, dya, n_planes + 2)
    dxh = dy * gg
    m1, m2 = dxh.mean(1, keepdim=True), (dxh * xx).mean(1, keepdim=True)
    want = rr[:, None] * (dxh - m1 - xx * m2)
    dxa = dya * gg.abs()
    absref = rr[:, None] * (dxa + dxa.mean(1, keepdim=True) + xx.abs() * (dxa * xx.abs()).mean(1, keepdim=True))
    _check("ln_tanh_bwd dz", dz[:B * F].view(B, F).cpu(), want, absref, n_planes + F)
    wd = torch.zeros(dz.numel(), dtype=torch.bool, device=dev)
    wd[:2 * B * F] = True
    assert_sentinel_outside(dz, wd, "dz / dy")
    assert bits_equal(zb.view(0)[:B, :F], dz[:B * F].view(B, F).to(torch.bfloat16)), "dz_bf16 != RN-bf16(dz)"
    assert_sentinel_outside(zb.buf, _tb_written(zb, [0], B, F), "dz_bf16")
    if with_param:
        dyg = dz[B * F:2 * B * F].view(B, F).double().cpu()           # the kernel reduces the dy it staged
        _check("ln_param_grad dgamma", dgamma[:F].cpu(), (dyg * xx).sum(0), (dyg * xx).abs().sum(0), B // 256 + 8)
        _check("ln_param_grad dbeta", dbeta[:F].cpu(), dyg.sum(0), dyg.abs().sum(0), B // 256 + 8)
        for t in (dgamma, dbeta):
            w = torch.zeros(F + 4, dtype=torch.bool, device=dev)
            w[:F] = True
            assert_sentinel_outside(t, w, "dgamma / dbeta")


# ---------------------------------------------------------------- scalar Q heads
@pytest.mark.parametrize("sign", [1, -1], ids=["target_above", "target_below"])
@pytest.mark.parametrize("H", [8, 56, 1024])
@pytest.mark.parametrize("B", [1, 31, 33, 256, 513])
def test_q_head_fwd(dev, B, H, sign):
    g = torch.Generator().manual_seed(B * 7 + H + (sign > 0))
    c2 = _tb(B, H, dev, batch=4)
    x = torch.relu(_rand(g, 4, B, H))
    for z in range(4):
        c2.load(x[z].float().to(dev), z)
    xb = x.to(torch.bfloat16).double()
    ws = H + 8                                                        # Q1 -> Q2 distance of the parameters (floats)
    wo = sign * 2 * ws                                                # critic -> target
    base = 0 if sign > 0 else 2 * ws
    w = _rand(g, 4 * ws).float().to(dev)
    b = _rand(g, 4 * ws).float().to(dev)
    q = fill_sentinel(torch.empty(5, B, device=dev))
    _call("drq_q_head_fwd_bf16", c2.buf.data_ptr(), c2.units, c2.stride, w.data_ptr() + 4 * base, b.data_ptr() + 4 * base,
          q.data_ptr(), B, H, 4, ws, 2, wo, _s())
    for z in range(4):
        off = base + (z % 2) * ws + (z // 2) * wo
        wz, bz = w[off:off + H].double().cpu(), b[off].double().cpu()
        _check("q_head_fwd", q[z].cpu(), xb[z] @ wz + bz, xb[z].abs() @ wz.abs() + bz.abs(), H // 8)
    wr = torch.zeros(5, B, dtype=torch.bool, device=dev)
    wr[:4] = True
    assert_sentinel_outside(q, wr, "q")


def _f(x):
    return torch.tensor(x, dtype=torch.float32)


def _loss_dq(loss, q, tq, reward, discount, B):
    """dq [2][B] exactly as loss_dq<LOSS> forms it (fp32, each step rounded), and the TD target"""
    q1, q2 = q[0], q[1]
    if loss == 1:
        tv = torch.minimum(tq[0], tq[1])
        t = reward + discount * tv                                    # __fmul_rn then __fadd_rn
        sc = _f(2.0) / _f(float(B))
        return torch.stack([sc * (q1 - t), sc * (q2 - t)]), t
    gm = _f(-1.0) / _f(float(B))
    half = _f(0.5) * gm
    d1 = torch.where(q1 < q2, gm, torch.where(q1 == q2, half, _f(0.0)))
    d2 = torch.where(q2 < q1, gm, torch.where(q1 == q2, half, _f(0.0)))
    return torch.stack([d1, d2]), None


def _scalars(g, B):
    q = (_rand(g, 2, B) * 4).float()
    q[1, ::3] = q[0, ::3]                                             # exact ties q1 == q2
    tq = (_rand(g, 2, B) * 4).float()
    tq[1, 1::4] = tq[0, 1::4]
    reward = _rand(g, B, lo=0, hi=1).float()
    discount = torch.where(torch.arange(B) % 5 == 0, 0.0, 0.99).float()
    return q, tq, reward, discount


@pytest.mark.parametrize("loss", [1, 2], ids=["critic", "actor"])
@pytest.mark.parametrize("B", [1, 255, 256, 257, 513])
def test_q_head_bwd_loss(dev, loss, B):
    H = 1024 if B % 2 == 0 else 56
    g = torch.Generator().manual_seed(B * 3 + loss)
    q, tq, reward, discount = _scalars(g, B)
    qd, tqd, rd, dd = (t.to(dev) for t in (q, tq, reward, discount))
    c2 = _tb(B, H, dev, batch=2)
    x = torch.relu(_rand(g, 2, B, H))
    for z in range(2):
        c2.load(x[z].float().to(dev), z)
    xb = x.to(torch.bfloat16).float()
    ws = H + 8
    w3 = _rand(g, 2 * ws).float().to(dev)
    dc2 = _tb(B, H, dev, batch=2)
    dw3 = fill_sentinel(torch.empty(2 * ws + 4, device=dev))
    db3 = fill_sentinel(torch.empty(2 * ws + 4, device=dev))
    tq_out = fill_sentinel(torch.empty(B + 1, device=dev))
    metrics = fill_sentinel(torch.empty(6, device=dev))
    if loss == 1:
        _call("drq_q_head_bwd_loss_bf16", 1, qd.data_ptr(), tqd.data_ptr(), rd.data_ptr(), dd.data_ptr(), tq_out.data_ptr(),
              metrics.data_ptr(), c2.buf.data_ptr(), c2.units, c2.stride, w3.data_ptr(), dc2.buf.data_ptr(),
              dw3.data_ptr(), db3.data_ptr(), B, H, ws, _s())
    else:
        _call("drq_q_head_bwd_loss_bf16", 2, qd.data_ptr(), None, None, None, None, metrics.data_ptr(), c2.buf.data_ptr(),
              c2.units, c2.stride, w3.data_ptr(), dc2.buf.data_ptr(), None, None, B, H, ws, _s())
    dq, t = _loss_dq(loss, q, tq, reward, discount, B)
    if loss == 2:                                                     # the tie rule is torch.min's gradient
        qq = q.double().requires_grad_(True)
        (-torch.minimum(qq[0], qq[1]).mean()).backward()
        assert torch.equal(qq.grad.float(), dq)
    w = w3.cpu()
    for z in range(2):
        wz = w[z * ws:z * ws + H]
        want = torch.where(xb[z] > 0, dq[z][:, None] * wz[None, :], _f(0.0)).to(torch.bfloat16)
        assert bits_equal(dc2.view(z)[:B, :H].cpu(), want), f"dc2[{z}] != RN-bf16(dq w3) masked by c2 > 0"
    assert_sentinel_outside(dc2.buf, _tb_written(dc2, [0, 1], B, H), "dc2")
    nm = 5 if loss == 1 else 1
    qq = q.double()
    if loss == 1:
        assert torch.equal(tq_out[:B].cpu(), t), "target_q_out is not bit-exact"
        dq64 = dq.double()
        for z in range(2):
            _check("q_head_bwd dw3", dw3[z * ws:z * ws + H].cpu(), dq64[z] @ xb[z].double(),
                   dq64[z].abs() @ xb[z].double(), B // 256 + 8)
            _check("q_head_bwd db3", db3[z * ws].cpu().view(1), dq64[z].sum().view(1), dq64[z].abs().sum().view(1), B // 256 + 8)
        e = (q - t).double()
        t64 = t.double()
        want = torch.stack([reward.double().mean(), t64.mean(), qq[0].mean(), qq[1].mean(), (e ** 2).mean(1).sum()])
        absref = torch.stack([reward.double().abs().mean(), t64.abs().mean(), qq[0].abs().mean(), qq[1].abs().mean(),
                              (e ** 2).mean(1).sum()])
        _check("q_head_bwd metrics", metrics[:5].cpu(), want, absref, B // 256 + 16)
        wd = torch.zeros(2 * ws + 4, dtype=torch.bool, device=dev)
        wd[:H] = True
        wd[ws:ws + H] = True
        assert_sentinel_outside(dw3, wd, "dw3")
        wb = torch.zeros(2 * ws + 4, dtype=torch.bool, device=dev)
        wb[0] = wb[ws] = True
        assert_sentinel_outside(db3, wb, "db3")
    else:
        mn = torch.minimum(qq[0], qq[1])
        _check("q_head_bwd metrics", metrics[:1].cpu(), -mn.mean().view(1), mn.abs().mean().view(1), B // 256 + 16)
    wm = torch.zeros(6, dtype=torch.bool, device=dev)
    wm[:nm] = True
    assert_sentinel_outside(metrics, wm, "metrics")


# ---------------------------------------------------------------- the fp32-mode twins (one block, a thread loop)
@pytest.mark.parametrize("B", [1, 257, 513])
def test_fp32_losses(dev, B):
    g = torch.Generator().manual_seed(B)
    q, tq, reward, discount = _scalars(g, B)
    qd, tqd, rd, dd = (t.to(dev).contiguous() for t in (q, tq, reward, discount))
    dq1, dq2, tq_out = (fill_sentinel(torch.empty(B + 1, device=dev)) for _ in range(3))
    metrics = fill_sentinel(torch.empty(6, device=dev))
    _call("drq_critic_loss", qd[0].data_ptr(), qd[1].data_ptr(), tqd[0].data_ptr(), tqd[1].data_ptr(), rd.data_ptr(),
          dd.data_ptr(), dq1.data_ptr(), dq2.data_ptr(), tq_out.data_ptr(), metrics.data_ptr(), B, _s())
    dq, t = _loss_dq(1, q, tq, reward, discount, B)
    assert torch.equal(dq1[:B].cpu(), dq[0]) and torch.equal(dq2[:B].cpu(), dq[1]) and torch.equal(tq_out[:B].cpu(), t)
    e = (q - t).double()
    want = torch.stack([reward.double().mean(), t.double().mean(), q.double()[0].mean(), q.double()[1].mean(),
                        (e ** 2).mean(1).sum()])
    absref = torch.stack([reward.double().mean(), t.double().abs().mean(), q.double()[0].abs().mean(),
                          q.double()[1].abs().mean(), (e ** 2).mean(1).sum()])
    _check("critic_loss metrics", metrics[:5].cpu(), want, absref, B // 256 + 16)
    for buf in (dq1, dq2, tq_out):
        w = torch.zeros(B + 1, dtype=torch.bool, device=dev)
        w[:B] = True
        assert_sentinel_outside(buf, w, "critic_loss outputs")
    dq1, dq2 = (fill_sentinel(torch.empty(B + 1, device=dev)) for _ in range(2))
    fill_sentinel(metrics)
    _call("drq_actor_loss", qd[0].data_ptr(), qd[1].data_ptr(), dq1.data_ptr(), dq2.data_ptr(), metrics.data_ptr(), B, _s())
    dq, _ = _loss_dq(2, q, tq, reward, discount, B)
    assert torch.equal(dq1[:B].cpu(), dq[0]) and torch.equal(dq2[:B].cpu(), dq[1])
    mn = torch.minimum(q[0], q[1]).double()
    _check("actor_loss metrics", metrics[:1].cpu(), -mn.mean().view(1), mn.abs().mean().view(1), B // 256 + 16)
    w = torch.zeros(6, dtype=torch.bool, device=dev)
    w[0] = True
    assert_sentinel_outside(metrics, w, "actor_loss metrics")


@pytest.mark.parametrize("B", [1, 257, 513])
def test_fp32_actor_sample(dev, B):
    A, clip, std = 6, 0.3, 0.5
    g = torch.Generator().manual_seed(B + 5)
    mu_pre = (_rand(g, B, A) * 3).float().to(dev)
    eps = _rand(g, B, A, lo=-2, hi=2).float().to(dev)
    stdd = torch.tensor([std], device=dev)
    act = fill_sentinel(torch.empty(B + 1, A + 2, device=dev))
    mu = fill_sentinel(torch.empty(B * A + 4, device=dev))
    metrics = fill_sentinel(torch.empty(3, device=dev))
    _call("drq_actor_sample", mu_pre.data_ptr(), eps.data_ptr(), stdd.data_ptr(), C.c_float(clip), act.data_ptr(), A + 2,
          mu.data_ptr(), metrics.data_ptr(), B, A, _s())
    m = torch.tanh(mu_pre.double().cpu())
    e = (eps.double().cpu() * std).clamp(-clip, clip)
    a = (m + e).clamp(-1 + 1e-6, 1 - 1e-6)
    _check("actor_sample mu", mu[:B * A].view(B, A).cpu(), m, torch.ones_like(m), 16)
    _check("actor_sample action", act[:B, :A].cpu(), a, torch.ones_like(a), 32)
    ga = act[:B, :A].double().cpu()
    gm = mu[:B * A].view(B, A).double().cpu()
    lp = (-((ga - gm) ** 2) / (2 * std * std) - torch.log(torch.tensor(std, dtype=torch.float64)) - 0.9189385332046727).sum(1).mean()
    _check("actor_sample logprob", metrics[:1].cpu(), lp.view(1), torch.tensor([A * 2.0]), B // 256 + A + 16)
    w = torch.zeros(B + 1, A + 2, dtype=torch.bool, device=dev)
    w[:B, :A] = True
    assert_sentinel_outside(act, w, "action")
    wm = torch.zeros(3, dtype=torch.bool, device=dev)
    wm[:2] = True
    assert_sentinel_outside(metrics, wm, "metrics")


# ---------------------------------------------------------------- actor sample backward
@pytest.mark.parametrize("B,A", [(1, 1), (7, 6), (129, 21), (256, 6), (513, 32)])
def test_actor_sample_bwd(dev, B, A):
    F, SX = 50, 8
    n_planes = 2 * SX
    ld = F + A
    PS = B * ld
    g = torch.Generator().manual_seed(B * 100 + A)
    dxf = fill_sentinel(torch.empty(n_planes * PS + 8, device=dev))
    planes = _rand(g, n_planes, B, ld) * 1e-2
    dxf[:n_planes * PS] = planes.float().reshape(-1).to(dev)
    mu = _rand(g, B, A, lo=-0.99, hi=0.99).float().to(dev)
    dmu_pre = fill_sentinel(torch.empty(B * A + 4, device=dev))
    dmu = _tb(B, A, dev)
    _call("drq_actor_sample_bwd", dxf.data_ptr() + 4 * F, ld, mu.data_ptr(), dmu_pre.data_ptr(), dmu.buf.data_ptr(),
          dmu.units, B, A, n_planes, PS, _s())
    P = planes.float().double()[:, :, F:]
    mm = mu.double().cpu()
    want = P.sum(0) * (1 - mm ** 2)
    _check("actor_sample_bwd", dmu_pre[:B * A].view(B, A).cpu(), want, P.abs().sum(0) * (1 - mm ** 2).abs(), n_planes + 2)
    w = torch.zeros(B * A + 4, dtype=torch.bool, device=dev)
    w[:B * A] = True
    assert_sentinel_outside(dmu_pre, w, "dmu_pre")
    assert bits_equal(dmu.view(0)[:B, :A], dmu_pre[:B * A].view(B, A).to(torch.bfloat16)), "dmu_bf16 != RN-bf16(dmu_pre)"
    assert_sentinel_outside(dmu.buf, _tb_written(dmu, [0], B, A), "dmu_bf16")


# ---------------------------------------------------------------- bias-gradient column sums
@pytest.mark.parametrize("M", [1, 64, 65, 129, 513])
def test_colsum_multi(dev, M):
    from drqv2_b200._bf16 import ColsumJob
    g = torch.Generator().manual_seed(M)
    spec = [(1, 1024, False), (1, 50, False), (1, 6, False), (0, 1000, False), (0, 21, True), (0, 50, True), (0, 6, False),
            (1, 21, False)]
    jobs, ref, keep = [], [], []
    for tb, N, with_y in spec:
        out = fill_sentinel(torch.empty(N + 4, device=dev))
        x = _rand(g, M, N)
        if tb:
            t = _tb(M, N, dev)
            t.buf.zero_()
            t.load(x.float().to(dev))
            xv = x.to(torch.bfloat16).double()
            jobs.append(ColsumJob(t.buf.data_ptr(), t.units, out.data_ptr(), M, N, 1, 0))
            keep.append(t)
            ref.append((out, xv.sum(0), xv.abs().sum(0), N, M // 64 + 64))
        else:
            ld = N + 3
            X = torch.zeros(M, ld, device=dev)
            X[:, :N] = x.float().to(dev)
            Y = torch.zeros(M, ld, device=dev)
            y = _rand(g, M, N)
            Y[:, :N] = y.float().to(dev)
            xv, yv = x.float().double(), y.float().double()
            if with_y:
                jobs.append(ColsumJob(X.data_ptr(), ld, out.data_ptr(), M, N, 0, 0, Y.data_ptr()))
                ref.append((out, (xv * yv).sum(0), (xv * yv).abs().sum(0), N, M // 8 + 8 + 2))
            else:
                jobs.append(ColsumJob(X.data_ptr(), ld, out.data_ptr(), M, N, 0, 0))
                ref.append((out, xv.sum(0), xv.abs().sum(0), N, M // 8 + 8))
            keep += [X, Y]
    arr = (ColsumJob * len(jobs))(*jobs)
    _call("drq_colsum_multi", arr, len(jobs), _s())
    for out, want, absref, N, n in ref:
        _check("colsum_multi", out[:N].cpu(), want, absref, n)
        w = torch.zeros(N + 4, dtype=torch.bool, device=dev)
        w[:N] = True
        assert_sentinel_outside(out, w, "colsum out")
