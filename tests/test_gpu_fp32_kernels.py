"""The fp32 mode's kernels (csrc/gemm_f32.cu, csrc/encoder_f32.cu, the single-job drq_ln_tanh_fwd, drq_copy2d_f32)
against fp64 at the shapes drqv2.py calls them with and at the edges of their tiling, then one fp32 update at the shape
only this mode runs.  The whole-update tests see these kernels only through per-tensor rel-L2; a dropped tile of a
weight gradient or a wrong row of a GEMM moves one tensor by far less than those bounds.

Bound: every fp32 result is within |got - want| <= 2 2^-24 (n + 8) A of fp64 math on the fp32 operands the kernel
received (tests/helpers.check_sum_bound), A the same operation on absolute values plus |bias| (and |C_old| when
accumulating), n the longest sequential fp32 chain behind the element (tests/test_fp32_schedule_cpu: the K chunk plus
bias / accumulate; 288 for a 3x3 conv; 9 cin for conv1; tiles per block x positions per tile + blocks for the weight
gradients).  conv1's reference input is the fp32 RN(RN(px / 255) - 0.5) its loader forms.

Sentinels and read extents: every output is one size too big and starts as a NaN sentinel; whatever a launch must not
write keeps it.  Every operand holds NaN outside what the kernel may read (a large finite 2^100 where the header only
asks for finite values), and the written outputs must equal, bit for bit, a run with zeros there."""
import pytest
import torch

from tests import test_fp32_schedule_cpu as S
from tests.helpers import assert_sentinel_outside, check_sum_bound, fill_sentinel

pytestmark = pytest.mark.gpu

SUM_C = 2.0
RATIOS = {}
LN_RATIOS = {}       # LayerNorm outputs: |got - want| / the propagated bound of tests/test_gpu_head_kernels.py
SUMMARY = []
BIG = 2.0 ** 100
PLANE, PW = S.PLANE, S.PW


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if SUMMARY:
        print("\nschedules run:\n  " + "\n  ".join(sorted(set(SUMMARY))))
    if RATIOS:
        print(f"largest c needed per kernel (bound c = {SUM_C:g}):")
        for k, v in sorted(RATIOS.items()):
            print(f"  {k:34s} {SUM_C * v:.4f}")
    if LN_RATIOS:
        print("LayerNorm forward, largest |got - want| / propagated bound:",
              {k: round(v, 4) for k, v in sorted(LN_RATIOS.items())})


def _s():
    return torch.cuda.current_stream().cuda_stream


def _call(name, *a):
    from drqv2_b200 import _lib
    _lib.call(name, *a)
    torch.cuda.synchronize()


def _check(kernel, got, want, absref, n):
    check_sum_bound(kernel, got, want, absref, n, RATIOS, SUM_C)


def _box(off, strides, extents, dev):
    """flat indices off + sum_d i_d stride_d over the box `extents` (int64, shaped like the box)"""
    t = torch.full((), off, dtype=torch.int64, device=dev)
    for d, (st, ex) in enumerate(zip(strides, extents)):
        shape = [1] * len(extents)
        shape[d] = ex
        t = t + torch.arange(ex, device=dev).view(shape) * st
    return t


class Poisoned:
    """an fp32 operand buffer: random values on the index set `idx` (aliases allowed), `fill` everywhere else"""

    def __init__(self, g, idx, dev, spare=37, lo=-1.0, hi=1.0):
        self.idx = idx
        n = int(idx.max()) + 1 + spare
        self.vals = (torch.rand(n, generator=g, dtype=torch.float64) * (hi - lo) + lo).float().to(dev)
        self.read = torch.zeros(n, dtype=torch.bool, device=dev)
        self.read[idx.reshape(-1)] = True

    def buf(self, fill):
        return torch.where(self.read, self.vals, torch.full_like(self.vals, fill))

    def dense(self):
        return self.vals.double()[self.idx]


# ================================================================= drq_gemm_f32
def _gemm_case(L, dev, seed):
    """run one launch of the table twice (NaN / zeros outside every operand's read set) and check it"""
    from drqv2_b200._lib import EPI_MASK_WIDE, EPI_RELU
    g = torch.Generator().manual_seed(seed)
    M, N, K = L.M, L.N, L.K
    nz = L.splitk if L.splitk > 1 else L.batch
    nb = 1 if L.splitk > 1 else L.batch
    a = Poisoned(g, _box(L.a_off, (L.bs[0], L.sa_m, L.sa_k), (nb, M, K), dev), dev)
    b = Poisoned(g, _box(L.b_off, (L.bs[1], L.sb_k, L.sb_n), (nb, K, N), dev), dev)
    bias = Poisoned(g, _box(0, (L.bs[3], 1), (nb, N), dev), dev, lo=-0.1, hi=0.1) if L.bias else None
    mask = Poisoned(g, _box(0, (L.bs[4], L.ldmask, 1), (nb, M, N), dev), dev) if L.ldmask else None
    col = torch.arange(N, device=dev)
    col = S.compact_to_wide(col) if L.epi == EPI_MASK_WIDE else col
    ic = (torch.arange(nz, device=dev).view(nz, 1, 1) * L.bs[2] + torch.arange(M, device=dev).view(1, M, 1) * L.ldc
          + col.view(1, 1, N))
    n_c = nz * L.bs[2] + (M + 1) * L.ldc                   # a spare entry / plane and a spare row
    written = torch.zeros(n_c, dtype=torch.bool, device=dev)
    written[ic.reshape(-1)] = True
    c_old = (torch.rand(n_c, generator=g, dtype=torch.float64) * 2 - 1).float().to(dev)
    outs = []
    for fill in (float("nan"), 0.0):
        C = fill_sentinel(torch.empty(n_c, device=dev))
        if L.acc:
            C[written] = c_old[written]
        bufs = [x.buf(fill) if x is not None else None for x in (a, b, bias, mask)]
        ptr = lambda t: t.data_ptr() if t is not None else None
        # the operand pointers carry their offsets as drqv2 passes them (dc1 + B H, W + w_col0, Q2.0.weight)
        _call("drq_gemm_f32", ptr(bufs[0]) + 4 * L.a_off, L.sa_m, L.sa_k, ptr(bufs[1]) + 4 * L.b_off, L.sb_k, L.sb_n,
              C.data_ptr(), L.ldc,
              ptr(bufs[2]), ptr(bufs[3]), L.ldmask, M, N, K, L.epi, L.acc, L.batch, *L.bs, L.splitk, _s())
        outs.append(C)
    C = outs[0]
    assert_sentinel_outside(C, written, L.name)
    assert torch.equal(C[written], outs[1][written]), f"{L.name}: NaN outside the read set changed the result"
    A64, B64 = a.dense(), b.dense()
    if L.splitk > 1:
        for z, (k0, k1) in enumerate(S.k_ranges(K, L.splitk)):
            want = A64[0, :, k0:k1] @ B64[0, k0:k1]
            absref = A64[0, :, k0:k1].abs() @ B64[0, k0:k1].abs()
            _check("gemm_f32 split plane", C[ic[z]], want, absref, S.gemm_chain(L))
        return
    want, absref = A64 @ B64, A64.abs() @ B64.abs()
    if bias is not None:
        want, absref = want + bias.dense()[:, None, :], absref + bias.dense().abs()[:, None, :]
    if L.epi == EPI_RELU:
        want = want.clamp_min(0)
    elif mask is not None:
        want = torch.where(mask.dense() > 0, want, torch.zeros_like(want))
    if L.acc:
        co = c_old.double()[ic]
        want, absref = want + co, absref + co.abs()
    kind = {0: "none", 1: "relu", 2: "mask", 3: "mask_wide"}[L.epi] + (" acc" if L.acc else "") + \
        (" batch2" if L.batch > 1 else "") + (" a^T" if L.sa_k != 1 else "")
    _check(f"gemm_f32 {kind}", C[ic], want, absref, S.gemm_chain(L))


@pytest.mark.parametrize("B", S.GEMM_BATCHES)
@pytest.mark.parametrize("shape", list(S.SHAPES))
def test_gemm_f32_launch_table(dev, shape, B):
    for i, L in enumerate(S.gemm_launches(B, *S.SHAPES[shape])):
        SUMMARY.append(f"B={B:3d} {shape:9s} " + S.gemm_schedule(L))
        _gemm_case(L, dev, seed=B * 1000 + i)


# ================================================================= drq_colsum_f32
@pytest.mark.parametrize("batch", [1, 2])
@pytest.mark.parametrize("M", S.COLSUM_M)
def test_colsum_f32(dev, M, batch):
    g = torch.Generator().manual_seed(M * 3 + batch)
    for A, F, H in S.SHAPES.values():
        qs = S.q_stride(A, F, H)
        for N in sorted({1, A, F, H}):
            ld = N + 3
            bs_x = M * ld + 5
            x = Poisoned(g, _box(0, (bs_x, ld, 1), (batch, M, N), dev), dev)
            bs_out = qs if batch > 1 else 0
            n_out = batch * (bs_out or N) + N
            io = _box(0, (bs_out, 1), (batch, N), dev)
            written = torch.zeros(n_out, dtype=torch.bool, device=dev)
            written[io.reshape(-1)] = True
            outs = []
            for fill in (float("nan"), 0.0):
                out = fill_sentinel(torch.empty(n_out, device=dev))
                xb = x.buf(fill)
                _call("drq_colsum_f32", xb.data_ptr(), ld, out.data_ptr(), M, N, batch, bs_x, bs_out, _s())
                outs.append(out)
            assert_sentinel_outside(outs[0], written, "colsum_f32")
            assert torch.equal(outs[0][written], outs[1][written])
            X = x.dense()
            _check("colsum_f32", outs[0][io], X.sum(1), X.abs().sum(1), S.colsum_chain(M))


# ================================================================= drq_ln_tanh_fwd (single job) and drq_copy2d_f32
@pytest.mark.parametrize("saved", [True, False], ids=["xhat_rstd", "no_xhat_rstd"])
@pytest.mark.parametrize("F", [50, 256])
@pytest.mark.parametrize("B,S_", S.LN_CASES)
def test_ln_tanh_fwd_single(dev, B, S_, F, saved):
    """the split planes as _trunk_fwd lays them out ([S][B][F], stride B F) and h_out inside [h | action] (ld F + A)"""
    from tests.test_gpu_head_kernels import check_ln_tanh_fwd
    assert S.splitk_for(B) == S_
    A = 38
    g = torch.Generator().manual_seed(B + S_ + F)
    part = torch.full(((S_ + 1) * B * F,), float("nan"), device=dev)      # NaN past the S planes
    p = (torch.rand(S_, B, F, generator=g, dtype=torch.float64) * 2 - 1) / S_ ** 0.5
    part[:S_ * B * F] = p.float().reshape(-1).to(dev)
    bias, gamma, beta = ((torch.rand(F, generator=g, dtype=torch.float64) * 2 - 1).float().to(dev) for _ in range(3))
    h = fill_sentinel(torch.empty(B + 1, F + A, device=dev))
    xhat = fill_sentinel(torch.empty(B * F + 8, device=dev)) if saved else None
    rstd = fill_sentinel(torch.empty(B + 1, device=dev)) if saved else None
    ptr = lambda t: t.data_ptr() if t is not None else None
    _call("drq_ln_tanh_fwd", part.data_ptr(), S_, B * F, bias.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
          h.data_ptr(), F + A, ptr(xhat), ptr(rstd), None, 0, B, F, 1e-5, _s())
    check_ln_tanh_fwd(part[:S_ * B * F].view(S_, B, F).double().cpu(), bias, gamma, beta, h, xhat, rstd, B, F, S_,
                      LN_RATIOS)


@pytest.mark.parametrize("B", [1, 65, 256])
def test_copy2d_f32(dev, B):
    """the action copy into [h | action] (drqv2.py:117): bit-exact, nothing outside the slice written"""
    for A, F, _ in S.SHAPES.values():
        g = torch.Generator().manual_seed(B * A)
        src = torch.full(((B + 1) * A,), float("nan"), device=dev)
        src[:B * A] = (torch.rand(B * A, generator=g) * 2 - 1).to(dev)
        dst = fill_sentinel(torch.empty(B + 1, F + A, device=dev))
        _call("drq_copy2d_f32", src.data_ptr(), A, dst.data_ptr() + 4 * F, F + A, B, A, _s())
        assert torch.equal(dst[:B, F:], src[:B * A].view(B, A))
        w = torch.zeros_like(dst, dtype=torch.bool)
        w[:B, F:] = True
        assert_sentinel_outside(dst, w, "copy2d")


# ================================================================= conv1 forward and weight gradient
def _conv1_input(obs, shift, pad=4):
    """[N][cin][84][84] u8 -> the fp32 values conv1's loader stages (RN(RN(px / 255) - 0.5), replicate pad + shift), as
    fp64"""
    x = torch.sub(torch.div(obs.float(), torch.tensor(255.0)), torch.tensor(0.5))
    xp = torch.nn.functional.pad(x, (pad, pad, pad, pad), mode="replicate")
    N = obs.shape[0]
    out = torch.empty_like(x)
    for n in range(N):
        sx, sy = (int(shift[n, 0]), int(shift[n, 1])) if shift is not None else (pad, pad)
        out[n] = xp[n, :, sy:sy + 84, sx:sx + 84]
    return out.double()


def _conv1_shifts(N, g):
    if N == 81:
        return torch.tensor([(sx, sy) for sy in range(9) for sx in range(9)], dtype=torch.int32)
    return torch.randint(0, 9, (N, 2), generator=g, dtype=torch.int32)


@pytest.mark.parametrize("N,use_shift", [(N, True) for N in S.CONV1_N] + [(5, False)],
                         ids=[f"N{N}" for N in S.CONV1_N] + ["N5_no_shift"])
@pytest.mark.parametrize("cin", S.CONV1_CIN)
def test_conv1_f32(dev, cin, N, use_shift):
    """the update's augmenting loader (N = 81: all 81 shifts) and the act path (shift = NULL); the forward writes
    [0, 1681) of each plane, the weight gradient reads dpre there only"""
    from drqv2_b200 import _lib
    g = torch.Generator().manual_seed(cin * 1000 + N)
    obs = torch.randint(0, 256, (N + 1, cin, 84, 84), dtype=torch.uint8, generator=g)   # a spare image
    shift = _conv1_shifts(N, g) if use_shift else None
    w = torch.full((32 * cin * 9 + 16,), float("nan"))
    w[:32 * cin * 9] = (torch.rand(32 * cin * 9, generator=g) * 2 - 1) * 0.2
    b = torch.full((40,), float("nan"))
    b[:32] = (torch.rand(32, generator=g) * 2 - 1) * 0.1
    obs_d, w_d, b_d = obs.to(dev), w.to(dev), b.to(dev)
    sh_d = shift.to(dev) if shift is not None else None
    out = fill_sentinel(torch.empty(N + 1, 32, PLANE, device=dev))
    _call("drq_conv1_fwd_f32", obs_d.data_ptr(), sh_d.data_ptr() if sh_d is not None else None, w_d.data_ptr(),
          b_d.data_ptr(), out.data_ptr(), N, cin, 4, _s())
    assert_sentinel_outside(out, S.plane_written(N + 1, N, 0, 41 * 41).to(dev), "conv1_fwd_f32")
    x = _conv1_input(obs[:N], shift).to(dev)
    wd, bd = w[:32 * cin * 9].double().view(32, cin, 3, 3).to(dev), b[:32].double().to(dev)
    want = torch.relu(torch.nn.functional.conv2d(x, wd, bd, stride=2))
    absref = torch.nn.functional.conv2d(x.abs(), wd.abs(), bd.abs(), stride=2)
    got = out[:N, :, :41 * 41].view(N, 32, 41, 41)
    _check("conv1_fwd_f32", got, want, absref, 9 * cin + 1)
    SUMMARY.append(f"conv1 cin={cin:2d} N={N:3d}: wgrad {S.conv1_wgrad_schedule(N)}")
    # weight gradient: dpre read on [0, 1681) of each plane only
    d = torch.rand(N, 32, 41, 41, generator=g, dtype=torch.float64) * 2 - 1
    outs = []
    for fill in (float("nan"), 0.0):
        dpre = torch.full((N, 32, PLANE), fill, device=dev)
        dpre[:, :, :41 * 41] = d.float().reshape(N, 32, -1).to(dev)
        part = fill_sentinel(torch.empty(int(_lib.lib().drq_conv_wgrad_ws_floats(cin)), device=dev))
        dw = fill_sentinel(torch.empty(32 * cin * 9 + 8, device=dev))
        db = fill_sentinel(torch.empty(40, device=dev))
        _call("drq_conv1_wgrad_f32", obs_d.data_ptr(), sh_d.data_ptr() if sh_d is not None else None, dpre.data_ptr(),
              part.data_ptr(), dw.data_ptr(), db.data_ptr(), N, cin, 4, _s())
        outs.append((dw, db))
    (dw, db), (dw0, db0) = outs
    nw = 32 * cin * 9
    assert torch.equal(dw[:nw], dw0[:nw]) and torch.equal(db[:32], db0[:32]), "conv1_wgrad read dpre past [0, 1681)"
    _wr = lambda n, size: torch.arange(size, device=dev) < n
    assert_sentinel_outside(dw, _wr(nw, dw.numel()), "conv1_wgrad dw")
    assert_sentinel_outside(db, _wr(32, 40), "conv1_wgrad db")
    dd = d.float().double().to(dev)
    cw = lambda xx, dy: torch.nn.grad.conv2d_weight(xx, (32, cin, 3, 3), dy, stride=2)
    n_chain = S.conv1_wgrad_chain(N)
    _check("conv1_wgrad_f32 dw", dw[:nw].view(32, cin, 3, 3), cw(x, dd), cw(x.abs(), dd.abs()), n_chain)
    _check("conv1_wgrad_f32 db", db[:32], dd.sum((0, 2, 3)), dd.abs().sum((0, 2, 3)), n_chain)


# ================================================================= conv2-4: forward, data gradient, weight gradient
def _wide(vals, N, fill, dev):
    """[N][32][h][w] values into a wide [N][32][PLANE] buffer holding `fill` everywhere else"""
    h, w = vals.shape[2:]
    buf = torch.full((N, 32, 41, 41), fill, device=dev)
    buf[:, :, :h, :w] = vals.float().to(dev)
    out = torch.full((N, 32, PLANE), fill, device=dev)
    out[:, :, :41 * 41] = buf.view(N, 32, -1)
    return out


def _weights(g, dev):
    w = torch.full((32 * 32 * 9 + 16,), float("nan"))
    w[:9216] = (torch.rand(9216, generator=g) * 2 - 1) * 0.1
    b = torch.full((40,), float("nan"))
    b[:32] = (torch.rand(32, generator=g) * 2 - 1) * 0.1
    return w.to(dev), b.to(dev), w[:9216].double().view(32, 32, 3, 3).to(dev), b[:32].double().to(dev)


@pytest.mark.parametrize("N", S.CONV_N)
@pytest.mark.parametrize("hout", S.CONV_HOUT)
def test_conv3x3_fwd_f32(dev, hout, N):
    g = torch.Generator().manual_seed(hout * 1000 + N)
    hin = hout + 2
    x = torch.rand(N, 32, hin, hin, generator=g, dtype=torch.float64).float()
    w, b, wd, bd = _weights(g, dev)
    xd = x.double().to(dev)
    want = torch.relu(torch.nn.functional.conv2d(xd, wd, bd))
    absref = torch.nn.functional.conv2d(xd.abs(), wd.abs(), bd.abs())
    valid = {}
    for fill in (float("nan"), 0.0):                   # outside hin x hin: NaN, then zeros
        inp = _wide(x, N, fill, dev)
        wide = fill_sentinel(torch.empty(N + 1, 32, PLANE, device=dev))
        _call("drq_conv3x3_fwd_f32", inp.data_ptr(), w.data_ptr(), b.data_ptr(), wide.data_ptr(), N, hout, 0, _s())
        compact = fill_sentinel(torch.empty(N + 1, 32, hout, hout, device=dev))
        _call("drq_conv3x3_fwd_f32", inp.data_ptr(), w.data_ptr(), b.data_ptr(), compact.data_ptr(), N, hout, 1, _s())
        assert_sentinel_outside(wide, S.plane_written(N + 1, N, 0, hout * PW).to(dev), "conv3x3_fwd wide")
        wc = torch.zeros_like(compact, dtype=torch.bool)
        wc[:N] = True
        assert_sentinel_outside(compact, wc, "conv3x3_fwd compact")
        got = wide[:N, :, :hout * PW].view(N, 32, hout, PW)[..., :hout]
        assert torch.equal(got, compact[:N]), "compact_out != the valid columns of the wide output"
        valid[fill == 0.0] = got.clone()
    assert torch.equal(valid[False], valid[True]), "NaN outside hin x hin changed a valid output"
    _check("conv3x3_fwd_f32", valid[False], want, absref, 288 + 1)


@pytest.mark.parametrize("N", S.CONV_N)
@pytest.mark.parametrize("hout", S.CONV_HOUT)
def test_conv3x3_dgrad_f32(dev, hout, N):
    """dout: valid hout x hout, +0 in rows hout, hout + 1 and columns >= hout, NaN past row hout + 1 (slack included);
    act_in NaN outside hin x hin"""
    g = torch.Generator().manual_seed(hout * 1000 + N + 7)
    hin = hout + 2
    d = (torch.rand(N, 32, hout, hout, generator=g, dtype=torch.float64) * 2 - 1).float()
    act = torch.relu(torch.rand(N, 32, hin, hin, generator=g, dtype=torch.float64) * 2 - 0.6).float()
    w, _, wd, _ = _weights(g, dev)
    outs = []
    for fill in (float("nan"), 0.0):
        dout = _wide(d, N, 0.0, dev)
        dout.view(N, 32, -1)[:, :, hin * PW:] = fill
        act_in = _wide(act, N, fill, dev)
        din = fill_sentinel(torch.empty(N + 1, 32, PLANE, device=dev))
        _call("drq_conv3x3_dgrad_f32", dout.data_ptr(), w.data_ptr(), act_in.data_ptr(), din.data_ptr(), N, hout, _s())
        outs.append(din)
    din = outs[0]
    written = S.dgrad_written(N + 1, N, hout).to(dev)
    assert_sentinel_outside(din, written, "conv3x3_dgrad")
    flat = din.view(-1)
    assert torch.equal(flat[written], outs[1].view(-1)[written]), "NaN outside the read extent changed din"
    rows = din[:N, :, :hin * PW].view(N, 32, hin, PW)
    assert bool((rows[..., hin:].view(torch.int32) == 0).all()), "columns >= hout + 2 are not +0"
    dd, ad = d.double().to(dev), act.double().to(dev)
    want = torch.where(ad > 0, torch.nn.functional.conv_transpose2d(dd, wd), torch.zeros_like(ad))
    absref = torch.nn.functional.conv_transpose2d(dd.abs(), wd.abs())
    _check("conv3x3_dgrad_f32", rows[..., :hin], want, absref, 288)


@pytest.mark.parametrize("N", S.CONV_N)
@pytest.mark.parametrize("hout", S.CONV_HOUT)
def test_conv3x3_wgrad_f32(dev, hout, N):
    """dpre: valid hout x hout, +0 at columns >= hout within [0, hout 41), NaN past it; in: 2^100 outside hin x hin
    (slack included) - dw / db must equal a run with zeros in both places"""
    from drqv2_b200 import _lib
    g = torch.Generator().manual_seed(hout * 1000 + N + 11)
    hin = hout + 2
    x = torch.rand(N, 32, hin, hin, generator=g, dtype=torch.float64).float()
    d = (torch.rand(N, 32, hout, hout, generator=g, dtype=torch.float64) * 2 - 1).float()
    outs = []
    for big, fill in ((BIG, float("nan")), (0.0, 0.0)):
        inp = _wide(x, N, big, dev)
        dpre = _wide(d, N, 0.0, dev)
        dpre.view(N, 32, -1)[:, :, hout * PW:] = fill
        part = fill_sentinel(torch.empty(int(_lib.lib().drq_conv_wgrad_ws_floats(32)), device=dev))
        dw = fill_sentinel(torch.empty(9216 + 8, device=dev))
        db = fill_sentinel(torch.empty(40, device=dev))
        _call("drq_conv3x3_wgrad_f32", inp.data_ptr(), dpre.data_ptr(), part.data_ptr(), dw.data_ptr(), db.data_ptr(),
              N, hout, _s())
        outs.append((dw, db))
    (dw, db), (dw0, db0) = outs
    assert torch.equal(dw[:9216], dw0[:9216]) and torch.equal(db[:32], db0[:32]), \
        "finite values outside hin x hin or NaN past hout rows of dpre changed dw / db"
    assert_sentinel_outside(dw, torch.arange(dw.numel(), device=dev) < 9216, "conv3x3_wgrad dw")
    assert_sentinel_outside(db, torch.arange(40, device=dev) < 32, "conv3x3_wgrad db")
    SUMMARY.append(f"conv3x3 wgrad hout={hout} N={N:3d}: {S.wgrad3_schedule(N, hout)}")
    xd, dd = x.double().to(dev), d.double().to(dev)
    cw = lambda xx, dy: torch.nn.grad.conv2d_weight(xx, (32, 32, 3, 3), dy)
    n_chain = S.wgrad3_chain(N, hout)
    _check("conv3x3_wgrad_f32 dw", dw[:9216].view(32, 32, 3, 3), cw(xd, dd), cw(xd.abs(), dd.abs()), n_chain)
    _check("conv3x3_wgrad_f32 db", db[:32], dd.sum((0, 2, 3)), dd.abs().sum((0, 2, 3)), n_chain)


# ================================================================= the fp32 escape hatch, end to end
def test_update_fp32_at_the_shape_only_fp32_runs(dev):
    """16 stacked channels, A = 129, F = 256, H = 1020 (every one refused or never reached by the tensor-core mode) at
    B = 65: two M tiles, S = 145 split planes, up to three weight-gradient tiles per block.  Then the wide-plane
    positions the fp32 backward reads but no kernel writes must still hold +0.0 (include/drqv2_b200.h: the data
    gradient's zero rows, the weight gradient's finite input)"""
    from drqv2_b200 import DrQV2Agent
    from oracle import drq_oracle as O
    from tests import test_gpu_parity as parity
    torch.set_num_threads(max(8, torch.get_num_threads()))
    C, A, F, H, B, lr = 16, 129, 256, 1020, 65, 1e-4
    assert S.splitk_for(B) == 145 and S.wgrad3_schedule(B, 39)["tpb_max"] == 3
    params = O.synthetic_params(C, A, F, H, seed=4)
    agent = DrQV2Agent((C, 84, 84), (A,), "cuda", lr, F, H, 0.01, 2000, 2, parity.SCHED, 0.3, True,
                       use_cuda_graph=False, seed=5, mode="fp32")
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    o32 = O.OracleAgent(params, lr, 0.01, parity.SCHED, 0.3, dtype=torch.float32)
    o64 = O.OracleAgent(params, lr, 0.01, parity.SCHED, 0.3, dtype=torch.float64)
    b = O.synthetic_batch(B, A, cin=C, seed=12)
    m_gpu = parity.run_update(agent, b, 0)
    args = (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 0, b["shift_obs"], b["shift_next"],
            b["eps_critic"], b["eps_actor"])
    m32, m64 = o32.update(*args), o64.update(*args)
    parity._check_update_against_oracle(agent, o32, o64, b, 0, lr, m_gpu, m32, m64)
    ws = agent.workspace(B)
    zero = lambda t, what: bool((t.contiguous().view(torch.int32) == 0).all()) or pytest.fail(f"{what} is not +0.0")
    dpre = [t.view(B, 32, PLANE) for t in ws.dpre]
    acts = [t.view(2 * B, 32, PLANE) for t in ws.acts]
    d3 = dpre[3][:, :, :41 * 41].reshape(B, 32, 41, 41)
    zero(d3[:, :, :, 35:], "dpre[3] columns >= 35")
    zero(d3[:, :, 35:, :], "dpre[3] rows >= 35")
    zero(dpre[3][:, :, 41 * 41:], "dpre[3] slack")
    zero(dpre[2][:, :, 37 * PW:39 * PW], "dpre[2] rows 37-38")
    zero(dpre[1][:, :, 39 * PW:41 * PW], "dpre[1] rows 39-40")
    zero(acts[0][:, :, 41 * 41:], "acts[0] slack")
    zero(acts[1][:, :, 39 * PW:], "acts[1] past row 38")
    zero(acts[2][:, :, 37 * PW:], "acts[2] past row 36")


def test_fp32_constructor_refuses_feature_dim_past_the_layernorm_kernels(dev):
    from drqv2_b200 import DrQV2Agent
    with pytest.raises(ValueError, match="F <= 256"):
        DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 257, 256, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, True,
                   mode="fp32")
