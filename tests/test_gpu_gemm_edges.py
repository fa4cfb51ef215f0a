"""Every instantiation of the tensor-core GEMM (drq_gemm_bf16, csrc/gemm_tc.cu) at the edges of its schedule, against
fp64 math on the bf16-rounded operands.

The launch table (tests/test_gemm_schedule_cpu.launches) restates the calls of twin_q_layers, actor_mlp_fwd,
critic_pass, _actor_pass and act_body with their modes, tiles, epilogues, batch_inner, inner / outer batch strides (the
negative outer weight stride of the merged trunk forward included), split-K and masks, at the update shapes (walker
B=256 A=6 F=50 H=1024, humanoid shard B=512 A=21 F=100 H=1024) and at odd ones (B = 1, 129, 200; A = 1, 32; H = 256).
Each runs at SM budgets 148, 140, 7, 2 and 1 (drq_set_sm_limit): from a 3-D grid of one tile per CTA down to one CTA
that runs every tile, so the operand ring, the TMEM accumulator ring and the bias double buffer wrap on every tile
boundary.  The four SMALL (two-stage) variants run at every budget too and must equal the normal variant bit for bit.
Each case prints its schedule from the CPU model.

Checks:
  - bf16 epilogues (RELU, MASK, TRUNK_DGRAD): |got - want| <= 2^-8 |want| + 2^-14 A (tests/helpers.assert_conv_bound);
  - fp32 epilogues (F32, TRUNK_WGRAD, split-K planes): |got - want| <= C_F32 2^-24 ceil(K_chunk / 16) A
    (tests/helpers.assert_f32_bound), A = the same GEMM on |operands| plus |bias|.  Split planes hold their chunk's sum
    without the bias;
  - every output is one size too big and starts as a NaN sentinel: fp32 outputs have a row past M, ldc > N padding
    columns, a spare batch entry / split plane; TB outputs a spare entry and spare units; whatever the launch must not
    write keeps the sentinel.  TB columns [N, n_store) are exact zeros;
  - the read contract of include/drqv2_b200.h: every operand holds NaN past its read extent (K-major: features past
    ceil(K/16)*16; MN-major: rows past ceil(K/16)*16 of the 128-row block) and past the rows / features that reach only
    unstored outputs, and rows [K, ceil(K/16)*16) of MN-major operands are zero; the result must not change when those
    NaN are zeros."""
import copy
import math
import zlib

import pytest
import torch

from tests import test_gemm_schedule_cpu as S
from tests.helpers import (assert_conv_bound, assert_f32_bound, assert_sentinel_outside, bits_equal, fill_sentinel,
                           wb_cs, wb_region, wb_written)

pytestmark = pytest.mark.gpu

# fp32 outputs: the accumulation error in units of 2^-24 * ceil(K_chunk / 16) * A.  Measured on one B200 (1,000 W power
# limit) over the whole table: at most 0.63 (KK128_F32; KK64_F32 0.56, TRUNK_WGRAD 0.23, KMN64_F32 0.22, MNMN 0.15-0.17).
# C_F32 = 2 leaves about 3x that (DESIGN.md §2).
C_F32 = 2.0
RATIOS = {}          # (instantiation, check) -> largest ratio observed
SUMMARY = []


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if SUMMARY:
        print("\nschedules run:\n  " + "\n  ".join(SUMMARY))
        print("largest ratio per instantiation (bf16: |got - want| / bound; fp32: the c needed):")
        for k, v in sorted(RATIOS.items()):
            print(f"  {k[0]:24s} {k[1]:5s} {v:.4f}")


@pytest.fixture
def sm_budget(request):
    """drq_set_sm_limit(request.param) for the test, the previous limit restored after it"""
    from drqv2_b200 import _lib
    prev = _lib.lib().drq_device_sm_count()
    _lib.call("drq_set_sm_limit", request.param)
    try:
        yield request.param
    finally:
        _lib.call("drq_set_sm_limit", prev)


@pytest.fixture
def gemm_small():
    """a setter of drq_set_gemm_small; the library default (off, its value outside the actor pass) is restored after
    the test"""
    from drqv2_b200 import _lib
    try:
        yield lambda on: _lib.call("drq_set_gemm_small", int(on))
    finally:
        _lib.call("drq_set_gemm_small", 0)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _note(inst, kind, r):
    k = (S.inst_name(inst), kind)
    RATIOS[k] = max(RATIOS.get(k, 0.0), r)


# ---------------------------------------------------------------- operands
class Operand:
    """one TB buffer of `n` entries of `rows` rows (row block rblk) and `feats` features + 2 spare units; entry e's
    matrix starts at row e * rows.  `dense` is the fp64 content with NaN -> 0, `flat` the bf16 buffer."""

    def __init__(self, g, dev, n, rows, rblk, feats, used, kmajor, K):
        """used: (row0, nrows, nfeats) regions of the entries; kmajor: contraction over features (K of them), else over
        rows (K of each region)"""
        self.rows, self.rblk = rows, rblk
        self.units = S._ceil(feats, 16) // 8 + 2
        W = self.units * 8
        d = torch.full((n * rows, W), float("nan"), dtype=torch.float64)
        for r0, nr, nf in used:
            v = (torch.rand(nr, nf, generator=g, dtype=torch.float64) * 2 - 1).to(torch.bfloat16).double()
            v[v.abs() < 0.02] = 0.0                                   # exact zeros (mask > 0 is strict)
            d[r0:r0 + nr, :nf] = v
            if kmajor:
                d[r0:r0 + nr, K:S._ceil(K, 16)] = 0.0                 # inside the read extent: zero padding
            else:
                d[r0 + K:r0 + S._ceil(K, 16), :] = 0.0
        if kmajor:
            d[:, S._ceil(K, 16):] = float("nan")                      # past the read extent
        self.dense = torch.nan_to_num(d, nan=0.0).to(dev)
        blocks = n * rows // rblk
        self.flat = d.to(torch.bfloat16).view(blocks, rblk, self.units, 8).permute(0, 2, 1, 3).contiguous().view(-1).to(dev)
        self.entry = rows * self.units * 8                            # elements per entry

    def ptr(self, e):
        return self.flat.data_ptr() + 2 * e * self.entry

    def clean(self):
        """the same operand with zeros where this one holds NaN"""
        c = copy.copy(self)
        c.flat = torch.nan_to_num(self.flat, nan=0.0)
        return c

    def mat(self, e, nrows, nfeats):
        return self.dense[e * self.rows:e * self.rows + nrows, :nfeats]


def _entries(place, batch, inner):
    """(zi, zo) -> entry index of an operand placed as (entries, base, inner stride, outer stride)"""
    _, base, si, so = place
    return {(zb % inner, zb // inner): base + (zb % inner) * si + (zb // inner) * so for zb in range(batch)}


class Case:
    """operands, references and output geometry of one launch of the table"""

    def __init__(self, key, dev):
        shape, name = key
        s = S.all_launches()[key]
        self.key, self.s = key, s
        mode, bn, epi, _ = s["inst"]
        M, N, K, batch, inner, sk = s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"]
        g = torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))
        ea, eb = _entries(s["a"], batch, inner), _entries(s["b"], batch, inner)
        # A: K-major activation [M][K] or MN-major activation [K rows][M]
        if mode == S.MNMN:
            ra = S._ceil(K, S.RA)
            self.A = Operand(g, dev, s["a"][0], ra, S.RA, M, [(e * ra, K, M) for e in set(ea.values())], False, K)
        else:
            ra = S._ceil(M, S.RA)
            self.A = Operand(g, dev, s["a"][0], ra, S.RA, K, [(e * ra, M, K) for e in set(ea.values())], True, K)
        if mode == S.KK:
            rb = s["b_rows"] or S._ceil(N, S.RW)
            self.B = Operand(g, dev, s["b"][0], rb, S.RW, K, [(e * rb, N, K) for e in set(eb.values())], True, K)
        elif mode == S.KMN:
            rb = S._ceil(K, S.RW)
            self.B = Operand(g, dev, s["b"][0], rb, S.RW, N, [(e * rb, K, N) for e in set(eb.values())], False, K)
        else:
            rb = S._ceil(K, S.RA)
            self.B = Operand(g, dev, s["b"][0], rb, S.RA, N, [(e * rb, K, N) for e in set(eb.values())], False, K)
        self.ea, self.eb = ea, eb
        self.mask = self.em = None
        if s["mask"]:
            self.em = _entries(s["mask"], batch, inner)
            rm = S._ceil(M, S.RA)
            self.mask = Operand(g, dev, s["mask"][0], rm, S.RA, N, [(e * rm, M, N) for e in set(self.em.values())], True, N)
        self.bias = self.eb_bias = None
        if s["bias"]:
            self.eb_bias = _entries(s["bias"], batch, inner)
            self.bias_w = N + 5
            bias = torch.full((s["bias"][0], self.bias_w), float("nan"), dtype=torch.float64)
            bias[:, :N] = torch.rand(s["bias"][0], N, generator=g, dtype=torch.float64) * 2 - 1
            self.bias = bias.float().to(dev)
        # the references, per (zi, zo, zs)
        ch = S.k_chunk(K, sk)
        self.chunks = [(zs * ch, min(K, (zs + 1) * ch)) for zs in range(sk)]
        self.want, self.absref = {}, {}
        for (zi, zo) in ea:
            Am, Bn = self._canon(zi, zo)
            for zs, (k0, k1) in enumerate(self.chunks):
                x, y = Am[:, k0:k1], Bn[:, k0:k1]
                w, a = x @ y.T, x.abs() @ y.abs().T
                if self.bias is not None and sk == 1:
                    b = self.bias[self.eb_bias[zi, zo], :N].double()
                    w, a = w + b, a + b.abs()
                if epi == S.RELU:
                    w = torch.relu(w)
                if epi in (S.MASK, S.TDGRAD):
                    keep = (self._mask(zi, zo) > 0).double()
                    w, a = w * keep, a * keep
                self.want[zi, zo, zs], self.absref[zi, zo, zs] = w, a

    def _canon(self, zi, zo):
        s = self.s
        mode = s["inst"][0]
        M, N, K = s["M"], s["N"], s["K"]
        a, b = self.ea[zi, zo], self.eb[zi, zo]
        Am = self.A.mat(a, M, K) if mode != S.MNMN else self.A.mat(a, K, M).T
        Bn = self.B.mat(b, N, K) if mode == S.KK else self.B.mat(b, K, N).T
        return Am, Bn

    def _mask(self, zi, zo):
        return self.mask.mat(self.em[zi, zo], self.s["M"], self.s["N"])

    # ---- one launch into a fresh sentinel output; returns the output buffer
    def run(self, A=None, B=None):
        from drqv2_b200 import _lib
        from drqv2_b200._bf16 import _strides
        s = self.s
        mode, bn, epi, _ = s["inst"]
        M, N, K, batch, inner, sk = s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"]
        dev = self.A.flat.device
        A, B = A or self.A, B or self.B
        ci, co, csp = s["c"]
        n_store = 0
        if epi in (S.F32, S.TWGRAD):
            self.ldc = ldc = N + 3 if epi == S.F32 else N + 8
            self.R = R = (M + 1) * ldc
            nreg = max(zi * ci + zo * co + zs * csp for (zi, zo) in self.ea for zs in range(sk)) + 2
            out = fill_sentinel(torch.empty(nreg * R, dtype=torch.float32, device=dev))
            cst = (ci * R, co * R, csp * R)
        elif epi in (S.RELU, S.MASK):
            self.rc = S._ceil(M, S.RA)
            self.uc = ldc = S._ceil(N, 16) // 8 + 2
            self.R = R = self.rc * ldc * 8
            nreg = max(zi * ci + zo * co for (zi, zo) in self.ea) + 2
            out = fill_sentinel(torch.empty(nreg * R, dtype=torch.bfloat16, device=dev))
            cst = (ci * R, co * R, 0)
            n_store = s.get("n_store", 0)
        else:                                                          # TRUNK_DGRAD: conv4's WB gradient, one image spare
            ldc = wb_cs(M)
            out = fill_sentinel(torch.empty(4 * ldc * 8 + 1776 * 8, dtype=torch.bfloat16, device=dev))
            cst = (0, 0, 0)
        pa, pb = s["a"], s["b"]
        ent = lambda op, p: (p[2] * op.entry, p[3] * op.entry)
        ai, ao = ent(A, pa)
        bi, bo = ent(B, pb)
        bias_p, bsi, bso = None, 0, 0
        if self.bias is not None:
            bias_p = self.bias.data_ptr() + 4 * s["bias"][1] * self.bias_w
            bsi, bso = s["bias"][2] * self.bias_w, s["bias"][3] * self.bias_w
        mask_p, mi, mo, mu = None, 0, 0, 0
        if self.mask is not None:
            mask_p = self.mask.ptr(s["mask"][1])
            mi, mo = ent(self.mask, s["mask"])
            mu = self.mask.units
        st = _strides((ai, bi, cst[0], bsi, mi), (ao, bo, cst[1], bso, mo), cst[2])
        _lib.call("drq_gemm_bf16", A.ptr(pa[1]), A.units, B.ptr(pb[1]), B.units, mode, out.data_ptr(), ldc, n_store,
                  bias_p, mask_p, mu, M, N, K, epi, 0, batch, inner, st, sk, bn, _stream())
        torch.cuda.synchronize()
        return out

    # ---- the checks
    def check(self, out):
        s = self.s
        inst = s["inst"]
        mode, bn, epi, _ = inst
        M, N, sk = s["M"], s["N"], s["splitk"]
        ci, co, csp = s["c"]
        what = f"{self.key} {S.inst_name(inst)}"
        written = torch.zeros(out.numel(), dtype=torch.bool, device=out.device)
        for (zi, zo, zs), w in self.want.items():
            a = self.absref[zi, zo, zs]
            k0, k1 = self.chunks[zs]
            if epi == S.F32:
                off = (zi * ci + zo * co + zs * csp) * self.R
                got = out[off:off + self.R].view(M + 1, self.ldc)[:M, :N]
                written[off:off + self.R].view(M + 1, self.ldc)[:M, :N] = True
                _note(inst, "fp32", assert_f32_bound(got, w, a, math.ceil((k1 - k0) / 16), C_F32, f"{what} {zi, zo, zs}"))
            elif epi == S.TWGRAD:
                got = out[:self.R].view(M + 1, self.ldc)[:M, :N]
                written[:self.R].view(M + 1, self.ldc)[:M, :N] = True
                ref = lambda x: x.view(M, 4, 1225, 8).permute(0, 1, 3, 2).reshape(M, N)   # encoder order -> reference order
                _note(inst, "fp32", assert_f32_bound(got, ref(w), ref(a), math.ceil((k1 - k0) / 16), C_F32, what))
            elif epi in (S.RELU, S.MASK):
                off = (zi * ci + zo * co) * self.R
                ent = out[off:off + self.R].view(self.rc // S.RA, self.uc, S.RA, 8).permute(0, 2, 1, 3).reshape(self.rc, -1)
                wcols = S._ceil(max(N, s.get("n_store", 0)), 8)
                wm = torch.zeros(self.rc, self.uc * 8, dtype=torch.bool, device=out.device)
                wm[:M, :wcols] = True                                  # rows < M, whole units below n_store
                written[off:off + self.R] = wm.view(self.rc // S.RA, S.RA, self.uc, 8).permute(0, 2, 1, 3).reshape(-1)
                r, _ = assert_conv_bound(ent[:M, :N].float(), w, a, what)
                _note(inst, "bf16", r)
                assert torch.count_nonzero(ent[:M, N:wcols].float()) == 0, what + ": columns [N, n_store) not zero"
            else:                                                      # TRUNK_DGRAD
                got = wb_region(out, M, 35, 35)
                to_nchw = lambda x: x.view(M, 4, 1225, 8).permute(0, 1, 3, 2).reshape(M, 32, 35, 35)
                r, _ = assert_conv_bound(got, to_nchw(w), to_nchw(a), what)
                _note(inst, "bf16", r)
                written = wb_written(out.numel(), M, 35, 35, out.device)
        assert_sentinel_outside(out, written, what)


_CACHE = {}


def _case(key, dev):
    if key not in _CACHE:
        _CACHE.clear()
        _CACHE[key] = Case(key, dev)
    return _CACHE[key]


KEYS = list(S.all_launches())
PARAMS = [(k, b) for k in KEYS for b in S.BUDGETS]


@pytest.mark.parametrize("key,sm_budget", PARAMS, indirect=["sm_budget"],
                         ids=[f"{k[0]}-{k[1]}-{b}" for k, b in PARAMS])
def test_gemm_instantiation_at_budget(dev, key, sm_budget, gemm_small):
    c = _case(key, dev)
    s = c.s
    out = c.run()
    c.check(out)
    sch = S.schedule(s["inst"], s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"], sm_budget)
    SUMMARY.append(f"{key[0]:8s} {key[1]:20s} {S.inst_name(s['inst']):22s} @{sm_budget:3d}: {S.fmt_schedule(sch)}")
    if s["small_ok"]:
        gemm_small(1)
        small = c.run()
        gemm_small(0)
        assert bits_equal(small, out) if small.dtype == torch.bfloat16 else \
            torch.equal(small.view(torch.int32), out.view(torch.int32)), f"{key}: SMALL variant differs"
        small_inst = s["inst"][:3] + (1,)
        sch = S.schedule(small_inst, s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"], sm_budget)
        SUMMARY.append(f"{key[0]:8s} {key[1]:20s} {S.inst_name(small_inst):22s} @{sm_budget:3d}: {S.fmt_schedule(sch)}")


@pytest.mark.parametrize("name", sorted(S.launches("b200")))
def test_nan_past_the_read_extent_changes_nothing(dev, name, gemm_small):
    """the same launch on operands whose NaN past the read extent are zeros gives the same bits (b200: the MN-major
    contraction ends 8 rows into a 16-row UMMA step)"""
    c = _case(("b200", name), dev)
    out = c.run()
    assert torch.isnan(c.A.flat.float()).any() and torch.isnan(c.B.flat.float()).any()
    ref = c.run(c.A.clean(), c.B.clean())
    view = (lambda t: t.view(torch.int32)) if out.dtype == torch.float32 else (lambda t: t.view(torch.int16))
    assert torch.equal(view(out), view(ref)), f"{name}: NaN past the read extent changed the result"
    if c.s["small_ok"]:
        gemm_small(1)
        small = c.run()
        gemm_small(0)
        assert torch.equal(view(small), view(ref)), f"{name} SMALL: NaN past the read extent changed the result"


def test_n_store_past_the_last_tile_is_refused(dev):
    """columns [N, n_store) are zero-filled by the tiles of N; an n_store past the last tile would leave columns unwritten"""
    from drqv2_b200 import _lib
    c = _case(("b200", "linear_bn128"), dev)
    s = c.s
    out = fill_sentinel(torch.empty(4 * c.A.entry, dtype=torch.bfloat16, device=dev))
    N = s["N"]
    with pytest.raises(_lib.DrqError, match="n_store"):
        _lib.call("drq_gemm_bf16", c.A.ptr(0), c.A.units, c.B.ptr(0), c.B.units, S.KK, out.data_ptr(), S._ceil(N, 16) // 8 + 4,
                  S._ceil(N, 128) + 8, c.bias.data_ptr(), None, 0, s["M"], N, s["K"], S.RELU, 0, 1, 1, None, 1, 128, _stream())
