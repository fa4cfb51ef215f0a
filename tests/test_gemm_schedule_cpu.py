"""A CPU model of the tensor-core GEMM's launch (csrc/gemm_tc.cu: launch_gemm_tc, tile_info, GemmCfg) and the launch
table of the GPU edge tests (tests/test_gpu_gemm_edges.py), checked without a GPU:

  - every (m tile, n tile, batch entry, split chunk) of every launch in the table is visited exactly once, by the 3-D
    grid or by the persistent 1-D grid, at every SM budget the GPU tests run;
  - the split-K chunking of the trunk forwards as the update issues them ends in a 32-column chunk;
  - the fp32 bound and the sentinels of the GPU tests accept a correct result and reject planted defects: a zeroed
    small element of the last partial m tile (which the older max-normalised bound accepts), a missing split plane,
    swapped inner and outer batch entries, a bias added to every split plane, and stores into row M or a spare plane.

The GPU tests print each case's schedule from `schedule()` below."""
import itertools
import math

import pytest
import torch

from tests.helpers import assert_f32_bound, assert_sentinel_outside, fill_sentinel, max_norm_ok

KK, KMN, MNMN = 0, 1, 2
F32, RELU, MASK, TWGRAD, TDGRAD = 0, 1, 2, 3, 4
RA, RW, BM = 128, 64, 128
REPR = 39200
BUDGETS = (148, 140, 7, 2, 1)

# every GT_SMALL / GT_CASE line of drq_gemm_bf16: (mode, bn, epilogue, small)
SMALL_INSTS = [(KK, 64, F32, 1), (KK, 64, RELU, 1), (KMN, 64, F32, 1), (KMN, 64, MASK, 1)]
NORMAL_INSTS = [(KK, 64, F32, 0), (KK, 64, RELU, 0), (KK, 128, F32, 0), (KK, 128, RELU, 0), (KMN, 64, F32, 0),
                (KMN, 64, MASK, 0), (KMN, 128, MASK, 0), (KMN, 128, TDGRAD, 0), (MNMN, 64, F32, 0), (MNMN, 128, F32, 0),
                (MNMN, 128, TWGRAD, 0)]
INSTANTIATIONS = SMALL_INSTS + NORMAL_INSTS
EPI_NAMES = {F32: "F32", RELU: "RELU", MASK: "MASK", TWGRAD: "TRUNK_WGRAD", TDGRAD: "TRUNK_DGRAD"}
MODE_NAMES = {KK: "KK", KMN: "KMN", MNMN: "MNMN"}


def inst_name(inst):
    mode, bn, epi, small = inst
    return f"{MODE_NAMES[mode]}{bn}_{EPI_NAMES[epi]}" + ("_SMALL" if small else "")


def stages(mode, bn, epi, small):
    """GemmCfg<MODE, BN, EPI, SMALL>::STAGES"""
    a_bytes = 16 * RA * 16 if mode == MNMN else 8 * RA * 16
    b_bytes = 8 * bn * 16 if mode == KK else (bn // 8) * (RW if mode == KMN else RA) * 16
    xp = 32 * (bn + 1) if epi == TWGRAD else (32 * 33 if epi == F32 else 0)
    budget = 196 * 1024 - (2 * bn * 4 + 4 * xp * 4)
    return 2 if small else min(6, budget // (a_bytes + b_bytes))


def k_chunk(K, splitk):
    """drq_gemm_bf16: the split-K chunk (a multiple of 128 columns); every chunk must be non-empty"""
    if splitk == 1:
        return K
    chunk = -(-(-(-K // splitk)) // 128) * 128
    assert chunk * (splitk - 1) < K, "empty split chunk"
    return chunk


def splitk_for(ctas_per_split, K=REPR, target_blocks=148):
    """drqv2_b200._bf16.splitk_for"""
    s0 = max(1, min(target_blocks // max(1, ctas_per_split), K // 128))
    chunk = -(-K // s0)
    chunk = -(-chunk // 128) * 128
    return -(-K // chunk)


def tile_info(t, nt, mt, splitk, batch_inner, grid3d, block=None):
    """tile_info<BN>: (m tile, n tile, inner batch entry, outer batch entry, split chunk) of tile t (or block (x, y, z))"""
    if grid3d:
        i_n, i_m, z = block
    else:
        i_m, z = 0, 0
        if nt > 1:
            rest = t // nt
            i_n, t = t - rest * nt, rest
        else:
            i_n = 0
        if mt > 1:
            z = t // mt
            i_m = t - z * mt
        else:
            z = t
    zs, zb = 0, z
    if splitk > 1:
        zb, zs = z // splitk, z % splitk
    zi, zo = zb, 0
    if zb >= batch_inner:
        zo, zi = zb // batch_inner, zb % batch_inner
    return i_m, i_n, zi, zo, zs


def cta_tiles(inst, M, N, K, batch, batch_inner, splitk, sms):
    """launch_gemm_tc + the kernel's tile loop: the list of tiles of every CTA, and whether the grid is 3-D"""
    mode, bn, epi, small = inst
    nt, mt = -(-N // bn), -(-M // BM)
    nz = splitk * batch
    tiles = nt * mt * nz
    grid3d = tiles <= sms
    if grid3d:
        ctas = [[tile_info(0, nt, mt, splitk, batch_inner, True, (x, y, z))]
                for z in range(nz) for y in range(mt) for x in range(nt)]
    else:
        ctas = [[tile_info(t, nt, mt, splitk, batch_inner, False) for t in range(b, tiles, sms)] for b in range(sms)]
    return ctas, grid3d


def schedule(inst, M, N, K, batch, batch_inner, splitk, sms):
    """what the GPU tests print: grid kind, tiles, CTAs, most tiles of one CTA, stages, how often that CTA's operand
    ring and TMEM accumulator ring wrap, the deepest UMMA accumulation chain (16-deep k steps of one tile)"""
    mode, bn, epi, small = inst
    ctas, grid3d = cta_tiles(inst, M, N, K, batch, batch_inner, splitk, sms)
    chunk = k_chunk(K, splitk)
    bk = RA if mode == MNMN else 64

    def depth(zs):
        return min(K, (zs + 1) * chunk) - zs * chunk

    busiest = max(ctas, key=len)
    kblocks = sum(-(-depth(t[4]) // bk) for t in busiest)
    st = stages(*inst)
    return dict(grid="3-D" if grid3d else "persistent", tiles=sum(len(c) for c in ctas), ctas=len(ctas),
                max_tiles=len(busiest), stages=st, ring_wraps=kblocks // st, acc_wraps=len(busiest) // 2,
                chain=-(-chunk // 16), last_chunk=depth(splitk - 1))


def fmt_schedule(s):
    return (f"{s['grid']} grid, {s['tiles']} tiles on {s['ctas']} CTAs (<= {s['max_tiles']} each), {s['stages']} stages, "
            f"ring wraps {s['ring_wraps']}, accumulator wraps {s['acc_wraps']}, chain {s['chain']}, "
            f"last chunk {s['last_chunk']}")


# ---------------------------------------------------------------- the launch table of the GPU tests
# An operand is one TB buffer of `entries` blocks of `rows` rows each (rows a multiple of its row block); the matrix of
# batch entry (zi, zo) starts at block base + zi * inner + zo * outer, as the strides of drq_gemm_bf16 place it.
# C (fp32) entries are regions of (M + 1) x ldc floats; the split plane of chunk s is `split` regions further.
SHAPES = {          # B, A, F, H
    "walker": (256, 6, 50, 1024),
    "humanoid": (512, 21, 100, 1024),
    "b1": (1, 1, 50, 256),
    "b129": (129, 32, 100, 256),
    "b200": (200, 1, 50, 256),
}


def _ceil(n, m):
    return -(-n // m) * m


def launches(shape):
    """the drq_gemm_bf16 calls of twin_q_layers, actor_mlp_fwd, critic_pass, _actor_pass and act_body at one shape:
    name -> dict(inst, M, N, K, batch, batch_inner, splitk, a / b / c / bias / mask placement)"""
    B, A, F, H = SHAPES[shape]
    RB, FP = _ceil(B, RA), _ceil(F, RW)
    NT = 2 * FP
    S2 = splitk_for(2 * (RB // RA) * (NT // 128))
    S1 = splitk_for((RB // RA) * (FP // 64))
    SX = 8 if H % 1024 == 0 else 1
    L = {}

    def add(name, mode, bn, epi, M, N, K, batch=1, inner=None, splitk=1, a=(1, 0, 0, 0), b=(1, 0, 0, 0), c=(0, 0, 0),
            bias=None, mask=None, small_ok=False, b_rows=None):
        """a / b / bias / mask: (entries, base, inner, outer) in entries; c: (inner, outer, split) in regions; b_rows:
        rows of one B entry when N spans several (the merged trunk weight's slots)"""
        L[name] = dict(inst=(mode, bn, epi, 0), M=M, N=N, K=K, batch=batch, batch_inner=inner or batch, splitk=splitk,
                       a=a, b=b, c=c, bias=bias, mask=mask, small_ok=small_ok, b_rows=b_rows)

    # critic_pass: the merged trunk forward (obs rows x [actor | critic], next rows x [target | actor])
    add("trunk_fwd_merged", KK, 128, F32, B, NT, REPR, batch=2, inner=1, splitk=S2, a=(2, 0, 0, 1), b=(3, 1, 0, -1),
        c=(0, 1, 2), b_rows=FP, bias=(2, 0, 0, 1))
    # (drq_gemm_bf16 ignores a bias when splitk > 1: the split forwards get one to show that no plane receives it)
    # _actor_pass / act_body: one trunk forward
    add("trunk_fwd", KK, 64, F32, B, FP, REPR, splitk=S1, c=(0, 0, 1), bias=(1, 0, 0, 0), small_ok=True)
    # twin_q_layers, nets = 2 (4 heads: x[0] for the critic's pair, x[1] for the target's) and nets = 1
    q = dict(batch=4, inner=2, a=(2, 0, 0, 1), b=(4, 0, 1, 2), bias=(4, 0, 1, 2), small_ok=True)
    add("q_l1_4heads", KK, 64, RELU, B, H, F + A, c=(1, 2, 0), **q)
    add("q_l2_4heads", KK, 64, RELU, B, H, H, c=(1, 2, 0), **q)
    q1 = dict(batch=2, inner=2, a=(1, 0, 0, 1), b=(2, 0, 1, 2), bias=(2, 0, 1, 2), small_ok=True)
    add("q_l1_2heads", KK, 64, RELU, B, H, F + A, c=(1, 2, 0), **q1)
    # actor_mlp_fwd on [obs | next] rows
    add("policy_l1", KK, 64, RELU, RB + B, H, F, bias=(1, 0, 0, 0))
    add("policy_l2", KK, 64, RELU, RB + B, H, H, bias=(1, 0, 0, 0))
    # the same Linear forward with the 128-wide tile (an instantiation no update path selects today)
    add("linear_bn128", KK, 128, RELU, B, H - 40, H, bias=(1, 0, 0, 0))      # N ends 24 or 88 columns into a tile
    add("linear_bn128_f32", KK, 128, F32, B, H, F + A, bias=(1, 0, 0, 0))
    # critic backward: Q heads' weight / data gradients, twin-head batched
    add("q_l2_wgrad", MNMN, 128, F32, H, H, B, batch=2, a=(2, 0, 1, 0), b=(2, 0, 1, 0), c=(1, 0, 0))
    add("q_l2_dgrad", KMN, 64, MASK, B, H, H, batch=2, a=(2, 0, 1, 0), b=(2, 0, 1, 0), c=(1, 0, 0), mask=(2, 0, 1, 0),
        small_ok=True)
    add("q_l1_wgrad", MNMN, 64, F32, H, F + A, B, batch=2, a=(2, 0, 1, 0), b=(1, 0, 0, 0), c=(1, 0, 0))
    add("q_l1_dgrad_critic", KMN, 64, F32, B, F, H, batch=2, splitk=SX, a=(2, 0, 1, 0), b=(2, 0, 1, 0), c=(1, 0, 2),
        small_ok=True)
    add("q_l1_dgrad_actor", KMN, 64, F32, B, F + A, H, batch=2, splitk=SX, a=(2, 0, 1, 0), b=(2, 0, 1, 0), c=(1, 0, 2),
        small_ok=True)
    add("trunk_wgrad", MNMN, 128, TWGRAD, F, REPR, B)
    add("trunk_dgrad", KMN, 128, TDGRAD, B, REPR, F, mask=(1, 0, 0, 0))
    # actor backward
    add("policy_l3_wgrad", MNMN, 128, F32, A, H, B)
    add("policy_l3_dgrad", KMN, 64, MASK, B, H, A, mask=(1, 0, 0, 0), small_ok=True)
    add("policy_l2_wgrad", MNMN, 128, F32, H, H, B)
    add("policy_l2_dgrad", KMN, 64, MASK, B, H, H, mask=(1, 0, 0, 0), small_ok=True)
    add("policy_l1_wgrad", MNMN, 64, F32, H, F, B)
    add("policy_l1_dgrad", KMN, 64, F32, B, F, H, small_ok=True)
    add("hidden_dgrad_bn128", KMN, 128, MASK, B, H, H, mask=(1, 0, 0, 0))
    L["linear_bn128"]["n_store"] = H - 24           # TB columns [N, n_store) are written as zeros
    return L


def all_launches():
    return {(shape, name): spec for shape in SHAPES for name, spec in launches(shape).items()}


# ---------------------------------------------------------------- tests of the model
def test_stages_of_every_instantiation():
    got = {inst_name(i): stages(*i) for i in INSTANTIATIONS}
    assert len(got) == 15
    assert all(v == 2 for k, v in got.items() if k.endswith("_SMALL"))
    # 64-wide K-major tiles: 24 KB per stage -> 6 (capped); 128-wide: 32 KB per stage -> 5 (fp32 epilogue scratch 17 KB)
    assert got["KK64_F32"] == 6 and got["KK128_F32"] == 5 and got["KK128_RELU"] == 6
    assert got["MNMN128_TRUNK_WGRAD"] == 2          # 64 KB stages + a 66 KB re-ordering scratch


def test_every_instantiation_is_in_the_table():
    insts = {spec["inst"] for spec in all_launches().values()}
    insts |= {(m, bn, e, 1) for (m, bn, e, _), spec in ((s["inst"], s) for s in all_launches().values())
              if spec["small_ok"]}
    assert insts == set(INSTANTIATIONS)


@pytest.mark.parametrize("sms", BUDGETS)
def test_every_tile_is_visited_once(sms):
    for (shape, name), s in all_launches().items():
        mode, bn, epi, _ = s["inst"]
        ctas, grid3d = cta_tiles(s["inst"], s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"], sms)
        seen = [t for c in ctas for t in c]
        nt, mt = -(-s["N"] // bn), -(-s["M"] // BM)
        inner = s["batch_inner"]
        want = [(im, i_n, zb % inner, zb // inner, zs) for im in range(mt) for i_n in range(nt)
                for zb in range(s["batch"]) for zs in range(s["splitk"])]
        assert sorted(seen) == sorted(want), (shape, name, sms)
        assert grid3d == (len(want) <= sms)
        if not grid3d:
            assert len(ctas) == sms and min(len(c) for c in ctas) >= 1


def test_trunk_forwards_end_in_a_32_column_chunk():
    w, h = launches("walker"), launches("humanoid")
    assert w["trunk_fwd_merged"]["splitk"] == 35 and h["trunk_fwd"]["splitk"] == 18
    for s in (w["trunk_fwd_merged"], h["trunk_fwd"]):
        assert REPR - (s["splitk"] - 1) * k_chunk(REPR, s["splitk"]) == 32
    # the merged humanoid forward: 2 n tiles x 4 m tiles x (2 entries x 9 chunks) = 144 tiles, 3-D at 148, persistent at 140
    s = h["trunk_fwd_merged"]
    sch = {sms: schedule(s["inst"], s["M"], s["N"], s["K"], 2, 1, s["splitk"], sms) for sms in (148, 140)}
    assert sch[148]["tiles"] == 144 and sch[148]["grid"] == "3-D" and sch[140]["grid"] == "persistent"


def test_budget_one_wraps_both_rings():
    s = launches("walker")["q_l2_4heads"]
    sch = schedule(s["inst"], s["M"], s["N"], s["K"], s["batch"], s["batch_inner"], s["splitk"], 1)
    assert sch["max_tiles"] == sch["tiles"] == 2 * 16 * 4 and sch["ring_wraps"] > sch["max_tiles"] and sch["acc_wraps"] > 1


# ---------------------------------------------------------------- the checks against planted defects
M, N, K, S = 200, 24, 300, 3       # a partial last m tile (200 = 128 + 72), three split chunks of 128 / 128 / 44
LDC = N + 3
R = (M + 1) * LDC                  # one C region: an extra row past M, padding columns past N


def _problem(seed=3):
    g = torch.Generator().manual_seed(seed)
    a = (torch.rand(2, 2, M, K, generator=g) - 0.5).to(torch.bfloat16).double()     # [outer][inner]
    b = (torch.rand(2, 2, N, K, generator=g) - 0.5).to(torch.bfloat16).double()
    bias = (torch.rand(N, generator=g) - 0.5).double()
    a[1, 1, M - 1, :] *= 2.0 ** -20  # one small row in the last partial m tile of the last entry
    return a, b, bias


def _chunks():
    ch = k_chunk(K, S)
    return [(s * ch, min(K, (s + 1) * ch)) for s in range(S)]


def _want(a, b, bias, split):
    """planes [zo][zi][s] of the reference and of the absolute reference"""
    want, absref = {}, {}
    for zo, zi in itertools.product(range(2), range(2)):
        for s, (k0, k1) in enumerate(_chunks() if split else [(0, K)]):
            x, y = a[zo, zi, :, k0:k1], b[zo, zi, :, k0:k1]
            want[zo, zi, s] = x @ y.T + (0 if split else bias)
            absref[zo, zi, s] = x.abs() @ y.abs().T + (0 if split else bias.abs())
    return want, absref


def _store(planes, split):
    """a sentinel fp32 buffer of 2 x 2 entries (x S planes) + a spare region, planes stored as the kernel stores them:
    entry (zi, zo) chunk s at region zi + 2 zo + 4 s"""
    n = 4 * (S if split else 1) + 1
    buf = fill_sentinel(torch.empty(n * R, dtype=torch.float32))
    for (zo, zi, s), v in planes.items():
        off = (zi + 2 * zo + 4 * s) * R
        buf[off:off + R].view(M + 1, LDC)[:M, :N] = v.float()
    return buf


def _check(buf, want, absref, split, c=8.0):
    written = torch.zeros(buf.numel(), dtype=torch.bool)
    need = 0.0
    for (zo, zi, s), w in want.items():
        off = (zi + 2 * zo + 4 * s) * R
        written[off:off + R].view(M + 1, LDC)[:M, :N] = True
        k0, k1 = (_chunks() if split else [(0, K)])[s]
        got = buf[off:off + R].view(M + 1, LDC)[:M, :N]
        need = max(need, assert_f32_bound(got, w, absref[zo, zi, s], math.ceil((k1 - k0) / 16), c, f"plane {zo, zi, s}"))
    assert_sentinel_outside(buf, written, "fp32 output")
    return need


@pytest.mark.parametrize("split", [False, True])
def test_correct_fp32_result_is_accepted(split):
    a, b, bias = _problem()
    want, absref = _want(a, b, bias, split)
    got = {k: v.float().double() for k, v in want.items()}          # fp32 rounding of the exact result
    need = _check(_store(got, split), want, absref, split)
    assert need < 1.0


def test_rejects_a_zeroed_small_element_of_the_last_partial_m_tile():
    a, b, bias = _problem()
    want, absref = _want(a, b, bias * 0, False)
    got = {k: v.clone() for k, v in want.items()}
    got[1, 1, 0][M - 1, N - 1] = 0.0
    # the older checks accept it: 2e-5 max|want| for fp32 outputs, 2^-8 max|want| for bf16 ones
    err = (got[1, 1, 0] - want[1, 1, 0]).abs().max()
    assert err <= 2e-5 * want[1, 1, 0].abs().max() and max_norm_ok(got[1, 1, 0], want[1, 1, 0])
    with pytest.raises(AssertionError, match="outside"):
        _check(_store(got, False), want, absref, False)


def test_rejects_a_missing_split_plane():
    a, b, bias = _problem()
    want, absref = _want(a, b, bias, True)
    got = {k: v for k, v in want.items() if k != (0, 1, S - 1)}      # never stored: the plane keeps the sentinel
    with pytest.raises(AssertionError, match="outside"):
        _check(_store(got, True), want, absref, True)


def test_rejects_swapped_inner_and_outer_batch_entries():
    a, b, bias = _problem()
    want, absref = _want(a, b, bias, False)
    got = dict(want)
    got[0, 1, 0], got[1, 0, 0] = want[1, 0, 0], want[0, 1, 0]
    with pytest.raises(AssertionError, match="outside"):
        _check(_store(got, False), want, absref, False)


def test_rejects_a_bias_added_to_every_split_plane():
    a, b, bias = _problem()
    want, absref = _want(a, b, bias, True)
    got = {k: v + bias for k, v in want.items()}
    with pytest.raises(AssertionError, match="outside"):
        _check(_store(got, True), want, absref, True)


@pytest.mark.parametrize("where", ["row_M", "padding_column", "spare_plane"])
def test_rejects_a_stray_store(where):
    a, b, bias = _problem()
    want, absref = _want(a, b, bias, True)
    buf = _store(want, True)
    off = (1 + 2 * 1 + 4 * (S - 1)) * R             # the last stored plane
    if where == "row_M":
        buf[off + M * LDC] = 0.0
    elif where == "padding_column":
        buf[off + 5 * LDC + N] = 0.0
    else:
        buf[4 * S * R + 7] = 0.0
    with pytest.raises(AssertionError, match="overwritten"):
        _check(buf, want, absref, True)
