"""A CPU model of the fp32 mode's schedules (drqv2_b200/drqv2.py: _splitk_for and the _gemm calls; csrc/gemm_f32.cu:
drq_gemm_f32's split-K chunking; csrc/encoder_f32.cu: the weight-gradient items and blocks) and the case tables of
tests/test_gpu_fp32_kernels.py, checked without a GPU:

  - every K index of the split-K trunk GEMM is in exactly one chunk at every batch size of the table, and no chunk is
    empty;
  - the GPU case tables reach each schedule edge: weight-gradient blocks that take 1, 2 and 10-12 tiles (2 at one layer
    only, 2 at every layer), S > 64 split planes, a partial last K chunk, 1, 2 and 3+ M tiles, K % 16 != 0;
  - the element-wise bound and the sentinels of the GPU tests accept a correct result and reject planted defects: a
    zeroed small element in the last partial M tile (which the update tests' rel-L2 accepts), a dropped split plane,
    swapped Q1 / Q2 batch entries, a 3x3 weight gradient that skips a block's second tile, and a data gradient that
    writes rows >= hout + 2.

The GPU tests take their chain lengths n (the bound |got - want| <= c 2^-24 (n + 8) A) and their printed schedules from
this model."""
import math
from collections import namedtuple

import pytest
import torch

from tests.helpers import assert_sentinel_outside, check_sum_bound, fill_sentinel, rel_l2

REPR, PLANE, PW = 39200, 1696, 41
BM, BN, BK = 64, 64, 16                    # gemm_f32.cu tile
TP = 128                                   # encoder_f32.cu kTP: output positions per 3x3 tile
WGRAD_BLOCKS = 296                         # kWgradBlocks
C1_TILES, C1_ROWS = 6, 7                   # conv1: 41 rows = 5 x 7 + 6
EPI_NONE, EPI_RELU, EPI_MASK, EPI_MASK_WIDE = 0, 1, 2, 3

# the shapes and batch sizes of the GPU GEMM table: walker, DMC dog, and one only the fp32 mode runs
SHAPES = {"walker": (6, 50, 1024), "dog": (38, 50, 1024), "fp32_only": (129, 256, 1020)}
GEMM_BATCHES = (1, 5, 63, 64, 65, 129, 256)
CONV_N = (1, 2, 5, 24, 25, 256)
CONV_HOUT = (39, 37, 35)
CONV1_CIN = (1, 9, 11, 16)
CONV1_N = (1, 5, 81, 256)                  # 81: every (sx, sy) shift once
COLSUM_M = (1, 7, 8, 9, 256, 513)
LN_CASES = ((64, 273), (65, 145), (256, 73), (512, 37))     # (B, S = _splitk_for(B))


# ---------------------------------------------------------------- split-K GEMM
def splitk_for(m_rows, K=REPR, target_blocks=296):
    """drqv2._splitk_for"""
    mblocks = (m_rows + 63) // 64
    s0 = max(1, min(target_blocks // mblocks, K // 64))
    chunk = -(-K // s0)
    chunk = -(-chunk // 16) * 16
    return -(-K // chunk)


def k_chunk(K, splitk):
    """drq_gemm_f32: ceil(K / splitk) rounded up to BK; DRQ_REQUIRE that no chunk is empty"""
    if splitk == 1:
        return K
    chunk = -(-(-(-K // splitk)) // BK) * BK
    assert chunk * (splitk - 1) < K, f"gemm: splitk {splitk} leaves empty chunks for K={K}"
    return chunk


def k_ranges(K, splitk):
    """[k_begin, k_end) of every split plane z, as gemm_f32_kernel forms them"""
    c = k_chunk(K, splitk)
    return [(z * c, min(K, z * c + c)) for z in range(splitk)]


def q_stride(A, F, H):
    """floats between the Q1.* and Q2.* tensors of the critic's arena segment (each tensor padded to 4 floats)"""
    pad4 = lambda n: (n + 3) // 4 * 4
    return pad4(H * (F + A)) + pad4(H) + pad4(H * H) + pad4(H) + pad4(H) + pad4(1)


Gemm = namedtuple("Gemm", "name M N K a_off sa_m sa_k b_off sb_k sb_n ldc bias ldmask epi acc batch bs splitk")


def _g(name, M, N, K, a, b, ldc, bias=False, ldmask=0, epi=EPI_NONE, acc=0, batch=1, bs=(0, 0, 0, 0, 0), splitk=1,
       a_off=0, b_off=0):
    return Gemm(name, M, N, K, a_off, a[0], a[1], b_off, b[0], b[1], ldc, bias, ldmask, epi, acc, batch, bs, splitk)


def gemm_launches(B, A, F, H):
    """every _gemm call of drqv2.py at (B, A, F, H), in the argument order of drq_gemm_f32 (a = (sa_m, sa_k), b = (sb_k,
    sb_n)); a_off / b_off are the pointer offsets in floats (the Q2 half of dc1, W + w_col0, Q2.0.weight = Q1 + qs)"""
    qs, BH, X = q_stride(A, F, H), B * H, F + A
    lin = lambda name, K, N, relu, **kw: _g(name, B, N, K, (K, 1), (1, K), N, bias=True,
                                             epi=EPI_RELU if relu else EPI_NONE, **kw)
    S = splitk_for(B)
    return [
        # _trunk_fwd: split-K partial planes
        _g("trunk_fwd", B, F, REPR, (REPR, 1), (1, REPR), F, bs=(0, 0, B * F, 0, 0), splitk=S),
        # _linear_fwd of the policy MLP (critic and actor passes, Actor.forward through _mlp_fwd)
        lin("policy0_fwd", F, H, True), lin("policy2_fwd", H, H, True), lin("policy4_fwd", H, A, False),
        # _twin_q_fwd: both heads per launch, the first layer's input shared (bs_a = 0)
        lin("q0_fwd_twin", X, H, True, batch=2, bs=(0, qs, BH, qs, 0)),
        lin("q2_fwd_twin", H, H, True, batch=2, bs=(BH, qs, BH, qs, 0)),
        lin("q4_fwd_twin", H, 1, False, batch=2, bs=(BH, qs, B, qs, 0)),
        # Critic.forward through _mlp_fwd: one head per launch
        lin("q0_fwd_mlp", X, H, True), lin("q4_fwd_mlp", H, 1, False),
        # _critic_pass backward (both heads per launch): wgrad's transposed A operand (sa_k = ld_dy)
        _g("q4_wgrad_twin", 1, H, B, (1, 1), (H, 1), H, batch=2, bs=(B, BH, qs, 0, 0)),
        _g("q4_dgrad_twin", B, H, 1, (1, 1), (H, 1), H, ldmask=H, epi=EPI_MASK, batch=2, bs=(B, qs, BH, 0, BH)),
        _g("q2_wgrad_twin", H, H, B, (1, H), (H, 1), H, batch=2, bs=(BH, BH, qs, 0, 0)),
        _g("q2_dgrad_twin", B, H, H, (H, 1), (H, 1), H, ldmask=H, epi=EPI_MASK, batch=2, bs=(BH, qs, BH, 0, BH)),
        _g("q0_wgrad_twin", H, X, B, (1, H), (X, 1), X, batch=2, bs=(BH, 0, qs, 0, 0)),
        _g("q0_dgrad_h_q1", B, F, H, (H, 1), (X, 1), X),
        _g("q0_dgrad_h_q2_acc", B, F, H, (H, 1), (X, 1), X, acc=1, a_off=BH, b_off=qs),
        # trunk weight gradient (critic and actor passes)
        _g("trunk_wgrad", F, REPR, B, (1, F), (REPR, 1), REPR),
        # _encoder_bwd: d(features) masked by conv4's ReLU, scattered into conv4's wide dpre
        _g("features_dgrad_mask_wide", B, REPR, F, (F, 1), (REPR, 1), 32 * PLANE, ldmask=REPR, epi=EPI_MASK_WIDE),
        # _actor_pass: d(action) from both heads into the action slice (w_col0 = F, n_cols = A)
        _g("q0_dgrad_action_q1", B, A, H, (H, 1), (X, 1), A, b_off=F),
        _g("q0_dgrad_action_q2_acc", B, A, H, (H, 1), (X, 1), A, acc=1, a_off=BH, b_off=qs + F),
        _g("policy4_wgrad", A, H, B, (1, A), (H, 1), H),
        _g("policy4_dgrad", B, H, A, (A, 1), (H, 1), H, ldmask=H, epi=EPI_MASK),
        _g("policy2_wgrad", H, H, B, (1, H), (H, 1), H),
        _g("policy2_dgrad", B, H, H, (H, 1), (H, 1), H, ldmask=H, epi=EPI_MASK),
        _g("policy0_wgrad", H, F, B, (1, H), (F, 1), F),
        _g("policy0_dgrad", B, F, H, (H, 1), (F, 1), F),
    ]


def gemm_chain(L):
    """the longest sequential fp32 chain behind one output element: the K chunk, the bias add, the accumulate"""
    return k_chunk(L.K, L.splitk) + int(L.bias) + L.acc


def gemm_schedule(L):
    mt, nt = -(-L.M // BM), -(-L.N // BN)
    s = f"{L.name}: M={L.M} N={L.N} K={L.K} grid {nt}x{mt}x{L.splitk if L.splitk > 1 else L.batch}"
    if L.splitk > 1:
        r = k_ranges(L.K, L.splitk)
        s += f" split {L.splitk} chunk {k_chunk(L.K, L.splitk)} last {r[-1][1] - r[-1][0]}"
    return s


def compact_to_wide(n):
    """gemm_f32.cu compact_to_wide (tensor or int): feature c*1225 + y*35 + x -> c*PLANE + y*41 + x"""
    c, r = n // 1225, n % 1225
    return c * PLANE + (r // 35) * PW + r % 35


# ---------------------------------------------------------------- encoder weight gradients
def wgrad3_schedule(N, hout):
    """conv3x3_wgrad_kernel: (image, 128-position tile) items over G <= 296 blocks; block g takes items g, g + G, ..."""
    ntiles = -(-hout * PW // TP)
    items = N * ntiles
    G = min(items, WGRAD_BLOCKS)
    return dict(ntiles=ntiles, items=items, G=G, tpb_max=-(-items // G), tpb_min=items // G)


def wgrad3_chain(N, hout):
    s = wgrad3_schedule(N, hout)
    return s["tpb_max"] * TP + s["G"]


def conv1_wgrad_schedule(N):
    """conv1_wgrad_kernel: (image, 7-row tile) items, 6 per image"""
    items = N * C1_TILES
    G = min(items, WGRAD_BLOCKS)
    return dict(items=items, G=G, tpb_max=-(-items // G), tpb_min=items // G)


def conv1_wgrad_chain(N):
    s = conv1_wgrad_schedule(N)
    return s["tpb_max"] * C1_ROWS * PW + s["G"]


def colsum_chain(M):
    return -(-M // 8) + 8


# ---------------------------------------------------------------- written sets (bool over a flat buffer)
def plane_written(N_buf, N, lo, hi):
    """positions [lo, hi) of every channel plane of images < N in a wide buffer of N_buf images"""
    w = torch.zeros(N_buf, 32, PLANE, dtype=torch.bool)
    w[:N, :, lo:hi] = True
    return w.reshape(-1)


def dgrad_written(N_buf, N, hout):
    """drq_conv3x3_dgrad_f32 writes [0, (hout + 2) 41) of each plane (+0 at columns >= hout + 2), nothing else"""
    return plane_written(N_buf, N, 0, (hout + 2) * PW)


# ================================================================= the model's own checks
def test_splitk_model_is_drqv2s():
    from drqv2_b200 import drqv2
    for B in list(range(1, 600)) + [1024, 4096]:
        assert splitk_for(B) == drqv2._splitk_for(B), B


@pytest.mark.parametrize("B", sorted(set(GEMM_BATCHES) | {b for b, _ in LN_CASES} | set(range(1, 520, 7))))
def test_every_k_index_in_exactly_one_chunk(B):
    S = splitk_for(B)
    cover = torch.zeros(REPR, dtype=torch.int32)
    for k0, k1 in k_ranges(REPR, S):
        assert k1 > k0, "empty chunk"
        cover[k0:k1] += 1
    assert bool((cover == 1).all())


def test_empty_chunk_is_refused():
    assert k_ranges(40, 3) == [(0, 16), (16, 32), (32, 40)]
    with pytest.raises(AssertionError, match="empty chunks"):
        k_chunk(33, 4)            # chunk 16: three planes cover 48 >= 33, the fourth would be empty


def test_tables_reach_the_schedule_edges():
    # split planes: S > 64, a partial last chunk; the LN cases take the S the trunk GEMM gives their B
    Ss = {splitk_for(B) for B in GEMM_BATCHES}
    assert max(Ss) > 64 and {273, 145, 73} <= Ss
    assert all(splitk_for(B) == S for B, S in LN_CASES)
    last = [r[1] - r[0] for r in (k_ranges(REPR, splitk_for(B))[-1] for B in GEMM_BATCHES)]
    assert any(n < k_chunk(REPR, splitk_for(B)) for n, B in zip(last, GEMM_BATCHES))
    assert k_ranges(REPR, 273)[-1] == (272 * 144, REPR) and REPR - 272 * 144 == 32
    # M tiles: 1, 2 and 3+; K % 16 != 0 among the GEMMs; a shared input (bs_a = 0) and transposed-A operands
    mts = {-(-L.M // BM) for B in GEMM_BATCHES for s in SHAPES.values() for L in gemm_launches(B, *s)}
    assert {1, 2, 3} <= mts and max(mts) >= 4
    launches = [L for B in GEMM_BATCHES for s in SHAPES.values() for L in gemm_launches(B, *s)]
    assert any(L.K % BK for L in launches if L.splitk == 1)
    assert any(L.batch == 2 and L.bs[0] == 0 for L in launches)
    assert any(L.sa_k != 1 for L in launches)
    assert any(L.acc and L.b_off for L in launches) and any(L.epi == EPI_MASK_WIDE for L in launches)
    # 3x3 weight gradients: one tile per block; two at one layer only (N = 24); two at every layer (N = 25); 10-12
    per_n = {N: [wgrad3_schedule(N, h)["tpb_max"] for h in CONV_HOUT] for N in CONV_N}
    assert per_n[5] == [1, 1, 1]
    assert per_n[24] == [2, 1, 1]
    assert per_n[25] == [2, 2, 2]
    s = [wgrad3_schedule(256, h) for h in CONV_HOUT]
    assert [(x["tpb_min"], x["tpb_max"]) for x in s] == [(11, 12), (10, 11), (10, 11)]
    # conv1: 81 images = 486 items on 296 blocks, 190 of which take two
    c = conv1_wgrad_schedule(81)
    assert (c["items"], c["G"], c["tpb_max"], c["items"] - c["G"]) == (486, 296, 2, 190)
    assert conv1_wgrad_schedule(256)["tpb_max"] == 6


# ================================================================= planted defects
def _gemm_case(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    a = (torch.rand(M, K, generator=g) * 2 - 1).double()
    b = (torch.rand(K, N, generator=g) * 2 - 1).double()
    bias = (torch.rand(N, generator=g) * 2 - 1).double() * 0.05
    want = a @ b + bias
    absref = a.abs() @ b.abs() + bias.abs()
    return a, b, bias, want, absref


def test_correct_gemm_output_is_accepted():
    a, b, bias, want, absref = _gemm_case(129, 70, 88, 1)
    got = (a.float() @ b.float() + bias.float()).double()
    r = check_sum_bound("planted", got, want, absref, 88 + 1)
    assert r < 0.5


def test_rejects_a_zeroed_small_element_of_the_last_partial_m_tile():
    M, N, K = 129, 64, 1020
    a, b, bias, want, absref = _gemm_case(M, N, K, 2)
    got = want.float().double()
    # the third M tile holds one row: its smallest element well above the bound
    bound = 2 * 2.0 ** -24 * (K + 1 + 8) * absref[128]
    j = int(torch.where(want[128].abs() > 4 * bound, want[128].abs(), torch.full_like(bound, math.inf)).argmin())
    assert float(want[128, j].abs()) < 0.1 * float(want.abs().max())
    got[128, j] = 0
    assert rel_l2(got.numpy(), want.numpy()) < 1e-3    # the whole-update tests' rel-L2 bounds accept it
    with pytest.raises(AssertionError, match="out of bound"):
        check_sum_bound("planted", got, want, absref, K + 1)


def test_rejects_a_dropped_split_plane():
    B, F = 5, 50
    S = splitk_for(B)
    g = torch.Generator().manual_seed(3)
    a = (torch.rand(B, REPR, generator=g) * 2 - 1).double()
    w = (torch.rand(REPR, F, generator=g) * 2 - 1).double() * 0.01
    planes = fill_sentinel(torch.empty(S + 1, B, F))
    for z, (k0, k1) in enumerate(k_ranges(REPR, S)):
        if z != S // 2:                                # that plane's block never stored
            planes[z] = (a[:, k0:k1] @ w[k0:k1]).float()
    with pytest.raises(AssertionError, match="out of bound"):
        for z, (k0, k1) in enumerate(k_ranges(REPR, S)):
            check_sum_bound("planted", planes[z], a[:, k0:k1] @ w[k0:k1], a[:, k0:k1].abs() @ w[k0:k1].abs(),
                            k_chunk(REPR, S))
    # ... and a plane stored as zeros (its NaN overwritten) is just as wrong
    planes[S // 2] = 0
    k0, k1 = k_ranges(REPR, S)[S // 2]
    with pytest.raises(AssertionError, match="out of bound"):
        check_sum_bound("planted", planes[S // 2], a[:, k0:k1] @ w[k0:k1], a[:, k0:k1].abs() @ w[k0:k1].abs(),
                        k_chunk(REPR, S))


def test_rejects_swapped_q1_q2_entries():
    outs = [_gemm_case(16, 64, 56, 10 + z) for z in range(2)]
    got = torch.stack([outs[1][3], outs[0][3]]).float().double()
    want = torch.stack([outs[0][3], outs[1][3]])
    absref = torch.stack([outs[0][4], outs[1][4]])
    with pytest.raises(AssertionError, match="out of bound"):
        check_sum_bound("planted", got, want, absref, 56 + 1)


def _wgrad3_case(N, hout, seed):
    g = torch.Generator().manual_seed(seed)
    hin = hout + 2
    x = (torch.rand(N, 32, hin, hin, generator=g)).double()
    d = (torch.rand(N, 32, hout, hout, generator=g) * 2 - 1).double()
    return x, d


def _tile_mask(N, hout, n, t):
    """dpre positions [t 128, t 128 + 128) of the wide plane of image n, as a mask over [N][1][hout][hout]"""
    p = torch.arange(hout).view(hout, 1) * PW + torch.arange(hout).view(1, hout)
    m = torch.zeros(N, 1, hout, hout, dtype=torch.float64)
    m[n, 0] = ((p >= t * TP) & (p < t * TP + TP)).double()
    return m


def test_rejects_a_wgrad_that_skips_a_blocks_second_tile():
    N, hout = 25, 35
    s = wgrad3_schedule(N, hout)
    assert s["tpb_max"] == 2 and s["items"] > s["G"]
    x, d = _wgrad3_case(N, hout, 4)
    cw = lambda xx, dd: torch.nn.grad.conv2d_weight(xx, (32, 32, 3, 3), dd)
    want, absref = cw(x, d), cw(x.abs(), d.abs())
    n_chain = wgrad3_chain(N, hout)
    check_sum_bound("planted", want.float(), want, absref, n_chain)
    item = s["G"]                                      # block 0's second item
    n, t = item // s["ntiles"], item % s["ntiles"]
    got = want - cw(x, d * _tile_mask(N, hout, n, t))
    with pytest.raises(AssertionError, match="out of bound"):
        check_sum_bound("planted", got.float(), want, absref, n_chain)


def test_rejects_a_dgrad_store_into_row_hout_plus_2():
    N, hout = 2, 37
    din = fill_sentinel(torch.empty(N + 1, 32, PLANE))
    din[:N, :, :(hout + 2) * PW] = 0.5
    assert_sentinel_outside(din, dgrad_written(N + 1, N, hout), "din")
    din[1, 7, (hout + 2) * PW + 3] = 0.0               # row hout + 2 of a plane: the next dgrad's zero row
    with pytest.raises(AssertionError, match="outside the written set"):
        assert_sentinel_outside(din, dgrad_written(N + 1, N, hout), "din")
