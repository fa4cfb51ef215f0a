"""The tensor-core conv kernels at the edges of their persistent schedules: reduced SM budgets (drq_set_sm_limit), every
image count mod 2 and 3, odd feature halves, and the stores a kernel must not make.

At the image counts of test_gpu_bf16.py every CTA takes one tile.  Here small budgets give each CTA 3-12 tiles, so the
shared-memory and TMEM rings wrap, pair rounds run into single-tile tails, a last grouped tile holds one or two real
images, and the budgets of the encoder backward (140) and of a data-parallel reservation reach every kernel that reads
sm_budget().  Each case prints its schedule as conv4x1_launch (csrc/conv4x1_tc.cu) computes it, through the CPU model
of tests/test_conv4x1_schedule_cpu.py.

Checks:
  - element-wise |got - want| <= 2^-8 |want| + 2^-14 A against fp64 math on bf16-rounded operands, A = the same
    operation on absolute values (tests/helpers.assert_conv_bound); the largest error-to-bound ratio of each kernel is
    printed at the end of the module.  Weight gradients (about 300 k terms per output) keep 2e-5 of max|want| and are
    checked bit for bit between the single-layer and the all-layers reduction;
  - every output buffer starts as a sentinel one size larger than needed, and everything outside the set a kernel writes
    must still hold the sentinel afterwards;
  - NHWC and TB outputs equal the WB output bit for bit; the ring-fed conv1 equals the gathered-stack one bit for bit."""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch

from tests import test_conv4x1_schedule_cpu as S
from tests.helpers import (assert_conv_bound, assert_sentinel_outside, bits_equal, check_conv_fwd_outputs, fill_sentinel,
                           wb_from_nchw, wb_region, wb_written)

pytestmark = pytest.mark.gpu

RATIOS = {}          # kernel -> largest |got - want| / bound observed
SUMMARY = []         # one line per case: the schedule it ran


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@pytest.fixture(scope="module", autouse=True)
def _restores_launch_state():
    """the SM limit and both kernel modes are what they were before this module ran; then the ratios and schedules"""
    if not torch.cuda.is_available():
        yield
        return
    from drqv2_b200 import _lib
    h = _lib.lib()
    before = (h.drq_device_sm_count(), h.drq_set_conv4x1(-1), h.drq_set_conv1_planes(-1))
    yield
    after = (h.drq_device_sm_count(), h.drq_set_conv4x1(-1), h.drq_set_conv1_planes(-1))
    print("\nschedules run:\n  " + "\n  ".join(SUMMARY))
    print("largest |got - want| / bound, and share of 2^-14 A beyond the bf16 round, per kernel:",
          {k: tuple(round(x, 4) for x in v) for k, v in sorted(RATIOS.items())})
    assert after == before, ("SM limit, conv4x1 mode, conv1 mode", before, after)


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
def conv4x1(request):
    """drq_set_conv4x1(request.param): 0 = one pixel per accumulator row, 2 = four-pixel columns, 1 = the latter from 48
    images, 3 = the default (1 for the forward, the one-pixel data gradient)"""
    from drqv2_b200 import _lib
    prev = _lib.lib().drq_set_conv4x1(request.param)
    try:
        yield request.param
    finally:
        _lib.lib().drq_set_conv4x1(prev)


@pytest.fixture
def conv1_planes(request):
    from drqv2_b200 import _lib
    prev = _lib.lib().drq_set_conv1_planes(request.param)
    try:
        yield request.param
    finally:
        _lib.lib().drq_set_conv1_planes(prev)


@contextlib.contextmanager
def _budget(n):
    from drqv2_b200 import _lib
    prev = _lib.lib().drq_device_sm_count()
    _lib.call("drq_set_sm_limit", n)
    try:
        yield
    finally:
        _lib.call("drq_set_sm_limit", prev)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _bf(x):
    return x.to(torch.bfloat16).double()


def _note(kernel, ratios):
    """ratios: (|got - want| / bound, share of the absolute term beyond the bf16 round) of one case"""
    old = RATIOS.get(kernel, (0.0, 0.0))
    RATIOS[kernel] = tuple(max(a, b) for a, b in zip(old, ratios))


def _tb_row(n, fh, fhr):
    return n if n < fh else n - fh + fhr


def schedule(N, hout, dgrad, budget, feat_half=0, feat_half_row=0):
    """conv4x1_launch's schedule through the CPU model: tiles, CTAs, pair rounds, tiles of the single-tile tail, the most
    tiles of one CTA, TB tile epilogues with one 32-byte store per pixel ("paired", two tiles each) and with 16-byte stores
    ("single"), and the real images of the last grouped tile"""
    h = hout + 2 if dgrad else hout
    block_rows, tpi, total = S.conv_tiles(N, h)
    grid = min(total, budget)
    p = dict(N=N, tpi=tpi, total=total, pair_tiles=(N & ~1) * tpi, grid=grid, pair_rounds=total // (2 * grid))
    fh = feat_half if feat_half > 0 else N
    paired = single = 0
    for b in range(grid):
        k = 0
        while (t := S.tile_at(p, b, k)) < total:
            two = False
            if not dgrad and k % 2 == 0 and k < 2 * p["pair_rounds"] and t < p["pair_tiles"]:
                n = S.tile_pos(p, t)[0]
                two = _tb_row(n + 1, fh, feat_half_row) == _tb_row(n, fh, feat_half_row) + 1 and _tb_row(n, fh, feat_half_row) % 2 == 0
            paired += two
            single += not two
            k += 2 if two else 1
    return dict(tiles=total, ctas=grid, pair_rounds=p["pair_rounds"], tail=total - 2 * p["pair_rounds"] * grid,
                per_cta=-(-total // grid), paired=paired, single=single,
                last_group=(N % 3 or 3) if block_rows % 3 == 1 else None)


def _record(what, sch):
    SUMMARY.append(f"{what}: " + ", ".join(f"{k}={v}" for k, v in sch.items()))


def _pack_w(w):
    from drqv2_b200 import _lib
    wf = torch.zeros(36 * 32 * 8, dtype=torch.bfloat16, device=w.device)
    wd = torch.zeros_like(wf)
    _lib.call("drq_pack_conv_w_bf16", w.data_ptr(), wf.data_ptr(), wd.data_ptr(), _stream())
    return wf, wd


def _column_kernel(mode, N, dgrad):
    """whether drq_conv3x3_{fwd,dgrad}_bf16 launch the four-pixel-column kernel (use_conv4x1, csrc/conv_tc.cu)"""
    if mode == 3 and dgrad:
        return False
    return mode == 2 or (mode >= 1 and N >= 48)


# ----------------------------------------------------------------------------------------------------- conv2-4 forward
FWD_SIZES = [(1, 148), (2, 148), (3, 148), (4, 148), (5, 148), (7, 148),
             (4, 4), (7, 5), (11, 4), (14, 4), (24, 8),
             (256, 140), (257, 140), (49, 148)]
FWD_CASES = [(N, b, m) for m in (0, 2) for N, b in FWD_SIZES] + [(49, 148, 1)]


def _conv_fwd_all_outputs(x, w, b, N, hout, feat_half, feat_half_row):
    """the three output modes of one forward; returns (WB, NHWC, TB view, TB rows) with every buffer one size too big
    and filled with the sentinel before the call"""
    from drqv2_b200 import _lib
    from drqv2_b200._bf16 import TB
    dev = x.device
    xin = wb_from_nchw(x)
    wf, _ = _pack_w(w)
    out = fill_sentinel(torch.empty(_lib.lib().drq_wb_elems(N + 1), dtype=torch.bfloat16, device=dev))
    _lib.call("drq_conv3x3_fwd_bf16", xin.data_ptr(), wf.data_ptr(), b.data_ptr(), out.data_ptr(), N, hout, 0, 0, 0, 0, _stream())
    feat = fill_sentinel(torch.empty(N + 1, hout * hout, 32, dtype=torch.bfloat16, device=dev))
    _lib.call("drq_conv3x3_fwd_bf16", xin.data_ptr(), wf.data_ptr(), b.data_ptr(), feat.data_ptr(), N, hout, 1, 0, 0, 0, _stream())
    fh = feat_half if feat_half > 0 else N
    rows = [_tb_row(n, fh, feat_half_row) for n in range(N)]
    fb = TB(max(rows) + 2, hout * hout * 32, dev)         # rows up to the next 128 boundary, at least one past the last
    fill_sentinel(fb.buf)
    _lib.call("drq_conv3x3_fwd_bf16", xin.data_ptr(), wf.data_ptr(), b.data_ptr(), fb.ptr(), N, hout, 2, fb.units,
              feat_half, feat_half_row, _stream())
    torch.cuda.synchronize()
    return out, feat, fb, rows


def _check_fwd_outputs(out, feat, fb, rows, want, absref, N, hout, column, what):
    # the four-pixel-column kernel stores the valid pixels only; the one-pixel kernel stores whole 41-pixel rows of the
    # valid rows (drq_conv3x3_fwd_bf16, include/drqv2_b200.h)
    return check_conv_fwd_outputs(out, feat, fb.view(), rows, want, absref, N, hout, hout if column else 41, what)


def _fwd_inputs(N, hout, seed, dev):
    g = torch.Generator().manual_seed(seed)
    hin = hout + 2
    x = torch.rand(N, 32, hin, hin, generator=g).to(dev)
    w = ((torch.rand(32, 32, 3, 3, generator=g) * 2 - 1) * 0.1).to(dev)
    b = ((torch.rand(32, generator=g) * 2 - 1) * 0.1).to(dev)
    xr, wr = _bf(x), _bf(w)
    want = torch.relu(torch.nn.functional.conv2d(xr, wr, b.double()))
    absref = torch.nn.functional.conv2d(xr.abs(), wr.abs(), b.double().abs())
    return x, w, b, want, absref


@pytest.mark.parametrize("N,sm_budget,conv4x1", FWD_CASES, indirect=["sm_budget", "conv4x1"])
@pytest.mark.parametrize("hout", [39, 37, 35])
def test_conv3x3_fwd_schedule_edges(dev, hout, N, sm_budget, conv4x1):
    x, w, b, want, absref = _fwd_inputs(N, hout, 1000 * hout + N, dev)
    half = N // 2
    fhr = -(-half // 128) * 128 if half else 0           # the update's layout: the second half on its own row block
    out, feat, fb, rows = _conv_fwd_all_outputs(x, w, b, N, hout, half, fhr)
    column = _column_kernel(conv4x1, N, False)
    what = f"fwd hout={hout} N={N} budget={sm_budget} mode={conv4x1}"
    ratio = _check_fwd_outputs(out, feat, fb, rows, want, absref, N, hout, column, what)
    _note("conv3x3 fwd, " + ("four-pixel columns" if column else "one pixel"), ratio)
    if column:
        _record(what, schedule(N, hout, False, sm_budget, half, fhr))


# TB feature epilogue: the exact cases of test_tb_feature_epilogue_writes_every_unit_once, and an update-shaped odd batch
TB_CASES = [(24, 12, 128, 8), (14, 7, 128, 4), (14, 7, 129, 5), (11, 11, 0, 4), (50, 25, 128, 8)]


@pytest.mark.parametrize("conv4x1", [2], indirect=True)
@pytest.mark.parametrize("N,feat_half,feat_half_row,sm_budget", TB_CASES, indirect=["sm_budget"])
def test_tb_feature_epilogue_paired_stores(dev, N, feat_half, feat_half_row, sm_budget, conv4x1):
    hout = 35
    sch = schedule(N, hout, False, sm_budget, feat_half, feat_half_row)
    what = f"TB hout={hout} N={N} half={feat_half}@{feat_half_row} budget={sm_budget}"
    _record(what, sch)
    assert sch["paired"] > 0, "the case must run the 32-byte stores"
    x, w, b, want, absref = _fwd_inputs(N, hout, 77 * N + feat_half_row, dev)
    out, feat, fb, rows = _conv_fwd_all_outputs(x, w, b, N, hout, feat_half, feat_half_row)
    _note("conv3x3 fwd, four-pixel columns", _check_fwd_outputs(out, feat, fb, rows, want, absref, N, hout, True, what))


# ------------------------------------------------------------------------------------------------ conv2-4 data gradient
DGRAD_SIZES = [(2, 148), (3, 148), (4, 148), (5, 148), (7, 5), (256, 140)]


@pytest.mark.parametrize("conv4x1", [2, 3], indirect=True)
@pytest.mark.parametrize("N,sm_budget", DGRAD_SIZES, indirect=["sm_budget"])
@pytest.mark.parametrize("hout", [39, 37, 35])
def test_conv3x3_dgrad_schedule_edges(dev, hout, N, sm_budget, conv4x1):
    from drqv2_b200 import _lib
    g = torch.Generator().manual_seed(3000 + 7 * hout + N)
    hin = hout + 2
    # every image carries a gradient: a window that reaches into the next image's rows shows up
    dout = ((torch.rand(N, 32, hout, hout, generator=g) * 2 - 1) * 1e-3).to(dev)
    act = (torch.rand(N + 1, 32, hin, hin, generator=g) - 0.4).clamp_min(0).to(dev)
    w = ((torch.rand(32, 32, 3, 3, generator=g) * 2 - 1) * 0.1).to(dev)
    d_wb, a_wb = wb_from_nchw(dout), wb_from_nchw(act)
    _, wd = _pack_w(w)
    din = fill_sentinel(torch.empty(_lib.lib().drq_wb_elems(N + 1), dtype=torch.bfloat16, device=dev))
    _lib.call("drq_conv3x3_dgrad_bf16", d_wb.data_ptr(), wd.data_ptr(), a_wb.data_ptr(), N + 1, din.data_ptr(), N, hout, _stream())
    torch.cuda.synchronize()
    dr, wr = _bf(dout), _bf(w)
    mask = (_bf(act[:N]) > 0).double()
    want = torch.nn.functional.conv_transpose2d(dr, wr) * mask
    absref = torch.nn.functional.conv_transpose2d(dr.abs(), wr.abs()) * mask
    column = _column_kernel(conv4x1, N, True)
    what = f"dgrad hout={hout} N={N} budget={sm_budget} mode={conv4x1}"
    ratio = assert_conv_bound(wb_region(din, N, hin, hin), want, absref, what)
    _note("conv3x3 dgrad, " + ("four-pixel columns" if column else "one pixel"), ratio)
    # whole rows < hin of images < N: the columns past the valid width are exact zeros (the next layer's windows read
    # them); nothing else is written
    assert torch.count_nonzero(wb_region(din, N, hin, 41)[..., hin:].float()) == 0, what
    assert_sentinel_outside(din, wb_written(din.numel(), N, hin, 41, dev), what)
    if column:
        _record(what, schedule(N, hout, True, sm_budget))
    else:
        ntiles = -(-hin * 41 // 128)
        _record(what + " (one pixel)", dict(tiles=N * ntiles, ctas=min(N * ntiles, 2 * sm_budget)))


# ------------------------------------------------------------------- weight gradients and the all-layers reduction
def _ring(dev, A=6):
    from tests.test_gpu_ring_direct import _ring_with_wrapping_episodes
    return _ring_with_wrapping_episodes("/test/conv_schedule_edges", A, dev)


def _ring_batch(ring, B, nstep, seed, dev):
    """B samples (episode start slot, idx) over the ring's episodes and the drq_ring_src; sample 0 is the last window of
    the episode that wraps past the end of the ring"""
    from drqv2_b200.replay_buffer import RingSrc
    g = np.random.default_rng(seed)
    eps = [ring.episodes[i] for i in g.integers(0, len(ring.episodes), B)]
    ix = [int(g.integers(1, r - nstep + 1)) for _, r in eps]
    eps[0] = next((s, r) for s, r in ring.episodes if s + r > ring.capacity)
    ix[0] = eps[0][1] - nstep
    es = np.array([s for s, _ in eps], np.int32)
    ix = np.array(ix, np.int32)
    es_d, ix_d = torch.from_numpy(es).to(dev), torch.from_numpy(ix).to(dev)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    src = RingSrc(ring.frames.data_ptr(), ring.action.data_ptr(), ring.reward.data_ptr(), ring.discount.data_ptr(),
                  ring.capacity, ring.frame_c, ring.stack, ring.A, nstep, 0.99, 0, ring.ep_table.data_ptr(),
                  ring.n_episodes.data_ptr(), 0, counter.data_ptr(), es_d.data_ptr(), ix_d.data_ptr())
    keep = (es_d, ix_d, counter)
    return src, es, ix, keep


def _gathered(ring, es, ix, nstep):
    from oracle import drq_oracle as O
    obs, _, _, _, nxt = O.ring_gather(ring.frames.cpu().numpy(), ring.action.cpu().numpy(), ring.reward.cpu().numpy(),
                                      ring.discount.cpu().numpy(), es, ix, nstep, 0.99)
    return torch.from_numpy(obs), torch.from_numpy(nxt)


def _conv1_input(obs_u8, shift):
    from oracle import drq_oracle as O
    return O.random_shift_exact(obs_u8.float(), shift.cpu()).double() / 255.0 - 0.5


def _wgrad_tol(tiles, budget):
    """2e-5 of max|want| for up to 32 tiles per CTA - the update's grids: at most 25 at B = 256 on 140 or 148 SMs - and
    in proportion to the tiles beyond.  Each CTA accumulates all of its tiles in one fp32 TMEM accumulator (8 UMMA
    accumulations per tile) before the fixed-order reduction of the G partials, and that chain's rounding grows with its
    length: at 7 CTAs and B = 256 a CTA takes 439-512 tiles, and the weight gradients measured up to 6.7e-5 of max|want|
    on a B200."""
    per_cta = -(-tiles // min(tiles, budget))
    return 2e-5 * max(1.0, per_cta / 32)


@pytest.mark.parametrize("B", [1, 24, 256])
@pytest.mark.parametrize("sm_budget", [148, 140, 7], indirect=True)
def test_encoder_wgrad_partials_and_reduce_multi(dev, B, sm_budget):
    """The encoder backward's weight gradients as encoder_backward (drqv2_b200/_bf16.py) issues them: three conv3x3 and the
    ring-fed conv1 weight gradient leave their per-CTA partials, one drq_conv_wgrad_reduce_multi reduces all four.  That
    equals the single-layer calls bit for bit (same reduction, same partial count G at the same budget) and fp64."""
    from drqv2_b200 import _lib
    from drqv2_b200._bf16 import WgReduceJob
    g = torch.Generator().manual_seed(500 + B + sm_budget)
    nstep, pad = 3, 4
    ring = _ring(dev)
    src, es, ix, keep = _ring_batch(ring, B, nstep, B + sm_budget, dev)
    shift = torch.randint(0, 2 * pad + 1, (B, 2), dtype=torch.int32, generator=g).to(dev)
    acts, ds = {}, {}
    for layer, hout in ((1, 39), (2, 37), (3, 35)):
        hin = hout + 2
        acts[layer] = (torch.rand(2 * B, 32, hin, hin, generator=g) - 0.3).clamp_min(0).to(dev)   # n_in = 2B images
        ds[layer] = ((torch.rand(B, 32, hout, hout, generator=g) * 2 - 1) * 1e-2).to(dev)
    d0 = ((torch.rand(B, 32, 41, 41, generator=g) * 2 - 1) * 1e-2).to(dev)
    a_wb = {k: wb_from_nchw(v) for k, v in acts.items()}
    d_wb = {k: wb_from_nchw(v) for k, v in ds.items()}
    d0_wb = wb_from_nchw(d0)
    z = lambda *s: torch.zeros(*s, device=dev)
    ws3, ws1 = _lib.lib().drq_conv_wgrad_bf16_ws_floats(), _lib.lib().drq_conv1_wgrad_bf16_ws_floats()

    # all layers: partials, then one reduction
    part = {k: z(ws3) for k in (1, 2, 3)}
    part0 = z(ws1)
    dw_m = {k: z(32, 32, 3, 3) for k in (1, 2, 3)}
    db_m = {k: z(32) for k in (1, 2, 3)}
    dw0_m, db0_m = z(32, 9, 3, 3), z(32)
    jobs = []
    for layer, hout in ((3, 35), (2, 37), (1, 39)):
        _lib.call("drq_conv3x3_wgrad_bf16", a_wb[layer].data_ptr(), 2 * B, d_wb[layer].data_ptr(), part[layer].data_ptr(),
                  None, None, B, hout, _stream())
        jobs.append(WgReduceJob(part[layer].data_ptr(), dw_m[layer].data_ptr(), db_m[layer].data_ptr(), B, hout, 0, 0))
    _lib.call("drq_conv1_wgrad_bf16_ring", C.byref(src), B, shift.data_ptr(), d0_wb.data_ptr(), part0.data_ptr(), None, None,
              B, pad, _stream())
    jobs.append(WgReduceJob(part0.data_ptr(), dw0_m.data_ptr(), db0_m.data_ptr(), B, 0, 9, 0))
    _lib.call("drq_conv_wgrad_reduce_multi", (WgReduceJob * 4)(*jobs), 4, _stream())
    # one layer at a time, reduced by each entry point itself
    dw_s = {k: z(32, 32, 3, 3) for k in (1, 2, 3)}
    db_s = {k: z(32) for k in (1, 2, 3)}
    for layer, hout in ((3, 35), (2, 37), (1, 39)):
        _lib.call("drq_conv3x3_wgrad_bf16", a_wb[layer].data_ptr(), 2 * B, d_wb[layer].data_ptr(), z(ws3).data_ptr(),
                  dw_s[layer].data_ptr(), db_s[layer].data_ptr(), B, hout, _stream())
    dw0_s, db0_s = z(32, 9, 3, 3), z(32)
    _lib.call("drq_conv1_wgrad_bf16_ring", C.byref(src), B, shift.data_ptr(), d0_wb.data_ptr(), z(ws1).data_ptr(),
              dw0_s.data_ptr(), db0_s.data_ptr(), B, pad, _stream())
    torch.cuda.synchronize()

    for layer, hout in ((3, 35), (2, 37), (1, 39)):
        what = f"conv{layer + 1} wgrad B={B} budget={sm_budget}"
        assert torch.equal(dw_m[layer], dw_s[layer]) and torch.equal(db_m[layer], db_s[layer]), what + ": multi != single"
        xr, dr = _bf(acts[layer][:B]), _bf(ds[layer])
        want_w = torch.nn.grad.conv2d_weight(xr, (32, 32, 3, 3), dr)
        want_b = dr.sum(dim=(0, 2, 3))
        tiles = B * -(-hout * 41 // 128)
        tol = _wgrad_tol(tiles, sm_budget)
        err_w = float((dw_m[layer].double() - want_w).abs().max() / want_w.abs().max())
        err_b = float((db_m[layer].double() - want_b).abs().max() / want_b.abs().max())
        _record(what, dict(tiles=tiles, G=min(tiles, sm_budget), err_w=f"{err_w:.1e}", err_b=f"{err_b:.1e}", tol=f"{tol:.1e}"))
        assert err_w <= tol and err_b <= tol, (what, err_w, err_b, tol)
    what = f"conv1 wgrad (ring) B={B} budget={sm_budget}"
    assert torch.equal(dw0_m, dw0_s) and torch.equal(db0_m, db0_s), what + ": multi != single"
    obs, _ = _gathered(ring, es, ix, nstep)
    x = _conv1_input(obs, shift).to(dev)
    dr = _bf(d0)
    want_w = torch.nn.grad.conv2d_weight(x, (32, 9, 3, 3), dr, stride=2)
    want_b = dr.sum(dim=(0, 2, 3))
    tol = _wgrad_tol(14 * B, sm_budget)
    err_w = float((dw0_m.double() - want_w).abs().max() / want_w.abs().max())
    err_b = float((db0_m.double() - want_b).abs().max() / want_b.abs().max())
    _record(what, dict(tiles=14 * B, G=min(14 * B, sm_budget), err_w=f"{err_w:.1e}", err_b=f"{err_b:.1e}", tol=f"{tol:.1e}"))
    assert err_w <= tol and err_b <= tol, (what, err_w, err_b, tol)
    del keep


# ------------------------------------------------------------------------------------ conv1 forward, parity planes
CONV1_GRIDS = [(3, 7), (96, 140), (48, 148)]


@pytest.mark.parametrize("conv1_planes", [2], indirect=True)
@pytest.mark.parametrize("N,sm_budget", CONV1_GRIDS, indirect=["sm_budget"])
def test_conv1_planes_fwd_schedule_edges(dev, N, sm_budget, conv1_planes):
    """the CPU model's grids of the planes kernel's row producer (test_conv1_producer_index_cpu.py): fp64 bound, sentinels"""
    from drqv2_b200 import _lib
    from oracle import drq_oracle as O
    g = torch.Generator().manual_seed(N + sm_budget)
    obs = torch.randint(0, 256, (N, 9, 84, 84), dtype=torch.uint8, generator=g)
    shift = torch.randint(0, 9, (N, 2), dtype=torch.int32, generator=g)
    w = ((torch.rand(32, 9, 3, 3, generator=g) - 0.5) * 0.3).to(dev)
    b = ((torch.rand(32, generator=g) - 0.5) * 0.1).to(dev)
    wp = torch.zeros(_lib.lib().drq_conv1_w_packed_elems(), dtype=torch.bfloat16, device=dev)
    _lib.call("drq_pack_conv1_w_bf16", w.data_ptr(), b.data_ptr(), wp.data_ptr(), 9, _stream())
    out = fill_sentinel(torch.empty(_lib.lib().drq_wb_elems(N + 1), dtype=torch.bfloat16, device=dev))
    obs_d, shift_d = obs.to(dev), shift.to(dev)
    _lib.call("drq_conv1_fwd_bf16", obs_d.data_ptr(), shift_d.data_ptr(), wp.data_ptr(), out.data_ptr(), N, 9, 4, _stream())
    torch.cuda.synchronize()
    x = (O.random_shift_exact(obs.float(), shift).double() / 255.0 - 0.5).to(dev)
    wr = _bf(w)
    want = torch.relu(torch.nn.functional.conv2d(x, wr, b.double(), stride=2))
    absref = torch.nn.functional.conv2d(x.abs(), wr.abs(), b.double().abs(), stride=2)
    what = f"conv1 fwd planes N={N} budget={sm_budget}"
    _note("conv1 fwd, planes", assert_conv_bound(wb_region(out, N, 41, 41), want, absref, what))
    assert_sentinel_outside(out, wb_written(out.numel(), N, 41, 41, dev), what)
    _record(what, dict(tiles=14 * N, ctas=min(14 * N, sm_budget), per_cta=-(-14 * N // min(14 * N, sm_budget))))


@pytest.mark.parametrize("conv1_planes", [2], indirect=True)
@pytest.mark.parametrize("B,N", [(2, 3), (48, 96)])
def test_conv1_planes_ring_equals_gathered_at_budget_7(dev, B, N, conv1_planes):
    """with 7 CTAs each takes 6-192 tiles and the row producer's four-tile prefetch crosses images, the obs / next_obs
    boundary and episodes that wrap around the ring"""
    from drqv2_b200 import _lib
    nstep, pad = 3, 4
    g = torch.Generator().manual_seed(N)
    ring = _ring(dev)
    src, es, ix, keep = _ring_batch(ring, B, nstep, 11 * N, dev)
    obs, nxt = _gathered(ring, es, ix, nstep)
    stacks = torch.cat([obs, nxt])[:N].contiguous().to(dev)
    shift = torch.randint(0, 2 * pad + 1, (N, 2), dtype=torch.int32, generator=g).to(dev)
    w = ((torch.rand(32, 9, 3, 3, generator=g) - 0.5) * 0.3).to(dev)
    b = ((torch.rand(32, generator=g) - 0.5) * 0.1).to(dev)
    wp = torch.zeros(_lib.lib().drq_conv1_w_packed_elems(), dtype=torch.bfloat16, device=dev)
    _lib.call("drq_pack_conv1_w_bf16", w.data_ptr(), b.data_ptr(), wp.data_ptr(), 9, _stream())
    y0 = fill_sentinel(torch.empty(_lib.lib().drq_wb_elems(N + 1), dtype=torch.bfloat16, device=dev))
    y1 = fill_sentinel(torch.empty_like(y0))
    with _budget(7):
        _lib.call("drq_conv1_fwd_bf16", stacks.data_ptr(), shift.data_ptr(), wp.data_ptr(), y0.data_ptr(), N, 9, pad, _stream())
        _lib.call("drq_conv1_fwd_bf16_ring", C.byref(src), B, shift.data_ptr(), wp.data_ptr(), y1.data_ptr(), N, pad, _stream())
    torch.cuda.synchronize()
    what = f"conv1 fwd planes, ring B={B} N={N} budget=7"
    assert bits_equal(y0, y1), what
    assert wb_region(y0, N, 41, 41).float().abs().sum() > 0
    assert_sentinel_outside(y1, wb_written(y1.numel(), N, 41, 41, dev), what)
    assert ((es.astype(np.int64) + ix + nstep - 1) >= ring.capacity).any(), "a sampled window must wrap"
    _record(what, dict(tiles=14 * N, ctas=7, per_cta=-(-14 * N // 7)))
    del keep
