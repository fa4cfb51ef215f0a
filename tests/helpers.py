"""Shared test helpers: the integer formulas the golden inputs were generated with
(tests/golden/make_golden.py) and probe positions; WB / TB layout conversions; the element-wise error bounds and the
stray-store sentinels of the kernel tests (self-tested in test_conv_checks_cpu.py, test_gemm_schedule_cpu.py and
test_fp32_schedule_cpu.py)."""
import numpy as np


def frame_formula(e, t):
    c = np.arange(3).reshape(3, 1, 1)
    y = np.arange(84).reshape(1, 84, 1)
    x = np.arange(84).reshape(1, 1, 84)
    return ((31 * e + 17 * t + 7 * c + 3 * y + 5 * x + (x * y) % 11 + (e + 1) * (t + 2) * (x + y) % 13) % 256).astype(np.uint8)


def scalar_formula(e, t, A):
    action = (((np.arange(A) * 37 + e * 11 + t * 5) % 200) / 100.0 - 1.0).astype(np.float32)
    reward = np.float32(((e * 7 + t * 13) % 97) / 97.0)
    discount = np.float32(1.0 if (t + e) % 5 else 0.9)
    return action, reward, discount


def episode_arrays(e, T, A):
    """Per-row single frames + scalars of golden episode e (rows 0..T; row 0 = reset dummy:
    action 0, reward 0, discount 1 — dmc.py:160-168)."""
    frames = np.stack([frame_formula(e, t) for t in range(T + 1)])
    action = np.zeros((T + 1, A), np.float32)
    reward = np.zeros((T + 1, 1), np.float32)
    discount = np.ones((T + 1, 1), np.float32)
    for t in range(1, T + 1):
        a, r, d = scalar_formula(e, t, A)
        action[t], reward[t, 0], discount[t, 0] = a, r, d
    return frames, action, reward, discount


def aug_input(N, C):
    n = np.arange(N).reshape(N, 1, 1, 1)
    c = np.arange(C).reshape(1, C, 1, 1)
    y = np.arange(84).reshape(1, 1, 84, 1)
    x = np.arange(84).reshape(1, 1, 1, 84)
    return ((n * 53 + c * 29 + y * y * 3 + x * 7 + (x * y) % 17) % 256).astype(np.uint8)


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ---- bf16 "WB" layout helpers (see include/drqv2_b200.h): torch-side conversions for tests
PLB, GUARD, WB_SLACK = 1776, 88, 128


def wb_from_nchw(x):
    """x float [N,32,H,W] (H,W <= 41) -> WB bf16 tensor [4][N*PLB+SLACK][8] on x.device."""
    import torch
    N, C, H, W = x.shape
    wide = torch.zeros(N, C, 41, 41, dtype=torch.float32, device=x.device)
    wide[:, :, :H, :W] = x
    rows = torch.zeros(N, PLB, C, dtype=torch.float32, device=x.device)
    rows[:, GUARD:GUARD + 1681, :] = wide.view(N, C, 1681).permute(0, 2, 1)
    wb = torch.zeros(4, N * PLB + WB_SLACK, 8, dtype=torch.bfloat16, device=x.device)
    wb[:, :N * PLB, :] = rows.view(N * PLB, 4, 8).permute(1, 0, 2).to(torch.bfloat16)
    return wb.contiguous()


def nchw_from_wb(wb, N, H, W):
    """inverse of wb_from_nchw: float32 [N,32,H,W] (only the valid region)."""
    rows = wb[:, :N * PLB, :].float().permute(1, 0, 2).reshape(N, PLB, 32)
    wide = rows[:, GUARD:GUARD + 1681, :].permute(0, 2, 1).reshape(N, 32, 41, 41)
    return wide[:, :, :H, :W].contiguous()


# ---- element-wise error bound and stray-store sentinels for the bf16 conv kernels
# A bf16 NaN that no kernel computes: every output buffer is filled with it before a call, and every element the call
# must not write has to hold it afterwards, bit for bit.
SENTINEL_BITS = 0x7FA5
F32_SENTINEL_BITS = 0x7FA5A5A5      # the same for fp32 outputs


def _sentinel_view(buf):
    import torch
    if buf.dtype == torch.float32:
        return buf.view(torch.int32), F32_SENTINEL_BITS
    return buf.view(torch.int16), SENTINEL_BITS


def fill_sentinel(buf):
    """bf16 or fp32 buffer -> every element the sentinel NaN of its type"""
    bits, s = _sentinel_view(buf)
    bits.fill_(s)
    return buf


def assert_sentinel_outside(buf, written, what):
    """every element of `buf` (bf16 or fp32, any shape) where the bool tensor `written` (same number of elements) is False
    still holds the sentinel"""
    bits, s = _sentinel_view(buf.reshape(-1))
    stray = (bits != s) & ~written.reshape(-1)
    n = int(stray.sum())
    assert n == 0, f"{what}: {n} elements outside the written set were overwritten, first at flat index " \
                   f"{int(stray.nonzero()[0])}"


def assert_conv_bound(got, want, absref, what, rel=2.0 ** -8, absc=2.0 ** -14):
    """|got - want| <= rel * |want| + absc * absref element-wise.  Returns (the largest |got - want| / bound, the largest
    share of the absolute term absc * absref used by what the bf16 round does not explain).

    want is fp64 math on the bf16-rounded operands and absref the same operation on their absolute values (the sum of
    |products|, plus |bias|).  The products are exact in fp32, so the kernel's error is the fp32 sum - at most about
    terms * 2^-24 * absref, 1.7e-5 * absref for a 288-term sum - and the final bf16 round.  bf16 keeps 8 significant
    bits, so that round alone is up to 2^-8 / (1 + 2^-8) relative: the first ratio reaches ~0.9 on a correct kernel."""
    import torch
    got, want, absref = got.double(), want.double(), absref.double()
    err = (got - want).abs()
    bound = rel * want.abs() + absc * absref
    bad = ~(err <= bound)                       # a NaN (an unwritten sentinel) fails too
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside |got - want| <= {rel:g}|want| + {absc:g}A, "
                             f"first at {i}: got {float(got[i])!r}, want {float(want[i])!r}, A {float(absref[i])!r}")
    if not err.numel():
        return 0.0, 0.0
    live = bound > 0
    ratio = torch.where(live, err / bound.clamp_min(1e-300), torch.zeros_like(err))
    rounding = 2.0 ** -8 / (1 + 2.0 ** -8) * want.abs()
    rest = torch.where(live, (err - rounding).clamp_min(0) / (absc * absref).clamp_min(1e-300), torch.zeros_like(err))
    return float(ratio.max()), float(rest.max())


def assert_f32_bound(got, want, absref, chain, c, what):
    """|got - want| <= c * 2^-24 * chain * A element-wise, for fp32 outputs of the tensor-core GEMM.  chain is the UMMA
    accumulation chain of the element's tile, ceil(K_chunk / 16) (scalar or broadcastable), A the same GEMM on absolute
    values plus |bias|.  The bf16 products are exact in fp32, so the error is the fp32 accumulation alone.  Returns the
    largest |got - want| / (2^-24 * chain * A): the c this output needed."""
    import torch
    got, want, absref = got.double(), want.double(), absref.double()
    unit = 2.0 ** -24 * chain * absref
    err = (got - want).abs()
    bad = ~(err <= c * unit)                    # a NaN (an unwritten sentinel) fails too
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside |got - want| <= {c:g} 2^-24 chain A, first at "
                             f"{i}: got {float(got[i])!r}, want {float(want[i])!r}, A {float(absref[i])!r}")
    if not err.numel():
        return 0.0
    need = torch.where(unit > 0, err / unit.clamp_min(1e-300), torch.zeros_like(err))
    return float(need.max())


def check_sum_bound(kernel, got, want, absref, n, ratios=None, c=2.0):
    """|got - want| <= c 2^-24 (n + 8) A element-wise, for fp32 results that are sums along chains of at most n
    sequential fp32 steps; A the same sum over absolute values (a NaN fails).  The largest |got - want| / bound goes into
    ratios[kernel] (the share of c the kernel needed)."""
    import torch
    got, want = got.double(), want.double()
    bound = c * 2.0 ** -24 * (n + 8) * absref.double()
    err = (got - want).abs()
    bad = ~(err <= bound)
    if bad.any():
        i = int(bad.reshape(-1).nonzero()[0])
        raise AssertionError(f"{kernel}: {int(bad.sum())} elements out of bound, first at flat {i}: got "
                             f"{float(got.reshape(-1)[i])!r} want {float(want.reshape(-1)[i])!r}")
    r = float(torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.zeros_like(err)).max()) if err.numel() else 0.0
    if ratios is not None:
        ratios[kernel] = max(ratios.get(kernel, 0.0), r)
    return r


def max_norm_ok(got, want):
    """the older, max-normalised check: |got - want| <= 2^-8 max|want| everywhere"""
    return bool((got.double() - want.double()).abs().max() <= 2.0 ** -8 * want.double().abs().max())


def wb_cs(N):
    """pixel rows per channel block of a WB buffer of N images (the block stride a kernel derives from N)"""
    return N * PLB + WB_SLACK


def wb_written(n_elems, N, rows, cols, device=None):
    """bool [n_elems] over a bf16 buffer holding (at its start) a WB layout of N images: True at the pixels
    (y < rows, x < cols) of images < N, in all four channel blocks"""
    import torch
    cs = wb_cs(N)
    unit = torch.zeros(n_elems // 8, dtype=torch.bool, device=device)
    n = torch.arange(N, device=device).view(N, 1, 1)
    y = torch.arange(rows, device=device).view(1, rows, 1)
    x = torch.arange(cols, device=device).view(1, 1, cols)
    pix = (n * PLB + GUARD + y * 41 + x).reshape(-1)
    for c in range(4):
        unit[c * cs + pix] = True
    return unit.repeat_interleave(8)


def wb_region(buf, N, H, W):
    """the bf16 values of images < N, rows < H, columns < W of a WB buffer of N images -> [N][32][H][W] (bf16)"""
    cs = wb_cs(N)
    rows = buf.reshape(-1)[:4 * cs * 8].view(4, cs, 8)[:, :N * PLB, :].permute(1, 0, 2).reshape(N, PLB, 32)
    wide = rows[:, GUARD:GUARD + 41 * 41, :].permute(0, 2, 1).reshape(N, 32, 41, 41)
    return wide[:, :, :H, :W]


def tb_feature_rows(tb_view, rows, hout):
    """rows of a TB feature matrix view [rpad][4*hout*hout*8] in the encoder-output feature order
    (c/8)*hout*hout*8 + (y*hout + x)*8 + c%8 -> [len(rows)][32][hout][hout] (bf16)"""
    r = tb_view[list(rows), :hout * hout * 32]
    return r.reshape(len(rows), 4, hout * hout, 8).permute(0, 1, 3, 2).reshape(len(rows), 32, hout, hout)


def bits_equal(a, b):
    import torch
    return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))


def check_conv_fwd_outputs(out, feat, tb_view, tb_rows, want, absref, N, hout, wb_cols, what):
    """the three outputs of one conv2-4 forward, each in a sentinel-filled buffer one size too big: `out` WB of N + 1
    images, `feat` NHWC [N + 1][hout*hout][32], `tb_view` the [rpad][units*8] view of a TB feature matrix whose image n
    is row tb_rows[n].  WB within the error bound, and the set it writes is rows < hout, columns < wb_cols of images < N;
    NHWC images < N and TB rows tb_rows equal WB bit for bit; nothing else is written.  Returns the error-to-bound ratio."""
    import torch
    dev = out.device
    got = wb_region(out, N, hout, hout)
    ratio = assert_conv_bound(got, want, absref, what)
    assert_sentinel_outside(out, wb_written(out.numel(), N, hout, wb_cols, dev), what + " WB")
    assert bits_equal(feat[:N].view(N, hout, hout, 32).permute(0, 3, 1, 2), got), what + ": NHWC != WB"
    written = torch.zeros(feat.shape, dtype=torch.bool, device=dev)
    written[:N] = True
    assert_sentinel_outside(feat, written, what + " NHWC")
    assert bits_equal(tb_feature_rows(tb_view, tb_rows, hout), got), what + ": TB != WB"
    rows = torch.zeros(tb_view.shape[0], dtype=torch.bool, device=dev)
    rows[list(tb_rows)] = True
    assert_sentinel_outside(tb_view, rows.view(-1, 1).expand(tb_view.shape), what + " TB")
    return ratio
