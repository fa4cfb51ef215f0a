"""The checks of test_gpu_conv_schedule_edges.py against planted defects, without a GPU.  A correct "kernel output" is
built from the fp64 reference, rounded to bf16 and stored as the kernels store it (WB, NHWC and TB buffers one size too
big, sentinel everywhere else); the checks must accept it and reject each defect below - evidence that the GPU tests
can fail."""
import pytest
import torch

from tests.helpers import (GUARD, PLB, WB_SLACK, check_conv_fwd_outputs, fill_sentinel, max_norm_ok, wb_cs)


def _wb_store(vals, N_buf):
    """a sentinel WB buffer of N_buf images holding vals [N][32][H][W] (bf16) at the pixels of images < N"""
    N, _, H, W = vals.shape
    buf = fill_sentinel(torch.empty(4 * (N_buf * PLB + WB_SLACK) * 8, dtype=torch.bfloat16))
    cs = wb_cs(N)
    blk = buf[:4 * cs * 8].view(4, cs, 8)
    pix = (torch.arange(N).view(N, 1, 1) * PLB + GUARD + torch.arange(H).view(1, H, 1) * 41 + torch.arange(W).view(1, 1, W))
    blk[:, pix.reshape(-1), :] = vals.reshape(N, 4, 8, H, W).permute(1, 0, 3, 4, 2).reshape(4, -1, 8)
    return buf


def _outputs(vals, tb_rows, tb_vals=None):
    """WB, NHWC and TB buffers as a correct kernel leaves them; tb_vals [rows][32][H][W] overrides what lands in the TB
    rows (row order of tb_rows)"""
    N, _, H, _ = vals.shape
    out = _wb_store(vals, N + 1)
    feat = fill_sentinel(torch.empty(N + 1, H * H, 32, dtype=torch.bfloat16))
    feat[:N] = vals.permute(0, 2, 3, 1).reshape(N, H * H, 32)
    rpad = -(-(max(tb_rows) + 2) // 128) * 128
    tb = fill_sentinel(torch.empty(rpad, H * H * 32, dtype=torch.bfloat16))
    src = vals if tb_vals is None else tb_vals
    tb[list(tb_rows)] = src.reshape(len(tb_rows), 4, 8, H * H).permute(0, 1, 3, 2).reshape(len(tb_rows), -1)
    return out, feat, tb


def _case(N, hout, seed):
    g = torch.Generator().manual_seed(seed)
    hin = hout + 2
    x = torch.rand(N, 32, hin, hin, generator=g).to(torch.bfloat16).double()
    w = ((torch.rand(32, 32, 3, 3, generator=g) * 2 - 1) * 0.1).to(torch.bfloat16).double()
    b = ((torch.rand(32, generator=g) * 2 - 1) * 0.1).double()
    want = torch.relu(torch.nn.functional.conv2d(x, w, b))
    absref = torch.nn.functional.conv2d(x.abs(), w.abs(), b.abs())
    return x, w, b, want, absref


def _check(vals, want, absref, N, hout, tb_rows, tb_vals=None):
    out, feat, tb = _outputs(vals, tb_rows, tb_vals)
    return check_conv_fwd_outputs(out, feat, tb, tb_rows, want, absref, N, hout, hout, "planted")


def _rows(N, fh, fhr):
    return [n if n < fh else n - fh + fhr for n in range(N)]


N, HOUT = 14, 39          # 39 rows = 10 block rows: grouped last block rows; N = 14 = 1 mod 3: a one-image last group
FH, FHR = 7, 128          # an odd first half: images 6 and 7 are a pair of tiles whose TB rows (6, 128) are not adjacent


@pytest.fixture(scope="module")
def case():
    return _case(N, HOUT, 5)


def test_correct_output_is_accepted(case):
    _, _, _, want, absref = case
    ratio, rest = _check(want.to(torch.bfloat16), want, absref, N, HOUT, _rows(N, FH, FHR))
    # the bf16 round of the exact value: up to 2^-8 / (1 + 2^-8) relative, nothing left for the absolute term
    assert ratio < 1 and rest < 1e-6


def test_rejects_a_zeroed_row_of_the_last_grouped_block_row(case):
    _, _, _, want, absref = case
    vals = want.to(torch.bfloat16)
    vals[N - 1, :, 37, :] = 0            # block row 9 = rows 36..38 of the last image: its grouped tile holds it alone
    with pytest.raises(AssertionError, match="outside"):
        _check(vals, want, absref, N, HOUT, _rows(N, FH, FHR))


def test_rejects_the_two_images_of_a_pair_swapped_in_tb(case):
    _, _, _, want, absref = case
    vals = want.to(torch.bfloat16)
    tb_vals = vals.clone()
    tb_vals[[2, 3]] = vals[[3, 2]]
    with pytest.raises(AssertionError, match="TB != WB"):
        _check(vals, want, absref, N, HOUT, _rows(N, FH, FHR), tb_vals)


def test_rejects_a_paired_store_into_a_non_adjacent_partners_row(case):
    """images 6 and 7 are the tiles of one pair round, but their rows are 6 and 128: a 32-byte store at row 6 writes
    image 7 into row 7 (the first row of nothing) and leaves row 128 unwritten"""
    _, _, _, want, absref = case
    vals = want.to(torch.bfloat16)
    rows = _rows(N, FH, FHR)
    out, feat, tb = _outputs(vals, rows)
    tb[7] = tb[128]
    fill_sentinel(tb[128])
    with pytest.raises(AssertionError, match="TB"):
        check_conv_fwd_outputs(out, feat, tb, rows, want, absref, N, HOUT, HOUT, "planted")
    # the stray store alone (row 128 right as well) is caught by the sentinel
    out, feat, tb = _outputs(vals, rows)
    tb[7] = tb[128]
    with pytest.raises(AssertionError, match="outside the written set"):
        check_conv_fwd_outputs(out, feat, tb, rows, want, absref, N, HOUT, HOUT, "planted")


def test_rejects_one_channel_blocks_bias_dropped(case):
    x, w, b, want, absref = case
    b2 = b.clone()
    b2[8:16] = 0
    vals = torch.relu(torch.nn.functional.conv2d(x, w, b2)).to(torch.bfloat16)
    with pytest.raises(AssertionError, match="outside"):
        _check(vals, want, absref, N, HOUT, _rows(N, FH, FHR))


def test_rejects_a_zeroed_small_pixel_the_max_normalised_bound_accepts(case):
    _, _, _, want, absref = case
    # an output well above the absolute term 2^-14 A and well below the old bound's 2^-8 max|want|
    small = (want > 4 * 2.0 ** -14 * absref) & (want < 0.5 * 2.0 ** -8 * want.abs().max())
    assert small.any()
    i = tuple(int(v) for v in small.nonzero()[0])
    vals = want.to(torch.bfloat16)
    vals[i] = 0
    assert max_norm_ok(vals, want)
    with pytest.raises(AssertionError, match="outside"):
        _check(vals, want, absref, N, HOUT, _rows(N, FH, FHR))


def test_rejects_a_store_past_the_valid_width_and_into_the_next_image(case):
    """the four-pixel-column forward writes valid pixels only: a value at x = hout, or in image N, is a stray store"""
    _, _, _, want, absref = case
    vals = want.to(torch.bfloat16)
    for n, y, x in ((0, 0, HOUT), (N, 0, 0)):
        out, feat, tb = _outputs(vals, _rows(N, FH, FHR))
        out.view(-1)[(0 * wb_cs(N) + n * PLB + GUARD + y * 41 + x) * 8] = 0
        with pytest.raises(AssertionError, match="outside the written set"):
            check_conv_fwd_outputs(out, feat, tb, _rows(N, FH, FHR), want, absref, N, HOUT, HOUT, "planted")
