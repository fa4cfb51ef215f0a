"""CPU check of the tile schedule and the TB feature epilogue of csrc/conv4x1_tc.cu, statement by statement: tile_pos /
tile_at (image-pair-major tile numbering, pair rounds, then single tiles), the epilogue's choice between one 32-byte
store for the same pixel of two images and 16-byte stores, and the TB addresses both write.  The tiles' sums themselves
are checked by test_conv4x1_index_cpu.py; here a tile's result is the reference output, so the test is about where every
value lands and that it lands once.  The second half emulates the stage layout and the UMMA operand offsets of the
grouped tiles against torch's convolutions."""
import numpy as np
import pytest
import torch

from tests.test_conv4x1_index_cpu import compact_weights, expand, win_cnt, win_oy0

TB_ACT = 128


def tiles_per_image(hout):
    return ((hout + 3) // 4 + 2) // 3


def launch_params(N, tpi, grid_budget=148):
    total = N * tpi
    grid = min(total, grid_budget)
    return dict(N=N, tpi=tpi, total=total, pair_tiles=(N & ~1) * tpi, grid=grid, pair_rounds=total // (2 * grid))


def tile_pos(p, t):
    if t < p["pair_tiles"]:
        q, rem = divmod(t, 2 * p["tpi"])
        return 2 * q + (rem & 1), rem >> 1
    return p["N"] - 1, t - p["pair_tiles"]


def tile_at(p, b, k):
    q2, g = 2 * p["pair_rounds"], p["grid"]
    return 2 * (b + (k >> 1) * g) + (k & 1) if k < q2 else q2 * g + b + (k - q2) * g


def cta_tiles(p, b):
    k, out = 0, []
    while (t := tile_at(p, b, k)) < p["total"]:
        out.append((k, t))
        k += 1
    return out


@pytest.mark.parametrize("N,hout,budget", [(512, 35, 148), (512, 39, 148), (512, 37, 148), (511, 35, 148), (7, 35, 148),
                                           (1, 35, 148), (10, 39, 4), (9, 6, 4), (256, 41, 140)])
def test_schedule_covers_every_tile_once(N, hout, budget):
    tpi = tiles_per_image(hout)
    p = launch_params(N, tpi, budget)
    seen = {}
    most = 0
    for b in range(p["grid"]):
        mine = cta_tiles(p, b)
        most = max(most, len(mine))
        for k, t in mine:
            assert t not in seen
            seen[t] = tile_pos(p, t)
            if k < 2 * p["pair_rounds"] and not (k & 1) and t < p["pair_tiles"]:
                (n0, tau0), (n1, tau1) = tile_pos(p, t), tile_pos(p, t + 1)
                assert (n1, tau1) == (n0 + 1, tau0) and n0 % 2 == 0 and mine[k + 1][1] == t + 1
    assert sorted(seen) == list(range(p["total"]))
    assert sorted(set(seen.values())) == [(n, tau) for n in range(N) for tau in range(tpi)]
    # as many tiles on the busiest CTA as a plain round robin over the grid
    assert most == -(-p["total"] // p["grid"])


def emulate_tb_epilogue(want, p, hout, feat_half, feat_half_row, n_rows_pad):
    """want [N][32][hout][hout]; returns the TB buffer [rows/128][4*hw][128][8] and the sizes of the stores issued"""
    hw = hout * hout
    feat_rpad = 4 * hw
    tb = np.full((n_rows_pad // TB_ACT, feat_rpad, TB_ACT, 8), np.nan)
    written = np.zeros(tb.shape[:3], int)
    sizes = []
    flat = tb.reshape(-1)
    wflat = written.reshape(-1)

    def tb_row(n):
        return n if n < feat_half else n - feat_half + feat_half_row

    def tb_unit(fr, c, u):                      # element offset, as the kernel's pointer arithmetic
        return (((fr >> 7) * feat_rpad + c * hw + u) * TB_ACT + (fr & 127)) * 8

    def store(off, vals):
        assert off % len(vals) == 0              # a 16-byte store on 16 bytes, a 32-byte store on 32
        assert np.isnan(flat[off:off + len(vals)]).all()
        flat[off:off + len(vals)] = vals
        wflat[off // 8:(off + len(vals)) // 8] += 1
        sizes.append(len(vals) * 2)

    def pixel(n, y, x, c):
        return want[n, 8 * c:8 * c + 8, y, x]

    for b in range(p["grid"]):
        k = 0
        while (t := tile_at(p, b, k)) < p["total"]:
            n, tau = tile_pos(p, t)
            two = ((k & 1) == 0 and k < 2 * p["pair_rounds"] and t < p["pair_tiles"] and
                   tb_row(n + 1) == tb_row(n) + 1 and (tb_row(n) & 1) == 0)
            for half in range(2):
                for m in range(123):
                    r, x = divmod(m, 41)
                    y0 = 4 * (tau * 3 + r) + 2 * half
                    for o in range(2):
                        y = y0 + o
                        if y >= hout or x >= hout:
                            continue
                        u = y * hout + x
                        for c in range(4):
                            if two:
                                store(tb_unit(tb_row(n), c, u), np.concatenate([pixel(n, y, x, c), pixel(n + 1, y, x, c)]))
                            else:
                                store(tb_unit(tb_row(n), c, u), pixel(n, y, x, c))
            k += 2 if two else 1
    return tb, written, sizes


@pytest.mark.parametrize("N,hout,feat_half,feat_half_row,budget", [
    (24, 35, 12, 128, 8),        # an update's [obs | next] halves, B even
    (14, 35, 7, 128, 4),         # B odd: the pair that straddles the halves goes one image at a time
    (14, 35, 7, 129, 5),         # the second half starts on an odd row: no pair is adjacent there
    (11, 35, 11, 0, 4),          # odd N: the last image has no partner; pair rounds and a tail of single tiles
    (9, 6, 9, 0, 2),             # one tile per image
])
def test_tb_feature_epilogue_writes_every_unit_once(N, hout, feat_half, feat_half_row, budget):
    g = torch.Generator().manual_seed(N * 100 + hout)
    want = torch.rand(N, 32, hout, hout, generator=g, dtype=torch.float64).numpy()
    p = launch_params(N, tiles_per_image(hout), budget)
    rows = [n if n < feat_half else n - feat_half + feat_half_row for n in range(N)]
    n_rows_pad = (max(rows) // TB_ACT + 1) * TB_ACT
    tb, written, sizes = emulate_tb_epilogue(want, p, hout, feat_half, feat_half_row, n_rows_pad)
    hw = hout * hout
    for n, fr in enumerate(rows):
        assert (written[fr // TB_ACT, :, fr % TB_ACT] == 1).all()
        # unit (c/8)*h*h + y*h + x holds channels 8(c/8) .. 8(c/8) + 7 of pixel (y, x)
        got = tb[fr // TB_ACT, :, fr % TB_ACT].reshape(4, hout, hout, 8).transpose(0, 3, 1, 2).reshape(32, hout, hout)
        assert np.array_equal(got, want[n])
    assert written.sum() == N * 4 * hw
    if p["pair_rounds"] > 0 and feat_half % 2 == 0 and feat_half_row % 2 == 0:
        assert 32 in sizes


# ---------------------------------------------------------------------------------------------------------------------
# The stage of a tile: six regions (window rows wy) x four channel blocks x three slots x 41 pixels, landed by three TMA
# boxes of two row planes; slots are three block rows of one image, or one block row of three images (grouped tiles).

PW, SLOTS, PAD_UNITS = 41, 3, 8
PLB, GUARD = 1776, 88                # WB pixel rows per image, zero guard rows in front of each
SLAB = SLOTS * PW                    # 16-byte units of one (region, channel block)
REGION = 4 * SLAB


def reorder_weights(wc, dgrad):
    """expand_weights: unit u = ((wx * 4 + ku) * 3 + j) * 32 + co of [wx][k/8][j][n][k%8] <- compact unit
    (tap * 4 + ku) * 32 + co, tap = dy * 3 + dx, dy = 2 - j (data gradient: j), dx = wx (2 - wx); [1152][8]"""
    buf = np.full((3 * 4 * 3 * 32, 8), np.nan)
    for u in range(buf.shape[0]):
        co, r = u & 31, u >> 5
        wk, j = divmod(r, 3)
        wx, ku = wk >> 2, wk & 3
        dy, dx = (j, 2 - wx) if dgrad else (2 - j, wx)
        buf[u] = wc[dy * 3 + dx, 8 * ku:8 * ku + 8, co]
    return buf


def b_operand(buf, wy, wx):
    """the UMMA's B for window element (wy, wx): K-major, start unit win_unit0, K units 96 rows apart -> [32 k][32 cnt n]"""
    u0, n = (wx * 12 + 2 - wy + win_oy0(wy)) * 32, 32 * win_cnt(wy)
    return np.concatenate([buf[u0 + 96 * ku:u0 + 96 * ku + n].T for ku in range(4)], axis=0)


@pytest.mark.parametrize("dgrad", [False, True])
def test_reordered_weights_give_every_window_element_its_operand(dgrad):
    """every (wy, wx) reads, through one descriptor, the B operand of the per-window-element expansion"""
    g = torch.Generator().manual_seed(7 + dgrad)
    w = (torch.rand(32, 32, 3, 3, generator=g, dtype=torch.float64) - 0.5).numpy()
    wc = compact_weights(w, dgrad)
    buf = reorder_weights(wc, dgrad)
    assert np.isfinite(buf).all()
    want = expand(wc, dgrad)
    for wy in range(6):
        for wx in range(3):
            assert np.array_equal(b_operand(buf, wy, wx), want[wy, wx])


def conv_tiles(N, h_out):
    """the launcher's tile counts: per-image tiles, and grouped tiles when block_rows % 3 == 1"""
    block_rows = (h_out + 3) // 4
    grouped = block_rows % 3 == 1
    tpi = block_rows // 3 if grouped else -(-block_rows // 3)
    return block_rows, tpi, N * tpi + (-(-N // 3) if grouped else 0)


def tile_pos_conv(N, tpi, block_rows, t):
    """tile_pos: (n, i0, grouped)"""
    pair_tiles, image_tiles = (N & ~1) * tpi, N * tpi
    if t < pair_tiles:
        q, rem = divmod(t, 2 * tpi)
        return 2 * q + (rem & 1), 3 * (rem >> 1), False
    if t < image_tiles:
        return N - 1, 3 * (t - pair_tiles), False
    return 3 * (t - image_tiles), block_rows - 1, True


def wb_row(wide, N, img, row):
    """pixel row `row` of image `img` as the WB buffer holds it [41][32]: rows 41..43 run into the next image's guard
    (zeros) and then its first pixels - NaN here, as is the slack past the last image: nothing may depend on them"""
    if row < PW:
        return wide[img, :, row, :].T
    out = np.full((PW, 32), np.nan)
    for x in range(PW):
        if GUARD + row * PW + x - PLB < GUARD:
            out[x] = 0.0
    return out


def stage_of_tile(wide, N, n, i0, grouped, dgrad, row_blocks):
    """the three boxes of the producer -> [PAD_UNITS zeros | 6 regions][32 channels as 4 blocks]; row blocks >= row_blocks
    and images >= N are the TMA's zero fill"""
    st = np.full((PAD_UNITS + 6 * REGION + 16, 8), np.nan)      # + what follows the stage
    st[:PAD_UNITS] = 0.0
    for b in range(3):
        plane0 = (0 if b == 1 else 2) if dgrad else (2 if b == 1 else 0)
        rb0 = i0 + ((-1 if b == 0 else 0) if dgrad else (1 if b == 2 else 0))
        for pl in range(2):
            for cb in range(4):
                for s in range(SLOTS):
                    img, rb = (n + s, rb0) if grouped else (n, rb0 + s)
                    row = 4 * rb + plane0 + pl
                    dst = PAD_UNITS + (2 * b + pl) * REGION + cb * SLAB + s * PW
                    if not (0 <= rb < row_blocks and img < N):
                        st[dst:dst + PW] = 0.0                    # TMA out-of-range fill
                    else:
                        st[dst:dst + PW] = wb_row(wide, N, img, row)[:, 8 * cb:8 * cb + 8]
    return st


def emulate_conv(wide, w, h_layer_out, dgrad):
    N = wide.shape[0]
    h_out = h_layer_out + 2 if dgrad else h_layer_out
    block_rows, tpi, total = conv_tiles(N, h_out)
    row_blocks = ((h_layer_out if dgrad else h_layer_out + 2) + 3) // 4      # the tensor maps: valid input rows only
    buf = reorder_weights(compact_weights(w, dgrad), dgrad)
    out = np.zeros((N, 32, h_out, h_out))
    written = np.zeros((N, h_out, h_out), bool)
    for t in range(total):
        n, i0, grouped = tile_pos_conv(N, tpi, block_rows, t)
        st = stage_of_tile(wide, N, n, i0, grouped, dgrad, row_blocks)
        D = np.zeros((128, 128))
        for wy in (2, 5, 3, 1, 4, 0):
            cnt, col = win_cnt(wy), 32 * win_oy0(wy)
            for wx in range(3):
                base = PAD_UNITS + wy * REGION + wx - (2 if dgrad else 0)
                # rows m of the A operand: K unit cb at base + cb * SLAB (the descriptor's leading-byte offset) + m
                A = np.concatenate([st[base + cb * SLAB:base + cb * SLAB + 128] for cb in range(4)], axis=1)
                prod = A @ b_operand(buf, wy, wx)
                if wx == 0 and wy in (2, 5):
                    D[:, col:col + 32 * cnt] = prod
                else:
                    D[:, col:col + 32 * cnt] += prod
        for m in range(123):
            r, x = divmod(m, PW)
            img, i = (n + r, i0) if grouped else (n, i0 + r)
            for oy in range(4):
                y = 4 * i + oy
                if img < N and y < h_out and (dgrad or x < h_out):
                    if x >= h_out:
                        assert np.all(D[m, oy * 32:oy * 32 + 32] == 0)   # the data gradient's zero columns
                        continue
                    assert not written[img, y, x]
                    written[img, y, x] = True
                    out[img, :, y, x] = D[m, oy * 32:oy * 32 + 32]
    assert written.all()
    return out, total


@pytest.mark.parametrize("hout,N", [(39, 3), (39, 4), (39, 5), (37, 3), (37, 4), (37, 2), (35, 3), (35, 2), (6, 1), (6, 3)])
def test_conv4x1_forward_grouped_stage(hout, N):
    g = torch.Generator().manual_seed(hout * 10 + N)
    hin = hout + 2
    x = torch.rand(N, 32, hin, hin, generator=g, dtype=torch.float64)
    w = torch.rand(32, 32, 3, 3, generator=g, dtype=torch.float64) - 0.5
    want = torch.nn.functional.conv2d(x, w).numpy()
    wide = np.full((N, 32, PW, PW), np.nan)              # columns and rows beyond the valid input: never needed
    wide[:, :, :hin, :hin] = x.numpy()
    got, total = emulate_conv(wide, w.numpy(), hout, False)
    assert np.isfinite(got).all()
    assert np.abs(got - want).max() <= 1e-10
    if hout in (39, 37):
        assert total == 3 * N + -(-N // 3)


@pytest.mark.parametrize("hout,N", [(39, 3), (39, 4), (37, 5), (35, 3), (35, 2), (6, 2)])
def test_conv4x1_dgrad_grouped_stage(hout, N):
    g = torch.Generator().manual_seed(200 + hout * 10 + N)
    d = torch.rand(N, 32, hout, hout, generator=g, dtype=torch.float64) - 0.5
    w = torch.rand(32, 32, 3, 3, generator=g, dtype=torch.float64) - 0.5
    want = torch.nn.functional.conv_transpose2d(d, w).numpy()
    wide = np.zeros((N, 32, PW, PW))                     # gradient buffers are zero outside the valid region
    wide[:, :, :hout, :hout] = d.numpy()
    got, _ = emulate_conv(wide, w.numpy(), hout, True)
    assert np.isfinite(got).all()
    assert np.abs(got - want).max() <= 1e-10


def test_grouped_tiles_per_sm_at_512_images():
    for hout in (39, 37):
        assert -(-conv_tiles(512, hout)[2] // 148) == 12
    assert -(-conv_tiles(512, 35)[2] // 148) == 11
