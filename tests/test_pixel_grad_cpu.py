"""Encoder(pixels=...) and DrQV2Agent(pixels=...) flag handling, and CPU restatements of the new kernels' index logic:
the random-shift backward's gather ranges against autograd of oracle.random_shift_exact (bit for bit on dyadic
gradients), and the tile / carry schedule of drq_conv1_dgrad_bf16 (every input pixel written exactly once)."""
import pickle

import pytest
import torch

from oracle import drq_oracle as O


def test_pixels_flag_validation_and_pickle_default():
    from drqv2_b200 import Encoder
    from drqv2_b200.drqv2 import DrQV2Agent
    assert Encoder((9, 84, 84)).pixels == "u8"
    assert Encoder((9, 84, 84), pixels="float").pixels == "float"
    for bad in ("f32", "U8", True, None, 1):
        with pytest.raises(ValueError):
            Encoder((9, 84, 84), pixels=bad)
        with pytest.raises(ValueError):
            DrQV2Agent((9, 84, 84), (6,), "cpu", 1e-4, 50, 1024, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, False,
                       pixels=bad)
    enc = Encoder((9, 84, 84), pixels="float")
    del enc.__dict__["pixels"]                  # an instance pickled before the flag existed
    back = pickle.loads(pickle.dumps(enc))
    assert back.pixels == "u8" and "pixels" not in back.__dict__
    assert pickle.loads(pickle.dumps(Encoder((9, 84, 84), pixels="float"))).pixels == "float"


def shift_bwd_formula(dout, shift, pad):
    """drq_random_shift_bwd_f32 restated: pixel (i, j) sums dout over the row range / column range whose clamped
    source it is, rows and columns ascending"""
    N, C, H, W = dout.shape
    dx = torch.zeros_like(dout)
    for n in range(N):
        dxs, dys = int(shift[n, 0]) - pad, int(shift[n, 1]) - pad
        for i in range(H):
            rlo, rhi = max(0 if i == 0 else i - dys, 0), min(H - 1 if i == H - 1 else i - dys, H - 1)
            for j in range(W):
                clo, chi = max(0 if j == 0 else j - dxs, 0), min(W - 1 if j == W - 1 else j - dxs, W - 1)
                acc = torch.zeros(C, dtype=dout.dtype)
                for r in range(rlo, rhi + 1):
                    for c in range(clo, chi + 1):
                        acc = acc + dout[n, :, r, c]
                dx[n, :, i, j] = acc
    return dx


@pytest.mark.parametrize("H", [7, 84])
@pytest.mark.parametrize("pad", [0, 1, 2, 3, 4])
def test_shift_backward_gather_formula(H, pad):
    sx, sy = torch.meshgrid(torch.arange(2 * pad + 1), torch.arange(2 * pad + 1), indexing="ij")
    shift = torch.stack([sx.reshape(-1), sy.reshape(-1)], 1)
    if H == 84:
        shift = shift[torch.randperm(shift.shape[0], generator=torch.Generator().manual_seed(pad))[:6]]
    n = shift.shape[0]
    g = torch.Generator().manual_seed(10 * H + pad)
    dout = torch.randint(-512, 513, (n, 2, H, H), generator=g).double() / 64
    x = torch.zeros(n, 2, H, H, dtype=torch.float64, requires_grad=True)
    want, = torch.autograd.grad(O.random_shift_exact(x, shift, pad), x, dout)
    assert torch.equal(shift_bwd_formula(dout, shift, pad), want)


def dgrad_bf16_schedule(N, grid):
    """drq_conv1_dgrad_bf16's schedule: CTA b takes images b, b + grid, ...; per image the 14 tiles of three output rows
    in order; tile t writes input rows 6t .. 6t+5 (and 78 .. 83 at t = 13: 78..82 from taps, 83 as +0) and carries
    row 6t+6.  Returns per image the write count of every input row, and checks each carried row is consumed by the
    next tile of the same CTA."""
    writes = [[0] * 84 for _ in range(N)]
    for b in range(min(N, grid)):
        for n in range(b, N, grid):
            carried = None
            for t in range(14):
                oy0 = 3 * t
                R = min(3, 41 - oy0)
                rows = list(range(2 * oy0, 2 * oy0 + 2 * R + 1))
                if t > 0:
                    assert carried == rows[0]
                carried = None
                for iy in rows:
                    if iy == rows[-1] and t < 13:
                        carried = iy
                    else:
                        writes[n][iy] += 1
                if t == 13:
                    writes[n][83] += 1
            assert carried is None
    return writes


def test_dgrad_bf16_taps_per_tile():
    """every (output row, ky) tap lands in the tile that holds its output row, and the rows a tile completes take all
    their taps from it and the carry"""
    for iy in range(84):
        taps = [(iy - ky) // 2 for ky in range(3) if (iy - ky) >= 0 and (iy - ky) % 2 == 0 and (iy - ky) // 2 < 41]
        tiles = {oy // 3 for oy in taps}
        if iy == 83:
            assert taps == []
        elif iy % 6 == 0 and iy > 0:
            assert tiles == {iy // 6 - 1, iy // 6}, iy       # the carried row: one tap from each neighbour tile
        else:
            assert len(tiles) <= 1


@pytest.mark.parametrize("N", [1, 2, 7, 48, 129, 256, 512, 1000])
@pytest.mark.parametrize("sms", [148, 140, 7, 1])
def test_dgrad_bf16_every_pixel_written_once(N, sms):
    grid = min(N, 2 * sms)
    writes = dgrad_bf16_schedule(N, grid)
    assert all(w == [1] * 84 for w in writes)
