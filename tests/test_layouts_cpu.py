"""CPU checks of the host-side mirror of the C ABI: the ctypes job structs have exactly the layout gcc gives the
header's structs, and the tile-blocked (TB) layout helpers address what include/drqv2_b200.h documents."""
import ctypes as C
import pathlib
import shutil
import subprocess

import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent

STRUCTS = {   # header struct -> (ctypes mirror, fields)
    "drq_pack_job": ("PackJob", ["kind", "rows", "cols", "reserved", "w", "bias", "out", "out2"]),
    "drq_colsum_job": ("ColsumJob", ["X", "ld", "out", "M", "N", "tb", "reserved", "Y"]),
    "drq_opt_seg": ("OptSeg", ["kind", "ema", "rows", "cols", "off", "n", "out", "out2"]),
    "drq_wgrad_reduce_job": ("WgReduceJob", ["partial", "dw", "db", "n_images", "hout", "cin", "reserved"]),
    "drq_ln_job": ("LnJob", ["partial", "ld_partial", "split_stride", "S", "bias", "gamma", "beta", "h_out", "ld_h", "xhat",
                             "rstd", "h_bf16", "units_bf16", "row0_bf16", "tail", "ld_tail", "n_tail"]),
    "drq_policy_sample": ("PolicySample", ["row0", "rows", "eps", "action_out", "ld_a", "mu_out", "metrics", "a_bf16",
                                           "units_a", "feat_off", "reserved"]),
    "drq_ring_src": ("replay_buffer.RingSrc", ["frames", "action", "reward", "discount", "capacity", "frame_c", "stack", "A",
                                               "nstep", "gamma", "reserved", "ep_table", "n_episodes", "seed", "counter",
                                               "ep_start", "idx"]),
}


@pytest.mark.skipif(shutil.which("gcc") is None, reason="gcc not available")
def test_ctypes_structs_match_the_header(tmp_path):
    from drqv2_b200 import _bf16, replay_buffer
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{ROOT / "include" / "drqv2_b200.h"}"', "int main(void) {"]
    for cname, (_, fields) in STRUCTS.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for f in fields:
            lines.append(f'  printf("{cname} {f} %zu\\n", offsetof({cname}, {f}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = {tuple(l.split()[:2]): int(l.split()[2]) for l in out if l.strip()}
    for cname, (pyname, fields) in STRUCTS.items():
        cls = getattr(replay_buffer, pyname.split(".")[1]) if "." in pyname else getattr(_bf16, pyname)
        assert C.sizeof(cls) == got[(cname, "size")], cname
        assert [f for f, _ in cls._fields_] == fields, cname
        for f in fields:
            assert getattr(cls, f).offset == got[(cname, f)], (cname, f)


def test_tb_layout_round_trip_and_addressing():
    """TB element (row, feat) of entry z sits at z*stride + ((row/R)*units + feat/8)*R*8 + (row%R)*8 + feat%8."""
    from drqv2_b200._bf16 import TB
    from drqv2_b200._lib import TB_ACT, TB_W
    g = torch.Generator().manual_seed(0)
    for rows, feats, batch, R in ((5, 56, 2, TB_W), (300, 50, 1, TB_ACT), (64, 1024, 4, TB_W), (130, 21, 1, TB_ACT)):
        t = TB(rows, feats, "cpu", batch=batch, rblk=R)
        assert t.units == (feats + 15) // 16 * 2 and t.rpad % R == 0 and t.rpad >= rows
        assert t.buf.numel() == batch * t.stride and t.stride == t.units * t.rpad * 8
        xs = []
        for z in range(batch):
            x = torch.randn(rows, feats, generator=g).to(torch.bfloat16)
            t.load(x, z)
            xs.append(x)
        for z in range(batch):
            assert torch.equal(t.dense(z), xs[z].float())
            for row, feat in ((0, 0), (rows - 1, feats - 1), (rows // 2, feats // 3)):
                idx = z * t.stride + ((row // R) * t.units + feat // 8) * R * 8 + (row % R) * 8 + feat % 8
                assert t.buf[idx] == xs[z][row, feat]
            # padding rows / features are zero
            assert float(t.view(z)[rows:].abs().sum()) == 0 and float(t.view(z)[:, feats:].abs().sum()) == 0
        assert t.off(batch - 1, R * ((rows - 1) // R), 8 * ((feats - 1) // 8)) < t.buf.numel()


def test_splitk_chunks_are_never_empty():
    """drq_gemm_bf16 rejects a split-K whose last chunk would be empty; the chooser must never produce one."""
    from drqv2_b200._bf16 import splitk_for
    from drqv2_b200._lib import REPR_DIM
    for ctas in range(1, 149):
        for K in (REPR_DIM, 1024, 4096):
            S = splitk_for(ctas, K)
            chunk = -(-(-(-K // S)) // 128) * 128
            assert S >= 1 and chunk * (S - 1) < K, (ctas, K, S)


def _lin_tile(cols, tile=1024):
    """Python restatement of lin_tile() in drqv2_b200/csrc/optim.cu (generic LINEAR segments of drq_adam_pack_step)."""
    c8 = (cols + 7) // 8 * 8
    CW = min(c8, 256)
    rt, p2 = tile // CW, 1
    while p2 * 2 <= rt and p2 < 32:
        p2 *= 2
    chunks = (cols + CW - 1) // CW
    width = cols if chunks == 1 else CW
    SW = (CW + 55) // 64 * 64 + 8
    return CW, p2, SW, chunks, width


def test_fused_optimiser_linear_tiling_covers_every_element_once():
    """The block -> (rows, columns) tiling of a generic Linear weight: every element is visited exactly once, the
    staged bf16 tile fits the kernel's shared buffer, 16-byte unit reads are aligned and bank-staggered."""
    SH_BF16 = 32 * 72                              # kOptShBf16
    for cols in list(range(1, 80)) + [100, 127, 255, 256, 257, 300, 511, 1000, 1025]:
        if cols % 8 == 0:
            continue                               # multiples of 8 take the flat float4 path
        CW, RT, SW, chunks, width = _lin_tile(cols)
        assert RT * width <= 1024 and RT * SW <= SH_BF16 and SW >= CW and SW % 8 == 0 and SW % 64 == 8
        rows = 37
        seen = {}
        blocks = ((rows + RT - 1) // RT) * chunks
        for b in range(blocks):
            rb, ch = divmod(b, chunks)
            r0, c0 = rb * RT, ch * CW
            for e in range(RT * width):
                lr, cc = divmod(e, width)
                r, c = r0 + lr, c0 + cc
                if r < rows and c < cols:
                    assert lr * SW + cc < RT * SW
                    seen[(r, c)] = seen.get((r, c), 0) + 1
            # units written by this block cover exactly its columns
            ul_n = (width + 7) // 8
            for ul in range(ul_n):
                if c0 + ul * 8 < cols:
                    assert (c0 // 8 + ul) * 8 < (cols + 15) // 16 * 16
        assert len(seen) == rows * cols and set(seen.values()) == {1}, cols
