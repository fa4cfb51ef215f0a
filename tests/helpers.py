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


# ---- exact reference of the random draws (csrc/ring.cu): Philox4x32-10 keyed by the seed, counter word
# (counter << 3) | stream, element index in the low 64 bits.  The integer draws are oracle.update_shifts and
# oracle.sample_indices (multiply-shift reductions, bit-exact); normals are Box-Muller on a pair of words with u formed
# in fp32 exactly as the kernels form it.
STREAM_SAMPLE, STREAM_SHIFT, STREAM_EPS, STREAM_NOISE = 0, 1, 3, 5
NORMAL_C = 8.0               # |got - want| <= NORMAL_C * 2^-24 * rad (sqrt(-2 ln u1))
INT_SENTINEL = 0x7FFFFFFF


def philox_words(seed, stream, counter, index):
    """uint64 [len(index)][4]: the four 32-bit words of key `seed` at counter word (counter << 3) | stream"""
    from oracle import drq_oracle as O
    return O.philox4x32(int(seed), (int(counter) << 3) | int(stream), np.asarray(index, np.uint64))


def uniform24(w):
    """((float)(w >> 8) + 0.5f) * 2^-24 in fp32: above 2^23 the + 0.5 rounds to even, so the upper half lies on a
    2^-23 grid and w >> 8 == 0xFFFFFF gives exactly 1.0"""
    u = (np.asarray(w, np.uint64) >> np.uint64(8)).astype(np.float32)
    return (u + np.float32(0.5)) * np.float32(2.0 ** -24)


def box_muller(w_rad, w_ang, odd, use_sin_for_odd=True):
    """(normal, rad) in fp64 from the fp32 uniforms of two words: rad * cos(2 pi u2), sin for odd elements"""
    u1 = uniform24(w_rad).astype(np.float64)
    u2 = uniform24(w_ang).astype(np.float64)
    rad = np.sqrt(-2.0 * np.log(u1))
    ang = 2.0 * np.pi * u2
    odd = np.asarray(odd, bool) & use_sin_for_odd
    return np.where(odd, rad * np.sin(ang), rad * np.cos(ang)), rad


def normals_ref(seed, stream, counter, n, words=(0, 1)):
    """element i of an N(0,1) draw: pair i >> 1 on words `words` of the Philox block"""
    i = np.arange(n, dtype=np.int64)
    r = philox_words(seed, stream, counter, i >> 1)
    return box_muller(r[:, words[0]], r[:, words[1]], (i & 1).astype(bool))


def update_draws_ref(seed, counter, pad, B, A):
    """the four draws of one update: dict of shift_obs, shift_next, eps_critic / eps_actor (words 0-1 / 2-3 of
    stream 3) and their rad"""
    from oracle import drq_oracle as O
    so, sn = O.update_shifts(seed, counter, pad, B)
    ec, rc = normals_ref(seed, STREAM_EPS, counter, B * A, (0, 1))
    ea, ra = normals_ref(seed, STREAM_EPS, counter, B * A, (2, 3))
    return dict(shift_obs=so, shift_next=sn, eps_critic=ec, rad_critic=rc, eps_actor=ea, rad_actor=ra)


def check_normals(got, want, rad, what):
    """|got - want| <= NORMAL_C 2^-24 rad element-wise (a NaN fails).  Returns the largest |got - want| / (2^-24 rad):
    the constant this draw needed.  A word or pair mix-up is off by O(1) and misses the bound by ~10^6."""
    got = np.asarray(got, np.float64).ravel()
    want, rad = np.asarray(want, np.float64).ravel(), np.asarray(rad, np.float64).ravel()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    unit = 2.0 ** -24 * rad
    err = np.abs(got - want)
    bad = ~(err <= NORMAL_C * unit)
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.size} normals outside |got - want| <= {NORMAL_C:g} "
                             f"2^-24 rad, first at {i}: got {got[i]!r}, want {want[i]!r}, rad {rad[i]!r}")
    live = unit > 0
    return float((err[live] / unit[live]).max()) if live.any() else 0.0


def assert_bits_equal(got, want, what):
    """integer draws and gathered values: equal bit for bit, with the first difference named"""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.dtype.kind == "f":
        got, want = got.view(np.int32 if got.itemsize == 4 else np.int64), want.astype(got.dtype).view(
            np.int32 if got.itemsize == 4 else np.int64)
    diff = got != want
    if diff.any():
        i = np.unravel_index(int(np.flatnonzero(diff)[0]), got.shape)
        raise AssertionError(f"{what}: {int(diff.sum())} of {got.size} differ, first at {tuple(int(v) for v in i)}: "
                             f"got {got[i]!r}, want {want[i]!r}")


# ---- the agent's key schedule: which (seed, stream, counter) keys each public call consumes
def key_schedule(calls, seed, loader_seed):
    """calls: sequence of "act", "act_eval", "update", "update_skip", "stage_critic", "stage_actor" -> list of
    (call, agent counter before, [keys consumed]) with a key (seed, stream, counter).  Each call that draws takes the
    agent counter once and advances it by one; an update also takes the loader's counter (its own seed, stream 0)."""
    c = lc = 0
    out = []
    for call in calls:
        keys = []
        if call in ("act", "stage_critic", "stage_actor"):
            keys = [(seed, STREAM_NOISE, c)]
        elif call == "update":
            keys = [(seed, STREAM_SHIFT, c), (seed, STREAM_EPS, c), (loader_seed, STREAM_SAMPLE, lc)]
            lc += 1
        else:
            assert call in ("act_eval", "update_skip"), call
        out.append((call, c, keys))
        if keys:
            c += 1
    return out


def assert_keys_disjoint(schedule):
    """no (seed, stream, counter) key is consumed twice"""
    seen = {}
    for k, (call, _, keys) in enumerate(schedule):
        for key in keys:
            assert key not in seen, f"key {key} of call {k} ({call}) was consumed before by call {seen[key]}"
            seen[key] = k


# ---- host model of the replay ring's episode bookkeeping (replay_buffer.GpuRing), by slot ownership
class RingModel:
    """Episodes are written one after another at the head, modulo capacity; an episode stays resident while every slot
    it was written to still holds it (FIFO eviction of whole episodes).  table(min_len) is what the sampler sees:
    (start slot, len = rows - 1) of the resident episodes with len >= min_len, the newest max_episodes of them."""

    def __init__(self, capacity, max_episodes):
        self.cap, self.max_episodes = capacity, max_episodes
        self.owner = np.full(capacity, -1, np.int64)
        self.head, self.n_added = 0, 0
        self.episodes = []                   # (episode id, start slot, rows), oldest first

    def add(self, rows):
        eid, start = self.n_added, self.head
        self.n_added += 1
        self.owner[(start + np.arange(rows)) % self.cap] = eid
        self.head = (start + rows) % self.cap
        self.episodes = [(e, s, r) for e, s, r in self.episodes + [(eid, start, rows)]
                         if (self.owner[(s + np.arange(r)) % self.cap] == e).all()]
        return eid

    def resident(self):
        return [(s, r) for _, s, r in self.episodes]

    def table(self, min_len):
        return [(s, r - 1) for _, s, r in self.episodes if r - 1 >= min_len][-self.max_episodes:]


def episode_content(eid, rows, A, frame_c=3):
    """distinct per-(episode, row) frames / action / reward / discount for the ring tests; discounts hold zeros"""
    t = np.arange(rows)
    frames = ((eid * 131 + t.reshape(-1, 1, 1, 1) * 7 + np.arange(frame_c).reshape(1, -1, 1, 1) * 3 +
               np.arange(84).reshape(1, 1, -1, 1) + 2 * np.arange(84).reshape(1, 1, 1, -1)) % 251).astype(np.uint8)
    action = (eid * 1000 + t.reshape(-1, 1) * 10 + np.arange(A).reshape(1, -1)).astype(np.float32)
    reward = (eid + t / 1024.0).astype(np.float32)
    discount = np.where((eid + t) % 4 == 0, 0.0, 1.0 - t / 4096.0).astype(np.float32)
    return frames, action, reward, discount


def check_ring_holds(table, frames, action, reward, discount, contents, cap, what):
    """every table entry (start, len) still holds, in slots [start, start + len + 1) mod cap, the frames / action /
    reward / discount of the episode written there.  contents: {start slot: (frames, action, reward, discount)} of the
    resident episodes"""
    for s, ln in table:
        want = contents.get(int(s))
        assert want is not None, f"{what}: table entry at slot {s} is no resident episode"
        rows = int(ln) + 1
        assert want[0].shape[0] == rows, f"{what}: table entry at slot {s}: len {ln}, the episode has {want[0].shape[0]} rows"
        slots = (int(s) + np.arange(rows)) % cap
        for name, arr, w in (("frames", frames, want[0]), ("action", action, want[1]), ("reward", reward, want[2]),
                             ("discount", discount, want[3])):
            assert np.array_equal(arr[slots], w.reshape(arr[slots].shape)), \
                f"{what}: {name} of the episode at slot {s} was overwritten"


# the sequence of public calls whose keys test_gpu_draws.py reads back and test_draws_cpu.py models: two exploration
# acts, an eval act, a step update() skips, updates (eager warm-up, graph capture + replay, replays), a batched
# exploration act and the stage API's two noise draws
AGENT_SCRIPT = ("act", "act", "act_eval", "update_skip", "update", "update", "update", "update", "act",
                "stage_critic", "stage_actor")
