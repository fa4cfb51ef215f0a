"""The values the update's random draws, replay sample and scalar ring produce, against the exact reference of
tests/helpers.py (Philox4x32-10 restated on the host).  The whole-update tests feed the oracle the draws and the batch
the update actually used, so a draw that is consistent but wrong (repeated noise, eps_critic equal to eps_actor, shifts
that repeat past the first pass of a loop, a sample from an overwritten episode) passes all of them; here every producer
is held to what it must draw: integers bit for bit, normals within NORMAL_C 2^-24 rad (a word or pair mix-up is off by
O(1)).  Every output buffer is one element too big and holds a sentinel that must survive, and every counter / cursor
must move by exactly one per call.  Run on the B200 box: pytest -m gpu tests/test_gpu_draws.py."""
import ctypes
import pathlib

import numpy as np
import pytest
import torch

from oracle import drq_oracle as O
from tests.helpers import (AGENT_SCRIPT, F32_SENTINEL_BITS, INT_SENTINEL, STREAM_NOISE, RingModel, assert_bits_equal,
                           assert_keys_disjoint, check_normals, check_ring_holds, episode_content, key_schedule,
                           normals_ref, update_draws_ref)

pytestmark = pytest.mark.gpu

SCHED = "linear(1.0,0.1,100000)"
SHAPES = [(1, 1), (2, 1), (1, 128), (255, 6), (256, 6), (171, 6), (257, 3), (512, 21), (512, 80), (1023, 1),
          (1024, 1), (1025, 1), (4097, 1)]
SEEDS = (0, 77, 2 ** 32 + 5, None, 2 ** 63 - 1)          # None: dist.rank_seed(123, 1)
COUNTERS = (0, 1, 2 ** 29 - 1, 2 ** 29, 2 ** 32 + 3, 2 ** 40)
PADS = (0, 1, 4)
# (seed 77) counters at which pair 0 of a normal draw has w >> 8 == 0xFFFFFF (u1 = 1.0: a normal of +-0) or 0 (the
# largest rad), found by an exhaustive search of the reference: stream 5 word 0; stream 3 words 0 (critic) and 2 (actor)
EDGE_NOISE = (456791, 24107590)
EDGE_EPS = (2371879, 12129983, 6767034, 11946318)
RING_CAP = 97
RING_TABLE = [(0, 40), (41, 7), (49, 30), (80, 35)]          # the last episode wraps past the ring end
RATIOS = {}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _call(name, *args):
    from drqv2_b200 import _lib
    _lib.call(name, *args)


def _seed(s):
    from drqv2_b200 import dist
    return dist.rank_seed(123, 1) if s is None else s


def f32_out(n, dev):
    return torch.empty(n + 1, dtype=torch.float32, device=dev).view(torch.int32).fill_(F32_SENTINEL_BITS).view(torch.float32)


def i32_out(shape, dev):
    return torch.full(tuple(np.atleast_1d(shape)), INT_SENTINEL, dtype=torch.int32, device=dev)


def assert_f32_tail(buf, n, what):
    assert int(buf.view(torch.int32)[n]) == F32_SENTINEL_BITS, f"{what}: element {n} (one past the end) was written"


def ratio(entry, r):
    RATIOS[entry] = max(RATIOS.get(entry, 0.0), r)
    return r


def report(capsys, line):
    with capsys.disabled():
        print("\n" + line, end="")


# ----------------------------------------------------------------------------- the ring source of the prologue
class RingSource:
    """a device ring with RING_TABLE as its episode table, a scalar ring and the drq_ring_src over it"""

    def __init__(self, dev, A, B, nstep=3, gamma=0.99, seed=5, slots=3):
        from drqv2_b200 import replay_buffer as R
        g = np.random.default_rng(A * 7 + B)
        self.A, self.B, self.nstep, self.gamma, self.seed = A, B, nstep, gamma, seed
        self.host = dict(action=(g.random((RING_CAP, A), dtype=np.float32) * 2 - 1),
                         reward=g.random(RING_CAP, dtype=np.float32),
                         discount=np.where(g.random(RING_CAP) < 0.2, 0.0, 0.97).astype(np.float32))
        self.frames = torch.zeros(RING_CAP, 16, dtype=torch.uint8, device=dev)      # the prologue reads no frames
        self.action, self.reward, self.discount = (torch.from_numpy(self.host[k]).to(dev) for k in ("action", "reward", "discount"))
        self.table = torch.full((8, 2), -1, dtype=torch.int32, device=dev)
        self.table[:len(RING_TABLE)] = torch.tensor(RING_TABLE, dtype=torch.int32)
        self.n_ep = torch.tensor([len(RING_TABLE)], dtype=torch.int32, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.ep_start, self.idx = i32_out(B + 1, dev), i32_out(B + 1, dev)
        self.src = R.RingSrc(self.frames.data_ptr(), self.action.data_ptr(), self.reward.data_ptr(), self.discount.data_ptr(),
                             RING_CAP, 3, 3, A, nstep, gamma, 0, self.table.data_ptr(), self.n_ep.data_ptr(), seed,
                             self.counter.data_ptr(), self.ep_start.data_ptr(), self.idx.data_ptr())
        self.scal_ring = (torch.arange(slots * 32, dtype=torch.float32) + 1).view(slots, 32).pin_memory()
        self.slots = slots

    def scalars_want(self, B):
        """oracle.ring_gather's action / n-step reward / discount of the samples (ep_start, idx) the kernel wrote"""
        es, ix = self.ep_start[:B].cpu().numpy(), self.idx[:B].cpu().numpy()
        h = self.host
        frames = np.zeros((RING_CAP, 1, 84, 84), np.uint8)             # the prologue gathers no frames
        _, act, rew, disc, _ = O.ring_gather(frames, h["action"], h["reward"], h["discount"], es, ix, self.nstep,
                                             self.gamma, stack=1)
        return act.reshape(-1), rew.reshape(-1), disc.reshape(-1)


class DrawBufs:
    """the four draw outputs of one update, each one element too big and sentinel-filled"""

    def __init__(self, dev, B, A):
        self.B, self.A = B, A
        self.so, self.sn = i32_out((B + 1, 2), dev), i32_out((B + 1, 2), dev)
        self.ec, self.ea = f32_out(B * A, dev), f32_out(B * A, dev)
        self.scal = f32_out(32, dev)

    def ptrs(self):
        return self.so.data_ptr(), self.sn.data_ptr(), self.ec.data_ptr(), self.ea.data_ptr()

    def check(self, want, entry, what, shifts=True, eps=True):
        B, n = self.B, self.B * self.A
        if shifts:
            assert_bits_equal(self.so[:B].cpu().numpy(), want["shift_obs"], what + " shift_obs")
            assert_bits_equal(self.sn[:B].cpu().numpy(), want["shift_next"], what + " shift_next")
        else:
            assert (self.so[:B] == INT_SENTINEL).all() and (self.sn[:B] == INT_SENTINEL).all(), what + ": shifts written"
        assert (self.so[B] == INT_SENTINEL).all() and (self.sn[B] == INT_SENTINEL).all(), what + ": shift row B written"
        if eps:
            ratio(entry, check_normals(self.ec[:n].cpu().numpy(), want["eps_critic"], want["rad_critic"], what + " eps_critic"))
            ratio(entry, check_normals(self.ea[:n].cpu().numpy(), want["eps_actor"], want["rad_actor"], what + " eps_actor"))
        else:
            for t in (self.ec, self.ea):
                assert (t.view(torch.int32)[:n] == F32_SENTINEL_BITS).all(), what + ": noise written"
        assert_f32_tail(self.ec, n, what + " eps_critic")
        assert_f32_tail(self.ea, n, what + " eps_actor")


def _prologue_ring(rs, bufs, seed, counter, cursor, pad, part, draws=True, out=None):
    B, A = bufs.B, bufs.A
    so, sn, ec, ea = bufs.ptrs() if draws else (None, bufs.sn.data_ptr(), bufs.ec.data_ptr(), bufs.ea.data_ptr())
    act, rew, disc = out
    _call("drq_update_prologue_ring_part", rs.scal_ring.data_ptr(), rs.slots, cursor.data_ptr(), bufs.scal.data_ptr(),
          seed, counter.data_ptr(), pad, so, sn, ec, ea, B, A, ctypes.byref(rs.src), act.data_ptr(), rew.data_ptr(), disc.data_ptr(),
          part, _stream())


# ----------------------------------------------------------------------------- 1. every draw producer
@pytest.mark.parametrize("B, A", SHAPES)
def test_draw_producers_match_reference(dev, B, A, capsys):
    """drq_rng_update_draws, drq_update_prologue, drq_update_prologue_ring (part 3, and parts 1 + 2), drq_ring_sample,
    drq_ring_sample_step and drq_rng_normal_f32 at shapes where the one-block kernels' strided loops run 0, 1 or several
    extra passes (B*A past 1024, B past 256), at every seed, counter and pad"""
    k0 = SHAPES.index((B, A))
    combos = [(_seed(SEEDS[(k0 + j) % len(SEEDS)]), COUNTERS[j], PADS[(k0 + j) % len(PADS)]) for j in range(len(COUNTERS))]
    if 2 <= B * A <= 128:
        combos += [(77, c, 4) for c in EDGE_NOISE + EDGE_EPS]
    n = B * A
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    cursor = torch.zeros(1, dtype=torch.int64, device=dev)
    rs = RingSource(dev, A, B)
    for seed, c, pad in combos:
        tag = f"B={B} A={A} seed={seed} counter={c} pad={pad}"
        want = update_draws_ref(seed, c, pad, B, A)
        # drq_rng_update_draws: does not advance the counter
        bufs = DrawBufs(dev, B, A)
        counter.fill_(c)
        _call("drq_rng_update_draws", seed, counter.data_ptr(), pad, *bufs.ptrs(), B, A, _stream())
        bufs.check(want, "drq_rng_update_draws", "rng_update_draws " + tag)
        assert int(counter) == c
        # drq_update_prologue: draws, counter + 1, cursor + 1
        bufs = DrawBufs(dev, B, A)
        cursor.fill_(5)
        _call("drq_update_prologue", rs.scal_ring.data_ptr(), rs.slots, cursor.data_ptr(), bufs.scal.data_ptr(), seed,
              counter.data_ptr(), pad, *bufs.ptrs(), B, A, _stream())
        bufs.check(want, "drq_update_prologue", "update_prologue " + tag)
        assert int(counter) == c + 1 and int(cursor) == 6, tag
        # drq_update_prologue_ring part 3, then parts 1 + 2 on fresh buffers
        for parts in ((3,), (1, 2)):
            bufs = DrawBufs(dev, B, A)
            out = (f32_out(n, dev), f32_out(B, dev), f32_out(B, dev))
            rs.ep_start.fill_(INT_SENTINEL)
            rs.idx.fill_(INT_SENTINEL)
            counter.fill_(c)
            cursor.fill_(5)
            lc = (c * 3 + 1) % 2 ** 41
            rs.counter.fill_(lc)
            for part in parts:
                _prologue_ring(rs, bufs, seed, counter, cursor, pad, part, out=out)
                if part == 1:      # part 1: shifts and sample only; neither the counter nor the cursor moves
                    assert int(counter) == c and int(cursor) == 5 and int(rs.counter) == lc + 1, tag
                    bufs.check(want, None, "prologue_ring part 1 " + tag, eps=False)
            entry = "drq_update_prologue_ring part " + "+".join(map(str, parts))
            bufs.check(want, entry, entry + " " + tag)
            assert int(counter) == c + 1 and int(cursor) == 6 and int(rs.counter) == lc + 1, tag
            es, ix = O.sample_indices(RING_TABLE, rs.nstep, rs.seed, lc, B)
            assert_bits_equal(rs.ep_start[:B].cpu().numpy(), es, entry + " ep_start " + tag)
            assert_bits_equal(rs.idx[:B].cpu().numpy(), ix, entry + " idx " + tag)
            assert int(rs.ep_start[B]) == INT_SENTINEL and int(rs.idx[B]) == INT_SENTINEL, tag
            for got, w, m, name in zip(out, rs.scalars_want(B), (n, B, B), ("action", "reward", "discount")):
                assert_bits_equal(got[:m].cpu().numpy(), w, f"{entry} {name} {tag}")
                assert_f32_tail(got, m, f"{entry} {name}")
        # the two sampler kernels, with this combo's seed and counter
        for kern in ("drq_ring_sample", "drq_ring_sample_step"):
            rs.ep_start.fill_(INT_SENTINEL)
            rs.idx.fill_(INT_SENTINEL)
            rs.counter.fill_(c)
            _call(kern, rs.table.data_ptr(), rs.n_ep.data_ptr(), 3, seed, rs.counter.data_ptr(), rs.ep_start.data_ptr(),
                  rs.idx.data_ptr(), B, _stream())
            es, ix = O.sample_indices(RING_TABLE, 3, seed, c, B)
            assert_bits_equal(rs.ep_start[:B].cpu().numpy(), es, f"{kern} ep_start {tag}")
            assert_bits_equal(rs.idx[:B].cpu().numpy(), ix, f"{kern} idx {tag}")
            assert int(rs.ep_start[B]) == INT_SENTINEL and int(rs.idx[B]) == INT_SENTINEL, tag
            assert int(rs.counter) == c + (kern == "drq_ring_sample_step"), tag
        # drq_rng_normal_f32 (stream 5): does not advance the counter
        out = f32_out(n, dev)
        counter.fill_(c)
        _call("drq_rng_normal_f32", seed, counter.data_ptr(), out.data_ptr(), n, _stream())
        w, rad = normals_ref(seed, STREAM_NOISE, c, n)
        ratio("drq_rng_normal_f32", check_normals(out[:n].cpu().numpy(), w, rad, "rng_normal_f32 " + tag))
        assert_f32_tail(out, n, "rng_normal_f32")
        assert int(counter) == c
    report(capsys, f"draws B={B} A={A}: largest normal error / (2^-24 rad) so far: " +
           ", ".join(f"{k} {v:.2f}" for k, v in sorted(RATIOS.items())))


# ----------------------------------------------------------------------------- 2. the scalar ring and the injected path
@pytest.mark.parametrize("slots", [1, 3, 256])
def test_scalar_ring_slot_and_injected_path(dev, slots):
    """drq_scalars_fetch, drq_update_prologue and prologue-ring parts 2 / 3 read slot cursor % slots into out[0, 32)
    and nothing past it, cursor + 1; part 1 reads no scalars; the injected path (shift_obs == NULL) writes no draw and
    leaves the counter alone"""
    B, A = 5, 3
    rs = RingSource(dev, A, B, slots=slots)
    ring = rs.scal_ring
    counter = torch.zeros(1, dtype=torch.int64, device=dev)
    cursor = torch.zeros(1, dtype=torch.int64, device=dev)
    for cur in (0, 255, 256, 2 ** 32 - 1, 2 ** 32):
        want = ring[cur % slots].numpy()

        def check(entry, bufs, moved=True):
            got = bufs.scal
            if moved:
                assert_bits_equal(got[:32].cpu().numpy(), want, f"{entry} scalars, slots {slots}, cursor {cur}")
                assert int(cursor) == cur + 1, (entry, slots, cur)
            else:
                assert (got.view(torch.int32)[:32] == F32_SENTINEL_BITS).all(), entry
                assert int(cursor) == cur, (entry, slots, cur)
            assert_f32_tail(got, 32, entry + " scalars")

        bufs = DrawBufs(dev, B, A)
        cursor.fill_(cur)
        _call("drq_scalars_fetch", ring.data_ptr(), slots, cursor.data_ptr(), bufs.scal.data_ptr(), _stream())
        check("drq_scalars_fetch", bufs)
        for draws in (True, False):
            bufs = DrawBufs(dev, B, A)
            cursor.fill_(cur)
            counter.fill_(7)
            so, sn, ec, ea = bufs.ptrs()
            _call("drq_update_prologue", ring.data_ptr(), slots, cursor.data_ptr(), bufs.scal.data_ptr(), 77,
                  counter.data_ptr(), 4, so if draws else None, sn, ec, ea, B, A, _stream())
            check("drq_update_prologue", bufs)
            assert int(counter) == 7 + draws
            if not draws:
                bufs.check(None, None, "update_prologue injected", shifts=False, eps=False)
        for part in (1, 2, 3):
            for draws in (True, False):
                bufs = DrawBufs(dev, B, A)
                out = (f32_out(B * A, dev), f32_out(B, dev), f32_out(B, dev))
                cursor.fill_(cur)
                counter.fill_(7)
                rs.counter.fill_(0)
                if part == 2:          # part 2 gathers at the indices part 1 drew
                    rs.ep_start[:B] = 41
                    rs.idx[:B] = torch.arange(1, B + 1, dtype=torch.int32, device=dev)
                _prologue_ring(rs, bufs, 77, counter, cursor, 4, part, draws=draws, out=out)
                check(f"prologue_ring part {part}", bufs, moved=part != 1)
                assert int(counter) == 7 + (draws and part != 1), (part, draws)
                assert int(rs.counter) == (part != 2), part
                if not draws:
                    bufs.check(None, None, f"prologue_ring part {part} injected", shifts=False, eps=False)


# ----------------------------------------------------------------------------- 3. the sampler
def _tables():
    mixed = [(0, 10), (11, 11), (23, 40), (64, 13), (78, 97)]
    E = 50_000
    big = np.stack([(np.arange(E) * 37) % 99_991, 10 + (np.arange(E) * 7919) % 1013], 1)
    return [("E=1, span 1", None), ("mixed", mixed), ("E=50000", big)]


@pytest.mark.parametrize("nstep", [1, 3, 10])
def test_sampler_kernels_match_reference(dev, nstep):
    """drq_ring_sample, drq_ring_sample_step and prologue-ring part 1 against the reference, bit for bit; table rows
    past n_episodes hold -1 and must not be read"""
    from drqv2_b200 import replay_buffer as R
    for name, table in _tables():
        table = np.array([[5, nstep]] if table is None else table, np.int64)
        E = len(table)
        dtab = torch.full((E + 16, 2), -1, dtype=torch.int32, device=dev)
        dtab[:E] = torch.from_numpy(table.astype(np.int32))
        n_ep = torch.tensor([E], dtype=torch.int32, device=dev)
        for B in (1, 256, 257, 4097):
            seed, c = _seed(SEEDS[B % 5]), COUNTERS[B % 6]
            es_w, ix_w = O.sample_indices(table, nstep, seed, c, B)
            if name.startswith("E=1"):
                assert (ix_w == 1).all()
            ctr = torch.tensor([c], dtype=torch.int64, device=dev)
            es, ix = i32_out(B + 1, dev), i32_out(B + 1, dev)
            for kern in ("drq_ring_sample", "drq_ring_sample_step", "part 1"):
                ctr.fill_(c)
                es.fill_(INT_SENTINEL)
                ix.fill_(INT_SENTINEL)
                if kern == "part 1":
                    src = R.RingSrc(dtab.data_ptr(), dtab.data_ptr(), dtab.data_ptr(), dtab.data_ptr(), 1 << 30, 3, 3, 1,
                                    nstep, 0.99, 0, dtab.data_ptr(), n_ep.data_ptr(), seed, ctr.data_ptr(), es.data_ptr(),
                                    ix.data_ptr())
                    scal = torch.zeros(32, device=dev)
                    cur = torch.zeros(1, dtype=torch.int64, device=dev)
                    o = torch.zeros(B, device=dev)
                    _call("drq_update_prologue_ring_part", scal.data_ptr(), 1, cur.data_ptr(), scal.data_ptr(), 0, None, 0,
                          None, None, None, None, B, 1, ctypes.byref(src), o.data_ptr(), o.data_ptr(), o.data_ptr(), 1, _stream())
                else:
                    _call(kern, dtab.data_ptr(), n_ep.data_ptr(), nstep, seed, ctr.data_ptr(), es.data_ptr(), ix.data_ptr(),
                          B, _stream())
                what = f"{kern} {name} nstep={nstep} B={B}"
                assert_bits_equal(es[:B].cpu().numpy(), es_w, what + " ep_start")
                assert_bits_equal(ix[:B].cpu().numpy(), ix_w, what + " idx")
                assert int(es[B]) == INT_SENTINEL and int(ix[B]) == INT_SENTINEL, what
                assert int(ctr) == c + (kern != "drq_ring_sample"), what


def test_captured_sampler_follows_the_table(dev):
    """a graph captured over drq_ring_sample_step reads n_episodes and the table at replay: growing them moves the
    draws to the new E"""
    B, nstep, seed = 300, 3, 2 ** 63 - 1
    full = np.stack([np.arange(40) * 50, 3 + (np.arange(40) * 13) % 40], 1)
    dtab = torch.full((40, 2), -1, dtype=torch.int32, device=dev)
    dtab[:3] = torch.from_numpy(full[:3].astype(np.int32))
    n_ep = torch.tensor([3], dtype=torch.int32, device=dev)
    ctr = torch.zeros(1, dtype=torch.int64, device=dev)
    es, ix = i32_out(B + 1, dev), i32_out(B + 1, dev)
    launch = lambda: _call("drq_ring_sample_step", dtab.data_ptr(), n_ep.data_ptr(), nstep, seed, ctr.data_ptr(),
                           es.data_ptr(), ix.data_ptr(), B, _stream())
    launch()                                             # eager, counter 0
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for c, E in ((1, 3), (2, 3), (3, 17), (4, 40)):
        dtab[:E] = torch.from_numpy(full[:E].astype(np.int32))
        n_ep.fill_(E)
        g.replay()
        torch.cuda.synchronize()
        w_es, w_ix = O.sample_indices(np.asarray(full)[:E], nstep, seed, c, B)
        assert_bits_equal(es[:B].cpu().numpy(), w_es, f"replay at E={E}, counter {c}: ep_start")
        assert_bits_equal(ix[:B].cpu().numpy(), w_ix, f"replay at E={E}, counter {c}: idx")
        assert int(ctr) == c + 1
    assert int(es[:B].max()) >= 17 * 50, "the grown table was not sampled"


# ----------------------------------------------------------------------------- 4. gather and n-step
@pytest.mark.parametrize("frame_c, stack", [(1, 1), (1, 3), (1, 4), (3, 1), (3, 3), (3, 4)])
def test_gather_nstep_matches_oracle(dev, frame_c, stack):
    """drq_ring_gather_nstep and the action / reward / discount of prologue-ring part 2 against oracle.ring_gather,
    bit for bit: an episode of rows == capacity that starts mid-ring, idx = 1 and idx = len - nstep + 1, n-step chains
    across the ring end, discounts with zeros"""
    from drqv2_b200 import replay_buffer as R
    cap = 37
    g = np.random.default_rng(frame_c * 10 + stack)
    frames = g.integers(0, 256, (cap, frame_c, 84, 84), dtype=np.uint8)
    reward = g.random(cap, dtype=np.float32)
    discount = np.where(g.random(cap) < 0.25, 0.0, 0.95 + 0.05 * g.random(cap)).astype(np.float32)
    d_frames, d_rew, d_disc = (torch.from_numpy(x).to(dev) for x in (frames, reward, discount))
    for A in (1, 6, 80):
        action = (g.random((cap, A), dtype=np.float32) * 2 - 1)
        d_act = torch.from_numpy(action).to(dev)
        for nstep in (1, 3, 10):
            ln = cap - 1                                  # (start 17, rows = cap): every slot, across the end
            last = ln - nstep + 1
            starts = [17, 17, 17, 17, 0, 36, 30]
            idx = [1, last, 2, (last + 1) // 2, last, 1, last]
            B = len(idx)
            es = torch.tensor(starts, dtype=torch.int32, device=dev)
            ix = torch.tensor(idx, dtype=torch.int32, device=dev)
            C = frame_c * stack
            obs = torch.full((B + 1, C, 84, 84), 0xA5, dtype=torch.uint8, device=dev)
            nxt = torch.full_like(obs, 0xA5)
            act, rew, disc = f32_out(B * A, dev), f32_out(B, dev), f32_out(B, dev)
            _call("drq_ring_gather_nstep", d_frames.data_ptr(), d_act.data_ptr(), d_rew.data_ptr(), d_disc.data_ptr(), cap,
                  frame_c, stack, A, es.data_ptr(), ix.data_ptr(), B, nstep, 0.99, obs.data_ptr(), nxt.data_ptr(),
                  act.data_ptr(), rew.data_ptr(), disc.data_ptr(), _stream())
            want = O.ring_gather(frames, action, reward, discount, np.array(starts), np.array(idx), nstep, 0.99, stack=stack)
            what = f"gather frame_c={frame_c} stack={stack} A={A} nstep={nstep}"
            assert np.array_equal(obs[:B].cpu().numpy(), want[0]), what + " obs"
            assert np.array_equal(nxt[:B].cpu().numpy(), want[4]), what + " next_obs"
            assert (obs[B] == 0xA5).all() and (nxt[B] == 0xA5).all(), what + ": stack B written"
            for got, w, m, name in ((act, want[1], B * A, "action"), (rew, want[2], B, "reward"), (disc, want[3], B, "discount")):
                assert_bits_equal(got[:m].cpu().numpy(), w.reshape(-1), f"{what} {name}")
                assert_f32_tail(got, m, f"{what} {name}")
            # prologue-ring part 2 on the same (ep_start, idx)
            ctr = torch.zeros(1, dtype=torch.int64, device=dev)
            src = R.RingSrc(d_frames.data_ptr(), d_act.data_ptr(), d_rew.data_ptr(), d_disc.data_ptr(), cap, frame_c, stack,
                            A, nstep, 0.99, 0, es.data_ptr(), es.data_ptr(), 0, ctr.data_ptr(), es.data_ptr(), ix.data_ptr())
            scal = torch.zeros(33, device=dev)
            ring = torch.zeros(32).pin_memory()
            cur = torch.zeros(1, dtype=torch.int64, device=dev)
            act2, rew2, disc2 = f32_out(B * A, dev), f32_out(B, dev), f32_out(B, dev)
            _call("drq_update_prologue_ring_part", ring.data_ptr(), 1, cur.data_ptr(), scal.data_ptr(), 0, ctr.data_ptr(), 0,
                  None, None, None, None, B, A, ctypes.byref(src), act2.data_ptr(), rew2.data_ptr(), disc2.data_ptr(), 2, _stream())
            for got, w, m, name in ((act2, want[1], B * A, "action"), (rew2, want[2], B, "reward"),
                                    (disc2, want[3], B, "discount")):
                assert_bits_equal(got[:m].cpu().numpy(), w.reshape(-1), f"prologue_ring part 2 {what} {name}")
                assert_f32_tail(got, m, f"prologue_ring part 2 {what} {name}")
    assert (discount == 0).any()


# ----------------------------------------------------------------------------- 5. the episode table through eviction
def run_eviction_sequences(device):
    """Random sequences of episodes (rows 1 = len 0, rows == capacity, len < nstep) into small GpuRings (capacity 17 to
    100, max_episodes 3 and the default); after every add the host list, the device table and n_episodes equal the
    slot-ownership model, every table entry's slots hold that episode, and of two loaders with nsteps 1 and 3 on the
    ring the table is filtered for the one that called ring() last."""
    from drqv2_b200 import replay_buffer as R
    A = 2
    g = np.random.default_rng(21)
    for cap in (17, 23, 64, 100):
        for max_eps in (3, None):
            key = str(pathlib.Path(f"/test/draws/evict/{device}/{cap}/{max_eps}"))
            ring = R.GpuRing(cap, 3, 3, A, device, max_episodes=max_eps)
            R._RINGS[key] = dict(ring=ring, capacity=cap, storage=None)
            loaders = [R.RingLoader(key, cap, 4, nstep, 0.99, seed=1) for nstep in (1, 3)]
            model = RingModel(cap, ring.max_episodes)
            contents, last = {}, None
            try:
                for k in range(40):
                    rows = int(g.choice([1, 2, 3, 4, 7, cap // 2, cap - 1, cap]))
                    eid = model.add(rows)
                    start = model.episodes[-1][1]
                    ep = episode_content(eid, rows, A)
                    ring.add_episode(*ep)
                    contents = {s: c for s, c in contents.items() if s in {s_ for s_, _ in model.resident()}}
                    contents[start] = ep
                    what = f"capacity {cap} max_episodes {max_eps} add {k} (rows {rows})"
                    assert ring.episodes == model.resident(), what
                    host = [t.cpu().numpy() for t in (ring.frames, ring.action, ring.reward, ring.discount)]
                    for ld in ([last] if last is not None else []) + [loaders[k % 2]]:
                        if ld is not last:
                            ld.ring()
                        want = model.table(ld.nstep)
                        n = int(ring.n_episodes[0])
                        assert n == len(want), (what, ld.nstep, n, len(want))
                        assert ring.ep_table[:n].cpu().numpy().tolist() == [list(x) for x in want], (what, ld.nstep)
                        check_ring_holds(ring.ep_table[:n].cpu().numpy(), *host, contents, cap, what)
                    last = loaders[k % 2]
            finally:
                del R._RINGS[key]


def test_episode_table_through_eviction(dev):
    run_eviction_sequences("cuda")


# ----------------------------------------------------------------------------- 6. drq_random_shift_f32
def test_random_shift_matches_oracle(dev):
    """every (sx, sy) in [0, 2 pad]^2, pads up to 9 (beyond H), against oracle.random_shift_exact bit for bit; the image
    after the last holds the sentinel; H != W is refused"""
    from drqv2_b200 import _lib
    g = torch.Generator().manual_seed(3)
    for C in (1, 9):
        for H in (1, 2, 9, 84):
            for pad in (0, 1, 4, 9):
                allv = torch.tensor([[sx, sy] for sx in range(2 * pad + 1) for sy in range(2 * pad + 1)], dtype=torch.int32)
                for N in sorted({1, 65, 81, len(allv)}):
                    shift = allv[torch.arange(N) % len(allv)]
                    x = torch.randn(N, C, H, H, generator=g)
                    want = O.random_shift_exact(x, shift, pad)
                    out = f32_out(N * C * H * H + C * H * H - 1, dev)
                    dx, ds = x.to(dev), shift.to(dev)
                    _call("drq_random_shift_f32", dx.data_ptr(), ds.data_ptr(), out.data_ptr(), N, C, H, H, pad, _stream())
                    m = N * C * H * H
                    what = f"random_shift N={N} C={C} H={H} pad={pad}"
                    assert_bits_equal(out[:m].view(N, C, H, H).cpu().numpy(), want.numpy(), what)
                    assert (out.view(torch.int32)[m:] == F32_SENTINEL_BITS).all(), what + ": image N written"
    x = torch.zeros(2, 1, 2, 3, device=dev)
    s = torch.zeros(2, 2, dtype=torch.int32, device=dev)
    with pytest.raises(_lib.DrqError, match="h != w"):
        _call("drq_random_shift_f32", x.data_ptr(), s.data_ptr(), x.data_ptr(), 2, 1, 2, 3, 4, _stream())


# ----------------------------------------------------------------------------- 7. the agent's key use
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_agent_consumes_each_key_once(dev, mode, capsys):
    """AGENT_SCRIPT through the public API with CUDA graphs (bf16: ring-direct updates): after every call the agent's
    counter is the key schedule's, and the draws the call consumed (act's eps, the update's shifts and noise, the
    loader's (ep_start, idx), the stage API's noise) equal the reference at the counter before the call"""
    from drqv2_b200 import DrQV2Agent, make_replay_loader
    from tests.test_gpu_ring_direct import _ring_with_wrapping_episodes
    A, Fd, H, B = 6, 50, 64, 32
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, use_cuda_graph=True,
                       seed=2 ** 40 + 7, mode=mode)
    key = f"/test/draws/agent/{mode}"
    _ring_with_wrapping_episodes(key, A, dev)
    loader = make_replay_loader(key, 100, B, 0, False, 3, 0.99)
    it = iter(loader)
    ring = loader.ring()
    if mode == "bf16":
        assert agent.ring_direct
    E = int(ring.n_episodes[0])
    table = ring.ep_table[:E].cpu().numpy()
    obs = O.synthetic_batch(3, A, seed=2)["obs"].numpy()
    feat = (torch.rand(B, 39200, generator=torch.Generator().manual_seed(1)) * 0.1).to(dev)
    fb = O.synthetic_batch(B, A, seed=3)
    sched = key_schedule(AGENT_SCRIPT, agent._seed, loader.seed)
    assert_keys_disjoint(sched)
    step, n_act = 0, 0
    for k, (call, c_model, keys) in enumerate(sched):
        c0, lc0 = int(agent._counter[0]), int(loader._counter[0])
        what = f"{mode} call {k} ({call})"
        assert c0 == c_model, (what, "agent counter", c0, c_model)
        if call in ("act", "act_eval"):
            n = 1 if n_act < 3 else 3                     # the act after the updates is a batched one
            n_act += 1
            agent.act(obs[0] if n == 1 else obs, 5000, call == "act_eval")
            torch.cuda.synchronize()
            if call == "act":
                w, rad = normals_ref(agent._seed, STREAM_NOISE, c0, n * A)
                ratio(f"act eps ({mode})", check_normals(agent._act_ws[n]["eps"].cpu().numpy(), w, rad, what))
        elif call == "update_skip":
            assert agent.update(it, step + 1) == {}
        elif call == "update":
            agent.update(it, step)
            torch.cuda.synchronize()
            step += 2
            ws = agent.workspace(B)
            want = update_draws_ref(agent._seed, c0, agent.aug.pad, B, A)
            assert_bits_equal(ws.shift[:B].cpu().numpy(), want["shift_obs"], what + " shift_obs")
            assert_bits_equal(ws.shift[B:].cpu().numpy(), want["shift_next"], what + " shift_next")
            ratio(f"update eps ({mode})", check_normals(ws.eps_c.cpu().numpy(), want["eps_critic"], want["rad_critic"], what))
            ratio(f"update eps ({mode})", check_normals(ws.eps_a.cpu().numpy(), want["eps_actor"], want["rad_actor"], what))
            es, ix = O.sample_indices(table, loader.nstep, loader.seed, lc0, B)
            assert_bits_equal(loader._ep_start.cpu().numpy(), es, what + " ep_start")
            assert_bits_equal(loader._idx.cpu().numpy(), ix, what + " idx")
        elif call == "stage_critic":
            agent.update_critic(feat, fb["action"].to(dev), fb["reward"].to(dev), fb["discount"].to(dev), feat, step)
            torch.cuda.synchronize()
            w, rad = normals_ref(agent._seed, STREAM_NOISE, c0, B * A)
            ratio(f"stage noise ({mode})", check_normals(agent.workspace(B).eps_c.cpu().numpy(), w, rad, what))
        elif call == "stage_actor":
            agent.update_actor(feat, step)
            torch.cuda.synchronize()
            w, rad = normals_ref(agent._seed, STREAM_NOISE, c0, B * A)
            ratio(f"stage noise ({mode})", check_normals(agent.workspace(B).eps_a.cpu().numpy(), w, rad, what))
        assert int(agent._counter[0]) == c0 + bool(keys), (what, "agent counter after", int(agent._counter[0]), c0)
        assert int(loader._counter[0]) == lc0 + (call == "update"), (what, "loader counter after")
    assert any(isinstance(v, torch.cuda.CUDAGraph) for v in agent._graphs.values())
    assert all(isinstance(g, torch.cuda.CUDAGraph) for w in agent._act_ws.values() for g in w["graph"].values())
    report(capsys, f"agent key use ({mode}): largest normal error / (2^-24 rad): " +
           ", ".join(f"{k} {v:.2f}" for k, v in sorted(RATIOS.items()) if mode in k))
