"""The exact reference of the random draws (tests/helpers.py) on its own, on any machine: Philox4x32-10 against the
Random123 known-answer vectors, the key schedule of the agent's public calls, statistical properties of the reference
with fixed keys, and the power of the checks test_gpu_draws.py applies to the kernels: each rejects a planted
defect applied to the reference's own outputs."""
import numpy as np
import pytest
import torch
from scipy import stats

from oracle import drq_oracle as O
from tests.helpers import (AGENT_SCRIPT, STREAM_EPS, STREAM_NOISE, RingModel, assert_bits_equal, assert_keys_disjoint,
                           box_muller, check_normals, check_ring_holds, episode_content, key_schedule, normals_ref,
                           philox_words, uniform24, update_draws_ref)

SEED = 77


# ----------------------------------------------------------------------------- Philox and the uniform
@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's Philox4x32-10 vectors; counter = (index lo, index hi, stream lo, stream hi), key = (seed lo, seed hi)"""
    index = ctr[0] | (ctr[1] << 32)
    stream = ctr[2] | (ctr[3] << 32)
    seed = key[0] | (key[1] << 32)
    got = O.philox4x32(seed, stream, np.array([index], np.uint64))[0]
    assert [int(x) for x in got] == list(want)


def test_counter_word_layout():
    """the counter sits above the 3 stream bits: at counter 2^29 it reaches the stream's high word"""
    a = philox_words(5, STREAM_NOISE, 2 ** 29, [3])
    b = O.philox4x32(5, (1 << 32) | STREAM_NOISE, np.array([3], np.uint64))
    assert np.array_equal(a, b)
    assert not np.array_equal(philox_words(5, STREAM_NOISE, 2 ** 29, [3]), philox_words(5, STREAM_NOISE, 0, [3]))


def test_edge_counters_hit_the_u1_edges():
    """the EDGE counters of test_gpu_draws.py put w >> 8 == 0 / 0xFFFFFF on pair 0 of the noise (stream 5, word 0) and
    of both update draws (stream 3, words 0 and 2), so its shapes with 2 <= B*A <= 128 run the largest rad and u1 = 1"""
    from tests.test_gpu_draws import EDGE_EPS, EDGE_NOISE
    noise = {int(philox_words(77, STREAM_NOISE, c, [0])[0, 0]) >> 8 for c in EDGE_NOISE}
    critic = {int(philox_words(77, STREAM_EPS, c, [0])[0, 0]) >> 8 for c in EDGE_EPS}
    actor = {int(philox_words(77, STREAM_EPS, c, [0])[0, 2]) >> 8 for c in EDGE_EPS}
    for hit in (noise, critic, actor):
        assert {0, 0xFFFFFF} <= hit


def test_uniform_is_the_kernels_fp32():
    w = np.array([0, 0xFF, 0x7FFFFF00, 0x80000000, 0x80000100, 0xFFFFFEFF, 0xFFFFFF00, 0xFFFFFFFF], np.uint64)
    u = uniform24(w)
    assert u.dtype == np.float32
    assert u[0] == u[1] == np.float32(2.0 ** -25)                  # w >> 8 == 0: the smallest u1, the largest rad
    assert u[2] == np.float32((2 ** 23 - 1 + 0.5) * 2.0 ** -24)    # below 2^23 the + 0.5 is exact
    assert u[3] == u[4] - np.float32(2.0 ** -23) == np.float32(0.5)   # 2^23 + 0.5 rounds to even
    assert u[6] == u[7] == np.float32(1.0)                       # 0xFFFFFF + 0.5 rounds up: u1 = 1, a normal of +-0
    v, rad = box_muller(w[6:7], w[0:1], [True])
    assert rad[0] == 0.0 and v[0] == 0.0
    # formed in fp64, u differs by up to 2^-25: tens of thousands of ulp of the normal near u1 = 1
    u64 = ((w >> np.uint64(8)).astype(np.float64) + 0.5) * 2.0 ** -24
    assert np.abs(u64 - u.astype(np.float64)).max() == 2.0 ** -25


# ----------------------------------------------------------------------------- the agent's key schedule
def test_key_schedule_of_the_agent_script():
    sch = key_schedule(AGENT_SCRIPT, SEED, 1234)
    assert_keys_disjoint(sch)
    drawing = [c for c, _, keys in sch if keys]
    assert [c for _, c, keys in sch if keys] == list(range(len(drawing)))      # one counter per drawing call
    assert all(not keys for call, _, keys in sch if call in ("act_eval", "update_skip"))
    # an act graph that lost its counter advance replays the previous call's key
    stuck = [(call, 0 if call == "act" else c, keys if call != "act" else [(SEED, STREAM_NOISE, 0)])
             for call, c, keys in sch]
    with pytest.raises(AssertionError, match="consumed before"):
        assert_keys_disjoint(stuck)


# ----------------------------------------------------------------------------- properties of the reference
def test_sampler_and_shift_uniformity():
    """chi-square of the episode (E = 7 and 50 000), the start index and the shifts over 2^20 draws"""
    n = 1 << 20
    for E in (7, 50_000):
        lens = 3 + (np.arange(E) * 7919) % 997
        table = np.stack([np.arange(E) * 1000, lens], 1)
        es, ix = O.sample_indices(table, 1, SEED, 3, n)
        e = es // 1000
        assert stats.chisquare(np.bincount(e, minlength=E)).pvalue > 1e-3, E
    table = np.array([[0, 997]])
    _, ix = O.sample_indices(table, 3, SEED, 4, n)
    assert ix.min() == 1 and ix.max() == 995
    assert stats.chisquare(np.bincount(ix - 1, minlength=995)).pvalue > 1e-3
    so, sn = O.update_shifts(SEED, 5, 4, n // 2)
    for s in (so[:, 0], so[:, 1], sn[:, 0], sn[:, 1]):
        assert s.min() == 0 and s.max() == 8
        assert stats.chisquare(np.bincount(s, minlength=9)).pvalue > 1e-3


def test_normals_distribution_and_independence():
    n = 1 << 20
    x, _ = normals_ref(SEED, STREAM_NOISE, 6, n)
    assert stats.kstest(x, "norm").pvalue > 1e-3
    lim = lambda m: 5.0 / np.sqrt(m)
    corr = lambda a, b: float(np.corrcoef(a, b)[0, 1])
    d = update_draws_ref(SEED, 7, 4, n // 8, 8)
    assert abs(corr(d["eps_critic"], d["eps_actor"])) < lim(n)
    assert abs(corr(x[0::2], x[1::2])) < lim(n // 2)                         # elements i and i ^ 1: cos and sin of a pair
    y, _ = normals_ref(SEED, STREAM_NOISE, 7, n)
    assert abs(corr(x, y)) < lim(n)                                          # consecutive counters


# ----------------------------------------------------------------------------- the checks reject planted defects
def test_normal_bound_rejects_word_and_pair_mixups():
    B, A = 256, 6
    d = update_draws_ref(SEED, 11, 4, B, A)
    assert check_normals(d["eps_critic"].astype(np.float32), d["eps_critic"], d["rad_critic"], "fp32 round") < 1.0
    i = np.arange(B * A)
    r = philox_words(SEED, STREAM_EPS, 11, i >> 1)
    cos_odd, _ = box_muller(r[:, 0], r[:, 1], i & 1, use_sin_for_odd=False)     # odd elements take cos
    with pytest.raises(AssertionError, match="outside"):
        check_normals(cos_odd, d["eps_critic"], d["rad_critic"], "cos for odd elements")
    with pytest.raises(AssertionError, match="outside"):                        # eps_a on words 0-1
        check_normals(d["eps_critic"], d["eps_actor"], d["rad_actor"], "eps_actor on words 0-1")
    # the one-block prologue's strided loop indexed at i & 1023: wrong past element 1023 (the walker shape, B*A = 1536)
    wrap = d["eps_critic"][i & 1023]
    with pytest.raises(AssertionError, match="outside"):
        check_normals(wrap, d["eps_critic"], d["rad_critic"], "prologue loop at i & 1023")
    so, _ = O.update_shifts(SEED, 11, 4, 1025)
    with pytest.raises(AssertionError, match="differ"):
        assert_bits_equal(so[np.arange(1025) & 1023], so, "shifts at i & 1023")


def test_sampler_check_rejects_a_counter_off_by_one_past_the_first_pass():
    """the one-block sampler's loop reading c + (b >= 256): B = 257 is enough"""
    table = np.array([[0, 40], [41, 7], [49, 300]])
    es, ix = O.sample_indices(table, 3, SEED, 9, 257)
    es2, ix2 = O.sample_indices(table, 3, SEED, 10, 257)
    bad_es, bad_ix = es.copy(), ix.copy()
    bad_es[256:], bad_ix[256:] = es2[256:], ix2[256:]
    assert np.array_equal(bad_es[:256], es[:256])
    with pytest.raises(AssertionError, match="differ"):
        assert_bits_equal(np.stack([bad_es, bad_ix]), np.stack([es, ix]), "sample c + (b >= 256)")


def test_ring_model_and_holds_check():
    """RingModel (slot ownership) and the slot check on host arrays written from the model: every table entry the model
    keeps holds its episode after every add, and the check rejects a table that keeps an overwritten episode (what an
    eviction rule that misses a case leaves behind).  The real GpuRing.add_episode is held to the model in
    test_ring_eviction_on_host_tensors.  Its -capacity overlap shift cannot be caught there or anywhere: episodes are
    written in order at the head, so a wrapped episode's low part never lies past the head, and an episode the new
    rows overwrite is always found by the 0 or +capacity shift."""
    g = np.random.default_rng(5)
    cap, A = 23, 2
    m = RingModel(cap, 3)
    frames = np.zeros((cap, 3, 84, 84), np.uint8)
    act, rew, disc = np.zeros((cap, A), np.float32), np.zeros(cap, np.float32), np.zeros(cap, np.float32)
    contents, stale = {}, None
    for k in range(40):
        rows = int(g.choice([1, 2, 5, 9, cap]))
        before = m.resident()
        eid = m.add(rows)
        start = m.episodes[-1][1]
        f, a, r, d = episode_content(eid, rows, A)
        slots = (start + np.arange(rows)) % cap
        frames[slots], act[slots], rew[slots], disc[slots] = f, a, r, d
        contents = {s: c for s, c in contents.items() if s in {s_ for s_, _ in m.resident()}}
        contents[start] = (f, a, r, d)
        gone = [e for e in before if e not in m.resident()]
        if gone and stale is None:
            stale = gone[0]
        check_ring_holds(m.table(1), frames, act, rew, disc, contents, cap, f"add {k}")
    assert stale is not None
    with pytest.raises(AssertionError):
        check_ring_holds(m.table(0) + [(stale[0], stale[1] - 1)], frames, act, rew, disc, contents, cap, "stale")


def test_ring_eviction_on_host_tensors(monkeypatch):
    """the same sequences through replay_buffer.GpuRing itself, its buffers on the host"""
    from tests.test_gpu_draws import run_eviction_sequences
    from drqv2_b200 import _lib
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(_lib, "lib", lambda: None)
    run_eviction_sequences("cpu")
