"""The schedule of the captured tensor-core update (DESIGN.md section 4) changes WHEN kernels run, never what they compute:
stream priorities, the early fork of the encoder backward, the two-launch prologue and the 66 KB GEMM variants of the actor
pass leave every parameter of drqv2.py:230-262's update bit-identical to the plain three-stream schedule and to one stream.
(The SM limit of the encoder backward is held fixed: the conv weight-gradient partials are summed per CTA, so the number of
CTAs is part of the arithmetic.)"""
import numpy as np
import pytest
import torch

from oracle import drq_oracle as O

pytestmark = pytest.mark.gpu
SCHED = "linear(1.0,0.1,100000)"

PLAIN = {"DRQV2_B200_PRIO": "0,0,0", "DRQV2_B200_EARLY_ENC": "0", "DRQV2_B200_SPLIT_PROLOGUE": "0", "DRQV2_B200_SMALL_GEMMS": "0"}


def _run(monkeypatch, env, tag, overlap=True, steps=4):
    from drqv2_b200 import DrQV2Agent, make_replay_loader
    from drqv2_b200 import replay_buffer as R
    for k in PLAIN:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("DRQV2_B200_ENC_BWD_SMS", "140")
    A, Fd, H, B = 6, 50, 256, 64                      # >= 48 images: the parity-plane conv1 and the four-pixel-column forward
    dev = torch.device("cuda")
    g = np.random.default_rng(3)
    key = f"/test/schedule/{tag}"
    ring = R.GpuRing(400, 3, 3, A, dev)
    for e in range(4):
        rows = 90
        ring.add_episode(g.integers(0, 256, (rows, 3, 84, 84), dtype=np.uint8), g.random((rows, A), dtype=np.float32) * 2 - 1,
                         g.random(rows, dtype=np.float32), np.ones(rows, dtype=np.float32))
    R._RINGS[key] = dict(ring=ring, capacity=400, storage=None)
    np.random.seed(9)
    it = iter(make_replay_loader(key, 400, B, 0, False, 3, 0.99))
    agent = DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, True, use_cuda_graph=True, seed=5,
                       mode="bf16")
    agent.overlap_encoder_backward = overlap
    params = O.synthetic_params(9, A, Fd, H, seed=6)
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    ms = [agent.update(it, 2 * s) for s in range(steps)]
    torch.cuda.synchronize()
    assert steps < 2 or any(isinstance(v, torch.cuda.CUDAGraph) for v in agent._graphs.values())   # the first update runs eagerly
    state = {f"{net}.{n}": p.detach().clone() for net in ("encoder", "actor", "critic", "critic_target")
             for n, p in getattr(agent, net).named_parameters()}
    return ms, state


def test_schedule_switches_are_bit_identical(monkeypatch):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    base_m, base = _run(monkeypatch, {}, "default")                       # priorities, early fork, split prologue, small GEMMs
    assert all(np.isfinite(m["critic_loss"]) for m in base_m)
    ms, st = _run(monkeypatch, PLAIN, "plain")
    assert ms == base_m
    for k in base:
        assert torch.equal(base[k], st[k]), k


def test_one_stream_equals_three_streams_up_to_the_wgrad_grid(monkeypatch):
    """One stream sizes the conv backward grids for all 148 SMs, the overlapped schedule for 140: the only difference is the
    summation order of the conv weight-gradient partials (fp32), i.e. rounding noise on the encoder's gradients."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    m3, s3 = _run(monkeypatch, {}, "three", steps=1)
    m1, s1 = _run(monkeypatch, {}, "one", overlap=False, steps=1)
    for k in ("critic_loss", "critic_q1", "critic_target_q", "actor_loss"):
        assert m3[0][k] == m1[0][k], k                # the forward and both losses do not depend on the grids
    for k in s3:
        if k.startswith(("actor.", "critic.", "critic_target.")):
            assert torch.equal(s3[k], s1[k]), k
        else:                                         # encoder: one Adam step of lr = 1e-4 on gradients that differ in the last bits
            assert (s3[k] - s1[k]).abs().max().item() <= 2.5e-4, k
