"""The power of tests/test_gpu_update_chain.py, asserted on any machine with the oracle alone.

That module holds every update of a run to the oracle at the agent's own state, with bounds that a right answer meets
at single-update tightness.  A bound the wrong answer also meets proves nothing: its learning rate LR is chosen so
that one optimiser step moves the numbers a stage reads by at least POWER x those bounds.  Here the bf16-faithful fp64
oracle runs configuration 1's chain of updates (its shape, LR, step counts and Adam state), its own stepped parameters
standing in for the agent's, and at every update
  (a) the actor stage against the pre-step critic (instead of the critic after critic_opt.step(), drqv2.py:201,213),
  (b) from the second update on, the critic stage with the previous update's critic
must be at least POWER x the bound of the right reference's check away from it, in a metric or a gradient tensor (the
fp32 oracle's own distance to fp64 sets the gradient bounds, as on the GPU).  An edit that lowers LR or loosens the
bounds until a stale read would pass fails here."""
from collections import OrderedDict

import torch

from oracle import drq_oracle as O
from tests.test_gpu_update_chain import BF16, CONFIG1, LR, NETS, POWER, SCHED, TAU, references

UPDATES = 6           # configuration 1: eager warm-up, capture, four replays


def oracle_chain_margins(cfg, lr, updates, sched=SCHED, seed=4):
    """(a, b) power margins of each update of an oracle-only run (b is None on the first update)"""
    A, Fd, H, B = cfg["A"], cfg["F"], cfg["H"], cfg["B"]
    state = O.synthetic_params(9, A, Fd, H, seed=seed)
    zeros = lambda: {net: OrderedDict((k, torch.zeros_like(v)) for k, v in state[net].items()) for net in NETS}
    moments = (zeros(), zeros(), dict(encoder=0, critic=0, actor=0))
    prev, out = None, []
    for k in range(updates):
        b = O.synthetic_batch(B, A, seed=100 + k)
        ref = references(state, prev, b, 2 * k, BF16, sched=sched, moments=moments, lr=lr)
        o = ref["oracle"]
        with torch.no_grad():
            for name in o.p["critic"]:
                O.soft_update(o.p["critic"][name], o.p["critic_target"][name], TAU)
        prev = state
        state = OrderedDict((net, OrderedDict((n, v.clone()) for n, v in o.p[net].items()))
                            for net in NETS + ("critic_target",))
        moments = (o.m, o.v, dict(o.t))
        out.append((ref["margin_a"], ref["margin_b"]))
    return out


def test_update_chain_power_at_config1(capsys):
    torch.set_num_threads(max(8, torch.get_num_threads()))
    margins = oracle_chain_margins(CONFIG1, LR, UPDATES)
    with capsys.disabled():
        for k, (a, b) in enumerate(margins):
            print(f"\nupdate {k}: power margin (a) actor stage at the pre-step critic {a:.1f}, "
                  f"(b) critic stage at the previous critic {'-' if b is None else f'{b:.1f}'} (need >= {POWER:g})", end="")
        print()
    for k, (a, b) in enumerate(margins):
        assert a >= POWER, (k, "actor stage at the pre-step critic", a)
        assert b is None or b >= POWER, (k, "critic stage at the previous critic", b)
