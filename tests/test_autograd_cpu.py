"""The module API's autograd switch on the host side: refused combinations and the flag's defaults, without a device."""
import pytest


def test_differentiable_with_data_parallel_is_refused():
    """the optimisers' step() does not all-reduce: refused before anything touches a device"""
    from drqv2_b200 import DrQV2Agent
    with pytest.raises(ValueError, match="data_parallel"):
        DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, False,
                   data_parallel=True, differentiable=True)


def test_modules_are_plain_by_default():
    from drqv2_b200 import Actor, Critic, Encoder
    assert not Encoder((9, 84, 84)).differentiable
    assert not Actor(39200, (6,), 50, 64).differentiable
    assert not Critic(39200, (6,), 50, 64).differentiable
    assert Encoder((9, 84, 84), differentiable=True).differentiable
    assert Critic(39200, (6,), 50, 64, differentiable=True).differentiable
    # an instance without the attribute (pickled before the flag existed) reads the class default
    enc = Encoder((3, 84, 84))
    del enc.__dict__["differentiable"]
    assert enc.differentiable is False
