"""differentiable="bf16" on the host side: refused combinations and the stored flag, without a device."""
import pytest

SCHED = "linear(1.0,0.1,100000)"


def _agent(**kw):
    from drqv2_b200 import DrQV2Agent
    return DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, SCHED, 0.3, False, **kw)


def test_bf16_flag_refusals_before_any_device():
    with pytest.raises(ValueError, match="mode='bf16'"):
        _agent(mode="fp32", differentiable="bf16")
    with pytest.raises(ValueError, match="data_parallel"):
        _agent(mode="bf16", data_parallel=True, differentiable="bf16")
    with pytest.raises(ValueError, match="differentiable"):
        _agent(mode="bf16", differentiable="fp16")


def test_module_refusals_and_flag_values():
    from drqv2_b200 import Actor, Critic, Encoder
    with pytest.raises(ValueError, match="10 channels"):
        Encoder((11, 84, 84), differentiable="bf16")
    Encoder((11, 84, 84), differentiable=True)               # the fp32 kernels take up to 16
    with pytest.raises(ValueError, match="differentiable"):
        Encoder((9, 84, 84), differentiable="yes")
    with pytest.raises(ValueError, match="1 <= A <= 128"):
        Actor(39200, (129,), 50, 64, differentiable="bf16")
    with pytest.raises(ValueError, match="multiple of 8"):
        Critic(39200, (6,), 50, 60, differentiable="bf16")
    with pytest.raises(ValueError, match="feature_dim"):
        Critic(39200, (6,), 257, 64, differentiable="bf16")
    assert Encoder((10, 84, 84), differentiable="bf16").differentiable == "bf16"
    assert Actor(39200, (6,), 50, 64, differentiable="bf16").differentiable == "bf16"
    t = Critic(39200, (6,), 50, 64, differentiable=True).differentiable
    assert t is True and t != "bf16"
