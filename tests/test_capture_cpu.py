"""DrQV2Agent(capturable=True): the flag's refusals, which run before any device work, and the ctypes binding of the
device producer of the Adam scalars (no GPU needed)."""
import ctypes
import inspect

import pytest

from drqv2_b200 import DrQV2Agent, _lib

ARGS = ((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, False)


def test_capturable_is_keyword_only_and_off_by_default():
    p = inspect.signature(DrQV2Agent.__init__).parameters["capturable"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is False
    assert DrQV2Agent.capturable is False       # class default: agents pickled before the flag existed


@pytest.mark.parametrize("differentiable", [False, 0])
def test_capturable_needs_differentiable(differentiable):
    with pytest.raises(ValueError, match="capturable=True .*differentiable"):
        DrQV2Agent(*ARGS, differentiable=differentiable, capturable=True)


@pytest.mark.parametrize("differentiable", [True, "bf16"])
def test_capturable_refuses_data_parallel(differentiable):
    with pytest.raises(ValueError, match="capturable=True with data_parallel=True"):
        DrQV2Agent(*ARGS, differentiable=differentiable, data_parallel=True, capturable=True, mode="bf16")


@pytest.mark.parametrize("flag", ["yes", 2, None])
def test_capturable_must_be_a_bool(flag):
    with pytest.raises(ValueError, match="capturable must be False or True"):
        DrQV2Agent(*ARGS, differentiable=True, capturable=flag)


def test_scalars_advance_binding_takes_doubles():
    # lr and the betas cross as fp64, so that -(lr / bc1) starts from the value utils.adam_scalars uses
    assert _lib.SIGNATURES["drq_adam_scalars_advance"] == [ctypes.c_void_p] + [ctypes.c_double] * 4 + [ctypes.c_void_p] * 2
