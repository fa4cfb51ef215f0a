"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol the
header declares; host logic (schedule, Adam scalars, init order, loud failure without CUDA)."""
import ctypes
import json
import pathlib
import re

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent


def _header_symbols():
    text = (ROOT / "include" / "drqv2_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(drq_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_header_symbol():
    from drqv2_b200 import _lib
    syms = _header_symbols()
    assert len(syms) >= 25
    h = ctypes.CDLL(str(_lib.LIB_PATH))
    for s in syms:
        assert hasattr(h, s), f"{s} declared in include/drqv2_b200.h but not exported"
    # and the ctypes table binds exactly the declared set
    assert sorted(_lib.exported_symbols()) == syms
    assert _lib.lib().drq_abi_version() == 2


def test_no_cuda_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from drqv2_b200 import DrQV2Agent, _lib
    with pytest.raises(RuntimeError):
        DrQV2Agent((9, 84, 84), (6,), "cuda", 1e-4, 50, 64, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, False)
    with pytest.raises(RuntimeError):
        DrQV2Agent((9, 84, 84), (6,), "cpu", 1e-4, 50, 64, 0.01, 2000, 2, "linear(1.0,0.1,100000)", 0.3, False)
    # a compute entry point without a device reports an error status, it does not fall back
    buf = torch.zeros(64)
    with pytest.raises(_lib.DrqError):
        _lib.call("drq_soft_update", buf.data_ptr(), buf.data_ptr(), 64, 0.01, 0.99, None)


def test_schedule_and_adam_scalars(golden_dir):
    from drqv2_b200 import utils
    from oracle import drq_oracle as O
    g = json.loads((golden_dir / "schedule_golden.json").read_text())
    for s, vals in g.items():
        for st, v in zip((0, 1, 50000, 100000, 250000), vals):
            assert utils.schedule(s, st) == v
    with pytest.raises(NotImplementedError):
        utils.schedule("cosine(1,2,3)", 0)
    for t in (1, 2, 1000):
        assert np.array_equal(utils.adam_scalars(1e-4, t), O.adam_scalars(1e-4, t))


def test_module_structure_matches_oracle_param_order():
    """state_dict names / shapes / order are the reference's (drqv2.py:55-59,74-81,100-111)."""
    from drqv2_b200 import Actor, Critic, Encoder
    from oracle import drq_oracle as O
    shapes = O.param_shapes(9, 6, 50, 64)
    for mod, key in ((Encoder((9, 84, 84)), "encoder"), (Actor(39200, (6,), 50, 64), "actor"),
                     (Critic(39200, (6,), 50, 64), "critic")):
        got = [(k, tuple(v.shape)) for k, v in mod.named_parameters()]
        assert got == [(k, tuple(s)) for k, s in shapes[key].items()]
