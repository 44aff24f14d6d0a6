"""CPU checks of the fused rollout with values (bb_rollout_value): the exported symbol and its ctypes prototype against
the header, and the baseline TrajectoryBatch takes from a rollout's "value" output."""
import ctypes as C
import os
import re

import pytest
import torch

from deepgroebner_b200.rollout import TrajectoryBatch, compute_advantages, discount_rewards

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_params(name):
    """ctypes types of the parameters of `name` as declared in include/bbenv.h."""
    hdr = open(os.path.join(ROOT, "include", "bbenv.h")).read()
    m = re.search(r"\bint %s\(([^)]*)\);" % name, hdr)
    assert m, name
    out = []
    for p in m.group(1).split(","):
        p = " ".join(p.split())
        if "*" in p:
            out.append(C.c_void_p)
        elif p.startswith("uint64_t"):
            out.append(C.c_uint64)
        elif p.startswith("double"):
            out.append(C.c_double)
        else:
            assert p.startswith("int "), p
            out.append(C.c_int)
    return out


def test_rollout_value_is_exported_with_the_header_prototype():
    from deepgroebner_b200 import _lib
    assert "bb_rollout_value" in _lib.EXPORTS
    want = header_params("bb_rollout_value")
    # bb_rollout's arguments in the same order, then the value arguments, then the stream
    assert want[:-7] == header_params("bb_rollout")[:-1]
    assert want[-7:] == [C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libbbenv.so not built (run __graft_entry__.build())")
    lib = _lib.load()
    assert hasattr(C.CDLL(_lib.LIB_PATH), "bb_rollout_value")
    assert lib.bb_rollout_value.argtypes == want and lib.bb_rollout_value.restype == C.c_int


def batch(with_value):
    g = torch.Generator().manual_seed(3)
    N, T = 5, 12
    out = dict(actions=torch.randint(0, 3, (N, T), generator=g, dtype=torch.int32),
               logp=-torch.rand((N, T), generator=g), reward=-torch.randint(1, 6, (N, T), generator=g).float(),
               lengths=torch.randint(1, 4, (N, T), generator=g, dtype=torch.int32),
               done=(torch.rand((N, T), generator=g) < 0.2).to(torch.uint8))
    out["done"][:, -1] = 1
    out["actions"][4, 7:] = -1     # a slot that stopped running (auto-reset off): value 0 there
    if with_value:
        out["value"] = -10 * torch.rand((N, T), generator=g, dtype=torch.float64)
        out["value"][4, 7:] = 0.0
    return out


def test_trajectory_batch_uses_the_rollout_values():
    out = batch(True)
    tb = TrajectoryBatch(out)
    gam, lam = 0.9, 0.8
    rtg, adv = tb.finish(gam, lam)
    done = out["done"].bool()
    assert torch.equal(adv, compute_advantages(out["reward"], out["value"], done, gam, lam))
    assert torch.equal(rtg, discount_rewards(out["reward"], done, gam))
    assert not torch.equal(adv, compute_advantages(out["reward"], torch.zeros_like(out["value"]), done, gam, lam))
    # explicit values still win
    other = torch.ones_like(out["value"])
    assert torch.equal(tb.finish(gam, lam, values=other)[1], compute_advantages(out["reward"], other, done, gam, lam))
    obs, actions, logp, a, r = tb.get(gam, lam, normalize_advantages=False)
    keep = tb.finished
    multi = out["lengths"][keep] != 1
    assert torch.equal(a, adv[keep].to(torch.float32)[multi])
    assert torch.equal(r, rtg[keep][multi].to(torch.float32))
    assert torch.equal(actions, out["actions"][keep][multi])


def test_trajectory_batch_without_values_is_unchanged():
    out = batch(False)
    tb = TrajectoryBatch(out)
    assert tb.value is None
    done = out["done"].bool()
    rtg, adv = tb.finish(0.9, 0.8)
    assert torch.equal(adv, compute_advantages(out["reward"], torch.zeros_like(out["reward"]), done, 0.9, 0.8))
    got = tb.get(0.9, 0.8)
    ref = TrajectoryBatch(out).get(0.9, 0.8, values=torch.zeros_like(out["reward"]))
    for x, y in zip(got[1:], ref[1:]):
        assert torch.equal(x, y)
