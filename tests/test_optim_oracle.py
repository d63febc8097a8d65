"""CPU: the optimiser-tail oracle (oracle/optim_oracle.py) against the golden fixture generated with the reference's own
Queue / get_grad_norm, torch.optim.AdamW(amsgrad) and clip_grad_norm_ (tests/golden/make_golden_optim.py)."""
import os

import torch

import optim_oracle as OO
from conftest import GOLDEN


def load():
    """The fixture, its float16-stored inputs (exact: drawn on the float16 grid) widened to the float32 they are used in."""
    fx = torch.load(os.path.join(GOLDEN, "optim_steps.pt"), weights_only=False)
    fx["init"] = [p.float() for p in fx["init"]]
    fx["grads"] = [[g.float() for g in step] for step in fx["grads"]]
    return fx


def test_oracle_matches_reference_pieces():
    fx = load()
    o = OO.TrainTailOracle(fx["init"])
    for grads, ref in zip(fx["grads"], fx["log"]):
        got = o.step(grads)
        assert abs(got["norm"] - ref["norm"]) <= 1e-5 * ref["norm"]
        assert abs(got["limit"] - ref["limit"]) <= 1e-6 * ref["limit"]
        assert (got["norm"] > got["limit"]) == ref["clipped"]
    assert sum(r["clipped"] for r in fx["log"]) == 2           # the fixture exercises both branches
    for a, b in zip(o.p, fx["params"]):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-8)
    for a, b in zip(o.ema, fx["ema"]):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-8)
    for a, b in zip(o.m, fx["exp_avg"]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))     # sums of +- terms: absolute scale
    for a, b in zip(o.vmax, fx["max_exp_avg_sq"]):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-12)
    assert max(abs(x - y) for x, y in zip(sorted(o.queue.items), fx["history"])) <= 1e-3


def test_queue_is_fifo_of_fifty():
    q = OO.NormQueue(max_len=5)
    for v in range(10):
        q.add(v)
    assert q.items == [9.0, 8.0, 7.0, 6.0, 5.0]
