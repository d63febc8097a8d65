#!/usr/bin/env python
"""Golden fixture for the optimiser tail (SURVEY.md §8 a21), generated with the REFERENCE's own pieces in the build
container: `Queue` and `get_grad_norm` imported unmodified from /root/reference/src/models/__init__.py (through
oracle/ref_shim.py), torch.optim.AdamW(lr 1e-4, weight_decay 1e-12, amsgrad=True) and
torch.nn.utils.clip_grad_norm_ (what Lightning's clip_gradients(..., "norm") calls), and the EMA arithmetic of
src/utils/__init__.py:133-142.  Run:  python tests/golden/make_golden_optim.py"""
import os
import sys

import torch
import torch._dynamo  # noqa: F401  (torch.optim imports it lazily; must happen before the stub modules are installed)

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_shim  # noqa: E402

ref_shim.install()      # stub modules + /root/reference on sys.path
from src.models import Queue, get_grad_norm  # noqa: E402

torch.manual_seed(11)
# the inputs (initial parameters, gradients) are drawn on the float16 grid and stored as float16, which is exact and keeps
# the fixture small; the last tensor spans two chunks of the optimiser kernels (bdiff_optimizer_chunk = 16384)
shapes = [(64, 77), (64,), (32, 8), (1, 64), (17,), (20000,)]
init = [(torch.randn(s) * 0.1).half() for s in shapes]
params = [torch.nn.Parameter(p.float()) for p in init]
opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-12, amsgrad=True)
queue = Queue()
queue.add(3000)
ema = [p.detach().clone() for p in params]
decay = 0.9999
steps, log = [], []
scales = [1.0, 0.5, 2.0, 4000.0, 1.0, 300.0, 1.0, 1.0]          # two spikes exercise the clipping branch
for k, sc in enumerate(scales):
    grads = [(torch.randn(s) * sc).half() for s in shapes]
    for p, g in zip(params, grads):
        p.grad = g.float()
    limit = 1.5 * queue.mean() + 2 * queue.std()
    norm = get_grad_norm(params)
    torch.nn.utils.clip_grad_norm_(params, max_norm=float(limit), norm_type=2.0)
    queue.add(float(limit) if float(norm) > limit else float(norm))
    opt.step()
    for w, e in zip(params, ema):
        diff = e.data - w.data
        diff.mul_(1.0 - decay)
        e.sub_(diff)
    steps.append(grads)
    log.append({"norm": float(norm), "limit": float(limit), "clipped": bool(float(norm) > limit)})
out = {"shapes": shapes, "init": init, "grads": steps, "log": log,
       "params": [p.detach().clone() for p in params], "ema": ema,
       "exp_avg": [opt.state[p]["exp_avg"].clone() for p in params],
       "max_exp_avg_sq": [opt.state[p]["max_exp_avg_sq"].clone() for p in params],
       "history": sorted(float(x) for x in queue.items)}
torch.save(out, os.path.join(os.path.dirname(os.path.abspath(__file__)), "optim_steps.pt"))
print("wrote optim_steps.pt;", [(round(l["norm"], 2), round(l["limit"], 2), l["clipped"]) for l in log])
