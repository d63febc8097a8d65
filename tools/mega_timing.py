#!/usr/bin/env python
"""Timing of the layer megakernel k_layers_tc (BDIFF_TIMING=1), GPU only:
  * per item: for a few CTAs, the first 16 work items with their fetch time, dependency/fence wait and run time (cycles);
  * per phase: for one edge tile and one node tile per CTA, the time between consecutive stamps (one before and after
    every accumulator wait, one after every operand publication), averaged over the CTAs.  An edge GCP k has two
    accumulator waits: the U pass (gates, u_full) and the S pass + G(k)b (d_full);
  * MMA lane: per item, cycles spent waiting for weight chunks and for operand publications, the rest issuing."""
import os, sys
os.environ["BDIFF_TIMING"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "bio-diffusion_b200")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch, bdiff, gcpnet_oracle as O
name = sys.argv[1] if len(sys.argv) > 1 else "qm9"
cfg = O.config_named(name)
net = bdiff.GCPNetDynamicsB200(config=bdiff.DenoiserConfig.named(name), mode="tensor")
net.load_state_dict(O.random_state_dict(cfg, 7), strict=True); net.cuda()
b, n = (128, 19) if name == "qm9" else (64, 44)
bi = torch.repeat_interleave(torch.arange(b), torch.full((b,), n)).cuda()
mask = torch.ones(b * n, dtype=torch.bool, device="cuda")
xh = torch.randn(b * n, 3 + cfg.num_h, device="cuda"); t = torch.full((b * n, 1), 0.5, device="cuda")
for _ in range(3): net.denoise(bi, mask, xh, t)
torch.cuda.synchronize()
raw = net.debug_tap("dbg"); st = raw.contiguous().view(torch.int64).reshape(512, 64).cpu()
for c in (0, 1, 50, 100, 147):
    rows = st[c].reshape(16, 4).tolist()
    t0 = rows[0][1]
    out = []
    for code, tf, ts, te in rows:
        if tf == 0:
            break
        ty = "N" if (code >> 30) & 1 else "E"
        out.append(f"{ty}{(code >> 24) & 63}.{code & 0xffffff}: fetch+{tf - t0} wait {ts - tf} run {te - ts}")
    print(f"CTA {c}:\n   " + "\n   ".join(out))
# one label per interval between consecutive stamps: every wait has a stamp before and after it, every publication one after
# it ("-> ..." = the short stretch from the previous publication to the next wait)
EDGE = ["T0 assemble->publish", "E0 prefetch", "wait G0", "E0 silu->publish"]
for k in (1, 2, 3):
    EDGE += [f"-> wait U{k}", f"wait G{k}a U pass (u_full)", f"E{k}a gate/vec->publish",
             f"-> wait S{k}", f"wait G{k}a S pass + G{k}b", f"E{k}b residual->publish"]
EDGE += ["m.s reduction rounds 0-3", "wait G4", "E4 gate + m.v rounds"]
NODE = ["T0a->publish", "T0 vectors", "wait G1a", "T0b->publish"]
for g, e in (("G1bc", "E1"), ("G2", "E2"), ("G3a", "E3a"), ("G3b(+G4)", "E3b")):
    NODE += [f"-> wait {g}", f"wait {g}", f"{e}->publish"]
NODE += ["E4 PI", "wait G5", "E5 + zero"]
ph = st[256:512]
for kind, off, names in (("edge", 0, EDGE), ("node", 32, NODE)):
    rows = ph[:148, off:off + 32]
    ok = rows[:, 1] > 0
    rows = rows[ok].double()
    if rows.shape[0] == 0:
        continue
    nst = int((rows[0] > 0).sum())
    d = (rows[:, 1:nst] - rows[:, :nst - 1]).mean(0)
    tot = (rows[:, nst - 1] - rows[:, 0]).mean()
    print(f"{kind} tile: {rows.shape[0]} CTAs, {nst} stamps, total {tot:.0f} cycles")
    assert len(names) == nst - 1, f"{kind} tile: {nst} stamps but {len(names)} phase labels"
    for i, v in enumerate(d.tolist()):
        print(f"   {names[i]:32s} {v:9.0f}  {100 * v / tot:5.1f} %")

mm = st[256 + 148:256 + 148 + 19].reshape(-1, 4)[:148 * 2]
for kind, ty in (("edge", 0), ("node", 1)):
    sel = [(r[1], r[2], r[3]) for r in mm.tolist() if r[1] > 0 and ((r[0] >> 30) & 1) == ty]
    if sel:
        n = len(sel)
        print(f"MMA lane, {kind} items ({n}): item {sum(x[0] for x in sel) / n:.0f} cycles, waiting for weights {sum(x[1] for x in sel) / n:.0f}, "
              f"waiting for operands {sum(x[2] for x in sel) / n:.0f}, issuing {sum(x[0] - x[1] - x[2] for x in sel) / n:.0f}")
