"""GPU: bdiff_optimizer_step (clipping + AdamW(amsgrad) + EMA in three multi-tensor kernels) against the oracle and the
golden fixture produced with the reference's own pieces.  Tolerance: fp32 elementwise arithmetic, 2e-6 relative on
parameters / EMA (the kernel contracts a*b+c into FMAs; torch does not), gradient norm 1e-6 relative."""
import pytest
import torch

import optim_oracle as OO
from test_optim_oracle import load as load_fixture

pytestmark = pytest.mark.gpu


def test_train_tail_matches_oracle_and_fixture():
    import bdiff
    from bdiff.optim import GCDMTrainTail
    fx = load_fixture()
    params = [torch.nn.Parameter(p.clone().cuda()) for p in fx["init"]]
    opt = GCDMTrainTail(params)
    orc = OO.TrainTailOracle(fx["init"])
    for grads, ref in zip(fx["grads"], fx["log"]):
        opt.zero_grad()
        for p, g in zip(params, grads):
            p.grad.add_(g.cuda())                 # what autograd does: accumulate into the installed buffers
        opt.step()
        o = orc.step(grads)
        rep = opt.report()
        assert abs(rep["norm"] - ref["norm"]) <= 2e-6 * ref["norm"]
        assert abs(rep["limit"] - ref["limit"]) <= 2e-6 * ref["limit"]
        assert rep["clipped"] == ref["clipped"]
        assert abs(rep["coef"] - o["coef"]) <= 2e-6
    assert opt.report()["step"] == len(fx["grads"])
    for got, a, b in zip(params, orc.p, fx["params"]):
        g = got.detach().cpu()
        assert torch.allclose(g, a, rtol=2e-6, atol=1e-8) and torch.allclose(g, b, rtol=2e-6, atol=1e-8)
    for got, a in zip(opt.ema_parameters(), fx["ema"]):
        assert torch.allclose(got.cpu(), a, rtol=2e-6, atol=1e-8)
    for got, a in zip(opt.max_exp_avg_sq, fx["max_exp_avg_sq"]):
        assert torch.allclose(got.cpu(), a, rtol=5e-5, atol=1e-12)     # (g * coef)^2: twice the coefficient's rounding
    hist = opt.report()["history"]
    assert max(abs(x - y) for x, y in zip(hist, fx["history"])) <= 1e-2
    assert opt.kernel_launches == 3 * len(fx["grads"])


def test_train_tail_rejects_cpu_and_replaced_grads():
    import bdiff
    from bdiff.optim import GCDMTrainTail
    with pytest.raises(bdiff.BdiffError):
        GCDMTrainTail([torch.nn.Parameter(torch.zeros(4))])
    p = torch.nn.Parameter(torch.zeros(4, device="cuda"))
    opt = GCDMTrainTail([p])
    p.grad = torch.ones(4, device="cuda")
    with pytest.raises(bdiff.BdiffError):
        opt.step()


def test_full_denoiser_parameter_set_one_step():
    """All 432 QM9 parameter tensors (6.2 M elements) in one call: same result as torch.optim.AdamW on the GPU."""
    import bdiff
    from bdiff.optim import GCDMTrainTail
    import gcpnet_oracle as O
    net = bdiff.GCPNetDynamicsB200(config=bdiff.DenoiserConfig.named("qm9"), mode="parity")
    net.load_state_dict(O.random_state_dict(O.config_named("qm9"), 3), strict=True)
    net.cuda()
    ref_params = [torch.nn.Parameter(p.detach().clone()) for p in net.parameters()]
    ref = torch.optim.AdamW(ref_params, lr=1e-4, weight_decay=1e-12, amsgrad=True)
    opt = GCDMTrainTail(net.parameters(), clip_gradients=False)
    g = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(3):
        opt.zero_grad()
        for p, q in zip(net.parameters(), ref_params):
            gr = torch.randn(p.shape, device="cuda", generator=g)
            p.grad.add_(gr)
            q.grad = gr.clone()
        opt.step()
        ref.step()
    for p, q in zip(net.parameters(), ref_params):
        assert torch.allclose(p, q, rtol=2e-6, atol=1e-8)


def test_step_invalidates_the_denoisers_packed_weights():
    """ADVICE r1: forward -> optimiser step -> forward must see the new parameters (version counters are bumped)."""
    import bdiff
    import gcpnet_oracle as O
    net = bdiff.GCPNetDynamicsB200(config=bdiff.DenoiserConfig.named("geom"), mode="parity")
    net.load_state_dict(O.random_state_dict(O.config_named("geom"), 1), strict=True)
    net.cuda()
    bi = torch.repeat_interleave(torch.arange(2), torch.tensor([7, 5])).cuda()
    mask = torch.ones(12, dtype=torch.bool, device="cuda")
    g = torch.Generator().manual_seed(0)
    xh = torch.randn((12, 19), generator=g).cuda()
    t = torch.full((12, 1), 0.4, device="cuda")
    out0 = net.denoise(bi, mask, xh, t).clone()
    opt = bdiff.GCDMTrainTail(list(net.parameters()))
    for p in net.parameters():
        p.grad.copy_(torch.randn(p.shape, generator=g).to(p.device))
    opt.step()
    out1 = net.denoise(bi, mask, xh, t)
    assert not torch.equal(out0, out1), "the denoiser kept its old packed weights after an optimiser step"
