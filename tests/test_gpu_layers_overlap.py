"""The layer megakernel's edge tile runs each message GCP's gate pass (U) ahead of its S pass with a commit of its own, so the
gate epilogue overlaps the S MMAs.  These tests pin down what that reordering must not change: two runs give the same bits,
tensor mode stays within the forward tolerance of parity mode, and the edge weight stream that the packer writes, the TMA
producer streams and the peer CTA relays has one size and one chunk count."""
import ctypes as C

import pytest
import torch

import gcpnet_oracle as O

FWD_TOL = 1e-4


@pytest.mark.parametrize("e_hidden, xi_hidden", [(64, 16), (16, 8)])
def test_edge_stream_chunks_match_packed_bytes(e_hidden, xi_hidden):
    """CPU: the chunk table shared by the TMA producer and the peer's relay lane covers exactly the packed stream."""
    import bdiff
    lib = bdiff.load_library()
    out = (C.c_int64 * 3)()
    assert lib.bdiff_tc_edge_stream_layout(e_hidden, xi_hidden, out) == 0
    stream_bytes, chunks, chunk_bytes = out
    k0s = (e_hidden + (64 + xi_hidden) // 4 + 9 + 15) // 16
    assert chunks == k0s + 3 * (4 + 16 + 2) + 4
    assert chunk_bytes == stream_bytes
    # per CTA: G0 planes, per GCP 16 gate K steps (32 rows) + 16 S K steps (128 rows) + 2 extra K steps, 16 G4 steps (16 rows)
    per_cta = k0s * 2 * 128 * 32 + 3 * (16 * 2 * (128 + 32) * 32 + 2 * 2 * 128 * 32) + 16 * 2 * 16 * 32
    assert stream_bytes == 2 * per_cta
    assert lib.bdiff_tc_edge_stream_layout(32, 8, out) != 0


def _forward_pair(cname, seed, bi, mask, xh, t):
    import bdiff
    ocfg = O.config_named(cname)
    sd = O.random_state_dict(ocfg, seed)
    outs = {}
    for mode in ("tensor", "parity"):
        net = bdiff.GCPNetDynamicsB200(config=bdiff.DenoiserConfig.named(cname), mode=mode)
        net.load_state_dict(sd, strict=True)
        net.cuda()
        outs[mode] = net.denoise(bi, mask, xh, t)
        if mode == "tensor":
            assert torch.equal(net.denoise(bi, mask, xh, t), outs[mode]), "tensor mode must be bit-identical from run to run"
    return outs


def _inputs(sizes, nh, seed, drop=()):
    g = torch.Generator().manual_seed(seed)
    b = len(sizes)
    bi = torch.repeat_interleave(torch.arange(b), sizes)
    n = int(sizes.sum())
    mask = torch.ones(n, dtype=torch.bool)
    for i in drop:
        mask[i] = False
    xh = torch.randn((n, 3 + nh), generator=g) * mask[:, None]
    _, xc = O.centralize(xh[:, :3], bi, mask, b)
    xh = torch.cat((xc, xh[:, 3:]), -1)
    t = torch.rand((b, 1), generator=g)[bi]
    return bi.cuda(), mask.cuda(), xh.cuda(), t.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [[19] * 128, [5, 9, 3, 19], [1, 2, 3, 7, 11, 19, 19, 4]], ids=["b128", "mixed4", "tiny8"])
def test_qm9_sizes_deterministic_and_match_parity(sizes):
    sizes = torch.tensor(sizes)
    args = _inputs(sizes, 6, 21, drop=(1,))
    outs = _forward_pair("qm9", 7, *args)
    d = (outs["tensor"] - outs["parity"]).abs().max().item()
    scale = max(1.0, outs["parity"].abs().max().item())
    print(f"qm9 {len(sizes)} molecules: tensor vs parity max|diff| {d:.3e}")
    assert torch.isfinite(outs["tensor"]).all()
    assert d <= FWD_TOL * scale


@pytest.mark.gpu
def test_geom_histogram_batch_deterministic_and_matches_parity():
    """64 molecules with sizes from the GEOM number-of-atoms histogram: rows cut by tile borders and rows longer than one
    128-edge tile (n >= 130)."""
    from bdiff.datasets import GEOM_N_NODES, sample_num_nodes
    sizes = sample_num_nodes(GEOM_N_NODES, 64, seed=123)
    sizes[0], sizes[1] = 181, 150
    args = _inputs(sizes, 16, 5)
    outs = _forward_pair("geom", 3, *args)
    d = (outs["tensor"] - outs["parity"]).abs().max().item()
    scale = max(1.0, outs["parity"].abs().max().item())
    print(f"geom histogram batch ({int(sizes.sum())} atoms): tensor vs parity max|diff| {d:.3e}")
    assert torch.isfinite(outs["tensor"]).all()
    assert d <= FWD_TOL * scale
