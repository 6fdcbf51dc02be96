"""Host tests of the input-gradient work: the float64 references the GPU gradient tests use (tests/grad_reference.py) reproduce
oracle/port.py - the line-by-line port of the reference - bit for bit when fed port.py's own indices, and the C ABI binding
covers the two adjoint kernels."""
import numpy as np
import pytest
import torch

import grad_reference as gr
from oracle import port
from p3tok import _lib, synth


@pytest.mark.parametrize("C", [3, 4])
def test_apf_reference_reproduces_port(C):
    B, N, G, k, E = 2, 300, 19, 11, 32
    x = torch.from_numpy(synth.make_cloud("clustered", B, N, 41, C))
    start = torch.from_numpy(synth.start_indices(B, N, 41))
    sd = synth.to_torch_state(synth.apf_encoder_state(E, 2 * C, 41))
    xyz = x[:, :, :3].contiguous()
    fidx = port.fps_indices(xyz, G, start)
    knn = port.knn_apf(k, xyz, port.take(xyz, fidx))
    perm = port.morton_order(port.take(xyz, fidx))
    neigh, center = port.apf_group(x, G, k, start)
    n2, c2 = gr.apf_group_idx(x, fidx, knn, perm)
    assert torch.equal(n2, neigh) and torch.equal(c2, center)
    assert torch.equal(gr.pointnet_idx(sd, x, fidx, knn, perm), port.apf_pointnet(sd, x, G, k, start))


@pytest.mark.parametrize("stages", [1, 2])
def test_p3embed_reference_reproduces_port(stages):
    B, N, k, W = 2, 512, 8, 32
    p = torch.from_numpy(synth.make_cloud("uniform", B, N, 43, 3))
    f = p.transpose(1, 2).contiguous()
    ratio = 0.25 ** stages
    sd = synth.to_torch_state(synth.p3embed_state(3, ratio, 4, 4, W, 43))
    starts = [torch.from_numpy(synth.start_indices(B, N // 4 ** s, 43, s)) for s in range(stages)]
    ps, fs = port.p3embed(sd, p, f, k, stages, starts)
    idx, pts = [], p
    for s in range(stages):
        cidx = port.fps_indices(pts, min(N // 4 ** (s + 1), pts.shape[1]), starts[s], masked_update=True)
        ctr = torch.gather(pts, 1, cidx.unsqueeze(-1).expand(-1, -1, 3))
        idx.append((cidx, port.knn_p4p(k, pts, ctr)))
        pts = ctr
    ps2, fs2 = gr.p3embed_idx(sd, p, f, k, idx)
    for a, b in zip(ps + fs, ps2 + fs2):
        assert torch.equal(a, b)


def test_reference_differentiates_to_the_points():
    """The float64 reference carries gradients to the cloud, the parameters and the BatchNorm affines, not to the buffers."""
    B, N, C, G, k, E = 1, 128, 3, 8, 6, 16
    x = torch.from_numpy(synth.make_cloud("uniform", B, N, 47, C)).double().requires_grad_(True)
    sd = gr.state64(synth.apf_encoder_state(E, 2 * C, 47))
    xyz = x.detach().float()
    fidx = port.fps_indices(xyz, G, torch.zeros(B, dtype=torch.long))
    ctr = port.take(xyz, fidx)
    gr.pointnet_idx(sd, x, fidx, port.knn_apf(k, xyz, ctr), port.morton_order(ctr)).sum().backward()
    assert x.grad is not None and float(x.grad.abs().sum()) > 0
    assert sd["first_conv.1.weight"].grad is not None and not sd["first_conv.1.running_mean"].requires_grad


def test_adjoint_kernels_are_bound():
    declared = set(_lib.declared_symbols())
    for name in ("p3tok_apf_rows_bwd_f32", "p3tok_gather_points_bwd_f32"):
        assert name in declared and name in _lib._SIGNATURES
    assert declared == set(_lib._SIGNATURES)
    with open(_lib.HEADER_PATH) as fh:
        assert "#define P3TOK_ABI_VERSION 3" in fh.read()
