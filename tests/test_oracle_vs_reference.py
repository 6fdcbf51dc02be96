"""The port and the oracle against the live reference on fresh random shapes (skipped where no checkout of the
original project is present, see oracle/ref_loader.py; tests/test_oracle_vs_golden.py compares both with the
reference's stored outputs everywhere)."""
import numpy as np
import pytest
import torch

from oracle import oracle, port, ref_loader
from p3tok import synth

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")


@pytest.fixture(scope="module")
def ref():
    return ref_loader.load()


def _forced(draws):
    import make_golden
    return make_golden.forced_randint(draws)


@pytest.mark.parametrize("B,N,G,k,seed", [(3, 300, 20, 12, 1), (2, 1000, 100, 32, 2), (1, 4096, 64, 64, 3)])
def test_index_ops(ref, B, N, G, k, seed):
    x = synth.make_cloud("clustered", B, N, seed)
    st = synth.start_indices(B, N, seed)
    xt = torch.from_numpy(x)
    with _forced([st]):
        f = ref.furthest_point_sample(xt, G)
    assert np.array_equal(oracle.fps(x, st, G), f.numpy())
    assert torch.equal(port.fps_indices(xt, G, torch.from_numpy(st)), f)
    ctr = ref.index_points(xt, f)
    assert torch.equal(port.knn_apf(k, xt, ctr), ref.knn_point(k, xt, ctr))
    # BLAS-independent arithmetic spec == this host's matmul / cdist
    assert np.array_equal(oracle.pair_dist(x, ctr.numpy(), oracle.KNN_APF_SQ), ref.square_distance(ctr, xt).numpy())
    d_ref = torch.cdist(ctr, xt).numpy()
    d_orc = oracle.pair_dist(x, ctr.numpy(), oracle.KNN_P4P_CDIST)
    ulps = np.abs(d_ref.view(np.int32).astype(np.int64) - d_orc.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1          # torch's CPU sqrt is not correctly rounded (<= 1 ulp off)
    assert np.array_equal(np.square(d_orc.astype(np.float64)).round(3) >= 0, np.ones_like(d_orc, bool))


@pytest.mark.parametrize("D", list(range(1, 33)))
def test_fps_nd(ref, D):
    """farthest_point_sampling on D-dimensional points (pix4point.py:8-53, distance over ALL coordinates): the oracle's
    restatement of torch's CPU summation order gives the live reference's picks for every D, exact ties included."""
    B, N, G = 3, 500, 70
    pts = synth.make_points_nd(B, N, D, 40 + D)
    st = synth.start_indices(B, N, 40 + D)
    with _forced([st]), torch.no_grad():
        r = ref.farthest_point_sampling(torch.from_numpy(pts), G)
    assert np.array_equal(oracle.fps_nd(pts, st, G), r.numpy())
    sq = np.square(pts - pts[:, 3:4])
    assert np.array_equal(oracle.torch_row_sum(sq.reshape(-1, D)), torch.sum(torch.from_numpy(sq), -1).numpy().reshape(-1))


def test_p3embed_port_matches_reference(ref):
    B, N, k = 2, 512, 16
    x = synth.make_cloud("uniform", B, N, 9)
    sd = synth.to_torch_state(synth.p3embed_state(3, 1 / 16, 4, 4, 128, 9))
    mod = ref.P3Embed(sample_ratio=1 / 16, k=k, embed_dim=128).eval()
    mod.load_state_dict(sd)
    st = [synth.start_indices(B, N, 9, 0), synth.start_indices(B, N // 4, 9, 1)]
    xt = torch.from_numpy(x)
    ft = xt.transpose(1, 2).contiguous()
    with torch.no_grad():
        with _forced(st):
            rp, rf = mod(xt, ft)
        pp, pf = port.p3embed(sd, xt, ft, k, 2, [torch.from_numpy(s) for s in st])
    for a, b in zip(rp + rf, pp + pf):
        assert torch.equal(a, b)
