"""GPU parity of the two index entry points beside the tokenizer's own: farthest point sampling on D-dimensional points
(p3tok_fps_nd; farthest_point_sampling sums the distance over ALL coordinates, pix4point.py:44) and the materialised
squared-distance matrix (p3tok_square_distance; _square_distance, sampler.py:47-62).  Bit-exact against the oracle, against
the reference-generated fixture (tests/golden/fps_nd.npz) and against the tokenizer's own kernels where they overlap."""
import os

import numpy as np
import pytest
import torch

import cases
from helpers import dev, to_dev
from oracle import oracle
from p3tok import _lib, ops, synth
from p3tok import functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("D", list(range(1, 17)))
def test_fps_nd_matches_oracle(D):
    B, N, G = 3, 700, 90
    pts = synth.make_points_nd(B, N, D, 80 + D)          # a quarter of every cloud is duplicated: exact ties
    st = synth.start_indices(B, N, 80 + D)
    got = ops.fps_nd(to_dev(pts), to_dev(st), G)
    assert got.dtype == torch.int64 and tuple(got.shape) == (B, G)
    assert np.array_equal(got.cpu().numpy(), oracle.fps_nd(pts, st, G))


@pytest.mark.parametrize("name", list(cases.FPS_ND_CASES))
def test_fps_nd_matches_the_reference_fixture(golden_dir, name):
    c = cases.FPS_ND_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    st = synth.start_indices(c["B"], c["N"], c["seed"])
    for D in c["dims"]:
        pts = synth.make_points_nd(c["B"], c["N"], D, c["seed"])
        got = F.farthest_point_sampling(to_dev(pts), c["G"], to_dev(st)).cpu().numpy()
        assert np.array_equal(got, g[f"idx_D{D}"]), D        # == the reference's picks


@pytest.mark.parametrize("N", [1500, 6000])     # one point at a time / several points staged per thread (csrc/fps_nd.cu)
@pytest.mark.parametrize("D", list(range(1, 17)))
def test_fps_nd_distance_bits_follow_torchs_summation_order(D, N):
    """After ONE iteration the caller's scratch holds every point's distance to the start point: the kernel's arithmetic
    itself, compared bit for bit with the oracle's restatement of torch.sum((p - c) ** 2, -1) (which the CPU suite pins
    against torch) - index equality alone would not notice a different summation order."""
    B = 2
    pts = synth.make_points_nd(B, N, D, 300 + D)
    st = synth.start_indices(B, N, 300 + D)
    x, s = to_dev(pts), to_dev(st)
    out = torch.empty((B, 1), dtype=torch.int64, device=dev())
    ws = torch.full((B, N), -7.0, dtype=torch.float32, device=dev())      # contents on entry are ignored
    rc = _lib.lib().p3tok_fps_nd(x.data_ptr(), B, N, D, D, s.data_ptr(), 1, out.data_ptr(), ws.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "fps_nd")
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy()[:, 0], st)
    sq = np.square(pts - pts[np.arange(B), st][:, None, :])
    want = np.minimum(oracle.torch_row_sum(sq.reshape(-1, D)).reshape(B, N), np.float32(1e10))
    assert np.array_equal(ws.cpu().numpy().view(np.int32), want.view(np.int32))


def test_fps_nd_on_xyz_equals_the_tokenizers_fps_kernel():
    B, N, G = 4, 2048, 128
    for kind in ("clustered", "duplicates"):
        x = synth.make_cloud(kind, B, N, 17, 3)
        st = synth.start_indices(B, N, 17)
        a = ops.fps_nd(to_dev(x), to_dev(st), G).cpu().numpy()
        b = ops.fps(to_dev(x), to_dev(st), G).cpu().numpy()
        assert np.array_equal(a, b) and np.array_equal(a, oracle.fps(x, st, G))


@pytest.mark.parametrize("B,N,D,G", [(3, 1, 4, 1), (2, 33, 5, 33), (2, 40, 7, 64), (2, 5000, 6, 300), (1, 20011, 4, 50),
                                     (130, 256, 9, 32), (1, 9000, 16, 20)])
def test_fps_nd_shapes(B, N, D, G):
    """One point, N below a warp, G beyond N (the exhausted cloud repeats index 0 like the reference's argmax over zeros),
    several points per thread, more clouds than fit one wave."""
    pts = synth.make_points_nd(B, N, D, 500 + N % 89)
    st = synth.start_indices(B, N, 9)
    got = ops.fps_nd(to_dev(pts), to_dev(st), G).cpu().numpy()
    assert np.array_equal(got, oracle.fps_nd(pts, st, G))
    assert got.min() >= 0 and got.max() < N
    # the reference flavour clamps n_samples to N (pix4point.py:23)
    clamped = F.farthest_point_sampling(to_dev(pts), G, to_dev(st))
    assert tuple(clamped.shape) == (B, min(G, N)) and np.array_equal(clamped.cpu().numpy(), got[:, :min(G, N)])


def test_fps_nd_rejects_what_it_cannot_do():
    x = torch.zeros(2, 64, 17, device=dev())
    with pytest.raises(RuntimeError, match="16"):
        F.farthest_point_sampling(x, 8, torch.zeros(2, dtype=torch.long, device=dev()))
    with pytest.raises(RuntimeError, match="start_idx"):
        ops.fps_nd(x[..., :5].contiguous(), torch.zeros(3, dtype=torch.long, device=dev()), 8)
    # out-of-range start indices are clamped into the cloud (the C ABI cannot validate device data)
    pts = synth.make_points_nd(2, 100, 5, 3)
    got = ops.fps_nd(to_dev(pts), torch.tensor([-4, 1000], device=dev()), 10).cpu().numpy()
    assert np.array_equal(got, oracle.fps_nd(pts, np.array([0, 99]), 10))


def test_square_distance_matches_the_oracle_bit_for_bit():
    B, N, S = 2, 1500, 48
    x = synth.make_cloud("clustered", B, N, 21, 3)
    ctr = np.ascontiguousarray(x[:, 5:5 + S])
    got = F.square_distance(to_dev(ctr), to_dev(x))
    assert tuple(got.shape) == (B, S, N) and got.dtype == torch.float32
    want = oracle.pair_dist(x, ctr, oracle.KNN_APF_SQ)        # pinned against the reference's _square_distance (CPU suite)
    g = got.cpu().numpy()
    assert np.array_equal(g, want)                            # slightly negative entries included: no clamp
    # xyz + height rows are read in place through a [:, :, :3] view
    x4 = to_dev(synth.make_cloud("clustered", B, N, 21, 4))
    assert torch.equal(F.square_distance(to_dev(ctr), x4[:, :, :3]), got)
    # empty query set
    assert tuple(F.square_distance(to_dev(ctr[:, :0]), to_dev(x)).shape) == (B, 0, N)


@pytest.mark.parametrize("B,S,N", [(1, 700, 1027), (3, 5, 33), (1, 2000, 4096), (2, 300, 1024), (5, 1, 1), (2, 257, 2050)])
def test_square_distance_shapes(B, S, N):
    """N off the 4-point quads and the 1024-point tiles (scalar stores), several 256-row passes, src rows split over
    gridDim.y when the (tile, cloud) grid alone is small."""
    x = synth.make_cloud("uniform", B, max(N, S), 29, 3)
    pts, ctr = np.ascontiguousarray(x[:, :N]), np.ascontiguousarray(x[:, ::-1][:, :S]).copy()
    got = F.square_distance(to_dev(ctr), to_dev(pts)).cpu().numpy()
    assert np.array_equal(got, oracle.pair_dist(pts, ctr, oracle.KNN_APF_SQ))


def test_square_distance_is_the_knn_kernels_distance():
    """The matrix entry at every selected neighbour equals the distance the kNN kernel reports for it, and the selected
    set is the k smallest (distance, index) pairs of the row."""
    B, N, S, k = 2, 3000, 64, 32
    x = synth.make_cloud("uniform", B, N, 23, 3)
    xt = to_dev(x)
    ctr = xt[:, :S].contiguous()
    idx, dist = ops.knn(xt, ctr, k, _lib.KNN_APF_SQ, False, True)
    M = F.square_distance(ctr, xt)
    assert torch.equal(torch.gather(M, 2, idx), dist)
    kth = dist[..., -1:]
    assert bool(((M < kth).sum(-1) <= k - 1).all()) and bool(((M <= kth).sum(-1) >= k).all())
