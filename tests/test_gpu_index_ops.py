"""GPU parity of the index kernels (FPS, kNN, Morton, grouping) through the C ABI: bit-exact against
the oracle on seeded inputs, against the committed reference outputs (tests/golden), and through
size-independent properties at BASELINE.json's full sizes."""
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


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


@pytest.mark.parametrize("name", list(cases.INDEX_CASES))
def test_golden_index_cases(golden_dir, name):
    c, g = cases.INDEX_CASES[name], _golden(golden_dir, name)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    st = synth.start_indices(c["B"], c["N"], c["seed"])
    xt = to_dev(x)
    f1 = F.furthest_point_sample(xt, c["G"], to_dev(st))
    f2 = F.farthest_point_sampling(xt, c["G"], to_dev(st))
    assert f1.dtype == torch.int64 and torch.equal(f1, f2)
    assert np.array_equal(f1.cpu().numpy(), g["fps_idx"])                 # == the reference, bit-exact
    ctr = F.index_points(xt, f1)
    assert np.array_equal(ctr.cpu().numpy(), oracle.gather_points(x, g["fps_idx"].astype(np.int64)))
    for mode, key, ulp, fn in ((oracle.KNN_APF_SQ, "knn_apf", 0, lambda: F.knn_point(c["k"], xt, ctr)),
                               (oracle.KNN_P4P_CDIST, "knn_p4p", 1, lambda: F.knn_query(xt, ctr, c["k"]))):
        mine = fn().cpu().numpy().astype(np.int64)
        D = oracle.pair_dist(x, ctr.cpu().numpy(), mode)
        assert np.array_equal(mine, oracle.knn(x, ctr.cpu().numpy(), c["k"], mode))      # canonical, bit-exact
        ok, msg = oracle.knn_tie_equivalent(mine, g[key].astype(np.int64), D, ulp)       # vs the reference
        assert ok, msg
    perm = F.morton_order(ctr).cpu().numpy()
    codes, operm = oracle.morton(ctr.cpu().numpy())
    assert np.array_equal(perm, operm)
    assert np.array_equal(np.take_along_axis(codes, perm, 1), np.take_along_axis(codes, g["morton_perm"].astype(np.int64), 1))


@pytest.mark.parametrize("B,N,G,C,kind", [
    (3, 1, 1, 3, "uniform"), (2, 31, 31, 3, "uniform"), (5, 100, 40, 3, "clustered"), (2, 257, 64, 4, "uniform"),
    (4, 1024, 256, 3, "uniform"), (3, 2048, 128, 4, "clustered"), (2, 2050, 33, 3, "duplicates"),
    (2, 8192, 96, 3, "uniform"), (2, 8193, 50, 3, "uniform"), (1, 20000, 40, 4, "clustered"),
    (2, 65536, 24, 3, "uniform"), (1, 70001, 16, 3, "uniform"), (1, 131072, 8, 3, "uniform"),
])
def test_fps_matches_oracle(B, N, G, C, kind):
    x = synth.make_cloud(kind, B, N, 100 + N % 97, C)
    st = synth.start_indices(B, N, 5)
    got = ops.fps(to_dev(x), to_dev(st), G).cpu().numpy()
    assert np.array_equal(got, oracle.fps(x, st, G))


def test_fps_edge_cases():
    # exhausted cloud (G > N) repeats index 0; identical points tie -> lowest index; xyz view of (B,N,4)
    x = synth.make_cloud("uniform", 2, 8, 1)
    got = ops.fps(to_dev(x), to_dev(np.array([3, 7])), 12).cpu().numpy()
    assert np.array_equal(got, oracle.fps(x, np.array([3, 7]), 12)) and (got[:, 8:] == 0).all()
    z = np.zeros((1, 64, 3), np.float32)
    assert ops.fps(to_dev(z), to_dev(np.array([9])), 5).cpu().numpy().tolist() == [[9, 0, 0, 0, 0]]
    x4 = to_dev(synth.make_cloud("uniform", 2, 300, 2, 4))
    st = to_dev(np.array([0, 299]))
    assert torch.equal(ops.fps(x4[:, :, :3], st, 20), ops.fps(x4[:, :, :3].contiguous(), st, 20))
    assert ops.fps(x4[:0], st[:0], 4).shape == (0, 4)
    # fps(): gathers all channels (sampler.py:33-45)
    d = F.fps(x4, 16, st)
    assert d.shape == (2, 16, 4)


@pytest.mark.parametrize("mode", [oracle.KNN_APF_SQ, oracle.KNN_P4P_CDIST])
@pytest.mark.parametrize("B,N,G,k,kind", [
    (2, 40, 7, 1, "uniform"), (2, 100, 33, 8, "uniform"), (3, 257, 20, 16, "clustered"), (2, 512, 64, 32, "duplicates"),
    (1, 1000, 100, 33, "uniform"), (2, 2048, 128, 32, "uniform"), (1, 2100, 40, 64, "clustered"),
    (1, 4096, 10, 100, "uniform"), (1, 5000, 5, 128, "duplicates"), (1, 128, 128, 128, "uniform"),
])
def test_knn_matches_oracle(mode, B, N, G, k, kind):
    x = synth.make_cloud(kind, B, N, 7 + k, 3)
    ctr = np.ascontiguousarray(x[:, :G] if kind != "clustered" else synth.make_cloud("uniform", B, G, 9, 3))
    idx, dist = ops.knn(to_dev(x), to_dev(ctr), k, mode, mode == oracle.KNN_P4P_CDIST, True)
    oi, od = oracle.knn(x, ctr, k, mode, return_dist=True)
    assert idx.dtype == (torch.int32 if mode == oracle.KNN_P4P_CDIST else torch.int64)
    assert np.array_equal(idx.cpu().numpy().astype(np.int64), oi)
    assert np.array_equal(dist.cpu().numpy(), od)


def test_knn_errors_and_strided_input():
    x = to_dev(synth.make_cloud("uniform", 1, 16, 1, 4))
    with pytest.raises(RuntimeError):
        F.knn_point(17, x[..., :3], x[:, :2, :3])          # k > N, like torch.topk in the reference
    a = F.knn_point(4, x[..., :3], x[:, :5, :3])
    b = F.knn_point(4, x[..., :3].contiguous(), x[:, :5, :3].contiguous())
    assert torch.equal(a, b)


@pytest.mark.parametrize("name", list(cases.APF_CASES))
def test_group_forward_matches_oracle_and_reference(golden_dir, name):
    from p3tok.modules import Group
    c, g = cases.APF_CASES[name], _golden(golden_dir, name)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], c["C"])
    st = synth.start_indices(c["B"], c["N"], c["seed"])
    xt = to_dev(x)
    grp = Group(c["G"], c["k"])
    neigh, center = grp(xt, xt[:, :, :3], to_dev(st))
    o = oracle.group_apf(x, st, c["G"], c["k"])
    assert np.array_equal(neigh.cpu().numpy(), o["neigh"]) and np.array_equal(center.cpu().numpy(), o["center"])
    assert np.array_equal(center.cpu().numpy(), g["center"])              # reference's Morton-ordered centres
    fidx, _, kidx, perm = grp.indices(xt, to_dev(st))
    assert np.array_equal(fidx.cpu().numpy(), g["fps_idx"])


def test_group_knn_gather_matches_oracle():
    B, N, G, k, D = 2, 300, 20, 8, 5
    p = synth.make_cloud("uniform", B, N, 3)
    f = synth.uniform01(4, B * N * D).reshape(B, N, D)
    ctr = np.ascontiguousarray(p[:, :G])
    gp, gf = F.group_knn(to_dev(p), to_dev(ctr), to_dev(f), k)
    idx = oracle.knn(p, ctr, k, oracle.KNN_P4P_CDIST)
    assert np.array_equal(gp.cpu().numpy(), oracle.gather_points(p, idx))
    assert np.array_equal(gf.cpu().numpy(), oracle.gather_points(f, idx))


def test_full_size_properties_c2_and_c4():
    """BASELINE configs 2 and 4 (index half) through properties that do not need the oracle."""
    for (B, N, G, k, kind) in ((128, 2048, 128, 32, "uniform"), (2, 65536, 2048, 64, "clustered")):
        x = synth.make_cloud(kind, B, N, 1234, 3)
        xt = to_dev(x)
        st = to_dev(synth.start_indices(B, N, 1234))
        idx = ops.fps(xt, st, G)
        assert torch.equal(idx[:, 0], st)
        assert all(len(set(r.tolist())) == G for r in idx.cpu().numpy())          # distinct picks
        assert torch.equal(idx, ops.fps(xt, st, G))                               # deterministic
        # prefix property: FPS with fewer centres is a prefix of FPS with more
        assert torch.equal(idx[:, : G // 2], ops.fps(xt, st, G // 2))
        ctr = ops.gather_points(xt, idx)
        nn_idx, dist = ops.knn(xt, ctr, k, _lib.KNN_APF_SQ, False, True)
        assert bool((dist[..., 1:] >= dist[..., :-1]).all())                      # sortedness
        assert bool((nn_idx == idx.unsqueeze(-1)).any(-1).all())                  # a group contains its centre
        assert bool(((nn_idx >= 0) & (nn_idx < N)).all())
        s = nn_idx.sort(-1)[0]
        assert bool((s[..., 1:] != s[..., :-1]).all())                            # no repeated neighbour
        # spot-check 4 clouds' worth of centres against the oracle at full size
        sub = slice(0, 1)
        assert np.array_equal(nn_idx[sub, :64].cpu().numpy(),
                              oracle.knn(x[sub], ctr[sub, :64].cpu().numpy(), k, oracle.KNN_APF_SQ))
        assert np.array_equal(idx[sub].cpu().numpy(), oracle.fps(x[sub], st[sub].cpu().numpy(), G))


def test_fps_cluster_size_follows_the_batch():
    """p3tok_fps picks the cluster size per launch so that all clouds are resident at once (csrc/fps.cu: a B200 seats only
    15 clusters of 8 CTAs, so 16 clouds of 65536 points run as clusters of 6 with 10923-point slices - 8 register points +
    4 shared-memory points per thread).  Whatever the decomposition, the picks are the oracle's, bit for bit: the same
    clouds sampled alone (clusters of 8), in the full batch (wide slices), with 4-channel rows and with sizes around the
    8192 / 12288-point slice limits, uniform / clustered / duplicated points."""
    G = 96
    for (B, N, C, kind) in ((16, 65536, 3, "clustered"), (18, 65536, 4, "uniform"), (3, 9000, 3, "duplicates"),
                            (40, 12288, 3, "uniform"), (2, 12289, 4, "clustered"), (20, 50001, 3, "duplicates")):
        x = synth.make_cloud(kind, B, N, 4321 + B, C)
        st = synth.start_indices(B, N, 4321 + B)
        xt, stt = to_dev(x), to_dev(st)
        full = ops.fps(xt, stt, G).cpu().numpy()
        sub = [0, B - 1]
        assert np.array_equal(full[sub], oracle.fps(x[sub], st[sub], G)), (B, N, C, kind)
        alone = ops.fps(xt[:2].contiguous(), stt[:2].contiguous(), G).cpu().numpy()      # 2 clouds: the widest cluster
        assert np.array_equal(alone, full[:2]), (B, N, C, kind)
        assert all(len(set(r.tolist())) == min(G, N) for r in full) or kind == "duplicates"


def test_randomised_shapes_against_oracle():
    """Seeded sweep over ragged shapes (N, G, k not multiples of the tile sizes; 3- and 4-channel rows; all three
    cloud kinds): FPS, both kNN flavours, Morton order and APF grouping stay bit-exact against the oracle."""
    rng = np.random.RandomState(20261018)
    kinds = ["uniform", "clustered", "duplicates"]
    for trial in range(24):
        B = int(rng.randint(1, 5))
        N = int(rng.choice([17, 63, 129, 500, 1025, 3000, 8200, 12345]))
        G = int(rng.randint(1, min(N, 300) + 1))
        k = int(rng.randint(1, min(N, 128) + 1))
        C = int(rng.choice([3, 4]))
        kind = kinds[trial % 3]
        x = synth.make_cloud(kind, B, N, 1000 + trial, 3)
        if C == 4:
            x = np.concatenate([x, x[..., 1:2] - x[..., 1:2].min(1, keepdims=True)], -1).astype(np.float32)
        st = synth.start_indices(B, N, trial)
        xt = to_dev(x)
        fidx = ops.fps(xt, to_dev(st), G)
        assert np.array_equal(fidx.cpu().numpy(), oracle.fps(x, st, G)), (trial, "fps", B, N, G, C)
        ctr = ops.gather_points(xt, fidx)[..., :3].contiguous()
        for mode in (oracle.KNN_APF_SQ, oracle.KNN_P4P_CDIST):
            idx, dist = ops.knn(xt, ctr, k, mode, mode == 1, True)
            oi, od = oracle.knn(x, ctr.cpu().numpy(), k, mode, return_dist=True)
            assert np.array_equal(idx.cpu().numpy().astype(np.int64), oi), (trial, "knn", mode, B, N, G, k, C)
            assert np.array_equal(dist.cpu().numpy(), od), (trial, "dist", mode)
        perm, codes = ops.morton_order(ctr)
        oc, op_ = oracle.morton(ctr.cpu().numpy())
        assert np.array_equal(perm.cpu().numpy(), op_) and np.array_equal(codes.cpu().numpy(), oc), (trial, "morton")
        if k <= 32 and G <= 64:
            kidx = ops.knn(xt, ctr, k, _lib.KNN_APF_SQ, False, False)[0]
            neigh, center = ops.apf_group(xt.contiguous(), fidx, kidx, perm)
            o = oracle.group_apf(x, st, G, k)
            assert np.array_equal(neigh.cpu().numpy(), o["neigh"]) and np.array_equal(center.cpu().numpy(), o["center"]), (trial, "group")


def test_dataset_level_fps_downsample():
    """SURVEY 8f "next" #2: ScanObjectNN.__init__ with sampling_method='fps' (src/data/scanobjectnn.py:92-97) moves the
    whole split to the GPU and calls fps(points, num_points) once: B = 2309 clouds, N = 2048, number = 1024."""
    B, N, G = 2309, 2048, 1024
    x = synth.make_cloud("clustered", B, N, 77, 3)
    st = synth.start_indices(B, N, 77)
    xt, stt = to_dev(x), to_dev(st)
    F.fps(xt, G, stt)                                   # warm-up at full size: allocator growth / kernel load are not timed
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = F.fps(xt, G, stt)
    e1.record()
    torch.cuda.synchronize()
    assert out.shape == (B, G, 3)
    idx = F.furthest_point_sample(xt, G, stt)
    assert torch.equal(out, torch.gather(xt, 1, idx.unsqueeze(-1).expand(-1, -1, 3)))
    sub = slice(0, 24)                                  # oracle on a slice (the CPU loop is G x N per cloud)
    assert np.array_equal(idx[sub].cpu().numpy(), oracle.fps(x[sub], st[sub], G))
    assert all(len(set(r.tolist())) == G for r in idx[::97].cpu().numpy())
    print(f"dataset-level fps: {B} clouds x {N} pts -> {G}: {e0.elapsed_time(e1):.1f} ms")


def _knn_both(x, ctr, k, mode, i32):
    """(idx, dist) from the plain sweep (p3tok_knn) and from the Z-order sorted / culled variant (p3tok_knn_sorted),
    both through the C ABI."""
    L = ops._L()
    B, N, _ = x.shape
    G = ctr.shape[1]
    outs = []
    for sorted_variant in (False, True):
        idx = torch.empty((B, G, k), dtype=torch.int32 if i32 else torch.int64, device=x.device)
        dist = torch.empty((B, G, k), dtype=torch.float32, device=x.device)
        dt = _lib.I32 if i32 else _lib.I64
        if sorted_variant:
            nbytes = int(L.p3tok_knn_workspace_bytes(B, N))
            assert nbytes > 0
            ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
            _lib.check(L.p3tok_knn_sorted(x.data_ptr(), B, N, 3, ctr.data_ptr(), G, k, mode, idx.data_ptr(), dt,
                                          dist.data_ptr(), ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream),
                       "knn_sorted")
        else:
            _lib.check(L.p3tok_knn(x.data_ptr(), B, N, 3, ctr.data_ptr(), G, k, mode, idx.data_ptr(), dt, dist.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream), "knn")
        torch.cuda.synchronize()
        outs.append((idx.cpu(), dist.cpu()))
    return outs


@pytest.mark.parametrize("mode", [oracle.KNN_APF_SQ, oracle.KNN_P4P_CDIST])
@pytest.mark.parametrize("B,N,G,k,kind", [
    (3, 1000, 77, 32, "uniform"), (2, 8192, 300, 32, "clustered"), (2, 2048, 128, 64, "duplicates"),
    (4, 100, 100, 100, "uniform"), (2, 33, 5, 16, "clustered"), (1, 4096, 64, 128, "duplicates"),
    # beyond 8192 points: the cloud is sorted as segments of <= 8192 points and a query walks them (csrc/knn.cu)
    (2, 8193, 50, 32, "uniform"), (2, 20011, 130, 64, "duplicates"), (1, 65536, 96, 64, "clustered"), (1, 131072, 40, 17, "uniform"),
])
def test_sorted_knn_is_bit_identical_to_the_sweep(mode, B, N, G, k, kind):
    """The culled variant must return exactly the sweep's (distance, index) lists: ragged N, k = N, duplicated points
    (ties at the k-th distance), and query points that are NOT cloud points (outside the cloud's bounding box too)."""
    x = to_dev(synth.make_cloud(kind, B, N, 900 + N, 3))
    g = torch.Generator().manual_seed(N + G)
    pick = torch.randint(0, N, (B, G), generator=g)
    ctr = torch.gather(x.cpu(), 1, pick[..., None].expand(B, G, 3)).clone()
    ctr[:, ::3] += torch.randn(B, (G + 2) // 3, 3, generator=g) * 0.3          # every third centre is off-cloud
    ctr[:, 1::7] *= 3.0                                                          # some far outside the bounding box
    ctr = ctr.contiguous().to(dev())
    (i0, d0), (i1, d1) = _knn_both(x, ctr, k, mode, mode == oracle.KNN_P4P_CDIST)
    assert torch.equal(i0, i1)
    assert torch.equal(d0.view(torch.int32), d1.view(torch.int32))


def test_sorted_knn_workspace_contract():
    L = ops._L()
    assert int(L.p3tok_knn_workspace_bytes(4, 8193)) > 0           # two segments
    assert int(L.p3tok_knn_workspace_bytes(4, 131073)) == 0        # too many points: use the sweep
    x = to_dev(synth.make_cloud("uniform", 1, 64, 1, 3))
    idx = torch.empty((1, 4, 8), dtype=torch.int64, device=dev())
    ws = torch.empty(16, dtype=torch.uint8, device=dev())
    rc = L.p3tok_knn_sorted(x.data_ptr(), 1, 64, 3, x.data_ptr(), 4, 8, 0, idx.data_ptr(), _lib.I64, None, ws.data_ptr(), 16,
                            torch.cuda.current_stream().cuda_stream)
    assert rc == _lib.ERR_WORKSPACE


@pytest.mark.parametrize("mode", [oracle.KNN_APF_SQ, oracle.KNN_P4P_CDIST])
def test_knn_prepare_query_split_and_stream_overlap(mode):
    """p3tok_knn_prepare + p3tok_knn_query (the halves modules run on two streams) == p3tok_knn, bit for bit; and the
    overlapped FPS + preparation pair returns what the two calls return back to back."""
    B, N, G, k = 5, 1500, 70, 24
    x = to_dev(synth.make_cloud("clustered", B, N, 91, 3))
    start = to_dev(synth.start_indices(B, N, 91))
    fidx, ws = ops.fps_with_knn_prepare(x, start, G)
    assert torch.equal(fidx, ops.fps(x, start, G))
    ctr = ops.gather_points(x, fidx)
    got = ops.knn_query(x, ws, ctr, k, mode, mode == oracle.KNN_P4P_CDIST)
    ref = ops.knn(x, ctr, k, mode, mode == oracle.KNN_P4P_CDIST, False)[0]
    assert torch.equal(got, ref)
    assert np.array_equal(got.cpu().numpy().astype(np.int64), oracle.knn(x.cpu().numpy(), ctr.cpu().numpy(), k, mode))
    big = to_dev(synth.make_cloud("uniform", 1, 9000, 92, 3))          # 8192 < N <= 131072: two sorted segments
    ws2 = ops.knn_prepare(big)
    assert ws2.numel() > 0
    c2 = big[:, :10].contiguous()
    got2 = ops.knn_query(big, ws2, c2, 8, mode, False)
    assert torch.equal(got2, ops.knn(big, c2, 8, mode, False, False)[0])
    assert np.array_equal(got2.cpu().numpy().astype(np.int64), oracle.knn(big.cpu().numpy(), c2.cpu().numpy(), 8, mode))
    huge = torch.zeros((1, 131073, 3), device=dev())                   # beyond the segmented limit: empty workspace, the sweep answers
    assert ops.knn_prepare(huge).numel() == 0


# ------------------------------------------------------------------ round-1 advisor findings
def test_fps_with_non_finite_points_stays_in_range():
    """Non-finite coordinates are outside the contract (the reference assumes finite input), but every index the kernel
    writes must stay inside the cloud - single-CTA and cluster paths."""
    for N in (1000, 20000):
        x = synth.make_cloud("uniform", 2, N, 9, 3)
        x[0, 5] = np.nan
        x[0, 7, 1] = np.inf
        x[1] = np.nan                                     # a cloud with no finite point at all
        idx = ops.fps(to_dev(x), to_dev(np.array([3, 0], np.int64)), 64)
        torch.cuda.synchronize()
        a = idx.cpu().numpy()
        assert a.min() >= 0 and a.max() < N


def test_group_forward_honours_the_xyz_argument():
    """apf.py:64-71 runs FPS / kNN / Morton on the `xyz` argument; a caller passing coordinates that are not
    x[:, :, :3] (e.g. normalised) must get the groups of THOSE coordinates, gathered from x."""
    from p3tok.modules import Group
    B, N, G, k = 2, 512, 16, 8
    x = synth.make_cloud("uniform", B, N, 21, 4)
    xyz = (x[..., :3] * np.array([1.0, 0.25, 2.0], np.float32)).astype(np.float32)     # anisotropic: different neighbours
    st = synth.start_indices(B, N, 21)
    neigh, center = Group(G, k)(to_dev(x), to_dev(xyz), to_dev(st))
    fidx = oracle.fps(xyz, st, G)
    ctr = oracle.gather_points(xyz, fidx)
    kidx = oracle.knn(xyz, ctr, k, oracle.KNN_APF_SQ)
    _, perm = oracle.morton(ctr)
    cf = oracle.gather_points(x, fidx)                                                  # centre features come from x
    nb = oracle.gather_points(x, kidx.reshape(B, -1)).reshape(B, G, k, 4) - cf[:, :, None, :]
    ref = np.concatenate([nb, np.broadcast_to(cf[:, :, None, :], nb.shape)], -1)
    ref = np.take_along_axis(ref, perm[:, :, None, None], 1)
    assert np.array_equal(neigh.cpu().numpy(), ref.astype(np.float32))
    assert np.array_equal(center.cpu().numpy(), np.take_along_axis(ctr, perm[:, :, None], 1))
    # and the in-place fast path (xyz IS the view) still equals the oracle
    xt = to_dev(x)
    n2, c2 = Group(G, k)(xt, xt[:, :, :3], to_dev(st))
    o = oracle.group_apf(x, st, G, k)
    assert np.array_equal(n2.cpu().numpy(), o["neigh"]) and np.array_equal(c2.cpu().numpy(), o["center"])


def test_knn_query_rejects_a_foreign_workspace():
    B, N = 2, 1024
    x0, x1 = (to_dev(synth.make_cloud("uniform", B, N, s, 3)) for s in (1, 2))
    ws = ops.knn_prepare(x0)
    ctr = x0[:, :8].contiguous()
    ops.knn_query(x0, ws, ctr, 4, _lib.KNN_APF_SQ, False)
    with pytest.raises(RuntimeError, match="prepared from a different"):
        ops.knn_query(x1, ws, ctr, 4, _lib.KNN_APF_SQ, False)
    x0.add_(1.0)                                           # modified in place since the preparation
    with pytest.raises(RuntimeError, match="prepared from a different"):
        ops.knn_query(x0, ws, ctr, 4, _lib.KNN_APF_SQ, False)


def test_farthest_point_sampling_fewer_than_three_coordinates():
    """pix4point.py:44 sums over all D coordinates; D < 3 (the general-D kernel) equals the zero-padded xyz sampling:
    the padding only adds exact +0 terms.  D > 3: tests/test_gpu_xtra_index.py."""
    p2 = synth.make_cloud("uniform", 2, 300, 5, 3)[..., :2].copy()
    st = synth.start_indices(2, 300, 5)
    got = F.farthest_point_sampling(to_dev(p2), 40, to_dev(st)).cpu().numpy()
    ref = oracle.fps(np.concatenate([p2, np.zeros((2, 300, 1), np.float32)], -1), st, 40)
    assert np.array_equal(got, ref)
    assert np.array_equal(got, oracle.fps_nd(p2, st, 40))
    with pytest.raises(RuntimeError, match="16"):
        F.farthest_point_sampling(torch.zeros(1, 8, 17, device=dev()), 2)


def test_seeded_draw_reproduces_reference_semantics():
    """Without start_idx, furthest_point_sample takes its first index from torch's global CPU generator like
    sampler.py:20, so the same manual_seed gives the same centres as passing that draw explicitly."""
    x = to_dev(synth.make_cloud("uniform", 3, 256, 8, 3))
    torch.manual_seed(77)
    a = F.furthest_point_sample(x, 16)
    torch.manual_seed(77)
    st = torch.randint(0, 256, (3,), dtype=torch.long)
    assert torch.equal(a, F.furthest_point_sample(x, 16, st.to(dev())))


def test_fps_many_iterations_bit_exact_near_ties():
    """65536 dependent FPS iterations over full-mantissa coordinates: the running distances of the two best candidates
    come within one ulp of each other about once per 10^4 iterations, so a single mis-rounded distance (round 1: a
    contracted FFMA2) shows up as a flipped pick.  Single-CTA and cluster paths."""
    for (B, N, G) in ((64, 2048, 1024), (4, 20000, 2048)):
        x = synth.make_cloud("uniform", B, N, 777, 3)
        st = synth.start_indices(B, N, 777)
        ref = oracle.fps(x, st, G)
        got = ops.fps(to_dev(x), to_dev(st), G).cpu().numpy()
        bad = np.argwhere(got != ref)
        assert bad.size == 0, f"{len(bad)} picks differ; first at cloud {bad[0][0]} iteration {bad[0][1]}"


def test_fps_ragged_shapes_equal_the_oracle():
    """p3tok_fps against the oracle: ragged N (partial last warp, 8 and 16 points per thread, up to the largest
    single-CTA cloud), G up to N and beyond, 3- and 4-channel rows, all cloud kinds incl. exact duplicates (ties resolved
    by the lowest index)."""
    rng = np.random.RandomState(7)
    kinds = ["uniform", "clustered", "duplicates"]
    shapes = [(3, 33, 33), (2, 100, 40), (4, 256, 64), (2, 257, 257), (3, 1000, 999), (2, 1024, 256), (2, 2048, 128), (2, 2049, 300),
              (1, 4096, 1024), (2, 5000, 77), (1, 8191, 512), (2, 8192, 2048), (2, 64, 100)]
    for t, (B, N, G) in enumerate(shapes):
        C = 3 + (t % 2)
        x = synth.make_cloud(kinds[t % 3], B, N, 500 + t, 3)
        if C == 4:
            x = np.concatenate([x, x[..., 1:2] - x[..., 1:2].min(1, keepdims=True)], -1).astype(np.float32)
        st = rng.randint(0, N, size=B).astype(np.int64)
        got = ops.fps(to_dev(x), to_dev(st), G).cpu().numpy()
        ref = oracle.fps(x, st, G)
        assert np.array_equal(got, ref), (B, N, G, np.argwhere(got != ref)[:3])
