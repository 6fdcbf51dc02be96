"""Reproducible gradients under torch.use_deterministic_algorithms: the *_det_f32 entry points and the wrappers that route to them.

Host-only: the workspace size queries against a Python mirror of the slice / strip formulas.
GPU: the fixed-point scatters bit for bit against an int64 numpy emulation of their contract (include/p3tok.h), batch
invariance of the scatters, the ordered reductions' partial layout and summation order, repeatability under concurrent load,
routing (profiler kernel names), bit-identical training steps across processes, and accuracy against float64 at the bounds of
the default path."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import dev, to_dev
from p3tok import _lib, ops, synth, train

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


@pytest.fixture
def det(monkeypatch):
    """torch.use_deterministic_algorithms(True) for the test; the previous mode (and warn-only state) restored on exit.  torch
    refuses cuBLAS calls under the flag unless CUBLAS_WORKSPACE_CONFIG is set, so it is set for the test too."""
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=warn)


def _cdiv(a, b):
    return -(-a // b)


def tn_slices(M, N, K):
    """(slices, rows per slice) of p3tok_linear_tn_f32 / _det_f32: ~4 CTAs per SM of a B200 over the 64 x 64 output tiles."""
    tiles = _cdiv(N, 64) * _cdiv(K, 64)
    rows = _cdiv(_cdiv(M, _cdiv(148 * 4, tiles)), 256) * 256
    return _cdiv(M, rows), rows


def strips(M, N):
    """(strips, rows per strip) of the column-strip reductions (strip_rows in csrc/train.cu)."""
    rows = max(_cdiv(_cdiv(M, _cdiv(148 * 8, _cdiv(N, 32))), 64) * 64, 64)
    return _cdiv(M, rows), rows


# ------------------------------------------------------------------------------------------------ host-only
def test_det_workspace_queries_are_zero_for_empty_shapes():
    L = _lib.lib()
    assert L.p3tok_linear_tn_det_workspace_bytes(0, 64, 64) == 0
    assert L.p3tok_colsum_det_workspace_bytes(0, 64) == 0
    assert L.p3tok_scatter_det_workspace_bytes(0, 1024, 3) == 0
    assert L.p3tok_scatter_det_workspace_bytes(4, 0, 3) == 0


@pytest.mark.parametrize("M,N,K", [(1, 64, 64), (100, 64, 64), (1000, 64, 64), (1000, 7, 3), (524288, 128, 6), (524288, 64, 6),
                                   (16384, 1536, 384), (16384, 384, 1536), (4096, 384, 384), (131072, 256, 512)])
def test_linear_tn_workspace_matches_slice_mirror(M, N, K):
    s, rows = tn_slices(M, N, K)
    assert (s - 1) * rows < M <= s * rows
    assert _lib.lib().p3tok_linear_tn_det_workspace_bytes(M, N, K) == s * N * K * 4
    assert s * N * K <= (592 + _cdiv(N, 64) * _cdiv(K, 64)) * 4096


@pytest.mark.parametrize("M,N", [(1, 32), (64, 384), (1000, 64), (524288, 64), (524288, 128), (16384, 384), (262144, 384),
                                 (65536, 1536)])
def test_colsum_workspace_matches_strip_mirror(M, N):
    s, rows = strips(M, N)
    assert (s - 1) * rows < M <= s * rows
    assert _lib.lib().p3tok_colsum_det_workspace_bytes(M, N) == 2 * s * N * 8


@pytest.mark.parametrize("B,N,C", [(1, 1, 3), (128, 2048, 3), (32, 8192, 3), (16, 2048, 3 + 61)])
def test_scatter_workspace_bytes(B, N, C):
    assert _lib.lib().p3tok_scatter_det_workspace_bytes(B, N, C) == 12 * B * N * C + 4 * B


# ------------------------------------------------------------------------------------------------ numpy emulation
def fixed_point_sum(B, per_cloud, K, slot, v):
    """The fixed-point scatter of include/p3tok.h in int64 numpy: contributions v (float32) to slots (cloud = slot // per_cloud)
    -> float32 (B * per_cloud,)."""
    v = np.asarray(v, np.float32).ravel()
    slot = np.asarray(slot, np.int64).ravel()
    cloud = slot // per_cloud
    fin = np.isfinite(v)
    m = np.zeros(B, np.float32)
    np.maximum.at(m, cloud[fin], np.abs(v[fin]))
    cbits = (int(K) - 1).bit_length()
    s = np.where(m > 0, 61 - cbits - np.frexp(m.astype(np.float64))[1], 0).astype(np.int64)
    q = np.rint(np.ldexp(v[fin].astype(np.float64), s[cloud[fin]])).astype(np.int64)
    acc = np.zeros(B * per_cloud, np.int64)
    np.add.at(acc, slot[fin], q)
    out = np.ldexp(acc.astype(np.float32).astype(np.float64), -np.repeat(s, per_cloud)).astype(np.float32)
    flags = {}
    for name, sel in (("nan", np.isnan(v)), ("pos", v == np.inf), ("neg", v == -np.inf)):
        f = np.zeros(B * per_cloud, bool)
        f[slot[sel]] = True
        flags[name] = f
    out[flags["pos"]] = np.inf
    out[flags["neg"]] = -np.inf
    out[flags["nan"] | (flags["pos"] & flags["neg"])] = np.nan
    return out


def _bits_equal(got, ref, what):
    got = got.detach().float().cpu().numpy().ravel() if torch.is_tensor(got) else np.asarray(got, np.float32).ravel()
    ref = np.asarray(ref, np.float32).ravel()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(got), nan), what
    bad = got[~nan].view(np.uint32) != ref[~nan].view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} elements differ in their bits"


def gather_points_contribs(g, idx, N):
    """(slots, values) of gather_points_bwd: g (B,S,C), idx (B,S)."""
    B, S, C = g.shape
    dst = (np.arange(B)[:, None] * N + idx)[:, :, None] * C + np.arange(C)
    return dst.ravel(), g.ravel()


def apf_rows_contribs(gn, fidx, kidx, perm, N):
    """(slots, values) of apf_rows_bwd: gn (B,G,k,2C) in output group order; the centre term summed in float32 in ascending n."""
    B, G, k, C2 = gn.shape
    C = C2 // 2
    g_in = perm if perm is not None else np.broadcast_to(np.arange(G), (B, G))
    nbr = np.take_along_axis(kidx, np.broadcast_to(g_in[:, :, None], kidx.shape), 1)   # (B,G,k) neighbours of output group j
    ctr = np.take_along_axis(fidx, g_in, 1)                                        # (B,G)
    drel, dctr = gn[..., :C], gn[..., C:]
    acc = np.zeros((B, G, C), np.float32)
    for n in range(k):
        acc = (acc + (dctr[:, :, n] - drel[:, :, n])).astype(np.float32)
    bb = np.arange(B)[:, None, None]
    s_nbr = ((bb * N + nbr)[..., None] * C + np.arange(C)).ravel()
    s_ctr = ((np.arange(B)[:, None] * N + ctr)[..., None] * C + np.arange(C)).ravel()
    return np.concatenate([s_nbr, s_ctr]), np.concatenate([drel.ravel(), acc.ravel()])


def _rand(shape, seed, scale=1.0):
    if int(np.prod(shape)) == 0:
        return np.zeros(shape, np.float32)
    return ((synth.uniform01(seed, int(np.prod(shape)), 5).reshape(shape) - 0.5) * 2 * scale).astype(np.float32)


# ------------------------------------------------------------------------------------------------ scatters vs numpy
@gpu
@pytest.mark.parametrize("C", [3, 4])
def test_gather_points_bwd_bits_vs_numpy(det, C):
    B, N, S = 3, 97, 4096
    idx = (synth.uniform01(7, B * S, 1).reshape(B, S) * 5).astype(np.int64) * 11 % N   # 5 destinations take every contribution
    idx[1] = np.arange(S) % N
    g = _rand((B, S, C), 8)
    g[2] *= 1e-30                                                                        # one cloud at a tiny scale
    got = ops.gather_points_bwd(to_dev(g), to_dev(idx), N)
    _bits_equal(got, fixed_point_sum(B, N * C, S, *gather_points_contribs(g, idx, N)), f"gather_points_bwd C={C}")


def _apf_indices(B, N, C, G, k, seed, dup=True):
    from p3tok.modules import Group
    x = synth.make_cloud("clustered", B, N, seed, C)
    if dup:
        x[:, N // 2:] = x[:, :N // 2]                                                     # duplicated points: tied distances
    st = to_dev(synth.start_indices(B, N, seed))
    fidx, _, kidx, perm = Group(G, k).to(dev()).indices(to_dev(x), st)
    return x, fidx, kidx, perm


def _apf_bwd_ref(gn, gc, fidx, kidx, perm, N, C):
    B, G = kidx.shape[:2]
    f, kk, p = fidx.cpu().numpy(), kidx.cpu().numpy(), None if perm is None else perm.cpu().numpy()
    out = fixed_point_sum(B, N * C, G * (kk.shape[2] + 1), *apf_rows_contribs(gn, f, kk, p, N))
    if gc is not None:
        src = f if p is None else np.take_along_axis(f, p, 1)
        gcp = np.zeros((B, G, C), np.float32)
        gcp[..., :3] = gc
        out = (out + fixed_point_sum(B, N * C, G, *gather_points_contribs(gcp, src, N))).astype(np.float32)
    return out


@gpu
@pytest.mark.parametrize("idx_dtype", [torch.int64, torch.int32])
@pytest.mark.parametrize("use_perm", [True, False])
@pytest.mark.parametrize("with_center", [False, True])
def test_apf_group_bwd_bits_vs_numpy(det, idx_dtype, use_perm, with_center):
    B, N, C, G, k = 3, 1024, 3, 64, 16
    x, fidx, kidx, perm = _apf_indices(B, N, C, G, k, 31)
    perm = perm if use_perm else None
    gn = _rand((B, G, k, 2 * C), 32)
    gc = _rand((B, G, 3), 33) if with_center else None
    got = ops.apf_group_bwd(to_dev(gn), to_dev(gc) if gc is not None else None, fidx, kidx.to(idx_dtype), perm, N, C)
    _bits_equal(got, _apf_bwd_ref(gn, gc, fidx, kidx, perm, N, C), "apf_group_bwd")


@gpu
def test_apf_group_bwd_bits_vs_numpy_large_cloud(det):
    B, N, C, G, k = 1, 65536, 3, 2048, 64
    x, fidx, kidx, perm = _apf_indices(B, N, C, G, k, 41)
    gn = _rand((B, G, k, 2 * C), 42)
    got = ops.apf_group_bwd(to_dev(gn), None, fidx, kidx.to(torch.int32), perm, N, C)
    _bits_equal(got, _apf_bwd_ref(gn, None, fidx, kidx, perm, N, C), "apf_group_bwd 65536 points")


@gpu
@pytest.mark.parametrize("D", [0, 61, 128])
@pytest.mark.parametrize("need", [(True, True), (True, False), (False, True)])
def test_group_gather_bwd_bits_vs_numpy(det, D, need):
    need_p, need_f = need
    if need_f and not need_p and D == 0:
        pytest.skip("no output to scatter to")
    B, N, G, k = 2, 300, 40, 24
    idx = (synth.uniform01(51, B * G * k, 2).reshape(B, G, k) * N).astype(np.int64) % 37          # heavy repeats
    gp, gf = _rand((B, G, k, 3), 52), _rand((B, G, k, D), 53, 1e3)
    dp, df = ops.group_gather_bwd(to_dev(gp), to_dev(gf), to_dev(idx), N, D, need_p, need_f)
    W = (3 if need_p else 0) + (D if need_f else 0)
    bb = np.arange(B)[:, None, None]
    # one accumulator for both outputs: dP slots first, then dF; the per-cloud scale covers the columns scattered
    slots, vals, clouds = [], [], []
    if need_p:
        slots.append(((bb * N + idx)[..., None] * 3 + np.arange(3)).ravel())
        vals.append(gp.ravel())
    if need_f and D:
        slots.append(B * N * 3 + ((bb * N + idx)[..., None] * D + np.arange(D)).ravel())
        vals.append(gf.ravel())
    slot, val = np.concatenate(slots), np.concatenate(vals)
    cloud = np.where(slot < B * N * 3, slot // (N * 3), (slot - B * N * 3) // max(N * D, 1))
    # emulate with one per-cloud scale over both regions: slots remapped to (cloud, position) with a common per-cloud size
    per = N * (3 + D)
    local = np.where(slot < B * N * 3, slot - cloud * N * 3, N * 3 + (slot - B * N * 3) - cloud * N * D)
    ref = fixed_point_sum(B, per, G * k, cloud * per + local, val).reshape(B, per)
    assert W > 0
    if need_p:
        _bits_equal(dp, ref[:, :N * 3], f"group_gather_bwd dP D={D}")
    else:
        assert dp.numel() == 0
    if need_f:
        _bits_equal(df, ref[:, N * 3:], f"group_gather_bwd dF D={D}")
    else:
        assert df.numel() == 0


@gpu
def test_scatter_non_finite_contributions(det):
    B, N, S, C = 2, 64, 512, 3
    idx = np.tile(np.arange(S) % N, (B, 1)).astype(np.int64)
    g = _rand((B, S, C), 61)
    for s_, v in ((0, np.inf), (1, -np.inf), (2, np.inf), (2 + N, -np.inf), (3, np.nan), (4 + N, np.nan), (5, np.inf), (5 + N, np.inf)):
        g[0, s_, 1] = v                                        # destinations 0..5 of cloud 0, channel 1
    got = ops.gather_points_bwd(to_dev(g), to_dev(idx), N)
    ref = fixed_point_sum(B, N * C, S, *gather_points_contribs(g, idx, N))
    _bits_equal(got, ref, "gather_points_bwd with non-finite contributions")
    r = got[0, :6, 1].cpu().numpy()
    assert r[0] == np.inf and r[1] == -np.inf and np.isnan(r[2]) and np.isnan(r[3]) and np.isnan(r[4]) and r[5] == np.inf
    assert np.isfinite(got[0, 6:].cpu().numpy()).all() and np.isfinite(got[1].cpu().numpy()).all()


@gpu
def test_scatters_are_batch_invariant(det):
    B, N, C, G, k = 5, 2048, 3, 128, 32
    x, fidx, kidx, perm = _apf_indices(B, N, C, G, k, 71, dup=False)
    gn, gc = to_dev(_rand((B, G, k, 2 * C), 72)), to_dev(_rand((B, G, 3), 73, 1e4))
    gn[3] *= 1e-6
    full = ops.apf_group_bwd(gn, gc, fidx, kidx, perm, N, C)
    g2 = to_dev(_rand((B, G, 4), 74))
    full2 = ops.gather_points_bwd(g2, fidx, N)
    for b in range(B):
        one = ops.apf_group_bwd(gn[b:b + 1], gc[b:b + 1], fidx[b:b + 1], kidx[b:b + 1], perm[b:b + 1], N, C)
        assert torch.equal(one[0].view(torch.int32), full[b].view(torch.int32)), b
        one2 = ops.gather_points_bwd(g2[b:b + 1], fidx[b:b + 1], N)
        assert torch.equal(one2[0].view(torch.int32), full2[b].view(torch.int32)), b


# ------------------------------------------------------------------------------------------------ ordered reductions
def _ws(nbytes):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=dev())


def _seq_sum(parts):
    acc = torch.zeros_like(parts[0], dtype=torch.float64)
    for p in parts:
        acc = acc + p.double()
    return acc


def _busy_side_stream():
    """A large p3tok GEMM enqueued on a second stream, running while the call under test runs."""
    side = torch.cuda.Stream()
    a = torch.randn(65536, 512, device=dev())
    w = torch.randn(512, 512, device=dev())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        train.linear(a, w)
    return side


@gpu
@pytest.mark.parametrize("M,N,K", [(0, 64, 64), (100, 64, 64), (1000, 70, 33), (524288, 128, 6), (524288, 6, 128), (16384, 1536, 384)])
@pytest.mark.parametrize("accumulate", [0, 1])
def test_linear_tn_det_slice_layout_and_order(M, N, K, accumulate):
    L = _lib.lib()
    torch.manual_seed(M + N)
    dy, x = torch.randn(M, N, device=dev()), torch.randn(M, K, device=dev())
    dw0 = torch.randn(N, K, device=dev())
    nb = L.p3tok_linear_tn_det_workspace_bytes(M, N, K)
    ws = _ws(nb)
    s = torch.cuda.current_stream().cuda_stream

    def call():
        dw = dw0.clone()
        _lib.check(L.p3tok_linear_tn_det_f32(dy.data_ptr(), x.data_ptr(), M, N, K, dw.data_ptr(), accumulate, ws.data_ptr(), nb, s), "tn")
        return dw

    dw = call()
    ref64 = dy.double().t() @ x.double() + (dw0.double() if accumulate else 0)
    if M == 0:
        assert torch.equal(dw, dw0 if accumulate else torch.zeros_like(dw0))
        return
    nsl, rows = tn_slices(M, N, K)
    part = ws.view(torch.float32).view(nsl, N, K)
    sm = _seq_sum(list(part)).float()
    assert torch.equal(dw, dw0 + sm if accumulate else sm), "dW is not the ascending fp64 sum of the slices, rounded once"
    for z in range(nsl):
        r = slice(z * rows, min(M, (z + 1) * rows))
        ref = dy[r].double().t() @ x[r].double()
        err = float((part[z].double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
        assert err < 1e-5, (z, err)
    assert float((dw.double() - ref64).abs().max() / ref64.abs().max()) < 1e-5
    for _ in range(5):
        side = _busy_side_stream()
        again = call()
        torch.cuda.current_stream().wait_stream(side)
        assert torch.equal(again, dw)


def _strip_case(kind, M, N):
    torch.manual_seed(M * 7 + N)
    L = _lib.lib()
    x = torch.randn(M, N, device=dev()) + 0.5
    dy = torch.randn(M, N, device=dev())
    mean, rstd = torch.randn(N, device=dev()) * 0.1, torch.rand(N, device=dev()) + 0.5
    gamma, beta = torch.randn(N, device=dev()), torch.randn(N, device=dev()) * 0.1
    rmean, rrstd = torch.randn(M, device=dev()) * 0.1, torch.rand(M, device=dev()) + 0.5
    pre = ((x.double() - mean.double()) * rstd.double()) * gamma.double() + beta.double()
    dy = torch.where(pre.abs() < 1e-4, torch.zeros_like(dy), dy)   # no ReLU decision within rounding of 0: both sides agree
    s = torch.cuda.current_stream().cuda_stream
    nb = L.p3tok_colsum_det_workspace_bytes(M, N)
    ws = _ws(nb)
    out = torch.empty(2 * N, dtype=torch.float64, device=dev())
    o0, o1 = out.data_ptr(), out.data_ptr() + 8 * N
    if kind == "colstats":
        call = lambda: L.p3tok_colstats_det_f32(x.data_ptr(), M, N, o0, o1, ws.data_ptr(), nb, s)
        terms = lambda r: (x[r].double(), x[r].double() ** 2)
    elif kind == "bn_bwd_stats":
        call = lambda: L.p3tok_bn_bwd_stats_det_f32(dy.data_ptr(), x.data_ptr(), M, N, mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(),
                                                     beta.data_ptr(), 1, o0, o1, ws.data_ptr(), nb, s)

        def terms(r):
            xh = (x[r] - mean) * rstd
            d = torch.where(xh * gamma + beta > 0, dy[r], torch.zeros_like(dy[r])).double()
            return d, d * xh.double()
    else:
        call = lambda: L.p3tok_ln_param_grad_det_f32(dy.data_ptr(), x.data_ptr(), M, N, rmean.data_ptr(), rrstd.data_ptr(), o0, o1,
                                                      ws.data_ptr(), nb, s)
        terms = lambda r: (dy[r].double() * ((x[r] - rmean[r, None]) * rrstd[r, None]).double(), dy[r].double())
    return call, terms, ws, out


@gpu
@pytest.mark.parametrize("kind", ["colstats", "bn_bwd_stats", "ln_param_grad"])
@pytest.mark.parametrize("M,N", [(0, 64), (50, 64), (1000, 70), (524288, 64), (16384, 384)])
def test_strip_reductions_det_layout_and_order(kind, M, N):
    call, terms, ws, out = _strip_case(kind, M, N)
    _lib.check(call(), kind)
    if M == 0:
        assert torch.equal(out, torch.zeros_like(out))
        return
    ns, rows = strips(M, N)
    part = ws.view(torch.float64).view(2, ns, N)
    for q in range(2):
        assert torch.equal(out[q * N:(q + 1) * N], _seq_sum(list(part[q]))), f"{kind}: not the ascending sum of the strips"
        for y in range(ns):
            ref = terms(slice(y * rows, min(M, (y + 1) * rows)))[q].sum(0)
            err = float((part[q, y] - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
            assert err < 1e-4, (kind, q, y, err)
        full = terms(slice(0, M))[q].sum(0)
        assert float((out[q * N:(q + 1) * N] - full).abs().max() / full.abs().max()) < 1e-5
    first = out.clone()
    for _ in range(5):
        side = _busy_side_stream()
        _lib.check(call(), kind)
        torch.cuda.current_stream().wait_stream(side)
        assert torch.equal(out, first)


@gpu
def test_det_workspace_too_small_is_an_error():
    L = _lib.lib()
    x = torch.randn(1000, 64, device=dev())
    out = torch.empty(128, dtype=torch.float64, device=dev())
    nb = L.p3tok_colsum_det_workspace_bytes(1000, 64)
    ws = _ws(nb)
    rc = L.p3tok_colstats_det_f32(x.data_ptr(), 1000, 64, out.data_ptr(), out.data_ptr() + 512, ws.data_ptr(), nb - 8,
                                  torch.cuda.current_stream().cuda_stream)
    assert rc == _lib.ERR_WORKSPACE


# ------------------------------------------------------------------------------------------------ routing
ATOMIC = ("sgemm_tn_kernel<false>", "colstats_kernel<false>", "bn_bwd_stats_kernel<false>", "ln_param_grad_kernel<false>",
          "AtomicF32Add")
DET = ("sgemm_tn_kernel<true>", "colstats_kernel<true>", "bn_bwd_stats_kernel<true>", "ln_param_grad_kernel<true>", "FixedAdd",
       "CloudMaxAbs", "slice_sum_kernel", "strip_sum_kernel", "fixed_to_f32_kernel")


_ROUTING_CHILD = r"""
import json, os, sys
sys.path[:0] = [{root!r}, os.path.join({root!r}, "adapting-2d-vits-for-3d-point-cloud-understanding_b200"), os.path.join({root!r}, "tests")]
import torch
from p3tok import synth, train
from p3tok.apf_model import AdaptPointFormer
mode, out = sys.argv[1], sys.argv[2]
torch.use_deterministic_algorithms(mode != "off", warn_only=mode == "warn_only")
assert train.deterministic() == (mode != "off")
dev = torch.device("cuda:0")
torch.manual_seed(0)
B, N, G, k, E = 2, 512, 32, 16, 384
m = AdaptPointFormer(num_classes=7, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="fp32").to(dev).train()
m._freeze()
x = torch.from_numpy(synth.make_cloud("uniform", B, N, 5, 3)).to(dev).requires_grad_(True)
st = torch.from_numpy(synth.start_indices(B, N, 5)).to(dev)
w = torch.randn(B, 7, device=dev)
(m(x, st) * w).sum().backward()                                 # warm-up outside the trace
torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
    (m(x, st) * w).sum().backward()
    torch.cuda.synchronize()
prof.export_chrome_trace(out)
"""


def _apf_step_kernels(mode, tmp_path):
    """Kernel names of one APF training step (x requiring grad) under the given flag mode.  The trace is taken in a child
    process, so this test leaves the profiler state of the test process as it found it."""
    import json
    path = str(tmp_path / f"routing_{mode}.json")
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    subprocess.run([sys.executable, "-c", _ROUTING_CHILD.format(root=ROOT), mode, path], check=True, env=env, cwd=ROOT,
                   timeout=600)
    with open(path) as f:
        names = {e["name"] for e in json.load(f)["traceEvents"] if e.get("cat") == "kernel"}
    assert names, "the profiler recorded no kernels"
    return names


@gpu
@pytest.mark.parametrize("mode", ["off", "on", "warn_only"])
def test_routing_by_kernel_names(mode, tmp_path):
    names = _apf_step_kernels(mode, tmp_path)
    hit = lambda pats: sorted(n for n in names if any(p in n for p in pats))
    if mode == "off":
        assert not hit(DET), hit(DET)
        assert hit(ATOMIC)
    else:
        assert not hit(ATOMIC), hit(ATOMIC)
        for p in ("sgemm_tn_kernel<true>", "colstats_kernel<true>", "bn_bwd_stats_kernel<true>", "ln_param_grad_kernel<true>",
                  "FixedAdd", "fixed_to_f32_kernel"):
            assert any(p in n for n in names), p


# ------------------------------------------------------------------------------------------------ across processes
_CHILD = r"""
import os, sys
sys.path[:0] = [{root!r}, os.path.join({root!r}, "adapting-2d-vits-for-3d-point-cloud-understanding_b200"), os.path.join({root!r}, "tests")]
import numpy as np, torch
from p3tok import synth
from p3tok.apf_model import AdaptPointFormer
from p3tok.p4p_model import Pix4Point
torch.use_deterministic_algorithms(True)
torch.manual_seed(1234)
dev = torch.device("cuda:0")
case, out = sys.argv[1], sys.argv[2]
if case in ("apf", "apf_tc"):
    B, N, G, k, E = 16, 1024, 64, 16, 384
    m = AdaptPointFormer(num_classes=7, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="fp32",
                         dropout_rate=0.1, dropout_path_rate=0.2)
    m.blocks = m.blocks[:4]
    m = m.to(dev).train()
    m._freeze()
    nc = 7
elif case == "p4p":
    B, N, E = 4, 2048, 64
    m = Pix4Point(num_classes=5, embed_dim=E, depth=2, num_heads=2, k_neighbors=16, precision="fp32",
                  sample_ratio=0.0625).to(dev).train()
    nc = 5
else:
    B, N, G, k, E = 4, 512, 32, 16, 384
    m = AdaptPointFormer(num_classes=7, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="bf16",
                         block_precision="fp32tc").to(dev).eval()
    m._freeze()
    nc = 7
x = torch.from_numpy(synth.make_cloud("clustered", B, N, 9, 3)).to(dev).requires_grad_(True)
st = torch.from_numpy(synth.start_indices(B, N, 9)).to(dev)
w = torch.randn(B, nc, device=dev)
opt = torch.optim.AdamW([p for p in m.parameters() if p.requires_grad], lr=1e-3)
sts = [torch.from_numpy(synth.start_indices(B, N // 4 ** s, 9, s)).to(dev) for s in range(2)] if case == "p4p" else st
logits = m(x, sts)
(logits * w).sum().backward()
opt.step()
res = {{"logits": logits.detach(), "x.grad": x.grad}}
for n, p in m.named_parameters():
    if p.grad is not None:
        res["grad." + n] = p.grad
        res["param." + n] = p.detach()
for n, b in m.named_buffers():
    res["buf." + n] = b
np.savez(out, **{{k: v.detach().cpu().numpy() for k, v in res.items()}})
"""


def _child_run(case, path, env_extra):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8", **env_extra)
    subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT), case, path], check=True, env=env, cwd=ROOT, timeout=1200)
    return np.load(path)


@gpu
@pytest.mark.parametrize("case,env", [("apf", {}), ("p4p", {}), ("apf_eval_bf16", {}), ("apf_tc", {"P3TOK_TRAIN_TC": "1"})])
def test_training_step_bit_identical_across_processes(case, env, tmp_path):
    a = _child_run(case, str(tmp_path / "a.npz"), env)
    b = _child_run(case, str(tmp_path / "b.npz"), env)
    assert sorted(a.files) == sorted(b.files)
    assert "x.grad" in a.files and any(f.startswith("grad.") for f in a.files)
    for f in a.files:
        assert a[f].tobytes() == b[f].tobytes(), f"{case}: {f} differs between processes"


# ------------------------------------------------------------------------------------------------ accuracy unchanged
@gpu
def test_pointnet_train_gradients_vs_float64_under_the_flag(det):
    import grad_reference as gr
    from oracle import oracle, train as otrain
    from p3tok.modules import PointNet
    B, N, C, G, k, E = 3, 500, 3, 21, 12, 48
    x = synth.make_cloud("clustered", B, N, 91, C)
    st = to_dev(synth.start_indices(B, N, 91))
    sd = synth.apf_encoder_state(E, 2 * C, 91)
    gt = (synth.uniform01(91, B * G * E, 3).reshape(B, G, E) - 0.5).astype(np.float32)
    net = PointNet(E, G, k, 2 * C).to(dev()).train()
    net.encoder.load_state_dict(synth.to_torch_state(sd))
    xt = to_dev(x).requires_grad_(True)
    (net(xt, st) * to_dev(gt)).sum().backward()
    grp = oracle.group_apf(x, st.cpu().numpy(), G, k)
    _, ograds, _ = otrain.apf_encoder_train(sd, grp["neigh"], gt)
    scale = max(np.abs(v).max() for k_, v in ograds.items() if k_.endswith("weight") and "conv" in k_)
    for n, p_ in net.encoder.named_parameters():
        err = np.abs(p_.grad.double().cpu().numpy() - ograds[n].reshape(p_.shape)).max() / scale
        assert err <= 1e-4, (n, err)
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    gidx = [torch.from_numpy(np.asarray(grp[n])) for n in ("fps_idx", "knn_idx", "perm")]
    gr.apf_group_idx(x64, *gidx)[0].backward(torch.from_numpy(ograds["input"]))
    ref = x64.grad.numpy()
    assert np.abs(xt.grad.double().cpu().numpy() - ref).max() / np.abs(ref).max() <= 1e-4


@gpu
def test_p3embed_train_gradients_vs_reference_under_the_flag(det, golden_dir):
    import cases
    import make_golden
    from p3tok.modules import P3Embed
    c = cases.P4P_TRAIN_CASES["p4p_train"]
    g = np.load(os.path.join(golden_dir, "p4p_train.npz"))
    x, start, sd, go = make_golden.p4p_train_inputs(c)
    m = P3Embed(in_channels=3, sample_ratio=0.25, scale=4, k=c["k"], layers=4, embed_dim=c["W"]).to(dev()).train()
    m.load_state_dict(synth.to_torch_state(sd))
    p = to_dev(x).requires_grad_(True)
    fe = to_dev(np.ascontiguousarray(x.transpose(0, 2, 1))).requires_grad_(True)
    _, fs = m(p, fe, [to_dev(start)])
    (fs[-1].transpose(1, 2) * to_dev(go)).sum().backward()
    for got, key in ((p.grad, "grad.p"), (fe.grad.transpose(1, 2), "grad.f")):
        ref = g[key]
        assert np.abs(got.double().cpu().numpy() - ref).max() / np.abs(ref).max() <= 1e-4, key
    scale = max(np.abs(g[k_]).max() for k_ in g.files if k_.startswith("grad.convs") and k_.endswith("weight"))
    for name, q in m.named_parameters():
        err = np.abs(q.grad.cpu().numpy().astype(np.float64) - g["grad." + name]).max() / scale
        assert err <= 1e-4, (name, err)
