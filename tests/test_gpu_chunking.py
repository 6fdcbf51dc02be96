"""Patch-embedding tokens across row-chunk boundaries.

p3tok_patch_embed walks the groups in row chunks: bf16 / fp32tc in chunks sized by chunk_groups() (csrc/embed_tc.cu:
2^20 to 2^22 rows, then equal chunks of a multiple of 8 groups), fp32 in fixed chunks of 8192 groups (csrc/mlp_f32.cu).
Every chunk after the first depends on offset arithmetic the first never exercises: g_begin in each first-layer route,
the cloud b = bj / G and the Morton-permuted group of a chunk that starts inside a cloud, the token offset g0 * out_dim
(`tokb` for bf16 tokens), the in-kernel first-layer weights packed by chunk 0 only, and the short last chunk.

A. Forced small chunks (P3TOK_CHUNK_ROWS, latched on first use, so set in a subprocess): every first-layer / pooling route
   at small shapes with G = 100 (and P3Embed stage sizes 250 / 62), so chunk boundaries fall inside clouds and chunks
   straddle clouds.  Tokens must equal the default (one chunk) tokens bit for bit: every kernel's per-row arithmetic is
   independent of the chunk's row count.
B. The default chunking at bench batch sizes: sentinel clouds next to the boundaries that chunk_groups() below predicts
   must equal the same cloud tokenized alone (one chunk), bit for bit, and match the float64 oracle.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import assert_tokens_close, dev, to_dev
from oracle import oracle
from p3tok import ops, synth
from p3tok.modules import Encoder, P3Embed, PointNet

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "adapting-2d-vits-for-3d-point-cloud-understanding_b200"
RTOL = {"fp32": 1e-4, "fp32tc": 1e-4, "bf16": 1e-2}
F32_CHUNK_GROUPS = 8192                   # csrc/mlp_f32.cu


# ------------------------------------------------------------------ the chunk policy, mirrored from csrc/embed_tc.cu
def rows_target(wmax, rows_env=0):
    """Rows per chunk before the split into equal chunks (chunk_groups in csrc/embed_tc.cu)."""
    t = rows_env
    if t <= 0:
        t = min(max((1 << 20) * 768 // (wmax if wmax > 0 else 768), 1 << 20), 1 << 22)
    return max(t, 128)


def chunk_groups(ngroups, k, wmax, rows_env=0):
    """Groups per chunk for `ngroups` groups of k rows; wmax = the block's widest activation in bf16 columns."""
    cg = max(rows_target(wmax, rows_env) // k, 1)
    n = -(-ngroups // cg)
    if n > 1:
        cg = (-(-ngroups // n) + 7) // 8 * 8
    return min(ngroups, cg)


def chunk_wmax(meta, prec):
    """The `wmax` that bf_layout (bf16) / x3_layout (fp32tc) pass to chunk_groups, from a folded block's meta
    [cin, n_pre, pre_dim..., pre_relu..., mid_dim, out_dim, out_relu]."""
    cin, n = meta[0], meta[1]
    widths = list(meta[2:2 + n]) + [meta[2 + 2 * n]]
    if prec == "bf16":
        return max([0 if cin <= 16 else (cin + 7) // 8 * 8] + widths)
    assert prec == "fp32tc"
    return 2 * max([0 if cin <= 16 else (cin + 63) // 64 * 64] + widths)


def chunk_size(ngroups, k, meta, prec, rows_env=0):
    if prec == "fp32":
        return min(ngroups, F32_CHUNK_GROUPS)
    return chunk_groups(ngroups, k, chunk_wmax(meta, prec), rows_env)


def boundaries(ngroups, cg):
    return list(range(cg, ngroups, cg))


# ------------------------------------------------------------------ A. forced small chunks, every route
FORCED_ROWS = (1, 3000)     # 1: the 128-row floor (8 groups per chunk for k >= 16); 3000: multi-tile chunks, k = 24 -> 2496 rows
CASES = {}


def _case(fn):
    CASES[fn.__name__.lstrip("_")] = fn
    return fn


def _counted(run):
    """run() -> (list of tokens on the host, kernels libp3tok launched for it)."""
    n0 = ops.kernel_launches()
    out = run()
    torch.cuda.synchronize()
    return [t.cpu() for t in out], ops.kernel_launches() - n0


def _apf(C, k, E, prec, token_dtype=None, B=3, N=1024, G=100, seed=0):
    """APF PointNet on B clouds of C channels: (tokens, launches, oracle references as [(ref, rtol)])."""
    s = 500 + 7 * C + k + E + seed
    if C <= 4:
        x = synth.make_cloud("clustered", B, N, s, C)
    else:
        x = np.concatenate([synth.make_cloud("clustered", B, N, s, 3), synth.make_points_nd(B, N, C - 3, s + 1)], -1)
    st = synth.start_indices(B, N, s)
    sd = synth.apf_encoder_state(E, 2 * C, s)
    net = PointNet(E, G, k, 2 * C, precision=prec, token_dtype=token_dtype).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd), strict=True)
    xt, stt = to_dev(x), to_dev(st)
    tok, n = _counted(lambda: [net(xt, stt)])
    return tok, n, lambda: [(oracle.pointnet_apf(sd, x, st, G, k)[0], RTOL[prec])]


def _p3e(prec, D=3, embed=256, k=32, B=2, N=1000, seed=0):
    """Two-stage P3Embed (sample ratio 1/16; N = 1000 -> 250 -> 62 centres): the tokens of both stages."""
    s = 600 + D + embed + k + seed
    p = synth.make_cloud("clustered", B, N, s, 3)
    f = p.copy() if D == 3 else synth.make_points_nd(B, N, D, s + 1)
    starts = [synth.start_indices(B, N, s, 0), synth.start_indices(B, N // 4, s, 1)]
    sd = synth.p3embed_state(D, 1 / 16, 4, 4, embed, s)
    mod = P3Embed(in_channels=D, sample_ratio=1 / 16, k=k, embed_dim=embed, precision=prec).eval().to(dev())
    mod.load_state_dict(synth.to_torch_state(sd), strict=True)
    pt, ft, stt = to_dev(p), to_dev(f).transpose(1, 2).contiguous(), [to_dev(v) for v in starts]
    tok, n = _counted(lambda: mod(pt, ft, stt)[1][1:])

    def ref():
        _, of, _ = oracle.p3embed(sd, p, f, starts, k, 2)
        return [(np.ascontiguousarray(of[s_].transpose(0, 2, 1)), RTOL[prec] * s_) for s_ in (1, 2)]   # channel-first like `tok`
    return tok, n, ref


@_case
def _apf_c3_k32_bf16():
    """bf16, C = 3, k = 32, E = 384: in-kernel first layer (apf_rel_rows_kernel + FusedL1, packed weights written by chunk 0
    only), the "pre" and concat/output pair kernels, float32 tokens at tokens + g0 * out_dim."""
    return _apf(3, 32, 384, "bf16")


@_case
def _apf_c3_k32_bf16_tokens():
    """As apf_c3_k32_bf16 with token_dtype = bfloat16: the pair epilogue writes the tokens through `tokb`."""
    return _apf(3, 32, 384, "bf16", token_dtype=torch.bfloat16)


@_case
def _apf_c4_k64_bf16():
    """bf16, C = 4 (xyz + height), k = 64: in-kernel first layer, parts = 2 partial maxima (partial_max_bf16_kernel,
    group_max_f32_kernel) over the chunk's gc groups."""
    return _apf(4, 64, 384, "bf16")


@_case
def _apf_c3_k24_bf16():
    """bf16, k = 24 (not a multiple of 32): generic rows_first_layer_kernel, layer-by-layer tc_linear, unfused max through
    `scratch` + group_max_f32_kernel."""
    return _apf(3, 24, 384, "bf16")


@_case
def _apf_c6_bf16():
    """bf16, C = 6 (12 input channels): the generic CUDA-core first layer (rows_first_layer_kernel, 16 channels)."""
    return _apf(6, 32, 384, "bf16")


@_case
def _apf_c9_bf16():
    """bf16, C = 9 (18 input channels): gathered tensor-core rows (rows_gather_bf16_kernel, kind 0) + padded weight."""
    return _apf(9, 32, 384, "bf16")


@_case
def _apf_e48_bf16():
    """bf16, E = 48: rows_first_layer_apf_warp_kernel, then layer-by-layer tc_linear (no pair kernel fits these widths)."""
    return _apf(3, 32, 48, "bf16")


@_case
def _encoder_rows_bf16():
    """bf16 Encoder on a materialised (B, G, k, 6) row tensor (kind 2): rows_first_layer_narrow_kernel reads
    R.x[(g_begin * k + r) * cin]."""
    B, N, G, k, E, s = 3, 1024, 100, 32, 384, 701
    x = synth.make_cloud("uniform", B, N, s, 3)
    neigh = oracle.group_apf(x, synth.start_indices(B, N, s), G, k)["neigh"]
    sd = synth.apf_encoder_state(E, 6, s)
    enc = Encoder(E, 6, precision="bf16").eval().to(dev())
    enc.load_state_dict(synth.to_torch_state(sd), strict=True)
    nt = to_dev(neigh)
    tok, n = _counted(lambda: [enc(nt)])
    return tok, n, lambda: [(oracle.apf_encoder(sd, neigh), RTOL["bf16"])]


@_case
def _p3e_default_bf16():
    """bf16 P3Embed, in_channels 3, embed 256: stage 0 rows_first_layer_narrow_kernel with l1_gmax + tc_stage_kernel;
    stage 1 tc_gather_linear (feature width D = 128, g_begin in the GEMM producer) + the concat/output pair kernel."""
    return _p3e("bf16")


@_case
def _p3e_e192_bf16():
    """bf16 P3Embed, embed 192: stage 1 has D = 96, so rows_gather_p4p_bf16_kernel + tc_linear, and a tail that is
    neither the stage kernel nor the pair kernel."""
    return _p3e("bf16", embed=192)


@_case
def _p3e_in13_bf16():
    """bf16 P3Embed, in_channels 13 (16 input channels): the generic rows_first_layer_kernel for kind 1."""
    return _p3e("bf16", D=13)


@_case
def _p3e_in14_bf16():
    """bf16 P3Embed, in_channels 14 (17 input channels, D % 4 != 0): rows_gather_bf16_kernel for kind 1."""
    return _p3e("bf16", D=14)


@_case
def _p3e_k24_bf16():
    """bf16 P3Embed, k = 24: unfused max (group_max_bf16_kernel / group_max_f32_kernel) for kind 1 rows."""
    return _p3e("bf16", k=24)


@_case
def _apf_c3_k32_fp32tc():
    """fp32tc (patch_embed_x3), C = 3, k = 32: rows_first_layer_split_kernel, split-operand tc_linear, fused 32-row max."""
    return _apf(3, 32, 384, "fp32tc")


@_case
def _apf_c4_k64_fp32tc():
    """fp32tc, C = 4, k = 64: partial_max_kernel / group_max_f32_kernel over two 32-row parts per group."""
    return _apf(4, 64, 384, "fp32tc")


@_case
def _p3e_default_fp32tc():
    """fp32tc P3Embed: stage 0 first layer as the block's only per-point layer (fp32 scratch max); stage 1
    rows_gather_split_kernel (kind 1)."""
    return _p3e("fp32tc")


def _run_all(path):
    """Entry point of the forced-chunk subprocess: every case's tokens and launch count, saved to `path`."""
    torch.save({name: fn()[:2] for name, fn in CASES.items()}, path)


_SUBPROCESS = ("import os, sys; r = os.getcwd(); sys.path[:0] = [r, os.path.join(r, %r), os.path.join(r, 'tests')];"
               "import test_gpu_chunking as t; t._run_all(sys.argv[1])" % PKG)


@pytest.fixture(scope="module")
def forced(tmp_path_factory):
    """{P3TOK_CHUNK_ROWS: {case: (tokens, launches)}}, one subprocess per value (the variable is latched per process)."""
    out = {}
    for rows in FORCED_ROWS:
        path = str(tmp_path_factory.mktemp("chunks") / f"rows{rows}.pt")
        env = dict(os.environ, P3TOK_CHUNK_ROWS=str(rows))
        subprocess.run([sys.executable, "-c", _SUBPROCESS, path], check=True, env=env, cwd=ROOT, timeout=1200)
        out[rows] = torch.load(path)
    return out


@pytest.mark.parametrize("name", list(CASES))
def test_forced_chunks_match_one_chunk(name, forced):
    tok, launches, refs = CASES[name]()
    for rows, res in forced.items():
        ftok, flaunch = res[name]
        assert flaunch > launches, f"P3TOK_CHUNK_ROWS={rows}: {flaunch} launches, one chunk {launches}: the loop did not iterate"
        for i, (a, b) in enumerate(zip(ftok, tok)):
            assert a.dtype == b.dtype and a.shape == b.shape
            if not torch.equal(a, b):
                d = (a.float() - b.float()).abs().flatten(0, -2).amax(-1)
                bad = torch.nonzero(d).flatten()
                raise AssertionError(f"{name}, P3TOK_CHUNK_ROWS={rows}, output {i}: {bad.numel()} token rows differ from the "
                                     f"one-chunk run, first {bad[:8].tolist()}, max |diff| {float(d.max()):.3e}")
    for i, (t, (ref, rtol)) in enumerate(zip(tok, refs())):
        assert_tokens_close(t.float().numpy().reshape(ref.shape), ref, rtol, f"{name} output {i} vs oracle")


def test_forced_chunk_counts():
    """The forced values really split the case shapes into many chunks that straddle clouds (G = 100, stage sizes
    250 / 62 are not multiples of 8), with a short last chunk."""
    apf = [6, 3, 256, 512, 384, 1, 1, 0, 768, 384, 0]
    for k in (24, 32, 64):
        cg = chunk_size(300, k, apf, "bf16", rows_env=1)
        assert cg == 8 and -(-300 // cg) == 38 and 300 % cg
        cg = chunk_size(300, k, apf, "bf16", rows_env=3000)
        assert 3 <= -(-300 // cg) <= 7 and cg % 8 == 0 and any(b % 100 for b in boundaries(300, cg))
    assert (chunk_size(300, 24, apf, "bf16", rows_env=3000) * 24) % 256
    s0, s1 = [6, 1, 128, 1, 256, 128, 1], [131, 1, 256, 1, 512, 256, 1]
    for meta, ng, G in ((s0, 500, 250), (s1, 124, 62)):
        for rows in FORCED_ROWS:
            cg = chunk_size(ng, 32, meta, "bf16", rows_env=rows)
            assert cg < ng and any(b % G for b in boundaries(ng, cg))


# ------------------------------------------------------------------ B. default chunking at bench batch sizes
def _sentinels(ngroups, G, cg, per_boundary=2):
    """Clouds next to the chunk boundaries (the one holding each boundary's last group and the one holding its first;
    the same cloud when the boundary is inside it), for the first `per_boundary` boundaries, plus the last cloud."""
    s = set()
    for b in boundaries(ngroups, cg)[:per_boundary]:
        s |= {(b - 1) // G, b // G}
    return sorted(s | {ngroups // G - 1})


def _straddling(ngroups, G, cg):
    return [b // G for b in boundaries(ngroups, cg) if b % G]


_ORACLE = {}


def _memo(key, fn):
    if key not in _ORACLE:
        _ORACLE[key] = fn()
    return _ORACLE[key]


_C4 = dict(B=16, N=65536, G=2048, k=64, E=384, seed=4500)


def _c4_inputs():
    c = _C4
    return _memo("c4", lambda: (synth.make_cloud("uniform", c["B"], c["N"], c["seed"], 3), synth.start_indices(c["B"], c["N"], c["seed"]),
                                synth.apf_encoder_state(c["E"], 6, c["seed"])))


@pytest.mark.parametrize("prec", ["bf16", "fp32tc", "fp32"])
def test_c4_batch_chunks_against_single_clouds(prec):
    """c4 (APF B = 16, N = 65536, G = 2048, k = 64, E = 384): 2 chunks of 8 clouds in bf16 / fp32tc, 4 of 4 clouds in fp32.
    The clouds beside the boundaries and the last one equal the cloud tokenized alone; cloud 15 matches the oracle."""
    c = _C4
    B, N, G, k, E = c["B"], c["N"], c["G"], c["k"], c["E"]
    x, st, sd = _c4_inputs()
    net = PointNet(E, G, k, 6, precision=prec).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd), strict=True)
    cg = chunk_size(B * G, k, net.encoder.folded(dev()).meta(), prec)
    assert -(-B * G // cg) >= 2 and 15 * G >= cg           # cloud 15 lies in a later chunk than the first
    xt, stt = to_dev(x), to_dev(st)
    tok = net(xt, stt)
    for j in _sentinels(B * G, G, cg):
        assert torch.equal(tok[j], net(xt[j:j + 1], stt[j:j + 1])[0]), f"c4 {prec}: cloud {j} differs from the cloud alone"
    ref = _memo("c4_15", lambda: oracle.pointnet_apf(sd, x[15:16], st[15:16], G, k)[0])
    assert_tokens_close(tok[15:16].cpu().numpy(), ref, RTOL[prec], f"c4 {prec} cloud 15 (chunk {15 * G // cg}) vs oracle")


def _p3e_batch(prec, B, N, k, seed, mid_cloud=True):
    """P3Embed (1/16, embed 256) on B clouds: sentinels of both stages against the cloud alone, the first cloud that straddles
    a stage-0 boundary and the last cloud against the oracle."""
    p = synth.make_cloud("uniform", B, N, seed, 3)
    starts = [synth.start_indices(B, N, seed, 0), synth.start_indices(B, N // 4, seed, 1)]
    sd = synth.p3embed_state(3, 1 / 16, 4, 4, 256, seed)
    mod = P3Embed(sample_ratio=1 / 16, k=k, embed_dim=256, precision=prec).eval().to(dev())
    mod.load_state_dict(synth.to_torch_state(sd), strict=True)
    metas = [m.meta() for m in mod.folded(dev())]
    pt, stt = to_dev(p), [to_dev(s) for s in starts]
    fs = mod(pt, pt.transpose(1, 2).contiguous(), stt)[1]
    sentinels, straddle0 = {B - 1}, None
    for s, G in enumerate((N // 4, N // 16)):
        cg = chunk_size(B * G, k, metas[s], prec)
        mid = _straddling(B * G, G, cg)
        assert len(boundaries(B * G, cg)) >= 1 and (mid or not mid_cloud), f"stage {s}: {B} clouds give no mid-cloud boundary"
        sentinels |= set(mid[:3])
        if s == 0:
            straddle0 = mid[0] if mid else boundaries(B * G, cg)[0] // G
    for j in sorted(sentinels):
        one = mod(pt[j:j + 1], pt[j:j + 1].transpose(1, 2).contiguous(), [v[j:j + 1] for v in stt])[1]
        for s in (1, 2):
            assert torch.equal(fs[s][j], one[s][0]), f"P3Embed B={B} {prec}: stage {s - 1} tokens of cloud {j} differ from the cloud alone"
    for j in (straddle0, B - 1):
        _, of, _ = _memo(("p3e", B, N, k, seed, j), lambda: oracle.p3embed(sd, p[j:j + 1], p[j:j + 1].copy(), [v[j:j + 1] for v in starts], k, 2))
        for s in (1, 2):
            assert_tokens_close(fs[s][j:j + 1].transpose(1, 2).cpu().numpy(), of[s], RTOL[prec] * s,
                                f"P3Embed B={B} {prec} cloud {j} stage {s - 1} vs oracle")
    return sorted(sentinels)


@pytest.mark.parametrize("prec", ["bf16", "fp32tc"])
def test_c3_like_batch_chunks_against_single_clouds(prec):
    """P3Embed N = 8192, k = 32, B = 101: bf16 stage 0 splits at 33.67 / 67.34 clouds, stage 1 at 50.5 (fp32tc: stage 0 every
    20.2 clouds)."""
    got = _p3e_batch(prec, 101, 8192, 32, 3301)
    if prec == "bf16":
        assert got == [33, 50, 67, 100], got


def test_c5_batch_chunks_against_single_clouds():
    """c5 (P3Embed B = 4096, N = 1024, k = 32, bf16): 11 stage-0 chunks (first boundary at 372.375 clouds) and 6 stage-1
    chunks (682.75)."""
    got = _p3e_batch("bf16", 4096, 1024, 32, 5501)
    assert got[0] == 372 and 682 in got and got[-1] == 4095, got


def test_fp32_chunks_of_8192_groups():
    """The CUDA-core fp32 path above 8192 groups: APF N = 1024, G = 100, k = 32, B = 90 -> chunks of 8192 and 808 groups,
    the boundary inside cloud 81; clouds 81 and 89 equal the cloud alone and match the oracle."""
    B, N, G, k, E, seed = 90, 1024, 100, 32, 384, 8100
    assert _straddling(B * G, G, chunk_size(B * G, k, None, "fp32")) == [81]
    x = synth.make_cloud("clustered", B, N, seed, 3)
    st = synth.start_indices(B, N, seed)
    sd = synth.apf_encoder_state(E, 6, seed)
    net = PointNet(E, G, k, 6, precision="fp32").eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd), strict=True)
    xt, stt = to_dev(x), to_dev(st)
    tok = net(xt, stt)
    for j in (80, 81, 82, 89):
        assert torch.equal(tok[j], net(xt[j:j + 1], stt[j:j + 1])[0]), f"fp32: cloud {j} differs from the cloud alone"
    for j in (81, 89):
        ref, _ = oracle.pointnet_apf(sd, x[j:j + 1], st[j:j + 1], G, k)
        assert_tokens_close(tok[j:j + 1].cpu().numpy(), ref, RTOL["fp32"], f"fp32 B={B} cloud {j} vs oracle")
