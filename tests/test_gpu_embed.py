"""GPU parity of the patch embedding and of the whole tokenizer, through the module drop-ins
(which call the C ABI): fp32 path within rtol 1e-4, bf16 tensor-core path within rtol 1e-2."""
import os

import numpy as np
import pytest
import torch

import cases
from helpers import assert_tokens_close, bf16_emulation, dev, rel_err, to_dev
from oracle import oracle
from p3tok import _lib, ops, synth
from p3tok.modules import Encoder, P3Embed, PointNet

pytestmark = pytest.mark.gpu

PRECISIONS = [("fp32", 1e-4), ("bf16", 1e-2), ("fp32tc", 1e-4)]     # fp32tc: bf16x3 split operands on the tensor cores


def _skip_unless_x3_widths(prec, *widths):
    """The fp32tc mode needs every layer width to be a multiple of 64 (all BASELINE widths are); other widths raise."""
    if prec == "fp32tc" and any(w % 64 for w in widths):
        pytest.skip("fp32tc: widths not multiples of 64")


def _bf16_ready():
    try:
        e = Encoder(32, 6, precision="bf16").eval().to(dev())
        e(torch.zeros(1, 4, 8, 6, device=dev()))
        return True
    except Exception as ex:
        return "not built yet" not in str(ex)


def _skip_if_unbuilt(prec):
    if prec == "bf16" and not _bf16_ready():
        pytest.skip("bf16 tensor-core path not built yet")


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


def test_linear_and_group_max_blocks():
    torch.manual_seed(0)
    for (M, K, N) in ((1, 3, 5), (130, 6, 256), (257, 131, 96), (1000, 512, 384)):
        a = torch.randn(M, K, device=dev())
        w = torch.randn(N, K, device=dev())
        b = torch.randn(N, device=dev())
        got = ops.linear_f32(a, w, b, True)
        ref = torch.relu(a.double() @ w.double().T + b.double())
        assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 1e-5
    x = torch.randn(7 * 16, 33, device=dev())
    assert torch.equal(ops.group_max(x, 16), x.view(7, 16, 33).max(1)[0])


@pytest.mark.parametrize("prec,rtol", PRECISIONS)
@pytest.mark.parametrize("name", list(cases.APF_CASES))
def test_pointnet_golden(golden_dir, name, prec, rtol):
    _skip_if_unbuilt(prec)
    c, g = cases.APF_CASES[name], _golden(golden_dir, name)
    _skip_unless_x3_widths(prec, c["E"])
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], c["C"])
    st = synth.start_indices(c["B"], c["N"], c["seed"])
    sd = synth.apf_encoder_state(c["E"], 2 * c["C"], c["seed"])
    net = PointNet(c["E"], c["G"], c["k"], 2 * c["C"], precision=prec).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd), strict=True)
    tok = net(to_dev(x), to_dev(st))
    assert tok.shape == (c["B"], c["G"], c["E"]) and tok.dtype == torch.float32
    assert_tokens_close(tok.cpu().numpy(), g["tokens"], rtol, f"{name} vs reference")
    otok, grp = oracle.pointnet_apf(sd, x, st, c["G"], c["k"])
    assert_tokens_close(tok.cpu().numpy(), otok, rtol, f"{name} vs oracle")
    # Encoder.forward on the materialised groups gives the same tokens as the fused path
    tok2 = net.encoder(to_dev(grp["neigh"]))
    assert_tokens_close(tok2.cpu().numpy(), otok, rtol, f"{name} encoder-only")


@pytest.mark.parametrize("prec,rtol", PRECISIONS)
@pytest.mark.parametrize("name", list(cases.P4P_CASES))
def test_p3embed_golden(golden_dir, name, prec, rtol):
    _skip_if_unbuilt(prec)
    c, g = cases.P4P_CASES[name], _golden(golden_dir, name)
    stages, dims = synth.p3embed_dims(3, c["sample_ratio"], 4, 4, c["embed_dim"])
    _skip_unless_x3_widths(prec, *[d[1] for d in dims])
    sd = synth.p3embed_state(3, c["sample_ratio"], 4, 4, c["embed_dim"], c["seed"])
    mod = P3Embed(sample_ratio=c["sample_ratio"], k=c["k"], embed_dim=c["embed_dim"], precision=prec).eval().to(dev())
    mod.load_state_dict(synth.to_torch_state(sd), strict=True)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    starts, n = [], c["N"]
    for s in range(stages):
        starts.append(synth.start_indices(c["B"], n, c["seed"], s))
        n //= 4
    xt = to_dev(x)
    ps, fs = mod(xt, xt.transpose(1, 2).contiguous(), [to_dev(s) for s in starts])
    assert len(ps) == stages + 1 and ps[0] is xt
    for s in range(stages):
        assert np.array_equal(ps[s + 1].cpu().numpy(), g[f"centres{s}"])          # centres == reference
        assert fs[s + 1].shape == (c["B"], dims[s][1], c["N"] // 4 ** (s + 1))    # channel-first like the reference
        # stage error compounds through the previous stage's tokens -> loosen by stage
        assert_tokens_close(fs[s + 1].transpose(1, 2).cpu().numpy(), g[f"tokens{s}"], rtol * (1 + s), f"{name} stage {s}")


@pytest.mark.parametrize("prec,rtol", PRECISIONS)
def test_real_widths_against_oracle(prec, rtol):
    """The real channel widths of BASELINE's configs (E=384 APF; 128/256 P3Embed) at a reduced batch."""
    _skip_if_unbuilt(prec)
    B, N, G, k, E = 2, 2048, 128, 32, 384
    x = synth.make_cloud("clustered", B, N, 55, 3)
    st = synth.start_indices(B, N, 55)
    sd = synth.apf_encoder_state(E, 6, 55)
    net = PointNet(E, G, k, 6, precision=prec).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd))
    tok = net(to_dev(x), to_dev(st)).cpu().numpy()
    otok, _ = oracle.pointnet_apf(sd, x, st, G, k)
    assert_tokens_close(tok, otok, rtol, "APF C2 widths")
    sd2 = synth.p3embed_state(3, 1 / 16, 4, 4, 256, 56)
    mod = P3Embed(sample_ratio=1 / 16, k=32, precision=prec).eval().to(dev())
    mod.load_state_dict(synth.to_torch_state(sd2))
    p = synth.make_cloud("uniform", 2, 1024, 56, 3)
    starts = [synth.start_indices(2, 1024, 56, 0), synth.start_indices(2, 256, 56, 1)]
    ps, fs = mod(to_dev(p), to_dev(p).transpose(1, 2).contiguous(), [to_dev(s) for s in starts])
    op, of, _ = oracle.p3embed(sd2, p, p.copy(), starts, 32, 2)
    for s in (1, 2):
        assert np.array_equal(ps[s].cpu().numpy(), op[s])
        assert_tokens_close(fs[s].transpose(1, 2).cpu().numpy(), of[s], rtol * s, f"P3Embed stage {s - 1}")


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_token_properties_full_c2(prec):
    """Config 2 at full size: permutation invariance over neighbours and batch-slicing consistency."""
    _skip_if_unbuilt(prec)
    B, N, G, k, E = 128, 2048, 128, 32, 384
    x = to_dev(synth.make_cloud("uniform", B, N, 1236, 3))
    st = to_dev(synth.start_indices(B, N, 1236))
    net = PointNet(E, G, k, 6, precision=prec).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(synth.apf_encoder_state(E, 6, 0)))
    tok = net(x, st)
    assert tok.shape == (B, G, E) and bool(torch.isfinite(tok).all())
    # clouds are independent: tokenising a slice of the batch gives the same rows (bitwise)
    assert torch.equal(net(x[5:9], st[5:9]), tok[5:9])
    # neighbour order inside a group does not matter (max-pool)
    fidx, ctr, kidx, perm = net.group.indices(x[:4], st[:4])
    neigh, _ = ops.apf_group(x[:4].contiguous(), fidx, kidx, perm)
    t1 = net.encoder(neigh)
    t2 = net.encoder(neigh.flip(2))
    assert torch.equal(t1, t2) or rel_err(t1.cpu().numpy(), t2.cpu().numpy()) < 1e-6


@pytest.mark.parametrize("M,K,N", [(128, 64, 64), (128, 256, 256), (300, 48, 40), (1000, 512, 384), (4096, 768, 384),
                                   (37888, 384, 768), (33, 136, 256), (64, 8, 8)])
def test_tc_linear_building_block(M, K, N):
    """tcgen05 GEMM against torch on the same bf16 operands (fp32 accumulate on both sides)."""
    torch.manual_seed(M + K + N)
    a = (torch.randn(M, K, device=dev()) * 0.5).bfloat16()
    w = (torch.randn(N, K, device=dev()) * 0.1).bfloat16()
    b = torch.randn(N, device=dev())
    ob, of, om = ops.linear_bf16(a, w, b, True, True)
    ref = torch.relu(a.float() @ w.float().T + b)
    torch.cuda.synchronize()
    scale = float(ref.abs().max())
    assert float((of - ref).abs().max()) <= 2e-5 * max(scale, 1.0) + 1e-5 * K ** 0.5
    assert float((ob.float() - ref).abs().max()) <= 8e-3 * max(scale, 1.0)
    pad = (32 - M % 32) % 32
    refm = torch.cat([ref, ref.new_full((pad, N), -1.0)]).view(-1, 32, N).max(1)[0]
    assert float((om - refm).abs().max()) <= 2e-5 * max(scale, 1.0) + 1e-5 * K ** 0.5


@pytest.mark.parametrize("E,k,cin", [(64, 32, 6), (384, 32, 6), (48, 16, 8), (96, 64, 6), (384, 64, 6), (128, 32, 8),
                                     (128, 64, 6), (256, 32, 6), (320, 32, 6)])
def test_bf16_path_matches_its_arithmetic_model(E, k, cin):
    """Tight check of the tensor-core path: against a torch model of exactly its arithmetic (bf16 operands,
    fp32 accumulate) the only differences are accumulation order and bf16 ties -> 2e-3 of max."""
    _skip_if_unbuilt("bf16")
    from p3tok import fold
    torch.manual_seed(E)
    ng = 300
    rows = torch.randn(ng * k, cin, device=dev()) * 0.3
    sd = synth.to_torch_state(synth.apf_encoder_state(E, cin, 5))
    enc = Encoder(E, cin, precision="bf16").eval().to(dev())
    enc.load_state_dict(sd)
    tok = enc(rows.view(1, ng, k, cin))[0]
    model = bf16_emulation(fold.fold_apf_encoder(sd), rows, k)
    err = float((tok - model).abs().max() / model.abs().max())
    assert err < 2e-3, err


def test_cuda_graph_replay_matches_eager():
    """The serving wrapper: one tokenizer call captured into a CUDA graph returns the eager result bit-for-bit,
    also after the inputs change."""
    from p3tok.graph import GraphedTokenizer
    B, N, G, k, E = 8, 1024, 64, 32, 128
    net = PointNet(E, G, k, 6, precision="bf16" if _bf16_ready() else "fp32").eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(synth.apf_encoder_state(E, 6, 3)))
    x0, x1 = (to_dev(synth.make_cloud("uniform", B, N, s, 3)) for s in (1, 2))
    s0, s1 = (to_dev(synth.start_indices(B, N, s)) for s in (1, 2))
    g = GraphedTokenizer(lambda x, st: net(x, st), [x0, s0])
    assert torch.equal(g(x0, s0), net(x0, s0))
    assert torch.equal(g(x1, s1), net(x1, s1))
    assert torch.equal(g(x0, s0), net(x0, s0))


def test_fused_pair_kernel_matches_layerwise(monkeypatch, tmp_path):
    """embed_fused.cu (two layers per kernel, hidden activation kept on-chip; opt-in via P3TOK_FUSED=1) against the
    default layer-by-layer tensor-core path: same bf16 arithmetic, different accumulation grouping."""
    _skip_if_unbuilt("bf16")
    import subprocess, sys, os
    code = (
        "import sys, os; sys.path.insert(0, os.path.join(os.getcwd(), 'adapting-2d-vits-for-3d-point-cloud-understanding_b200'));"
        "import torch; from p3tok import synth; from p3tok.modules import PointNet;"
        "net = PointNet(384, 64, 32, 6, precision='bf16').eval().cuda();"
        "net.encoder.load_state_dict(synth.to_torch_state(synth.apf_encoder_state(384, 6, 9)));"
        "x = torch.from_numpy(synth.make_cloud('clustered', 4, 1024, 9, 3)).cuda();"
        "st = torch.from_numpy(synth.start_indices(4, 1024, 9)).cuda();"
        "torch.save(net(x, st).cpu(), sys.argv[1])")
    outs = []
    for flag in ("0", "1"):
        path = str(tmp_path / f"fused_{flag}.pt")
        env = dict(os.environ, P3TOK_FUSED=flag)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        outs.append(torch.load(path))
    err = float((outs[0] - outs[1]).abs().max() / outs[0].abs().max())
    assert err < 3e-3, err


def test_token_head_matches_oracle_and_golden(golden_dir):
    """SURVEY 8f next #1: proj + pos_embed + cls concat of PointViT.forward (pix4point.py:245-252), fp32, rtol 1e-4."""
    c = cases.HEAD_CASES["p4p_head"]
    g = _golden(golden_dir, "p4p_head")
    sd = synth.token_head_state(c["W"], c["E"], c["seed"])
    tokens = synth.uniform01(c["seed"], c["B"] * c["G"] * c["W"], 9).reshape(c["B"], c["G"], c["W"])
    centres = synth.make_cloud("uniform", c["B"], c["G"], c["seed"], 3)
    t = {k: to_dev(v) for k, v in sd.items()}
    feats, pos = ops.token_head(to_dev(tokens), to_dev(centres), t["proj.weight"], t["proj.bias"], t["pos_embed.0.weight"],
                                t["pos_embed.0.bias"], t["pos_embed.2.weight"], t["pos_embed.2.bias"], t["cls_token"], t["cls_pos"])
    of, op = oracle.token_head(sd, tokens, centres)
    for got, ref, gold in ((feats, of, g["feats"]), (pos, op, g["pos"])):
        assert_tokens_close(got.cpu().numpy(), ref, 1e-4, "token head vs oracle")
        assert_tokens_close(got.cpu().numpy(), gold, 1e-4, "token head vs torch.nn golden")


def test_pointvit_tokens_module():
    """PointViTTokens = P3Embed + token head behind PointViT's attribute names; BASELINE C1 shapes (embed dim 384)."""
    from p3tok.modules import PointViTTokens
    B, N, k, E = 4, 1024, 32, 384
    m = PointViTTokens(embed_dim=E, k_neighbors=k, sample_ratio=1 / 16).eval().to(dev())
    sd_p = synth.to_torch_state(synth.p3embed_state(3, 1 / 16, 4, 4, 256, 5))
    sd_h = synth.to_torch_state(synth.token_head_state(256, E, 5))
    m.patch_embed.load_state_dict(sd_p, strict=True)
    missing = m.load_state_dict(sd_h, strict=False)
    assert not missing.unexpected_keys and all(k_.startswith("patch_embed.") for k_ in missing.missing_keys)
    assert {"proj.weight", "pos_embed.0.weight", "pos_embed.2.bias", "cls_token", "cls_pos"} <= set(m.state_dict())
    p = synth.make_cloud("uniform", B, N, 5, 3)
    starts = [synth.start_indices(B, N, 5, 0), synth.start_indices(B, N // 4, 5, 1)]
    p_list, x_list, feats, pos = m(to_dev(p), None, [to_dev(s) for s in starts])
    assert feats.shape == pos.shape == (B, 1 + N // 16, E)
    op, of, _ = oracle.p3embed(synth.p3embed_state(3, 1 / 16, 4, 4, 256, 5), p, p.copy(), starts, k, 2)
    rf, rp = oracle.token_head(synth.token_head_state(256, E, 5), of[-1].astype(np.float32), op[-1])
    assert_tokens_close(feats.cpu().numpy(), rf, 2e-4, "PointViTTokens feats")
    assert_tokens_close(pos.cpu().numpy(), rp, 1e-4, "PointViTTokens pos_embed")


@pytest.mark.gpu
@pytest.mark.parametrize("W,ng", [(128, 8), (128, 4099), (64, 777)])
def test_stage_kernel_matches_arithmetic_model_and_layerwise(W, ng, tmp_path):
    """embed_stage.cu (concat + output layer + pool of a narrow P3Embed stage in one kernel, weights resident in
    shared memory) against a torch model of its arithmetic and against the layer-by-layer tensor-core path
    (P3TOK_STAGE=0 in a subprocess); ragged tile counts (ng not a multiple of 8 patches = 256 rows)."""
    _skip_if_unbuilt("bf16")
    import os, subprocess, sys
    from p3tok import fold
    k, cin = 32, 6
    sd = synth.p3embed_state(3, 0.25, 4, 4, W, 77)
    mlp = fold.fold_p3embed_stage(synth.to_torch_state(sd), 0)
    torch.manual_seed(W + ng)
    rows = (torch.randn(ng * k, cin) * 0.5)
    m = mlp.to(dev(), torch.bfloat16)
    tok = ops.patch_embed(_lib.ROWS_DIRECT, rows.to(dev()), None, None, None, None, ng, k, m.tensors(), m.meta(), True)
    model = bf16_emulation(mlp, rows.to(dev()), k)
    err = float((tok - model).abs().max() / model.abs().max())
    assert err < 2e-3, err
    path_in, path_out = str(tmp_path / "stage_in.pt"), str(tmp_path / "stage_out.pt")
    torch.save(rows, path_in)
    code = (
        "import sys, os; sys.path.insert(0, os.path.join(os.getcwd(), 'adapting-2d-vits-for-3d-point-cloud-understanding_b200'));"
        "import torch; from p3tok import synth, fold, ops, _lib;"
        f"mlp = fold.fold_p3embed_stage(synth.to_torch_state(synth.p3embed_state(3, 0.25, 4, 4, {W}, 77)), 0).to(torch.device('cuda:0'), torch.bfloat16);"
        "rows = torch.load(sys.argv[1]).cuda();"
        f"tok = ops.patch_embed(_lib.ROWS_DIRECT, rows, None, None, None, None, {ng}, 32, mlp.tensors(), mlp.meta(), True);"
        "torch.save(tok.cpu(), sys.argv[2])")
    env = dict(os.environ, P3TOK_STAGE="0")
    subprocess.run([sys.executable, "-c", code, path_in, path_out], check=True, env=env,
                   cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ref = torch.load(path_out)
    err2 = float((tok.cpu() - ref).abs().max() / ref.abs().max())
    assert err2 < 2e-3, err2


# ------------------------------------------------------------------ BASELINE configs[2] / configs[3] shapes, end to end
_C4_ORACLE = {}


def _c4_oracle(kind):
    """One cloud of BASELINE configs[3] (N = 65536, G = 2048, k = 64, E = 384) through the oracle (~10 s), cached per kind."""
    if kind not in _C4_ORACLE:
        B, N, G, k, E = 1, 65536, 2048, 64, 384
        x = synth.make_cloud(kind, B, N, 4400 + len(kind), 3)
        st = synth.start_indices(B, N, 4400)
        sd = synth.apf_encoder_state(E, 6, 44)
        tok, grp = oracle.pointnet_apf(sd, x, st, G, k)
        _C4_ORACLE[kind] = (x, st, sd, tok, grp)
    return _C4_ORACLE[kind]


@pytest.mark.parametrize("prec,rtol", PRECISIONS)
@pytest.mark.parametrize("kind", ["uniform", "clustered", "duplicates"])
def test_c4_shape_pointnet_against_oracle(kind, prec, rtol):
    """BASELINE configs[3] at its real per-cloud shape (cluster FPS over 65536 points -> sweep kNN with k = 64 -> fused
    embed at E = 384): indices bit-exact, tokens in tolerance, all three cloud kinds (duplicates = exact distance ties)."""
    _skip_if_unbuilt(prec)
    x, st, sd, otok, grp = _c4_oracle(kind)
    G, k, E = 2048, 64, 384
    net = PointNet(E, G, k, 6, precision=prec).eval().to(dev())
    net.encoder.load_state_dict(synth.to_torch_state(sd), strict=True)
    xt, stt = to_dev(x), to_dev(st)
    fidx, ctr, kidx, perm = net.group.indices(xt, stt)
    assert np.array_equal(fidx.cpu().numpy(), grp["fps_idx"]), "FPS indices"
    assert np.array_equal(kidx.cpu().numpy(), grp["knn_idx"]), "kNN indices"
    assert np.array_equal(perm.cpu().numpy(), grp["perm"]), "Morton order"
    tok = net(xt, stt)
    assert tok.shape == (1, G, E)
    assert_tokens_close(tok.cpu().numpy(), otok, rtol, f"c4 shape ({kind}, {prec}) vs oracle")


@pytest.mark.parametrize("prec,rtol", PRECISIONS)
@pytest.mark.parametrize("kind", ["uniform", "clustered"])
def test_c3_shape_p3embed_against_oracle(kind, prec, rtol):
    """BASELINE configs[2] at its real per-cloud shape: P3Embed 2-stage 8192 -> 2048 -> 512, k = 32, widths 128 / 256
    (Z-order culled kNN at N = 8192, stage kernel, gathered stage-1 rows, fused pair), B = 2 clouds."""
    _skip_if_unbuilt(prec)
    B, N, k = 2, 8192, 32
    p = synth.make_cloud(kind, B, N, 3300 + len(kind), 3)
    starts = [synth.start_indices(B, N, 33, 0), synth.start_indices(B, N // 4, 33, 1)]
    sd = synth.p3embed_state(3, 1 / 16, 4, 4, 256, 33)
    mod = P3Embed(sample_ratio=1 / 16, k=k, embed_dim=256, precision=prec).eval().to(dev())
    mod.load_state_dict(synth.to_torch_state(sd), strict=True)
    pt = to_dev(p)
    ps, fs = mod(pt, pt.transpose(1, 2).contiguous(), [to_dev(s) for s in starts])
    op, of, aux = oracle.p3embed(sd, p, p.copy(), starts, k, 2)
    assert [tuple(f.shape) for f in fs[1:]] == [(B, 128, N // 4), (B, 256, N // 16)]
    for s in (1, 2):
        assert np.array_equal(ps[s].cpu().numpy(), op[s]), f"centres of stage {s - 1}"
        assert_tokens_close(fs[s].transpose(1, 2).cpu().numpy(), of[s], rtol * s, f"c3 shape ({kind}, {prec}) stage {s - 1} vs oracle")


def test_bf16_token_output_is_the_rounded_fp32_output():
    """token_dtype=torch.bfloat16 (bf16 path): the patch max is rounded once by the epilogue that produces it, so the
    result equals the float32 tokens rounded to bf16 - for the APF tokenizer (fused pair epilogue, k = 32 and k = 64
    partial-max reduction) and for the last P3Embed stage; the fp32 path refuses the option."""
    _skip_if_unbuilt("bf16")
    for (G, k) in ((64, 32), (32, 64)):
        x = to_dev(synth.make_cloud("uniform", 3, 1024, 61, 3))
        st = to_dev(synth.start_indices(3, 1024, 61))
        sd = synth.to_torch_state(synth.apf_encoder_state(384, 6, 61))
        nets = [PointNet(384, G, k, 6, precision="bf16", token_dtype=dt).eval().to(dev()) for dt in (None, torch.bfloat16)]
        for n in nets:
            n.encoder.load_state_dict(sd)
        t32, t16 = nets[0](x, st), nets[1](x, st)
        assert t16.dtype == torch.bfloat16 and t32.dtype == torch.float32
        assert torch.equal(t16, t32.bfloat16())
    p = to_dev(synth.make_cloud("uniform", 2, 1024, 62, 3))
    starts = [to_dev(synth.start_indices(2, 1024, 62, 0)), to_dev(synth.start_indices(2, 256, 62, 1))]
    sd = synth.to_torch_state(synth.p3embed_state(3, 1 / 16, 4, 4, 256, 62))
    outs = []
    for dt in (None, torch.bfloat16):
        m = P3Embed(sample_ratio=1 / 16, k=32, precision="bf16", token_dtype=dt).eval().to(dev())
        m.load_state_dict(sd)
        outs.append(m(p, p.transpose(1, 2).contiguous(), starts)[1])
    assert outs[1][1].dtype == torch.float32 and outs[1][2].dtype == torch.bfloat16     # only the last stage changes dtype
    assert torch.equal(outs[1][1], outs[0][1]) and torch.equal(outs[1][2], outs[0][2].bfloat16())
    with pytest.raises(ValueError):
        PointNet(64, 8, 8, 6, precision="fp32", token_dtype=torch.bfloat16).eval().to(dev())(x, st)


def test_fp32tc_rejects_widths_it_cannot_tile():
    """The bf16x3 mode has no fallback: widths that are not multiples of 64 raise instead of silently taking another path."""
    _skip_if_unbuilt("bf16")
    enc = Encoder(48, 6, precision="fp32tc").eval().to(dev())
    with pytest.raises(RuntimeError, match="multiples of 64"):
        enc(torch.zeros(1, 4, 32, 6, device=dev()))


def test_fp32tc_is_close_to_the_cuda_core_fp32_path_at_c2():
    """BASELINE configs[1] shapes: the tensor-core fp32-accurate mode against the CUDA-core fp32 mode on the same inputs
    (both are held to rtol 1e-4 against the oracle; against each other the difference is the split's ~7e-6)."""
    _skip_if_unbuilt("bf16")
    B, N, G, k, E = 16, 2048, 128, 32, 384
    x = to_dev(synth.make_cloud("uniform", B, N, 12, 3))
    st = to_dev(synth.start_indices(B, N, 12))
    sd = synth.to_torch_state(synth.apf_encoder_state(E, 6, 12))
    toks = []
    for prec in ("fp32", "fp32tc"):
        net = PointNet(E, G, k, 6, precision=prec).eval().to(dev())
        net.encoder.load_state_dict(sd)
        toks.append(net(x, st))
    err = float((toks[0] - toks[1]).abs().max() / toks[0].abs().max())
    print(f"[parity] fp32tc vs fp32 at c2 shapes: {err:.2e} of max")
    assert err < 5e-5, err
