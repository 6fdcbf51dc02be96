"""The fp32-accurate ViT block stacks: block_precision="fp32tc" (p3tok::apf_vit_x3 / p3tok::vit_blocks_x3, bf16x3 split
operands on the stack's own kernels) held to the fp32 contract, rtol 1e-4 (helpers.assert_tokens_close).

  1. host only: the x3 folds reconstruct the float64 folded matrices, their padding is zero, their shapes are the ones the
     ops validate;
  2. the split attention kernels alone against the float64 softmax, persistent form past one pass, and the persistent form
     equal to the general one bit for bit;
  3-5. the APF and Pix4Point stacks against the float64 oracle and the reference goldens, and both models end to end;
  6. serving properties: batch invariance at c2v, CUDA-graph replay, empty batch, errors.
Every stack comparison also prints the error of the fp32 autograd forward (train_vit, CUDA cores) on the same inputs.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import cases
from helpers import assert_tokens_close, dev, rel_err, to_dev
from oracle import oracle
from p3tok import fold, ops, synth
from p3tok.apf_model import (AdapterLayer, AdaptPointFormer, APFViTLayer, ClassificationHead, fold_vit_layer64,
                             fold_vit_layer_x3, run_blocks)
from p3tok.p4p_model import PointViT, TimmBlock, fold_timm_block64, fold_timm_block_x3

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "adapting-2d-vits-for-3d-point-cloud-understanding_b200"
RTOL = 1e-4
gpu = pytest.mark.gpu


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------ 1. the x3 folds (host only)
def _random_apf_layer(D, heads, R, seed):
    torch.manual_seed(seed)
    layer = APFViTLayer(D, heads)
    layer.adapter = AdapterLayer(D, R)
    with torch.no_grad():
        for p in layer.parameters():          # up_proj / biases start at zero: give every entry a value
            p.copy_(torch.randn_like(p) * 0.05)
        layer.adapter.scale.fill_(0.7)
    return layer.eval()


def _check_x3_fold(mats64, x3, D, R):
    HR = mats64[2][0].shape[0]
    HRp = fold.pad64(HR)
    want = ops.vit_layer_shapes(D, HRp, True)
    for name, t in zip(ops.VIT_LAYER_TENSORS, x3):
        assert tuple(t.shape) == want[name], (name, tuple(t.shape), want[name])
        assert t.dtype == (torch.bfloat16 if name.endswith("_w") else torch.float32), name
    for (w64, b64), w3, b3 in zip(mats64, x3[0::2], x3[1::2]):
        n, k = w64.shape
        kp = fold.pad64(k)
        hi, hi2, lo = w3[:, :kp].double(), w3[:, kp:2 * kp].double(), w3[:, 2 * kp:].double()
        assert torch.equal(hi, hi2)
        rec = hi[:n, :k] + lo[:n, :k]
        assert ((rec - w64).abs() <= 2.0 ** -16 * w64.abs()).all(), f"hi + lo off by {float(((rec - w64).abs() / w64.abs()).max()):.2e}"
        assert not hi[:, k:].any() and not lo[:, k:].any(), "padded columns must be zero"
        assert not hi[n:].any() and not lo[n:].any(), "padded rows must be zero"
        assert torch.equal(b3[:n].double(), b64.float().double()) and not b3[n:].any()
    H = HR - R
    assert x3[4].shape[0] == HRp and (HRp - R) // 64 * 64 == H     # the H the ops recover from the padded width


@pytest.mark.parametrize("R", [64, 8])
def test_x3_fold_apf_layer(R):
    D = 128
    layer = _random_apf_layer(D, 2, R, 5 + R)
    _check_x3_fold(fold_vit_layer64(layer), fold_vit_layer_x3(layer), D, R)


def test_x3_fold_timm_block():
    D = 192
    torch.manual_seed(3)
    blk = TimmBlock(D, 3).eval()
    with torch.no_grad():
        for p in blk.parameters():
            p.copy_(torch.randn_like(p) * 0.05)
    _check_x3_fold(fold_timm_block64(blk), fold_timm_block_x3(blk), D, 0)


def test_patch_mlp_x3_uses_the_split_helper():
    """PatchMLP.to_x3 and the ViT folds share fold.split_x3: [W_hi | W_hi | W_lo] of a float32 matrix, unchanged."""
    torch.manual_seed(1)
    w = torch.randn(96, 100)
    x3 = fold.split_x3(w)
    hi, kp = w.bfloat16(), 128
    assert tuple(x3.shape) == (96, 3 * kp) and x3.dtype == torch.bfloat16
    assert torch.equal(x3[:, :100], hi) and torch.equal(x3[:, kp:kp + 100], hi)
    assert torch.equal(x3[:, 2 * kp:2 * kp + 100], (w - hi.float()).bfloat16())
    m = fold.PatchMLP(cin=100, pre_dims=[96], pre_relu=[1], mid_dim=64, out_dim=64, out_relu=0, w_pre=[w], b_pre=[torch.zeros(96)],
                      w_mid_g=torch.randn(64, 96), w_mid_f=torch.randn(64, 96), b_mid=torch.zeros(64), w_out=torch.randn(64, 64),
                      b_out=torch.zeros(64))
    assert torch.equal(m.to_x3("cpu").w_pre[0], x3)


def test_block_precision_values():
    with pytest.raises(ValueError):
        AdaptPointFormer(num_classes=15, embedding_dim=64, npoint=32, nsample=16, block_precision="fp16")
    with pytest.raises(ValueError):
        PointViT(embed_dim=64, depth=1, num_heads=2, block_precision="fp16")
    with pytest.raises(ValueError):
        run_blocks([APFViTLayer(64, 2).eval()], torch.zeros(1, 4, 64), None, None, "fp32")


# ------------------------------------------------------------------ 2. the split attention kernels alone
def _split(t):
    hi = t.bfloat16()
    return hi, (t - hi.float()).bfloat16()


def _attn_inputs(B, G, heads, hd):
    g = torch.Generator().manual_seed(7919 * G + 31 * hd + heads)     # CPU generator: the same values in every process
    v = torch.randn(B * G, 3 * heads * hd, generator=g) * 1.5
    hi, lo = _split(v)
    return torch.cat([hi, lo], 1).to(dev()), (hi.double() + lo.double()).to(dev())


def _attention_ref(qkv, B, G, heads):
    D = qkv.shape[1] // 3
    hd = D // heads
    t = qkv.reshape(B, G, 3, heads, hd).permute(2, 0, 3, 1, 4)
    att = ((t[0] @ t[1].transpose(-2, -1)) * hd ** -0.5).softmax(-1)
    return (att @ t[2]).transpose(1, 2).reshape(B * G, D)


def _merge(out):
    D = out.shape[1] // 2
    return out[:, :D].double() + out[:, D:].double()


ATTN_G = [1, 2, 63, 64, 65, 127, 128, 129, 197, 513]
ATTN_CASES = [(G, hd) for hd in (32, 64) for G in ATTN_G]
HEADS = 4


def _attn_batch(G):
    """G <= 128 (persistent form, one CTA per SM in x3): at least 2.5 passes over the (cloud, head) items."""
    if G <= 128:
        return cdiv(5 * torch.cuda.get_device_properties(dev()).multi_processor_count, 2 * HEADS) + 1
    return 3


def _run_attention_cases(path):
    """Entry point of the P3TOK_ATTN_SMALL=0 subprocess: the persistent cases through the general kernel."""
    out = {}
    for G, hd in ATTN_CASES:
        if G <= 128:
            B = _attn_batch(G)
            out[f"{G}-{hd}"] = ops.attention_x3(_attn_inputs(B, G, HEADS, hd)[0], B, G, HEADS).cpu()
    torch.save(out, path)


_SUBPROCESS = ("import os, sys; r = os.getcwd(); sys.path[:0] = [r, os.path.join(r, %r), os.path.join(r, 'tests'), os.path.join(r, 'tests', 'golden')];"
               "import test_gpu_vit_x3 as t; t._run_attention_cases(sys.argv[1])" % PKG)


@pytest.fixture(scope="module")
def attention_general_form(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("attn_x3") / "general.pt")
    env = dict(os.environ, P3TOK_ATTN_SMALL="0")
    subprocess.run([sys.executable, "-c", _SUBPROCESS, path], check=True, env=env, cwd=ROOT, timeout=1200)
    return torch.load(path)


@gpu
@pytest.mark.parametrize("G,hd", ATTN_CASES, ids=lambda v: str(v))
def test_attention_x3(G, hd, attention_general_form):
    B = _attn_batch(G)
    qkv, exact = _attn_inputs(B, G, HEADS, hd)
    got = ops.attention_x3(qkv, B, G, HEADS)
    assert tuple(got.shape) == (B * G, 2 * HEADS * hd)
    ref = _attention_ref(exact, B, G, HEADS)
    assert_tokens_close(_merge(got).cpu().numpy(), ref.cpu().numpy(), RTOL, f"attention x3 G={G} hd={hd} B={B}")
    bf16 = ops.attention_bf16(qkv[:, :3 * HEADS * hd].contiguous(), B, G, HEADS)
    print(f"[attention] G={G} hd={hd}: bf16 kernel on the hi half max|err|/max|ref| {rel_err(bf16.float().cpu().numpy(), ref.cpu().numpy()):.2e}")
    if G <= 128:
        items, slots = B * HEADS, torch.cuda.get_device_properties(dev()).multi_processor_count
        assert items > 2 * slots, (items, slots)           # the persistent form walks more than two passes
        other = attention_general_form[f"{G}-{hd}"]
        assert torch.equal(got.cpu(), other), f"G={G} hd={hd}: the persistent and the general x3 kernels differ"


@gpu
def test_layernorm_split():
    torch.manual_seed(4)
    x = torch.randn(1000, 768, device=dev()) * 3 + 1
    out = ops.layernorm_split(x, None, None, 1e-5)
    ref = torch.nn.functional.layer_norm(x.double(), (768,), None, None, 1e-5)
    assert torch.equal(out[:, :768], ops.layernorm_bf16(x, None, None, 1e-5))   # hi is the bf16 stack's operand
    assert_tokens_close(_merge(out).cpu().numpy(), ref.cpu().numpy(), 1e-5, "layernorm split")


# ------------------------------------------------------------------ 3. the APF stack
def _apf_stack(D, heads, depth, sd, R=64):
    blocks = torch.nn.Sequential(*[APFViTLayer(D, heads) for _ in range(depth)])
    if R != 64:
        for blk in blocks:
            blk.adapter = AdapterLayer(D, R)
    blocks = blocks.eval().to(dev())
    norm = torch.nn.LayerNorm(D).eval().to(dev())
    head = ClassificationHead(D, 15).eval().to(dev())
    tsd = synth.to_torch_state(sd)
    for mod, prefix in ((blocks, "blocks."), (norm, "encoder_norm."), (head, "head.")):
        mod.load_state_dict({k[len(prefix):]: v for k, v in tsd.items() if k.startswith(prefix)}, strict=True)
    return blocks, norm, head


def _autograd_forward(blocks, tok, norm):
    """The fp32 autograd forward (train_vit, CUDA cores) on the same eval-mode stack: the input asks for a gradient."""
    t = tok.clone().requires_grad_(True)
    with torch.enable_grad():
        x, pooled = run_blocks(blocks, t, norm)
    return x.detach(), pooled.detach()


def _check_apf(c, sd, tok, what, golden=None, R=64):
    blocks, norm, head = _apf_stack(c["D"], c["heads"], c["depth"], sd, R)
    tokd = to_dev(tok)
    with torch.no_grad():
        x, pooled = run_blocks(blocks, tokd, norm, None, "fp32tc")
        logits = head(pooled)
    ax, ap = _autograd_forward(blocks, tokd, norm)
    with torch.no_grad():
        al = head(ap)
    ox, op, ol = oracle.apf_vit(sd, tok, c["depth"], c["heads"])
    for got, aut, orc, key in ((x, ax, ox, "x"), (pooled, ap, op, "pooled"), (logits, al, ol, "logits")):
        print(f"[{what}] {key}: fp32 autograd forward max|err|/max|ref| {rel_err(aut.cpu().numpy(), orc):.2e}")
        assert_tokens_close(got.cpu().numpy(), orc, RTOL, f"{what}:{key} x3 vs oracle")
        if golden is not None:
            assert_tokens_close(got.cpu().numpy(), golden[key], RTOL, f"{what}:{key} x3 vs reference golden")
    return x, pooled


@gpu
@pytest.mark.parametrize("name", list(cases.VIT_CASES))
def test_apf_x3_golden(golden_dir, name):
    c = cases.VIT_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    sd = synth.apf_vit_state(c["D"], c["depth"], c["classes"], c["seed"])
    _check_apf(c, sd, synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"]), name, g)


@gpu
def test_apf_x3_vit_b_width():
    """D = 768, G = 196: qkv (2304) and fc1d (3136) are column slices of the split outputs; the general attention kernel."""
    c = dict(B=2, G=196, D=768, heads=12, depth=2, seed=61)
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
    _check_apf(c, sd, synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"]), "vit-b")


@gpu
@pytest.mark.parametrize("G", [1, 2, 63, 64, 65, 127, 129])
def test_apf_x3_sequence_lengths(G):
    c = dict(B=2, G=G, D=64, heads=2, depth=2, seed=70 + G)
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
    _check_apf(c, sd, synth.vit_tokens(c["B"], G, c["D"], c["seed"]), f"G={G}")


@gpu
def test_apf_x3_bottleneck_8():
    """R = 8: H + R = 520 is padded to 576 fc1d rows / fc2u columns."""
    c = dict(B=2, G=50, D=128, heads=2, depth=2, seed=88)
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"], bottleneck=8)
    _check_apf(c, sd, synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"]), "R=8", R=8)


# ------------------------------------------------------------------ 4. the Pix4Point stack
@gpu
@pytest.mark.parametrize("name", list(cases.P4P_VIT_CASES))
def test_pointvit_x3_golden(golden_dir, name):
    import make_golden
    c = cases.P4P_VIT_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    feats, pos, sd = make_golden.p4p_vit_inputs(c)
    tsd = synth.to_torch_state(sd)
    blocks = torch.nn.ModuleList([TimmBlock(c["D"], c["heads"]) for _ in range(c["depth"])]).eval().to(dev())
    blocks.load_state_dict({k[len("vit.blocks."):]: v for k, v in tsd.items() if k.startswith("vit.blocks.")}, strict=True)
    norm = torch.nn.LayerNorm(c["D"], eps=1e-6).eval().to(dev())
    norm.load_state_dict({k[len("vit.norm."):]: v for k, v in tsd.items() if k.startswith("vit.norm.")}, strict=True)
    params = [t for blk in blocks for t in fold_timm_block_x3(blk)]
    out, pooled = ops.vit_blocks_x3(to_dev(feats), to_dev(pos), params, c["heads"], norm.weight.detach(), norm.bias.detach(), 1e-6, 1)
    ox, og = oracle.pointvit_blocks(sd, feats, pos, c["depth"], c["heads"])
    from p3tok import train_vit
    f = to_dev(feats).requires_grad_(True)
    with torch.enable_grad():
        aout = train_vit.timm_blocks_train(blocks, norm, f, to_dev(pos)).detach()
    print(f"[{name}] fp32 autograd forward normed feats max|err|/max|ref| {rel_err(aout.cpu().numpy(), ox):.2e}")
    D = c["D"]
    assert_tokens_close(out.cpu().numpy(), ox, RTOL, f"{name} x3 normed feats vs oracle")
    assert_tokens_close(out.cpu().numpy(), g["feats"], RTOL, f"{name} x3 normed feats vs golden")
    assert_tokens_close(pooled.cpu().numpy(), og[:, :D], RTOL, f"{name} x3 token max vs oracle")
    assert_tokens_close(torch.cat([pooled, out[:, 0]], 1).cpu().numpy(), g["glob"], RTOL, f"{name} x3 'max,cls' vs golden")


# ------------------------------------------------------------------ 5. end to end
def _check_argmax(logits, ref):
    top2 = np.sort(ref, 1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 1e-3 * np.abs(ref).max()
    assert clear.any()
    assert np.array_equal(logits.argmax(1)[clear], ref.argmax(1)[clear])


@gpu
def test_adaptpointformer_x3_end_to_end():
    B, N, G, k, E = 3, 512, 32, 16, 64
    x = synth.make_cloud("clustered", B, N, 71, 3)
    start = synth.start_indices(B, N, 71)
    sd_enc = synth.apf_encoder_state(E, 6, 71)
    sd_vit = synth.apf_vit_state(E, 12, 15, 71)
    tok64, _ = oracle.pointnet_apf(sd_enc, x, start, G, k)
    _, op, ol = oracle.apf_vit(sd_vit, tok64, 12, 2)
    m = AdaptPointFormer(num_classes=15, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="fp32tc",
                         block_precision="fp32tc")
    for blk in m.blocks:
        blk.attention.num_heads = 2
    state = {"point_encoder.encoder." + k_: v for k_, v in synth.to_torch_state(sd_enc).items()}
    state.update(synth.to_torch_state(sd_vit))
    m.load_state_dict(state, strict=True)
    m = m.eval().to(dev())
    with torch.no_grad():
        feats = m.features(to_dev(x), to_dev(start))
        logits = m(to_dev(x), to_dev(start))
    assert_tokens_close(feats.cpu().numpy(), op, RTOL, "APF x3 pooled features")
    assert_tokens_close(logits.cpu().numpy(), ol, RTOL, "APF x3 logits")
    _check_argmax(logits.cpu().numpy(), ol)


@gpu
def test_pointvit_x3_end_to_end():
    B, N, k, E = 2, 1024, 32, 384
    m = PointViT(embed_dim=E, k_neighbors=k, sample_ratio=1 / 16, precision="fp32", block_precision="fp32tc").eval().to(dev())
    sd_p = synth.p3embed_state(3, 1 / 16, 4, 4, 256, 7)
    sd_h = synth.token_head_state(256, E, 7)
    sd_v = synth.pointvit_state(E, 12, 7)
    m.patch_embed.load_state_dict(synth.to_torch_state(sd_p), strict=True)
    miss = m.load_state_dict({**synth.to_torch_state(sd_h), **synth.to_torch_state(sd_v)}, strict=False)
    assert not miss.unexpected_keys
    p = synth.make_cloud("uniform", B, N, 7, 3)
    starts = [synth.start_indices(B, N, 7, 0), synth.start_indices(B, N // 4, 7, 1)]
    with torch.no_grad():
        glob = m.forward_cls_feat(to_dev(p), None, [to_dev(s) for s in starts])
    op, of, _ = oracle.p3embed(sd_p, p, p.copy(), starts, k, 2)
    hf, hp = oracle.token_head(sd_h, of[-1].astype(np.float32), op[-1])
    _, og = oracle.pointvit_blocks(sd_v, hf, hp, 12, 6)
    assert_tokens_close(glob.cpu().numpy(), og, RTOL, "PointViT x3 'max,cls' vs oracle")


# ------------------------------------------------------------------ 6. serving properties
C2V = dict(D=384, heads=12, depth=12, B=128, G=128, seed=0, tok_seed=128)


@pytest.fixture(scope="module")
def c2v():
    c = C2V
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
    blocks, norm, _ = _apf_stack(c["D"], c["heads"], c["depth"], sd)
    tok = to_dev(synth.vit_tokens(c["B"], c["G"], c["D"], c["tok_seed"]))
    cache = {}
    fn = lambda t: run_blocks(blocks, t, norm, cache, "fp32tc")     # noqa: E731
    with torch.no_grad():
        return fn, tok, fn(tok)


@gpu
def test_x3_batch_invariance_c2v(c2v):
    fn, tok, (x, pooled) = c2v
    with torch.no_grad():
        for i in range(0, tok.shape[0], 4):
            px, pp = fn(tok[i:i + 4])
            assert torch.equal(px, x[i:i + 4]) and torch.equal(pp, pooled[i:i + 4]), f"clouds {i}..{i + 3} differ between B = 128 and 4"
        ax, ap = fn(tok)
    assert torch.equal(ax, x) and torch.equal(ap, pooled), "two identical runs differ"


@gpu
def test_x3_cuda_graph_replay(c2v):
    fn, tok, (x, pooled) = c2v
    static = tok.clone()
    with torch.no_grad():
        s = torch.cuda.Stream(device=dev())
        s.wait_stream(torch.cuda.current_stream(dev()))
        with torch.cuda.stream(s):
            fn(static)                                      # warm-up: fold cache filled, kernels configured
        torch.cuda.current_stream(dev()).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            gx, gp = fn(static)
        static.copy_(tok * 0.5)                             # replay on other data first, then on the original tokens
        g.replay()
        torch.cuda.synchronize()
        hx, hp = fn(tok * 0.5)
        assert torch.equal(gx, hx) and torch.equal(gp, hp)
        static.copy_(tok)
        g.replay()
        torch.cuda.synchronize()
    assert torch.equal(gx, x) and torch.equal(gp, pooled), "graph replay differs from the eager result"


@gpu
def test_x3_empty_batch_and_errors():
    sd = synth.apf_vit_state(64, 1, 15, 69)
    blocks, norm, _ = _apf_stack(64, 2, 1, sd)
    with torch.no_grad():
        x, pooled = run_blocks(blocks, torch.zeros(0, 4, 64, device=dev()), norm, None, "fp32tc")
    assert tuple(x.shape) == (0, 4, 64) and tuple(pooled.shape) == (0, 64)
    blk = APFViTLayer(192, 2).eval().to(dev())             # head dim 96
    with torch.no_grad(), pytest.raises(RuntimeError, match="head dim"):
        run_blocks([blk], torch.zeros(1, 4, 192, device=dev()), None, None, "fp32tc")
    with torch.no_grad(), pytest.raises(RuntimeError):     # CPU tensors: no fallback
        run_blocks([APFViTLayer(64, 2).eval()], torch.zeros(1, 4, 64), None, None, "fp32tc")
    with pytest.raises(RuntimeError):
        ops.attention_x3(torch.zeros(8, 384, dtype=torch.bfloat16), 2, 4, 2)
    qkv = torch.zeros(8, 6 * 96, dtype=torch.bfloat16, device=dev())
    with pytest.raises(RuntimeError, match="head dim"):
        ops.attention_x3(qkv, 2, 4, 1)
