"""CPU-only checks of the host side: C-ABI library loads and exports what include/p3tok.h declares,
struct layouts, weight folding algebra, module state_dict compatibility, error behaviour."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from helpers import folded_forward
from oracle import oracle, ref_loader
from p3tok import _build, _lib, fold, synth
from p3tok.modules import Encoder, Group, P3Embed, PointNet


@pytest.fixture(scope="module")
def built():
    return _build.build_library()


def test_library_exports_every_declared_symbol(built):
    L = ctypes.CDLL(built)
    names = _lib.declared_symbols()
    assert len(names) >= 12
    for n in names:
        assert hasattr(L, n), n
    assert sorted(_lib._SIGNATURES) == names      # the Python binding covers the whole header
    L.p3tok_abi_version.restype = ctypes.c_int
    assert L.p3tok_abi_version() == 2             # host-only call, no GPU needed


def test_host_only_size_queries(built):
    """Size queries are host computations (no GPU): the sorted-kNN scratch follows the segment layout of csrc/knn.cu -
    21 bytes per point plus per-segment tables, segments of at most 8192 points, nothing beyond 131072 points."""
    L = ctypes.CDLL(built)
    L.p3tok_knn_workspace_bytes.restype = ctypes.c_int64
    L.p3tok_knn_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64]
    ws = L.p3tok_knn_workspace_bytes
    assert ws(0, 1024) > 0 and ws(4, 0) == 0 and ws(-1, 8) == 0
    one, two = ws(1, 8192), ws(1, 8193)
    assert 8192 * 21 <= one <= 8192 * 21 + 4096             # pts 16 B + ids 4 B + boxes 1 B per point, cell table, meta
    assert two > one and two - one < 2 * (32 * 21) + 4096    # a second segment: two more padded blocks and a second table
    assert ws(16, 65536) >= 16 * 65536 * 21 and ws(1, 131072) > 0 and ws(1, 131073) == 0
    assert ws(7, 20011) - ws(6, 20011) == ws(3, 20011) - ws(2, 20011)   # linear in the number of clouds


def test_patch_embed_workspace_is_bounded_by_one_chunk(built):
    """The patch embedding is chunked so any B fits (DESIGN.md §3): p3tok_patch_embed_workspace_bytes (a host computation)
    never exceeds the workspace of one full chunk, whatever the number of groups.  bf16 / fp32tc chunks hold at most
    cg_max = ceil8(rows_target / k) groups: chunks are sized equally and rounded up to 8 groups, so the size dips and rises
    with n and its maximum is reached at n = 2 * (rows_target // k) (two chunks of cg_max groups); fp32 chunks hold 8192.
    The Python mirror of the policy (tests/test_gpu_chunking.py, which picks the sentinel clouds of the GPU tests) must
    predict the size: ws(n) == ws(mirror(n)) where mirror(n) is one chunk."""
    import random
    from test_gpu_chunking import F32_CHUNK_GROUPS, chunk_size, chunk_wmax, rows_target
    if os.environ.get("P3TOK_CHUNK_ROWS"):
        pytest.skip("P3TOK_CHUNK_ROWS overrides the default chunk policy")
    L = _lib.lib()

    def mlp(meta):
        m = _lib.MlpStruct()
        n = meta[1]
        m.cin, m.n_pre = meta[0], n
        for i in range(n):
            m.pre_dim[i], m.pre_relu[i] = meta[2 + i], meta[2 + n + i]
        m.mid_dim, m.out_dim, m.out_relu = meta[2 + 2 * n:5 + 2 * n]
        return m

    layouts = {"APF E=384": [6, 3, 256, 512, 384, 1, 1, 0, 768, 384, 0],
               "P3Embed stage 0": [6, 1, 128, 1, 256, 128, 1], "P3Embed stage 1": [131, 1, 256, 1, 512, 256, 1]}
    precs = {"bf16": _lib.BF16, "fp32tc": _lib.BF16X3, "fp32": _lib.F32}
    rnd = random.Random(2026)
    full_sizes = {}
    for lname, meta in layouts.items():
        m = mlp(meta)
        for pname, prec in precs.items():
            for k in (1, 5, 24, 32, 64, 128):
                ws = lambda n: int(L.p3tok_patch_embed_workspace_bytes(ctypes.byref(m), n, k, prec))
                if pname == "fp32":
                    cg0 = cg_max = F32_CHUNK_GROUPS
                else:
                    cg0 = rows_target(chunk_wmax(meta, pname)) // k
                    cg_max = (cg0 + 7) // 8 * 8
                what = f"{lname} {pname} k={k}"
                n_full = cg0 if pname == "fp32" else 2 * cg0
                assert chunk_size(n_full, k, meta, pname) == cg_max, what
                full = ws(n_full)
                full_sizes[(lname, pname, k)] = full
                assert ws(cg0) <= full and ws(1) <= full, what
                # around every change of the chunk count (n = c * cg0 + d) and at random n up to 2^26 groups
                ns = [c * cg0 + d for c in range(1, 64) for d in range(-9, 10)] + [rnd.randint(1, 1 << 26) for _ in range(300)]
                worst = max(ws(n) for n in ns if 0 < n <= 1 << 26)
                assert worst == full, (what, worst, full)          # never above one full chunk, and reached
                if pname == "fp32":
                    assert ws(1 << 26) == full and ws(F32_CHUNK_GROUPS + 1) == full, what
                elif k in (32, 64):                   # rows_target / k is a multiple of 8: mirror(n) is itself one chunk
                    for n in ns[-200:]:
                        assert ws(n) == ws(chunk_size(n, k, meta, pname)), f"{what}: n={n}"
    gb = lambda key: full_sizes[key] / 1e9
    assert 3.3 < gb(("APF E=384", "bf16", 32)) < 3.5 and 8.8 < gb(("APF E=384", "bf16", 1)) < 9.0
    assert 8.2 < gb(("APF E=384", "fp32tc", 32)) < 8.4 and 1.6 < gb(("APF E=384", "fp32", 32)) < 1.7
    assert max(full_sizes.values()) < 16e9                  # fits beside the model on one 180 GB device, any B


def test_apf_fold_moves_the_feature_bias_into_the_concat_layer():
    """fold_apf_encoder (p3tok/fold.py): first_conv.6's bias is folded through the max and the concat into second_conv.0 -
    the folded feature layer carries a zero bias and the folded network still equals the oracle (checked above); here: the
    moved term is exactly (Wm_g + Wm_f) b3."""
    sd = synth.to_torch_state(synth.apf_encoder_state(64, 6, 3))
    m = fold.fold_apf_encoder(sd)
    assert float(m.b_pre[2].abs().max()) == 0.0
    sd0 = {k: v.clone() for k, v in sd.items()}
    sd0["first_conv.6.bias"] = torch.zeros_like(sd0["first_conv.6.bias"])
    m0 = fold.fold_apf_encoder(sd0)
    b3 = sd["first_conv.6.bias"].double()
    moved = (m0.w_mid_g.double() + m0.w_mid_f.double()) @ b3
    assert torch.allclose(m.b_mid.double() - m0.b_mid.double(), moved, rtol=1e-5, atol=1e-6)


def test_struct_layouts_match_header(tmp_path, built):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "p3tok.h"\nint main(){printf("%zu %zu %zu %zu\\n",'
                   'sizeof(p3tok_mlp),sizeof(p3tok_rows),offsetof(p3tok_mlp,w_pre),offsetof(p3tok_rows,x));'
                   'printf("%zu %zu %zu\\n",sizeof(p3tok_vit_layer),offsetof(p3tok_vit_layer,fc1d_w),'
                   'offsetof(p3tok_vit_layer,fc2u_b));return 0;}')
    exe = tmp_path / "sz"
    inc = os.path.join(os.path.dirname(_lib.HEADER_PATH))
    subprocess.run(["gcc", "-I", inc, str(src), "-o", str(exe)], check=True)
    a, b, c, d, e, f, g = (int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split())
    assert ctypes.sizeof(_lib.MlpStruct) == a and ctypes.sizeof(_lib.RowsStruct) == b
    assert _lib.MlpStruct.w_pre.offset == c and _lib.RowsStruct.x.offset == d
    assert ctypes.sizeof(_lib.VitLayerStruct) == e and _lib.VitLayerStruct.fc1d_w.offset == f
    assert _lib.VitLayerStruct.fc2u_b.offset == g


def test_fold_apf_matches_oracle():
    sd = synth.apf_encoder_state(40, 6, 3)
    x = synth.make_cloud("uniform", 2, 96, 3)
    grp = oracle.group_apf(x, np.zeros(2, np.int64), 6, 8)
    ref = oracle.apf_encoder(sd, grp["neigh"])
    m = fold.fold_apf_encoder(synth.to_torch_state(sd))
    got = folded_forward(m, torch.from_numpy(grp["neigh"]).reshape(-1, 6), 8).numpy().reshape(ref.shape)
    assert np.abs(got - ref).max() <= 2e-6 * np.abs(ref).max()   # fp32-rounded folded weights
    assert m.meta() == [6, 3, 256, 512, 40, 1, 1, 0, 80, 40, 0]


def test_fold_p3embed_matches_oracle():
    sd = synth.p3embed_state(3, 1 / 16, 4, 4, 64, 4)
    pts = synth.make_cloud("uniform", 2, 128, 4)
    ctr, ref, fidx, kidx = oracle.p3embed_stage(sd, 0, pts, pts, np.zeros(2, np.int64), 8)
    m = fold.fold_p3embed_stage(synth.to_torch_state(sd), 0)
    rows = np.concatenate([oracle.gather_points(pts, kidx), oracle.gather_points(pts, kidx)], -1).reshape(-1, 6)
    got = folded_forward(m, torch.from_numpy(rows), 8).numpy().reshape(ref.shape)
    assert np.abs(got - ref).max() <= 2e-6 * np.abs(ref).max()
    assert m.out_relu == 1 and m.pre_dims == [32]


def test_state_dict_keys_match_reference_layout():
    keys = set(PointNet(64, 8, 4, 6).state_dict())
    assert keys == {"encoder." + k for k in synth.apf_encoder_state(64, 6)}
    assert set(P3Embed(sample_ratio=1 / 16, embed_dim=64).state_dict()) == set(synth.p3embed_state(3, 1 / 16, 4, 4, 64))
    e = P3Embed()
    assert e.out_channels == 256 and e.channel_list == [3, 256] and len(e.convs) == 1
    e2 = P3Embed(sample_ratio=1 / 16)
    assert e2.channel_list == [3, 128, 256]


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_state_dict_loads_from_reference_modules():
    ref = ref_loader.load()
    r = ref.PointNet(48, 8, 4, 8)
    mine = PointNet(48, 8, 4, 8)
    mine.load_state_dict(r.state_dict(), strict=True)
    r2 = ref.P3Embed(sample_ratio=1 / 16, k=8, embed_dim=128)
    mine2 = P3Embed(sample_ratio=1 / 16, k=8, embed_dim=128)
    mine2.load_state_dict(r2.state_dict(), strict=True)
    assert mine2.out_channels == r2.out_channels and mine2.channel_list == r2.channel_list


def test_state_dicts_have_the_layouts_the_reference_modules_accepted():
    """tests/golden/make_golden.py loaded these synthetic state dicts into the reference's own modules with strict=True
    (apf_height: PointNet encoder E=48 on 8 channels; p4p_2stage / p4p_2stage_k32: P3Embed 1/16 with E=64 / 256;
    vit_small: APFViTLayer(64, 2) and ClassificationHead(64, 15)), so their key -> shape maps are the reference's.
    The modules here must have exactly those maps and load them strictly."""
    from p3tok.apf_model import APFViTLayer, ClassificationHead

    def same_layout(module, sd):
        shapes = lambda d: {k: tuple(v.shape) or (1,) for k, v in d.items()}     # num_batches_tracked: () here, (1,) stored
        assert shapes(module.state_dict()) == shapes(sd)
        module.load_state_dict(sd, strict=True)

    same_layout(PointNet(48, 24, 16, 8).encoder, synth.to_torch_state(synth.apf_encoder_state(48, 8, 12)))
    for E in (64, 256):
        same_layout(P3Embed(sample_ratio=1 / 16, k=8, embed_dim=E), synth.to_torch_state(synth.p3embed_state(3, 1 / 16, 4, 4, E, 21)))
    vit = synth.to_torch_state(synth.apf_vit_state(64, 2, 15, 51))
    for p, m in (("blocks.0.", APFViTLayer(64, 2)), ("blocks.1.", APFViTLayer(64, 2)), ("head.", ClassificationHead(64, 15))):
        same_layout(m, {k[len(p):]: v for k, v in vit.items() if k.startswith(p)})


def test_no_cpu_fallback():
    from p3tok import functional as F
    x = torch.zeros(1, 16, 3)
    with pytest.raises((NotImplementedError, RuntimeError)):
        F.furthest_point_sample(x, 4, torch.zeros(1, dtype=torch.long))
    with pytest.raises((NotImplementedError, RuntimeError)):
        F.knn_point(4, x, x[:, :2])
    with pytest.raises((NotImplementedError, RuntimeError)):
        PointNet(32, 4, 4, 6).eval()(x)


def test_train_mode_has_no_cpu_fallback_either():
    with pytest.raises(RuntimeError, match="CUDA"):          # train mode runs csrc/train.cu: CPU tensors are refused, not emulated
        Encoder(32, 6).train()(torch.zeros(1, 2, 4, 6))
    with pytest.raises(ValueError):
        Encoder(32, 6, precision="fp16").eval()(torch.zeros(1, 2, 4, 6))


def test_product_never_imports_oracle():
    pkg = os.path.dirname(_lib.__file__)
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            src = open(os.path.join(pkg, f)).read()
            assert "oracle" not in src.replace("# oracle", ""), f


def test_apf_model_state_dict_keys():
    """AdaptPointFormer drop-in: parameter names of the reference (src/models/apf.py:296-317, apf_utils.py:236-266)."""
    from p3tok.apf_model import AdaptPointFormer
    m = AdaptPointFormer(num_classes=15, embedding_dim=64, npoint=8, nsample=4, in_channels=3)
    keys = set(m.state_dict())
    want = set(synth.apf_vit_state(64, 12, 15)) | {"point_encoder.encoder." + k for k in synth.apf_encoder_state(64, 6)}
    assert keys == want, (sorted(keys - want)[:5], sorted(want - keys)[:5])
    m.load_state_dict(synth.to_torch_state(synth.apf_vit_state(64, 12, 15)), strict=False)
    with pytest.raises(RuntimeError):
        m.train()(torch.zeros(1, 16, 3))
    with pytest.raises(RuntimeError):
        AdaptPointFormer(pretrained=True)


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_apf_model_keys_match_reference_modules():
    from p3tok.apf_model import APFViTLayer, ClassificationHead
    ref = ref_loader.load()
    assert set(APFViTLayer(64, 2).state_dict()) == set(ref.apf_utils.APFViTLayer(dim=64, num_heads=2).state_dict())
    assert set(ClassificationHead(64, 15).state_dict()) == set(ref.apf.ClassificationHead(64, 15).state_dict())
    sd = ref.apf_utils.APFViTLayer(dim=64, num_heads=2).state_dict()
    APFViTLayer(64, 2).load_state_dict(sd, strict=True)


def test_fold_vit_layer_matches_oracle():
    """The four folded GEMMs of a layer (p3tok.apf_model.fold_vit_layer) evaluated in float64 equal the oracle's layer."""
    from p3tok.apf_model import APFViTLayer, fold_vit_layer
    D, heads, R = 64, 2, 64
    sd = synth.apf_vit_state(D, 1, 15, 9)
    blk = APFViTLayer(D, heads).eval()
    blk.load_state_dict({k[len("blocks.0."):]: v for k, v in synth.to_torch_state(sd).items() if k.startswith("blocks.0.")})
    x = torch.from_numpy(synth.vit_tokens(2, 10, D, 9)).double()
    ref = oracle.apf_vit_layer(sd, "blocks.0.", x.numpy(), heads)
    qw, qb, pw, pb, f1w, f1b, f2w, f2b = [t.double() for t in fold_vit_layer(blk)]
    ln = lambda t: torch.nn.functional.layer_norm(t, (D,), None, None, 1e-5)
    qkv = (ln(x) @ qw.T + qb).reshape(2, 10, 3, heads, D // heads).permute(2, 0, 3, 1, 4)
    att = ((qkv[0] @ qkv[1].transpose(-2, -1)) * (D // heads) ** -0.5).softmax(-1)
    x = x + ((att @ qkv[2]).transpose(1, 2).reshape(2, 10, D) @ pw.T + pb)
    h = ln(x) @ f1w.T + f1b
    h = torch.cat([torch.nn.functional.gelu(h[..., :-R]), torch.relu(h[..., -R:])], -1)
    got = 2 * x + (h @ f2w.T + f2b)
    assert np.abs(got.numpy() - ref).max() <= 1e-2 * np.abs(ref).max()      # bf16-rounded folded weights
    assert np.linalg.norm(got.numpy() - ref) <= 5e-3 * np.linalg.norm(ref)


def test_fold_uses_the_modules_bn_eps():
    """ADVICE r1: BatchNorm eps comes from the module, not a constant (a checkpoint built with eps = 1e-3 must fold with it)."""
    from p3tok.modules import _bn_eps
    enc = Encoder(32, 6).eval()
    enc.load_state_dict(synth.to_torch_state(synth.apf_encoder_state(32, 6, 4)))
    for m in enc.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.eps = 1e-3
    eps = _bn_eps(enc)
    assert set(eps) == {"first_conv.1", "first_conv.4", "second_conv.1"} and set(eps.values()) == {1e-3}
    rows = torch.randn(4 * 8, 6)
    with torch.no_grad():                     # the container modules ARE the reference arithmetic (same nn layers)
        f = enc.first_conv(rows.view(4, 8, 6).transpose(1, 2))
        g = f.max(2, keepdim=True)[0]
        ref = enc.second_conv(torch.cat([g.expand(-1, -1, 8), f], 1)).max(2)[0]
    got = folded_forward(fold.fold_apf_encoder(enc.state_dict(), eps), rows, 8)
    assert float((got - ref.double()).abs().max()) <= 1e-5 * float(ref.abs().max())
    wrong = folded_forward(fold.fold_apf_encoder(enc.state_dict()), rows, 8)       # default 1e-5: measurably different
    assert float((wrong - ref.double()).abs().max()) > 1e-4 * float(ref.abs().max())


def test_start_index_draws_mirror_the_reference():
    """furthest_point_sample draws on the global CPU generator (sampler.py:20); an explicit start_idx is used as is."""
    from p3tok.functional import _start
    x = torch.zeros(5, 100, 3)
    torch.manual_seed(123)
    a = _start(x, None)
    torch.manual_seed(123)
    b = torch.randint(0, 100, (5,), dtype=torch.long)
    assert torch.equal(a, b)
    assert torch.equal(_start(x, torch.tensor([1, 2, 3, 4, 5], dtype=torch.int32)), torch.tensor([1, 2, 3, 4, 5]))


def test_fps_kernel_sass_has_no_fused_multiply_add(built):
    """Regression (round 2): ptxas contracted the packed distance arithmetic of fps_kernel into FFMA2, so ~19 % of the
    squared distances differed from ((dx*dx)+(dy*dy))+(dz*dz) in the last bit and FPS picks flipped on near-ties."""
    import __graft_entry__ as entry
    assert entry.fps_fused_multiply_adds(built) == 0


def test_general_d_fps_and_square_distance_validate_on_the_host(built):
    """p3tok_fps_nd / p3tok_square_distance: argument validation and the empty cases return before any CUDA call, so the
    error behaviour of the C ABI is checkable without a GPU (status codes of include/p3tok.h, text from p3tok_last_error)."""
    L = _lib.lib()
    assert L.p3tok_fps_nd(None, 0, 16, 5, 5, None, 4, None, None, None) == _lib.OK            # no clouds: nothing to do
    assert L.p3tok_fps_nd(None, 2, 16, 5, 5, None, 0, None, None, None) == _lib.OK            # no samples asked for
    assert L.p3tok_fps_nd(None, 2, 16, 17, 17, None, 4, None, None, None) == _lib.ERR_UNSUPPORTED
    assert b"D=17" in L.p3tok_last_error()
    assert L.p3tok_fps_nd(None, 2, 16, 5, 4, None, 4, None, None, None) == _lib.ERR_INVALID   # rows shorter than D
    assert L.p3tok_fps_nd(None, 2, 0, 5, 5, None, 4, None, None, None) == _lib.ERR_INVALID    # empty clouds cannot be sampled
    assert L.p3tok_fps_nd(None, 2, 16, 5, 5, None, 4, None, None, None) == _lib.ERR_INVALID   # null pointers
    assert L.p3tok_square_distance(None, 2, 0, None, 16, 3, None, None) == _lib.OK            # empty matrix
    assert L.p3tok_square_distance(None, 2, 4, None, 16, 2, None, None) == _lib.ERR_INVALID   # dst rows shorter than xyz
    assert L.p3tok_square_distance(None, 2, 4, None, 16, 3, None, None) == _lib.ERR_INVALID   # null pointers
    assert L.p3tok_square_distance(None, 1 << 14, 1 << 14, None, 1 << 14, 3, None, None) == _lib.ERR_INVALID  # nulls first
    from p3tok import functional as F
    with pytest.raises(RuntimeError, match="16"):
        F.farthest_point_sampling(torch.zeros(1, 8, 17), 4, torch.zeros(1, dtype=torch.long))
    with pytest.raises((NotImplementedError, RuntimeError)):                                  # CPU tensors: no fallback
        F.farthest_point_sampling(torch.zeros(1, 8, 5), 4, torch.zeros(1, dtype=torch.long))
    with pytest.raises((NotImplementedError, RuntimeError)):
        F.square_distance(torch.zeros(1, 2, 3), torch.zeros(1, 8, 3))


def test_bn_statistics_combination_matches_batchnorm():
    """Host logic of the train-mode BatchNorm (p3tok.train.combine_stats): (sum, sum of squares, rows) -> mean, rstd and the
    unbiased variance nn.BatchNorm1d puts into running_var; summing the per-shard triples first (SyncBN) gives the same."""
    from p3tok import train
    torch.manual_seed(3)
    x = torch.randn(200, 7, dtype=torch.float64) * 3 + 1
    bn = torch.nn.BatchNorm1d(7).double().train()
    y = bn(x)
    mean, rstd, var_unb = train.combine_stats(x.sum(0), (x * x).sum(0), 200.0, bn.eps)
    assert torch.allclose((x - mean) * rstd, y, atol=1e-10)
    assert torch.allclose(bn.running_var, 0.9 * torch.ones(7, dtype=torch.float64) + 0.1 * var_unb, atol=1e-12)
    a, b = x[:80], x[80:]
    m2, r2, v2 = train.combine_stats(a.sum(0) + b.sum(0), (a * a).sum(0) + (b * b).sum(0), 200.0, bn.eps)
    assert torch.allclose(m2, mean) and torch.allclose(r2, rstd) and torch.allclose(v2, var_unb)
