"""GPU tests of the gradients with respect to the input points: the point-op drop-ins (gather_points, apf_group, group_gather
and the functions over them), PointNet in train mode, the eval-mode tokenizers and heads (running-statistics BatchNorm), and
AdaptPointFormer / Pix4Point end to end - against torch float64 autograd of oracle/port.py's functions with the kernels'
indices injected (tests/grad_reference.py), of torch.nn heads, and of the float64 oracle.  Also: eval-mode calls that want no
input gradient still run the serving kernels, bit for bit."""
import copy

import numpy as np
import pytest
import torch

import grad_reference as gr
from helpers import dev, to_dev
from oracle import oracle, port, train as otrain
from p3tok import functional, ops, synth, train_vit
from p3tok.apf_model import AdaptPointFormer, ClassificationHead, run_blocks
from p3tok.modules import Encoder, Group, P3Embed, PointNet
from p3tok.p4p_model import ClsHead, Pix4Point

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _close(got, ref, what, tol=TOL, scale=None):
    got = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    ref = ref.detach().double().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert np.isfinite(got).all(), what
    err = np.abs(got - ref).max() / max(np.abs(ref).max() if scale is None else scale, 1e-30)
    print(f"[grad parity] {what}: max|err|/max|ref| {err:.2e}")
    assert err <= tol, (what, err)


def _close_picks(got, ref, what, share=0.99, fro_tol=2e-2):
    """For the tokenizer stage of the end-to-end tests, whose arg-max pools make tens of thousands of picks: an fp32 kernel
    and the float64 reference can resolve a near-tie differently, which moves one row's gradient to another point.  So at
    least `share` of the elements within 1e-4 of max, and the relative Frobenius error within fro_tol (a handful of moved
    picks); the element-wise 1e-4 contract is held by the module tests above, on shapes with fewer picks."""
    got = got.detach().double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    ref = ref.detach().double().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    assert got.shape == ref.shape and np.isfinite(got).all(), what
    diff = np.abs(got - ref)
    ok = float((diff <= TOL * np.abs(ref).max()).mean())
    fro = float(np.linalg.norm(got - ref) / max(np.linalg.norm(ref), 1e-30))
    print(f"[grad parity] {what}: max|err|/max|ref| {diff.max() / np.abs(ref).max():.2e}, share within 1e-4 of max {ok:.5f}, "
          f"relative Frobenius {fro:.2e}")
    assert ok >= share and fro <= fro_tol, (what, ok, fro)


def _rand(shape, seed):
    return torch.from_numpy((synth.uniform01(seed, int(np.prod(shape)), 61).reshape(shape) - 0.5).astype(np.float32))


def _x64(x):
    return x.detach().double().cpu().requires_grad_(True)


def _params_close(module, sd64, what, prefix=""):
    """Every parameter gradient of the module against the float64 reference's, on the scale of the largest weight gradient (a
    conv bias in front of a BatchNorm has an exactly-zero gradient, whose fp32 noise has no scale of its own)."""
    named = [(n, p_) for n, p_ in module.named_parameters() if p_.requires_grad]
    scale = max(float(sd64[prefix + n].grad.abs().max()) for n, _ in named if n.endswith("weight"))
    for n, p_ in named:
        assert p_.grad is not None, n
        _close(p_.grad, sd64[prefix + n].grad, f"{what} grad {n}", scale=scale)


def _buffers(module):
    return {n: b.detach().clone() for n, b in module.named_buffers()}


def _buffers_unchanged(module, before):
    for n, b in module.named_buffers():
        assert torch.equal(b, before[n]), n


# ------------------------------------------------------------------------------------------------ functional drop-ins
@pytest.mark.parametrize("B,N,C,shape", [(2, 300, 3, (37,)), (3, 500, 4, (13, 7)), (2, 9000, 3, (64,))])
def test_index_points_and_fps_gradients(B, N, C, shape):
    x = to_dev(synth.make_cloud("uniform", B, N, 3, C)).requires_grad_(True)
    idx = to_dev(synth.randint(5, B * int(np.prod(shape)), N, 9).reshape(B, *shape).astype(np.int64))
    g = to_dev(_rand((B, *shape, C), 7).numpy())
    (functional.index_points(x, idx) * g).sum().backward()
    x64 = _x64(x)
    (port.take(x64, idx.cpu()) * g.double().cpu()).sum().backward()
    _close(x.grad, x64.grad, f"index_points B{B} N{N} C{C}", 1e-6)
    # fps: FPS picks (no gradient) then the gather of all C channels
    x.grad = None
    st = to_dev(synth.start_indices(B, N, 3))
    S = shape[0]
    out = functional.fps(x, S, st)
    gs = to_dev(_rand((B, S, C), 8).numpy())
    (out * gs).sum().backward()
    x64 = _x64(x)
    (port.take(x64, ops.fps(x.detach(), st, S).cpu()) * gs.double().cpu()).sum().backward()
    _close(x.grad, x64.grad, f"fps B{B} N{N} C{C}", 1e-6)


@pytest.mark.parametrize("need", ["both", "feats"])
def test_group_knn_gradients(need):
    B, N, D, G, k = 2, 700, 5, 29, 13
    p = to_dev(synth.make_cloud("clustered", B, N, 11, 3)).requires_grad_(need == "both")
    f = to_dev(_rand((B, N, D), 12).numpy()).requires_grad_(True)
    ctr = functional.index_points(p.detach(), to_dev(synth.randint(11, B * G, N, 13).reshape(B, G).astype(np.int64)))
    gp, gf = functional.group_knn(p, ctr, f, k)
    wp, wf = to_dev(_rand((B, G, k, 3), 14).numpy()), to_dev(_rand((B, G, k, D), 15).numpy())
    ((gp * wp).sum() + (gf * wf).sum()).backward()
    nidx = functional.knn_query(p.detach(), ctr, k).long().cpu()
    p64, f64 = _x64(p), _x64(f)
    bi = torch.arange(B).view(B, 1, 1).expand(-1, G, k)          # pix4point.py:92-102
    ((p64[bi, nidx] * wp.double().cpu()).sum() + (f64[bi, nidx] * wf.double().cpu()).sum()).backward()
    _close(f.grad, f64.grad, "group_knn d feats", 1e-6)
    if need == "both":
        _close(p.grad, p64.grad, "group_knn d pnts", 1e-6)
    else:
        assert p.grad is None


@pytest.mark.parametrize("B,N,C,G,k", [(2, 400, 3, 37, 13), (2, 400, 4, 21, 16), (2, 9000, 3, 64, 16)])
@pytest.mark.parametrize("route", ["view", "xyz"])
def test_group_forward_gradients(B, N, C, G, k, route):
    """Both routes of Group.forward: xyz = the x[:, :, :3] view (p3tok::apf_group in place) and a separate xyz tensor (indices
    and centres from xyz through gather_points, the neighbourhood from x)."""
    x = to_dev(synth.make_cloud("clustered", B, N, 17, C)).requires_grad_(True)
    st = to_dev(synth.start_indices(B, N, 17))
    grp = Group(G, k)
    xyz = x[:, :, :3] if route == "view" else x[:, :, :3] * 0.5
    neigh, center = grp(x, xyz, st)
    wn, wc = to_dev(_rand((B, G, k, 2 * C), 18).numpy()), to_dev(_rand((B, G, 3), 19).numpy())
    ((neigh * wn).sum() + (center * wc).sum()).backward()
    fidx, _, kidx, perm = grp.indices(x.detach() if route == "view" else xyz.detach().contiguous(), st)
    x64 = _x64(x)
    n64, c64 = gr.apf_group_idx(x64, fidx, kidx, perm)
    if route == "xyz":
        c64 = gr.apf_group_idx(x64[:, :, :3] * 0.5, fidx, kidx, perm)[1]
    _close(neigh, n64, "Group neighbourhood", 1e-6)
    _close(center, c64, "Group centres", 1e-6)
    ((n64 * wn.double().cpu()).sum() + (c64 * wc.double().cpu()).sum()).backward()
    _close(x.grad, x64.grad, f"Group.forward ({route}) d x", 1e-5)


def test_opcheck_of_the_differentiable_gathers():
    x = to_dev(synth.make_cloud("uniform", 2, 64, 4, 4)).requires_grad_(True)
    fidx = to_dev(synth.randint(1, 2 * 8, 64, 2).reshape(2, 8).astype(np.int64))
    kidx = to_dev(synth.randint(1, 2 * 8 * 5, 64, 3).reshape(2, 8, 5).astype(np.int64))
    perm = torch.stack([torch.randperm(8, generator=torch.Generator().manual_seed(i)) for i in range(2)]).to(dev())
    f = to_dev(_rand((2, 64, 6), 4).numpy()).requires_grad_(True)
    for op, args in ((ops.gather_points, (x, fidx)), (ops.apf_group, (x, fidx, kidx, perm)),
                     (ops.group_gather, (x[..., :3].contiguous().detach().requires_grad_(True), f, kidx.int()))):
        torch.library.opcheck(op, args, test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))


# ------------------------------------------------------------------------------------------------ PointNet in train mode
@pytest.mark.parametrize("C", [3, 4])
def test_pointnet_train_fills_input_gradient(C):
    B, N, G, k, E = 3, 500, 21, 12, 48
    x = synth.make_cloud("clustered", B, N, 91, C)
    st = to_dev(synth.start_indices(B, N, 91))
    sd = synth.apf_encoder_state(E, 2 * C, 91)
    gt = (synth.uniform01(91, B * G * E, 3).reshape(B, G, E) - 0.5).astype(np.float32)

    def run(want):
        net = PointNet(E, G, k, 2 * C).to(dev()).train()
        net.encoder.load_state_dict(synth.to_torch_state(sd))
        xt = to_dev(x).requires_grad_(want)
        tok = net(xt, st)
        (tok * to_dev(gt)).sum().backward()
        return net, xt, tok

    net, xt, tok = run(True)
    net0, _, tok0 = run(False)
    assert torch.equal(tok, tok0), "tokens change when x requires grad"
    grp = oracle.group_apf(x, st.cpu().numpy(), G, k)
    _, ograds, _ = otrain.apf_encoder_train(sd, grp["neigh"], gt)
    scale = max(np.abs(v).max() for k_, v in ograds.items() if k_.endswith("weight") and "conv" in k_)
    for (n, a), (_, b) in zip(net.encoder.named_parameters(), net0.encoder.named_parameters()):
        _close(a.grad, b.grad, f"train grad {n} with / without x.requires_grad", 1e-6, scale)
    for n, p_ in net.encoder.named_parameters():
        _close(p_.grad, ograds[n].reshape(p_.shape), f"train grad {n} vs oracle", scale=scale)
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    gidx = [torch.from_numpy(np.asarray(grp[n])) for n in ("fps_idx", "knn_idx", "perm")]
    gr.apf_group_idx(x64, *gidx)[0].backward(torch.from_numpy(ograds["input"]))
    _close(xt.grad, x64.grad, "PointNet.train() d x vs float64")


# ------------------------------------------------------------------------------------------------ eval mode
def test_encoder_eval_gradients():
    B, G, k, C, E = 3, 17, 12, 3, 64
    sd = synth.apf_encoder_state(E, 2 * C, 23)
    enc = Encoder(E, 2 * C).to(dev()).eval()
    enc.load_state_dict(synth.to_torch_state(sd))
    before = _buffers(enc)
    pg = to_dev(_rand((B, G, k, 2 * C), 24).numpy()).requires_grad_(True)
    gt = to_dev(_rand((B, G, E), 25).numpy())
    tok = enc(pg)
    (tok * gt).sum().backward()
    sd64 = gr.state64(sd)
    pg64 = _x64(pg)
    tok64 = port.apf_encode(sd64, pg64)
    (tok64 * gt.double().cpu()).sum().backward()
    _close(tok, tok64, "Encoder.eval tokens")
    _close(pg.grad, pg64.grad, "Encoder.eval d point_groups")
    _params_close(enc, sd64, "Encoder.eval")
    _buffers_unchanged(enc, before)


def _pointnet_eval_case(C, kind, precision, seed, B=3, N=500, G=21, k=12, E=48):
    x = to_dev(synth.make_cloud(kind, B, N, seed, C)).requires_grad_(True)
    st = to_dev(synth.start_indices(B, N, seed))
    sd = synth.apf_encoder_state(E, 2 * C, seed)
    net = PointNet(E, G, k, 2 * C, precision=precision).to(dev()).eval()
    net.encoder.load_state_dict(synth.to_torch_state(sd))
    before = _buffers(net)
    gt = to_dev(_rand((B, G, E), seed).numpy())
    tok = net(x, st)
    (tok * gt).sum().backward()
    _buffers_unchanged(net, before)
    fidx, _, kidx, perm = net.group.indices(x.detach(), st)
    sd64 = gr.state64(sd)
    x64 = _x64(x)
    tok64 = gr.pointnet_idx(sd64, x64, fidx, kidx, perm)
    (tok64 * gt.double().cpu()).sum().backward()
    return net, x, tok, sd64, x64, tok64


@pytest.mark.parametrize("C,precision", [(3, "fp32"), (4, "bf16")])
def test_pointnet_eval_gradients(C, precision):
    """The gradient path is fp32 whatever `precision` says (bf16 here: tokens still within 1e-4 and float32)."""
    net, x, tok, sd64, x64, tok64 = _pointnet_eval_case(C, "clustered", precision, 31)
    assert tok.dtype == torch.float32
    _close(tok, tok64, f"PointNet.eval C{C} tokens")
    _close(x.grad, x64.grad, f"PointNet.eval C{C} d x")
    _params_close(net.encoder, sd64, f"PointNet.eval C{C}")


def test_pointnet_eval_gradients_on_duplicated_points():
    """Coincident points are interchangeable for kNN and the max-pools, so the gradient may move between them: compare the
    gradient summed over every set of coincident points."""
    B = 3
    net, x, tok, sd64, x64, tok64 = _pointnet_eval_case(3, "duplicates", "fp32", 37, B=B)
    _close(tok, tok64, "PointNet.eval duplicates tokens")
    xs, got, ref = x.detach().cpu().numpy(), x.grad.cpu().numpy().astype(np.float64), x64.grad.numpy()
    for b in range(B):
        _, inv = np.unique(xs[b], axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        sg, sr = np.zeros((inv.max() + 1, 3)), np.zeros((inv.max() + 1, 3))
        np.add.at(sg, inv, got[b])
        np.add.at(sr, inv, ref[b])
        _close(sg, sr, f"PointNet.eval duplicates cloud {b}: d x summed per coincident set", scale=np.abs(ref).max())


def _p3embed_indices(p, starts, k, stages):
    idx, pts, N = [], p.detach(), p.shape[1]
    for s in range(stages):
        N //= 4
        cidx = ops.fps(pts, starts[s], min(N, pts.shape[1]))
        ctr = ops.gather_points(pts, cidx)
        idx.append((cidx, functional.knn_query(pts, ctr, k)))
        pts = ctr
    return idx


@pytest.mark.parametrize("stages", [1, 2])
def test_p3embed_eval_gradients(stages):
    B, N, k, W = 2, 1024, 16, 64
    sd = synth.p3embed_state(3, 0.25 ** stages, 4, 4, W, 53)
    m = P3Embed(in_channels=3, sample_ratio=0.25 ** stages, k=k, embed_dim=W, precision="bf16",
                token_dtype=torch.bfloat16).to(dev()).eval()
    m.load_state_dict(synth.to_torch_state(sd))
    before = _buffers(m)
    p = to_dev(synth.make_cloud("clustered", B, N, 53, 3)).requires_grad_(True)
    f = to_dev(_rand((B, 3, N), 54).numpy()).requires_grad_(True)
    starts = [to_dev(synth.start_indices(B, N // 4 ** s, 53, s)) for s in range(stages)]
    ps, fs = m(p, f, starts)
    assert fs[-1].dtype == torch.float32
    gf, gc = to_dev(_rand(tuple(fs[-1].shape), 55).numpy()), to_dev(_rand(tuple(ps[-1].shape), 56).numpy())
    ((fs[-1] * gf).sum() + (ps[-1] * gc).sum()).backward()
    _buffers_unchanged(m, before)
    sd64 = gr.state64(sd)
    p64, f64 = _x64(p), _x64(f)
    ps64, fs64 = gr.p3embed_idx(sd64, p64, f64, k, _p3embed_indices(p, starts, k, stages))
    ((fs64[-1] * gf.double().cpu()).sum() + (ps64[-1] * gc.double().cpu()).sum()).backward()
    for s in range(1, stages + 1):
        _close(fs[s], fs64[s], f"P3Embed.eval stage {s} features")
    _close(p.grad, p64.grad, f"P3Embed.eval ({stages} stages) d p")
    _close(f.grad, f64.grad, f"P3Embed.eval ({stages} stages) d f")
    _params_close(m, sd64, f"P3Embed.eval ({stages} stages)")


# ------------------------------------------------------------------------------------------------ heads
def _randomise_bn_buffers(module, seed):
    for i, bn in enumerate(m for m in module.modules() if isinstance(m, torch.nn.BatchNorm1d)):
        c = bn.num_features
        bn.running_mean.copy_(torch.from_numpy(synth.uniform01(seed + i, c, 71) - 0.5).float())
        bn.running_var.copy_(torch.from_numpy(synth.uniform01(seed + i, c, 72) + 0.5).float())
        bn.weight.data.copy_(torch.from_numpy(synth.uniform01(seed + i, c, 73) + 0.5).float())
        bn.bias.data.copy_(torch.from_numpy(synth.uniform01(seed + i, c, 74) - 0.5).float())


@pytest.mark.parametrize("kind", ["ClassificationHead", "ClsHead"])
def test_heads_eval_gradients(kind):
    B, E, classes = 6, 96, 7
    torch.manual_seed(5)
    head = ClassificationHead(E, classes) if kind == "ClassificationHead" else ClsHead(E, classes)
    with torch.no_grad():
        _randomise_bn_buffers(head, 61)
    head = head.to(dev()).eval()
    seq = head.mlp_head if kind == "ClassificationHead" else head.head
    before = _buffers(head)
    x = to_dev(_rand((B, E), 62).numpy()).requires_grad_(True)
    gl = to_dev(_rand((B, classes), 63).numpy())
    logits = head(x)
    (logits * gl).sum().backward()
    _buffers_unchanged(head, before)
    ref = copy.deepcopy(seq).cpu().double().eval()
    for p_ in ref.parameters():
        p_.grad = None
    x64 = _x64(x)
    l64 = ref(x64)
    (l64 * gl.double().cpu()).sum().backward()
    _close(logits, l64, f"{kind}.eval logits")
    _close(x.grad, x64.grad, f"{kind}.eval d x")
    scale = max(float(p_.grad.abs().max()) for n, p_ in ref.named_parameters() if n.endswith("weight"))
    for (n, a), (_, b) in zip(seq.named_parameters(), ref.named_parameters()):
        _close(a.grad, b.grad, f"{kind}.eval grad {n}", scale=scale)


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("freeze", [False, True])
def test_adaptpointformer_eval_input_gradient(freeze):
    """AdaptPointFormer.eval() with x.requires_grad, checked stage by stage: the head (torch.nn float64) on the kernel's pooled
    features, the 12-block stack (float64 oracle) on the kernel's tokens fed the kernel's pooled gradient, the tokenizer (float64
    port) fed the kernel's token gradient.  Then the module's own forward gives the same logits and d x."""
    B, N, G, k, E = 4, 256, 16, 8, 384
    m = AdaptPointFormer(num_classes=7, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="fp32")
    sd = synth.apf_vit_state(E, 12, 7, 17)
    sd.update({"point_encoder.encoder." + k_: v for k_, v in synth.apf_encoder_state(E, 6, 17).items()})
    m.load_state_dict(synth.to_torch_state(sd), strict=True)
    m = m.to(dev()).eval()
    if freeze:
        m._freeze()
    before = _buffers(m)
    x = to_dev(synth.make_cloud("uniform", B, N, 17, 3)).requires_grad_(True)
    st = to_dev(synth.start_indices(B, N, 17))
    tok = m.point_encoder(x, st)
    tok.retain_grad()
    pooled = run_blocks(m.blocks, tok, m.encoder_norm, {}, m.block_precision)[1]
    pooled.retain_grad()
    logits = m.head(pooled)
    gl = to_dev(_rand((B, 7), 18).numpy())
    (logits * gl).sum().backward()
    _buffers_unchanged(m, before)
    for n, p_ in m.named_parameters():
        assert (p_.grad is not None) == p_.requires_grad, n
    # head
    ref = copy.deepcopy(m.head.mlp_head).cpu().double().eval()
    pin = _x64(pooled)
    l64 = ref(pin)
    (l64 * gl.double().cpu()).sum().backward()
    _close(logits, l64, "logits")
    _close(pooled.grad, pin.grad, "d pooled")
    # blocks
    po, dx, gn = otrain.apf_vit_backward(sd, tok.detach().cpu().numpy(), 12, 12, pooled.grad.cpu().numpy())
    _close(pooled, po, "pooled (12 layers)")
    _close(tok.grad, dx, "d tokens through 12 layers")
    _close(m.encoder_norm.weight.grad, gn["encoder_norm.weight"], "encoder_norm.weight grad")
    # tokenizer
    fidx, _, kidx, perm = m.point_encoder.group.indices(x.detach(), st)
    sd64 = gr.state64({k_[len("point_encoder.encoder."):]: v for k_, v in sd.items() if k_.startswith("point_encoder.encoder.")})
    x64 = _x64(x)
    tok64 = gr.pointnet_idx(sd64, x64, fidx, kidx, perm)
    (tok64 * tok.grad.double().cpu()).sum().backward()
    _close(tok, tok64, "tokens")
    _close_picks(x.grad, x64.grad, "AdaptPointFormer.eval d x")
    for n, p_ in m.point_encoder.encoder.named_parameters():
        _close_picks(p_.grad, sd64[n].grad, f"AdaptPointFormer.eval point_encoder grad {n}", 0.0)
    # the module's forward routes the same way
    x2 = x.detach().clone().requires_grad_(True)
    logits2 = m(x2, st)
    (logits2 * gl).sum().backward()
    _close(logits2, logits, "forward() logits vs stage by stage", 1e-6)
    _close(x2.grad, x.grad, "forward() d x vs stage by stage", 1e-5)


@pytest.mark.parametrize("frozen", [False, True])
def test_pix4point_eval_input_gradient(frozen):
    """Pix4Point.eval() with the points requiring grad, stage by stage: ClsHead (torch.nn float64) on the kernel's global
    features, the block loop (float64 oracle) on the kernel's feats / pos fed the global-feature gradient, the tokenizer
    (P3Embed + proj + pos_embed + cls concat in float64 on the kernel's indices) fed the kernel's feats / pos gradients."""
    B, N, k, E, depth, heads = 3, 512, 8, 64, 2, 2
    torch.manual_seed(3)
    m = Pix4Point(num_classes=5, embed_dim=E, depth=depth, num_heads=heads, k_neighbors=k, frozen=frozen, precision="fp32")
    with torch.no_grad():
        for i, bn in enumerate(mod for mod in m.modules() if isinstance(mod, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d))):
            c = bn.num_features
            bn.running_mean.copy_(torch.from_numpy(synth.uniform01(80 + i, c, 71) * 0.2 - 0.1).float())
            bn.running_var.copy_(torch.from_numpy(synth.uniform01(80 + i, c, 72) + 0.5).float())
        for n, t in synth.to_torch_state(synth.pointvit_state(E, depth, 3)).items():
            m.model.state_dict()[n].copy_(t)
    m = m.to(dev()).eval()
    before = _buffers(m)
    p = to_dev(synth.make_cloud("clustered", B, N, 81, 3)).requires_grad_(True)
    st = [to_dev(synth.start_indices(B, N, 81))]
    tokm = m.model.__dict__["_tok"]
    tokm.train(False)
    p_list, _, feats, pos = tokm(p, None, st)
    feats.retain_grad()
    pos.retain_grad()
    out = train_vit.timm_blocks_train(m.model.vit.blocks, m.model.norm, feats, pos)
    glob = torch.cat([train_vit.TokenMaxFn.apply(out, 1), out[:, 0, :]], 1)
    glob.retain_grad()
    logits = m.cls_head(glob)
    gl = to_dev(_rand((B, 5), 82).numpy())
    (logits * gl).sum().backward()
    _buffers_unchanged(m, before)
    for n, p_ in m.named_parameters():
        if n != "model.vit.pos_embed":                      # timm's position table: PointViT never reads it
            assert (p_.grad is not None) == p_.requires_grad, n
    if frozen:                                               # vit.cls_token is aliased as cls_token and stays trainable, as in
        assert all(p_.grad is None for p_ in m.model.vit.blocks.parameters())   # the reference (pix4point.py:224-233)
    # head
    ref = copy.deepcopy(m.cls_head.head).cpu().double().eval()
    g64 = _x64(glob)
    l64 = ref(g64)
    (l64 * gl.double().cpu()).sum().backward()
    _close(logits, l64, "logits")
    _close(glob.grad, g64.grad, "d global features")
    # blocks
    sd = {n: t.detach().cpu().numpy() for n, t in m.model.state_dict().items()}
    glob_o, dfe, dpo, _ = otrain.pointvit_backward(sd, feats.detach().cpu().numpy(), pos.detach().cpu().numpy(), depth, heads,
                                                   glob.grad.cpu().numpy())
    _close(glob, glob_o, "global features")
    _close(feats.grad, dfe, "d feats")
    _close(pos.grad, dpo, "d pos")
    # tokenizer
    sd64 = gr.state64(m.model.state_dict())
    p64 = _x64(p)
    idx = _p3embed_indices(p, st, k, 1)
    ps64, fs64 = gr.p3embed_idx({n[len("patch_embed."):]: t for n, t in sd64.items() if n.startswith("patch_embed.")},
                                p64, p64.transpose(1, 2), k, idx)
    lin = lambda t, n: t @ sd64[n + ".weight"].t() + sd64[n + ".bias"]
    x_tok = lin(fs64[-1].transpose(1, 2), "proj")
    pe = lin(torch.nn.functional.gelu(lin(ps64[-1], "pos_embed.0")), "pos_embed.2")
    f64 = torch.cat([sd64["vit.cls_token"].expand(B, -1, -1), x_tok], 1)
    q64 = torch.cat([sd64["cls_pos"].expand(B, -1, -1), pe], 1)
    ((f64 * feats.grad.double().cpu()).sum() + (q64 * pos.grad.double().cpu()).sum()).backward()
    _close(feats, f64, "feats")
    _close(pos, q64, "pos")
    _close_picks(p.grad, p64.grad, "Pix4Point.eval d p")
    for n, p_ in m.model.patch_embed.named_parameters():
        _close_picks(p_.grad, sd64["patch_embed." + n].grad, f"Pix4Point.eval patch_embed grad {n}", 0.0)
    # the module's forward routes the same way
    p2 = p.detach().clone().requires_grad_(True)
    logits2 = m(p2, st)
    (logits2 * gl).sum().backward()
    _close(logits2, logits, "forward() logits vs stage by stage", 1e-6)
    _close(p2.grad, p.grad, "forward() d p vs stage by stage", 1e-5)


# ------------------------------------------------------------------------------------------------ serving unchanged
def test_eval_without_input_gradient_keeps_serving_path():
    """Eval-mode calls that want no input gradient - an input without grad under grad mode (parameters still requiring grad),
    or an input with grad under no_grad / inference_mode - run the serving kernels: outputs bit-identical to the no_grad call
    and the same number of kernel launches."""
    B, N = 4, 512
    apf = AdaptPointFormer(num_classes=7, embedding_dim=384, npoint=32, nsample=16, in_channels=3).to(dev()).eval()
    p4p = Pix4Point(num_classes=5, embed_dim=64, depth=2, num_heads=2, k_neighbors=8).to(dev()).eval()
    x = to_dev(synth.make_cloud("clustered", B, N, 7, 3))
    st = to_dev(synth.start_indices(B, N, 7))
    for name, model, call in (("AdaptPointFormer", apf, lambda t: apf(t, st)), ("Pix4Point", p4p, lambda t: p4p(t, [st]))):
        with torch.no_grad():
            call(x)                                                 # warm the folded-weight caches
            n0 = ops.kernel_launches()
            ref = call(x)
            n_ref = ops.kernel_launches() - n0
        xg = x.clone().requires_grad_(True)
        for what, ctx, inp in (("grad mode, input without grad", torch.enable_grad(), x),
                               ("no_grad, input with grad", torch.no_grad(), xg),
                               ("inference_mode, input with grad", torch.inference_mode(), xg)):
            with ctx:
                n0 = ops.kernel_launches()
                out = call(inp)
                n = ops.kernel_launches() - n0
            assert not out.requires_grad, (name, what)
            assert torch.equal(out, ref), (name, what)
            assert n == n_ref, (name, what, n, n_ref)
