"""Generate tests/golden/*.npz from the UNMODIFIED reference.

Run:  python tests/golden/make_golden.py
Needs a checkout of the original project (read-only; oracle/ref_loader.py says where).  The reference's internal `torch.randint` draw for the
first FPS index (src/data/sampler.py:20, src/models/pix4point.py:30) is substituted by the
synthetic start indices for the duration of each call; nothing else is touched.
While generating, the script also asserts that oracle/port.py is bit-identical to the
reference on this host and that oracle/oracle.py agrees (indices up to exact ties, tokens
to 1e-5), i.e. it is the script that pins the oracle.
"""
import contextlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from p3tok import synth  # noqa: E402
from oracle import oracle, port, ref_loader  # noqa: E402
import cases  # noqa: E402


@contextlib.contextmanager
def forced_randint(draws):
    draws = [torch.as_tensor(d, dtype=torch.long) for d in draws]
    real = torch.randint
    it = iter(draws)

    def fake(low, high, size, **kw):
        d = next(it)
        assert tuple(size) == tuple(d.shape) and int(d.max()) < high
        return d.clone()

    torch.randint = fake
    try:
        yield
    finally:
        torch.randint = real


def apf_case(ref, name, c):
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], c["C"])
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    sd = synth.apf_encoder_state(c["E"], 2 * c["C"], c["seed"])
    tsd = synth.to_torch_state(sd)
    net = ref.PointNet(c["E"], c["G"], c["k"], 2 * c["C"]).eval()
    net.encoder.load_state_dict(tsd, strict=True)
    xt = torch.from_numpy(x)
    with torch.no_grad():
        with forced_randint([start]):
            fidx = ref.furthest_point_sample(xt[:, :, :3].contiguous(), c["G"])
        ctr = ref.index_points(xt[:, :, :3].contiguous(), fidx)
        kidx = ref.knn_point(c["k"], xt[:, :, :3].contiguous(), ctr)
        with forced_randint([start]):
            neigh, center = net.group(xt, xt[:, :, :3])
        tok = net.encoder(neigh)
        with forced_randint([start]):
            tok2 = net(xt)
        assert torch.equal(tok, tok2)
        # port == reference, bitwise, on this host
        pn, pc = port.apf_group(xt, c["G"], c["k"], torch.from_numpy(start))
        assert torch.equal(pn, neigh) and torch.equal(pc, center), name
        assert torch.equal(port.apf_encode(tsd, pn), tok), name
    # oracle vs reference
    o_tok, grp = oracle.pointnet_apf(sd, x, start, c["G"], c["k"])
    assert np.array_equal(grp["fps_idx"], fidx.numpy()), name
    D = oracle.pair_dist(x, grp["center"] if False else oracle.gather_points(x[..., :3], grp["fps_idx"]), oracle.KNN_APF_SQ)
    ok, msg = oracle.knn_tie_equivalent(grp["knn_idx"], kidx.numpy(), D, ulp=0)
    assert ok, (name, msg)
    ties = msg
    ref_tok = tok.numpy()
    # Morton order may differ only on equal codes
    codes, perm = grp["codes"], grp["perm"]
    ref_center = center.numpy()
    same_order = np.array_equal(grp["center"], ref_center)
    err = np.abs(o_tok - ref_tok).max() / np.abs(ref_tok).max()
    print(f"{name}: fps exact, knn {ties}, morton-order-identical={same_order}, token rel-max-err {err:.2e}")
    assert same_order and err < 2e-5, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), fps_idx=fidx.numpy().astype(np.int32),
                        knn_idx=kidx.numpy().astype(np.int32), center=ref_center,
                        neigh=neigh.numpy() if neigh.numel() < 70000 else np.zeros(0, np.float32),
                        tokens=ref_tok)


def p4p_case(ref, name, c):
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    stages, dims = synth.p3embed_dims(3, c["sample_ratio"], 4, 4, c["embed_dim"])
    starts, n = [], c["N"]
    for s in range(stages):
        starts.append(synth.start_indices(c["B"], n, c["seed"], s))
        n //= 4
    sd = synth.p3embed_state(3, c["sample_ratio"], 4, 4, c["embed_dim"], c["seed"])
    tsd = synth.to_torch_state(sd)
    mod = ref.P3Embed(in_channels=3, sample_ratio=c["sample_ratio"], k=c["k"], embed_dim=c["embed_dim"]).eval()
    mod.load_state_dict(tsd, strict=True)
    xt = torch.from_numpy(x)
    ft = xt.clone().transpose(1, 2).contiguous()
    rec = {"fps": [], "grp": []}
    real_s, real_g = mod.sample_fn, mod.grouper
    mod.sample_fn = lambda p, m: rec["fps"].append(real_s(p, m)) or rec["fps"][-1]
    mod.grouper = lambda p, cc, f, k: rec["grp"].append(real_g(p, cc, f, k)) or rec["grp"][-1]
    with torch.no_grad():
        with forced_randint(starts):
            rp, rf = mod(xt, ft)
        pp, pf = port.p3embed(tsd, xt, ft, c["k"], stages, [torch.from_numpy(s) for s in starts])
        for a, b in zip(rf, pf):
            assert torch.equal(a, b), name
        ref_knn = [torch.cdist(rp[s + 1], rp[s]).topk(k=c["k"], dim=-1, largest=False, sorted=True).indices
                   for s in range(stages)]
    for s in range(stages):  # the recorded grouper output is what those indices gather
        bi = torch.arange(c["B"]).view(-1, 1, 1)
        assert torch.equal(rec["grp"][s][0], rp[s][bi, ref_knn[s]]), name
    # oracle: drive each stage with the REFERENCE's previous-stage features so one stage's
    # tie-break differences cannot cascade
    out = {}
    for s in range(stages):
        pts = rp[s].numpy()
        feats = rf[s].transpose(1, 2).contiguous().numpy()
        ctr, tok, fidx, kidx = oracle.p3embed_stage(sd, s, pts, feats, starts[s], c["k"])
        assert np.array_equal(fidx, rec["fps"][s].numpy()), (name, s)
        D = oracle.pair_dist(pts, ctr, oracle.KNN_P4P_CDIST)
        ok, msg = oracle.knn_tie_equivalent(kidx, ref_knn[s].numpy(), D, ulp=1)
        assert ok, (name, s, msg)
        assert oracle.sorted_by_distance(ref_knn[s].numpy(), D, ulp=1), (name, s)
        rtok = rf[s + 1].transpose(1, 2).numpy()
        nbad = int((np.abs(tok - rtok).max(-1) > 2e-5 * np.abs(rtok).max()).sum())
        print(f"{name} stage {s}: fps exact, knn {msg}, groups with token diff > 2e-5: {nbad}")
        assert nbad == 0, name
        out[f"fps_idx{s}"] = rec["fps"][s].numpy().astype(np.int32)
        out[f"knn_idx{s}"] = ref_knn[s].numpy().astype(np.int32)
        out[f"centres{s}"] = rp[s + 1].numpy()
        out[f"tokens{s}"] = rtok
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)


def index_case(ref, name, c):
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    xt = torch.from_numpy(x)
    with torch.no_grad():
        with forced_randint([start]):
            f1 = ref.furthest_point_sample(xt, c["G"])
        with forced_randint([start]):
            f2 = ref.farthest_point_sampling(xt, c["G"])
        assert torch.equal(f1, f2)
        ctr = ref.index_points(xt, f1)
        k_apf = ref.knn_point(c["k"], xt, ctr)
        k_p4p = torch.cdist(ctr, xt).topk(k=c["k"], dim=-1, largest=False, sorted=True).indices
        mperm = ref.MortonEncoder.points_to_morton(ctr)
    assert np.array_equal(oracle.fps(x, start, c["G"]), f1.numpy()), name
    cn = ctr.numpy()
    for mode, r, ulp in ((oracle.KNN_APF_SQ, k_apf, 0), (oracle.KNN_P4P_CDIST, k_p4p, 1)):
        D = oracle.pair_dist(x, cn, mode)
        ok, msg = oracle.knn_tie_equivalent(oracle.knn(x, cn, c["k"], mode), r.numpy(), D, ulp=ulp)
        assert ok, (name, mode, msg)
        print(f"{name} mode {mode}: {msg}")
    codes, perm = oracle.morton(cn)
    rc = np.take_along_axis(codes, mperm.numpy(), 1)
    assert (np.diff(rc, axis=1) >= 0).all() and np.array_equal(np.sort(mperm.numpy(), 1), np.sort(perm, 1)), name
    print(f"{name}: fps exact; morton perm identical={np.array_equal(perm, mperm.numpy())}")
    np.savez_compressed(os.path.join(HERE, name + ".npz"), fps_idx=f1.numpy().astype(np.int32),
                        knn_apf=k_apf.numpy().astype(np.int32), knn_p4p=k_p4p.numpy().astype(np.int32),
                        morton_perm=mperm.numpy().astype(np.int32))


def fps_nd_case(ref, name, c):
    """farthest_point_sampling (pix4point.py:8-53) of the UNMODIFIED reference on (B,N,D) points for every D in c['dims']."""
    out = {}
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    for D in c["dims"]:
        pts = synth.make_points_nd(c["B"], c["N"], D, c["seed"])
        with torch.no_grad(), forced_randint([start]):
            r = ref.farthest_point_sampling(torch.from_numpy(pts), c["G"]).numpy()
        assert np.array_equal(oracle.fps_nd(pts, start, c["G"]), r), (name, D)
        sq = np.square(pts - pts[:, :1])
        assert np.array_equal(oracle.torch_row_sum(sq.reshape(-1, D)),
                              torch.sum(torch.from_numpy(sq), -1).numpy().reshape(-1)), (name, D)
        out[f"idx_D{D}"] = r.astype(np.int32)
    print(f"{name}: oracle.fps_nd == reference for D in {c['dims']}; row sums bit-equal to torch.sum")
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)


def head_case(name, c):
    """The reference builds these layers with plain torch.nn (pix4point.py:213-218) and applies them at 245-252; PointViT
    itself cannot be constructed here (timm.create_model), so the same torch.nn modules are evaluated directly."""
    import torch.nn as nn
    sd = synth.token_head_state(c["W"], c["E"], c["seed"])
    tsd = synth.to_torch_state(sd)
    proj = nn.Linear(c["W"], c["E"])
    pos = nn.Sequential(nn.Linear(3, 128, bias=True), nn.GELU(), nn.Linear(128, c["E"]))
    proj.load_state_dict({"weight": tsd["proj.weight"], "bias": tsd["proj.bias"]})
    pos.load_state_dict({"0.weight": tsd["pos_embed.0.weight"], "0.bias": tsd["pos_embed.0.bias"],
                         "2.weight": tsd["pos_embed.2.weight"], "2.bias": tsd["pos_embed.2.bias"]})
    tokens = synth.uniform01(c["seed"], c["B"] * c["G"] * c["W"], 9).reshape(c["B"], c["G"], c["W"])
    centres = synth.make_cloud("uniform", c["B"], c["G"], c["seed"], 3)
    with torch.no_grad():
        x = proj(torch.from_numpy(tokens))
        pe = pos(torch.from_numpy(centres))
        feats = torch.cat([tsd["cls_token"].expand(c["B"], -1, -1), x], dim=1)
        pemb = torch.cat([tsd["cls_pos"].expand(c["B"], -1, -1), pe], dim=1)
    of, op = oracle.token_head(sd, tokens, centres)
    e1 = np.abs(of - feats.numpy()).max() / np.abs(feats.numpy()).max()
    e2 = np.abs(op - pemb.numpy()).max() / np.abs(pemb.numpy()).max()
    print(f"{name}: oracle vs torch.nn head: feats {e1:.2e}, pos {e2:.2e}")
    assert e1 < 2e-6 and e2 < 2e-6, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), feats=feats.numpy(), pos=pemb.numpy())


def vit_case(ref, name, c):
    """The reference's AdaptPointFormer cannot be constructed here (its constructor downloads timm weights,
    src/models/apf.py:319-327), so its forward tail (apf.py:361-371) is evaluated on the reference's own modules:
    apf_utils.APFViTLayer x depth, nn.LayerNorm, max over tokens, apf.ClassificationHead."""
    import torch.nn as nn
    sd = synth.apf_vit_state(c["D"], c["depth"], c["classes"], c["seed"])
    tsd = synth.to_torch_state(sd)
    blocks = nn.Sequential(*[ref.apf_utils.APFViTLayer(dim=c["D"], num_heads=c["heads"], drop_path=0.0, dropout=0.1)
                             for _ in range(c["depth"])]).eval()
    norm = nn.LayerNorm(c["D"]).eval()
    head = ref.apf.ClassificationHead(c["D"], c["classes"]).eval()
    blocks.load_state_dict({k[len("blocks."):]: v for k, v in tsd.items() if k.startswith("blocks.")})
    norm.load_state_dict({k[len("encoder_norm."):]: v for k, v in tsd.items() if k.startswith("encoder_norm.")})
    head.load_state_dict({k[len("head."):]: v for k, v in tsd.items() if k.startswith("head.")})
    tok = synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"])
    with torch.no_grad():
        x = torch.from_numpy(tok)
        for i in range(len(blocks)):
            x = blocks[i](x)
        pooled = norm(x).max(-2)[0]
        logits = head(pooled)
    ox, op, ol = oracle.apf_vit(sd, tok, c["depth"], c["heads"])
    rel = lambda a, b: np.abs(a - b).max() / np.abs(b).max()
    e = (rel(ox, x.numpy()), rel(op, pooled.numpy()), rel(ol, logits.numpy()))
    print(f"{name}: oracle vs reference blocks: x {e[0]:.2e}, pooled {e[1]:.2e}, logits {e[2]:.2e}")
    assert max(e) < 2e-5, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), x=x.numpy(), pooled=pooled.numpy(), logits=logits.numpy())


def p4p_vit_inputs(c):
    """(feats (B,1+G,D), pos (B,1+G,D), state) of a P4P_VIT_CASES entry (shared with the tests)."""
    S = c["G"] + 1
    feats = synth.vit_tokens(c["B"], S, c["D"], c["seed"])
    pos = (0.3 * synth.vit_tokens(c["B"], S, c["D"], c["seed"] + 1000)).astype(np.float32)
    return feats, pos, synth.pointvit_state(c["D"], c["depth"], c["seed"])


def p4p_vit_case(name, c):
    """Pix4Point's blocks are timm `Block`s (pix4point.py:221-228); timm is neither in the reference tree nor installed, so
    the fixture comes from an INDEPENDENT implementation of the same published block - torch.nn.TransformerEncoderLayer
    (norm_first, exact GELU, eps 1e-6, packed q/k/v projection in timm's order) - driven exactly as the reference drives its
    blocks: `feats = blk(feats + pos_embed)` per block, final norm, 'max,cls' features (pix4point.py:254-271)."""
    import torch.nn as nn
    feats, pos, sd = p4p_vit_inputs(c)
    tsd = synth.to_torch_state(sd)
    D, H = c["D"], 4 * c["D"]
    layers = []
    for i in range(c["depth"]):
        l = nn.TransformerEncoderLayer(D, c["heads"], H, dropout=0.0, activation="gelu", layer_norm_eps=1e-6, batch_first=True,
                                       norm_first=True).eval()
        b = f"vit.blocks.{i}."
        l.load_state_dict({"self_attn.in_proj_weight": tsd[b + "attn.qkv.weight"], "self_attn.in_proj_bias": tsd[b + "attn.qkv.bias"],
                           "self_attn.out_proj.weight": tsd[b + "attn.proj.weight"], "self_attn.out_proj.bias": tsd[b + "attn.proj.bias"],
                           "linear1.weight": tsd[b + "mlp.fc1.weight"], "linear1.bias": tsd[b + "mlp.fc1.bias"],
                           "linear2.weight": tsd[b + "mlp.fc2.weight"], "linear2.bias": tsd[b + "mlp.fc2.bias"],
                           "norm1.weight": tsd[b + "norm1.weight"], "norm1.bias": tsd[b + "norm1.bias"],
                           "norm2.weight": tsd[b + "norm2.weight"], "norm2.bias": tsd[b + "norm2.bias"]})
        layers.append(l)
    norm = nn.LayerNorm(D, eps=1e-6).eval()
    norm.load_state_dict({"weight": tsd["vit.norm.weight"], "bias": tsd["vit.norm.bias"]})
    with torch.no_grad():
        x, p = torch.from_numpy(feats), torch.from_numpy(pos)
        for l in layers:
            x = l(x + p)
        x = norm(x)
        glob = torch.cat([x[:, 1:].max(1)[0], x[:, 0]], 1)
    ox, og = oracle.pointvit_blocks(sd, feats, pos, c["depth"], c["heads"])
    e1 = np.abs(ox - x.numpy()).max() / np.abs(x.numpy()).max()
    e2 = np.abs(og - glob.numpy()).max() / np.abs(glob.numpy()).max()
    print(f"{name}: oracle vs torch.nn.TransformerEncoderLayer stack: feats {e1:.2e}, global {e2:.2e}")
    assert max(e1, e2) < 2e-5, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), feats=x.numpy(), glob=glob.numpy())


def p4p_vit_train_case(name, c):
    """torch.nn.TransformerEncoderLayer stack (the independent implementation of timm's Block used by p4p_vit_case) in TRAIN mode
    (dropout 0) under autograd, driven as pix4point.py:254-271: loss = sum(global_features * grad_glob)."""
    import torch.nn as nn
    from oracle import train
    feats, pos, sd = p4p_vit_inputs(c)
    tsd = synth.to_torch_state(sd)
    D, H = c["D"], 4 * c["D"]
    gg = (synth.uniform01(c["seed"], c["B"] * 2 * D, 39).reshape(c["B"], 2 * D) - 0.5).astype(np.float32)
    names = {"self_attn.in_proj_weight": "attn.qkv.weight", "self_attn.in_proj_bias": "attn.qkv.bias",
             "self_attn.out_proj.weight": "attn.proj.weight", "self_attn.out_proj.bias": "attn.proj.bias",
             "linear1.weight": "mlp.fc1.weight", "linear1.bias": "mlp.fc1.bias", "linear2.weight": "mlp.fc2.weight",
             "linear2.bias": "mlp.fc2.bias", "norm1.weight": "norm1.weight", "norm1.bias": "norm1.bias",
             "norm2.weight": "norm2.weight", "norm2.bias": "norm2.bias"}
    layers = []
    for i in range(c["depth"]):
        l = nn.TransformerEncoderLayer(D, c["heads"], H, dropout=0.0, activation="gelu", layer_norm_eps=1e-6, batch_first=True,
                                       norm_first=True).train()
        l.load_state_dict({k: tsd[f"vit.blocks.{i}." + v] for k, v in names.items()})
        layers.append(l)
    norm = nn.LayerNorm(D, eps=1e-6).train()
    norm.load_state_dict({"weight": tsd["vit.norm.weight"], "bias": tsd["vit.norm.bias"]})
    x0, p0 = torch.from_numpy(feats).requires_grad_(True), torch.from_numpy(pos).requires_grad_(True)
    x = x0
    for l in layers:
        x = l(x + p0)
    x = norm(x)
    glob = torch.cat([x[:, 1:].max(1)[0], x[:, 0]], 1)
    (glob * torch.from_numpy(gg)).sum().backward()
    out = {"glob": glob.detach().numpy(), "grad.feats": x0.grad.numpy(), "grad.pos": p0.grad.numpy(),
           "grad.vit.norm.weight": norm.weight.grad.numpy(), "grad.vit.norm.bias": norm.bias.grad.numpy()}
    for i, l in enumerate(layers):
        for k, v in names.items():
            out[f"grad.vit.blocks.{i}.{v}"] = dict(l.named_parameters())[k].grad.numpy()
    og, dx, dp, grads = train.pointvit_backward(sd, feats, pos, c["depth"], c["heads"], gg)
    rel = lambda a, b: np.abs(np.asarray(a).reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-30)
    worst = max(rel(og, out["glob"]), rel(dx, out["grad.feats"]), rel(dp, out["grad.pos"]))
    scale = max(np.abs(v).max() for k_, v in out.items() if k_.endswith("weight") and v.ndim == 2)
    for n, v in grads.items():
        worst = max(worst, np.abs(v.reshape(out["grad." + n].shape) - out["grad." + n]).max() / scale)
    print(f"{name}: oracle/train.py pointvit_backward vs torch.nn.TransformerEncoderLayer autograd: worst error {worst:.2e}")
    assert worst < 1e-5, name
    small = {}
    for k_, v in out.items():
        if v.size > 5000:
            m = v.reshape(v.shape[0], -1)
            small[k_ + "#rowsum"] = m.sum(1)
            small[k_ + "#colsum"] = m.sum(0)
        else:
            small[k_] = v
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **small)


def train_inputs(c):
    """(neigh (B,G,k,2C) f32, grad_tokens (B,G,E) f32, encoder state) of a TRAIN_CASES entry (shared with the tests)."""
    x = synth.make_cloud("uniform", c["B"], c["N"], c["seed"], c["C"])
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    sd = synth.apf_encoder_state(c["E"], 2 * c["C"], c["seed"])
    neigh = oracle.group_apf(x, start, c["G"], c["k"])["neigh"].astype(np.float32)
    gt = (synth.uniform01(c["seed"], c["B"] * c["G"] * c["E"], 31).reshape(c["B"], c["G"], c["E"]) - 0.5).astype(np.float32)
    return neigh, gt, sd


def train_case(ref, name, c):
    """Reference Encoder in TRAIN mode (apf.py:114-181): forward with batch statistics, loss = sum(tokens * grad_tokens),
    autograd.  Stores what the reference returned; asserts oracle/train.py against it."""
    from oracle import train
    neigh, gt, sd = train_inputs(c)
    enc = ref.Encoder(c["E"], 2 * c["C"]).train()
    enc.load_state_dict(synth.to_torch_state(sd))
    xt = torch.from_numpy(neigh).requires_grad_(True)
    tok = enc(xt)
    (tok * torch.from_numpy(gt)).sum().backward()
    out = {"tokens": tok.detach().numpy(), "grad.input": xt.grad.numpy()}
    for n, p_ in enc.named_parameters():
        out["grad." + n] = p_.grad.numpy()
    for n, b in enc.named_buffers():
        if "num_batches" not in n:
            out["running." + n] = b.numpy()
    tk, grads, running = train.apf_encoder_train(sd, neigh, gt)
    scale = max(np.abs(v).max() for k_, v in out.items() if k_.startswith("grad.") and k_.endswith("weight"))
    worst = np.abs(tk - out["tokens"]).max() / np.abs(out["tokens"]).max()
    for n, v in grads.items():
        worst = max(worst, np.abs(v.reshape(out["grad." + n].shape) - out["grad." + n]).max() / scale)
    for n, v in running.items():
        worst = max(worst, np.abs(v - out["running." + n]).max() / np.abs(out["running." + n]).max())
    print(f"{name}: oracle/train.py vs reference autograd: worst error {worst:.2e}")
    assert worst < 1e-5, name
    # keep the fixture small: matrices above 20 k elements are stored as their row sums and column sums
    small = {}
    for k_, v in out.items():
        if v.size > 20000:
            m = v.reshape(v.shape[0], -1)
            small[k_ + "#rowsum"] = m.sum(1)
            small[k_ + "#colsum"] = m.sum(0)
        else:
            small[k_] = v
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **small)


def p4p_train_inputs(c):
    x = synth.make_cloud("uniform", c["B"], c["N"], c["seed"], 3)
    start = synth.start_indices(c["B"], c["N"], c["seed"], 0)
    sd = synth.p3embed_state(3, 0.25, 4, 4, c["W"], c["seed"])
    G = c["N"] // 4
    go = (synth.uniform01(c["seed"], c["B"] * G * c["W"], 33).reshape(c["B"], G, c["W"]) - 0.5).astype(np.float32)
    return x, start, sd, go


def p4p_train_case(ref, name, c):
    """Reference P3Embed.forward in TRAIN mode (pix4point.py:166-191, 1 stage) + autograd; loss = sum(out * grad_out)."""
    from oracle import train
    x, start, sd, go = p4p_train_inputs(c)
    m = ref.P3Embed(in_channels=3, sample_ratio=0.25, scale=4, k=c["k"], layers=4, embed_dim=c["W"]).train()
    m.load_state_dict(synth.to_torch_state(sd))
    p = torch.from_numpy(x).requires_grad_(True)
    fe = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).requires_grad_(True)
    with forced_randint([start]):
        _, fs = m(p, fe)
    (fs[-1].transpose(1, 2) * torch.from_numpy(go)).sum().backward()
    out = {"out": fs[-1].detach().transpose(1, 2).numpy(), "grad.p": p.grad.numpy(), "grad.f": fe.grad.transpose(1, 2).numpy()}
    for n, q in m.named_parameters():
        out["grad." + n] = q.grad.numpy()
    for n, b in m.named_buffers():
        if "num_batches" not in n:
            out["running." + n] = b.numpy()
    _, _, _, kidx = oracle.p3embed_stage(sd, 0, x, x.copy(), start, c["k"])
    rows = np.concatenate([oracle.gather_points(x, kidx), oracle.gather_points(x, kidx)], -1)
    o, grads, running = train.p3embed_stage_train(sd, 0, rows, go)
    dp, df = train.scatter_rows_grad(grads["rows"], kidx, c["N"])
    scale = max(np.abs(v).max() for k_, v in out.items() if k_.startswith("grad.convs") and k_.endswith("weight"))
    worst = max(np.abs(o - out["out"]).max() / np.abs(out["out"]).max(), np.abs(dp - out["grad.p"]).max() / np.abs(out["grad.p"]).max(),
                np.abs(df - out["grad.f"]).max() / np.abs(out["grad.f"]).max())
    for n, v in grads.items():
        if n != "rows":
            worst = max(worst, np.abs(v.reshape(out["grad." + n].shape) - out["grad." + n]).max() / scale)
    for n, v in running.items():
        worst = max(worst, np.abs(v - out["running." + n]).max() / np.abs(out["running." + n]).max())
    print(f"{name}: oracle/train.py vs reference P3Embed autograd: worst error {worst:.2e}")
    assert worst < 1e-5, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)


def vit_train_case(ref, name, c):
    """The reference's APFViTLayer stack (dropout / DropPath at 0: they are random in train mode) + nn.LayerNorm + max over
    tokens (apf.py:361-366) under autograd: gradient of sum(pooled * grad_pooled) w.r.t. the tokens and the encoder_norm."""
    import torch.nn as nn
    from oracle import train
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
    tsd = synth.to_torch_state(sd)
    blocks = nn.Sequential(*[ref.apf_utils.APFViTLayer(dim=c["D"], num_heads=c["heads"], drop_path=0.0, dropout=0.0)
                             for _ in range(c["depth"])]).train()
    blocks.load_state_dict({k[len("blocks."):]: v for k, v in tsd.items() if k.startswith("blocks.")})
    norm = nn.LayerNorm(c["D"]).train()
    norm.load_state_dict({"weight": tsd["encoder_norm.weight"], "bias": tsd["encoder_norm.bias"]})
    tok = synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"])
    gp = (synth.uniform01(c["seed"], c["B"] * c["D"], 35).reshape(c["B"], c["D"]) - 0.5).astype(np.float32)
    x = torch.from_numpy(tok).requires_grad_(True)
    h = x
    for i in range(c["depth"]):
        h = blocks[i](h)
    pooled = norm(h).max(-2)[0]
    (pooled * torch.from_numpy(gp)).sum().backward()
    po, dx, g = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], gp)
    rel = lambda a, b: np.abs(a - b).max() / np.abs(b).max()
    worst = max(rel(po, pooled.detach().numpy()), rel(dx, x.grad.numpy()), rel(g["encoder_norm.weight"], norm.weight.grad.numpy()),
                rel(g["encoder_norm.bias"], norm.bias.grad.numpy()))
    print(f"{name}: oracle/train.py vs reference autograd through the block stack: worst error {worst:.2e}")
    assert worst < 1e-5, name
    np.savez_compressed(os.path.join(HERE, name + ".npz"), pooled=pooled.detach().numpy(), grad_tokens=x.grad.numpy(),
                        grad_norm_w=norm.weight.grad.numpy(), grad_norm_b=norm.bias.grad.numpy())


def vit_full_train_inputs(c):
    """(state, tokens (B,G,D), grad_logits (B,classes), masks) of a VIT_FULL_TRAIN_CASES entry (shared with the tests).
    masks = dict(adapter=[(B*G, 64) per layer], pool=(B,D), head=((B,512), (B,256))) keep masks scaled by 1 / keep, or None."""
    sd = synth.apf_vit_state(c["D"], c["depth"], c["classes"], c["seed"])
    tok = synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"])
    gl = (synth.uniform01(c["seed"], c["B"] * c["classes"], 37).reshape(c["B"], c["classes"]) - 0.5).astype(np.float32)

    def keep(shape, p, stream):
        if p <= 0:
            return None
        u = synth.uniform01(c["seed"], int(np.prod(shape)), stream).reshape(shape)
        return ((u >= p).astype(np.float32) / np.float32(1.0 - p)).astype(np.float32)

    masks = dict(adapter=[keep((c["B"] * c["G"], 64), c["p_adapter"], 41 + i) for i in range(c["depth"])],
                 pool=keep((c["B"], c["D"]), c["p_pool"], 61), head=(keep((c["B"], 512), c["p_head"], 62), keep((c["B"], 256), c["p_head"], 63)))
    return sd, tok, gl, masks


@contextlib.contextmanager
def forced_dropout(masks):
    """torch.nn.functional.dropout (what nn.Dropout and the reference's adapter call, apf_utils.py:223) multiplies by the next
    forced keep mask instead of drawing one; a None entry means "dropout off" for that call."""
    import torch.nn.functional as F
    real = F.dropout
    it = iter(masks)

    def fake(input, p=0.5, training=True, inplace=False):
        m = next(it)
        if m is None:
            return input
        return input * torch.from_numpy(np.asarray(m)).reshape(input.shape)

    F.dropout = fake
    try:
        yield
    finally:
        F.dropout = real


def vit_full_train_case(ref, name, c):
    """The reference's APFViTLayer stack + nn.LayerNorm + max over tokens + nn.Dropout + ClassificationHead (apf.py:219-252,
    358-371) in TRAIN mode under autograd, every parameter asking for a gradient; dropout draws replaced by forced keep masks
    (DropPath is a timm class, absent here - its masks are exercised against the oracle only)."""
    import torch.nn as nn
    from oracle import train
    sd, tok, gl, masks = vit_full_train_inputs(c)
    tsd = synth.to_torch_state(sd)
    blocks = nn.Sequential(*[ref.apf_utils.APFViTLayer(dim=c["D"], num_heads=c["heads"], drop_path=0.0, dropout=max(c["p_adapter"], 0.0))
                             for _ in range(c["depth"])]).train()
    blocks.load_state_dict({k[len("blocks."):]: v for k, v in tsd.items() if k.startswith("blocks.")})
    norm = nn.LayerNorm(c["D"]).train()
    norm.load_state_dict({"weight": tsd["encoder_norm.weight"], "bias": tsd["encoder_norm.bias"]})
    drop = nn.Dropout(0.1).train()
    head = ref.apf.ClassificationHead(c["D"], c["classes"]).train()
    head.load_state_dict({k[len("head."):]: v for k, v in tsd.items() if k.startswith("head.")})
    x = torch.from_numpy(tok).requires_grad_(True)
    order = list(masks["adapter"]) + [masks["pool"], masks["head"][0], masks["head"][1]]
    with forced_dropout(order):
        h = x
        for i in range(c["depth"]):
            h = blocks[i](h)
        pooled = norm(h).max(-2)[0]
        logits = head(drop(pooled))
    (logits * torch.from_numpy(gl)).sum().backward()
    out = {"logits": logits.detach().numpy(), "pooled": pooled.detach().numpy(), "grad.tokens": x.grad.numpy()}
    for n, p_ in blocks.named_parameters():
        out["grad.blocks." + n] = p_.grad.numpy()
    for n, p_ in norm.named_parameters():
        out["grad.encoder_norm." + n] = p_.grad.numpy()
    for n, p_ in head.named_parameters():
        out["grad.head." + n] = p_.grad.numpy()
    for n, b in head.named_buffers():
        if "num_batches" not in n:
            out["running.head." + n] = b.numpy()
    # the oracle, held to the reference
    lm = [(None, masks["adapter"][i], None) for i in range(c["depth"])]
    po, _, _ = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], np.zeros((c["B"], c["D"])), lm)
    pin = po * (1.0 if masks["pool"] is None else masks["pool"])
    lo, hg, run = train.head_train(sd, pin, gl, masks["head"])
    dpool = hg.pop("input") * (1.0 if masks["pool"] is None else masks["pool"])
    _, dx, bg = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], dpool, lm, param_grads=True)
    rel = lambda a, b: np.abs(np.asarray(a).reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-30)
    worst = max(rel(lo, out["logits"]), rel(po, out["pooled"]), rel(dx, out["grad.tokens"]))
    scale = max(np.abs(v).max() for k_, v in out.items() if k_.startswith("grad.") and k_.endswith("weight") and v.ndim == 2)
    for n, v in list(bg.items()) + list(hg.items()):
        worst = max(worst, np.abs(v.reshape(out["grad." + n].shape) - out["grad." + n]).max() / scale)
    for n, v in run.items():
        worst = max(worst, rel(v, out["running." + n]))
    print(f"{name}: oracle/train.py vs reference autograd (blocks + encoder_norm + head, train mode): worst error {worst:.2e}")
    assert worst < 1e-5, name
    small = {}
    for k_, v in out.items():                      # matrices above 5 k elements are stored as their row sums and column sums
        if v.size > 5000:
            m = v.reshape(v.shape[0], -1)
            small[k_ + "#rowsum"] = m.sum(1)
            small[k_ + "#colsum"] = m.sum(0)
        else:
            small[k_] = v
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **small)


def main():
    """python tests/golden/make_golden.py [case names ...]  (no names: every case)."""
    assert ref_loader.available(), "reference tree not present"
    ref = ref_loader.load()
    torch.set_num_threads(os.cpu_count() or 1)
    only = set(sys.argv[1:])
    want = lambda name: not only or name in only
    for name, c in cases.INDEX_CASES.items():
        if want(name): index_case(ref, name, c)
    for name, c in cases.FPS_ND_CASES.items():
        if want(name): fps_nd_case(ref, name, c)
    for name, c in cases.APF_CASES.items():
        if want(name): apf_case(ref, name, c)
    for name, c in cases.P4P_CASES.items():
        if want(name): p4p_case(ref, name, c)
    for name, c in cases.HEAD_CASES.items():
        if want(name): head_case(name, c)
    for name, c in cases.VIT_CASES.items():
        if want(name): vit_case(ref, name, c)
    for name, c in cases.P4P_VIT_CASES.items():
        if want(name): p4p_vit_case(name, c)
    for name, c in cases.TRAIN_CASES.items():
        if want(name): train_case(ref, name, c)
    for name, c in cases.P4P_TRAIN_CASES.items():
        if want(name): p4p_train_case(ref, name, c)
    for name, c in cases.VIT_TRAIN_CASES.items():
        if want(name): vit_train_case(ref, name, c)
    for name, c in cases.VIT_FULL_TRAIN_CASES.items():
        if want(name): vit_full_train_case(ref, name, c)
    for name, c in cases.P4P_VIT_TRAIN_CASES.items():
        if want(name): p4p_vit_train_case(name, c)


if __name__ == "__main__":
    main()
