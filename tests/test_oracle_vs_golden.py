"""The oracle against the committed golden vectors (outputs of the reference itself, made by
tests/golden/make_golden.py).  Runs anywhere - no GPU, no reference tree."""
import os

import numpy as np
import pytest

import cases
from oracle import oracle
from p3tok import synth


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


@pytest.mark.parametrize("name", list(cases.INDEX_CASES))
def test_index_cases(golden_dir, name):
    c = cases.INDEX_CASES[name]
    g = _load(golden_dir, name)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    fidx = oracle.fps(x, start, c["G"])
    assert np.array_equal(fidx, g["fps_idx"])          # bit-exact incl. lowest-index ties
    ctr = oracle.gather_points(x, fidx)
    for mode, key, ulp in ((oracle.KNN_APF_SQ, "knn_apf", 0), (oracle.KNN_P4P_CDIST, "knn_p4p", 1)):
        D = oracle.pair_dist(x, ctr, mode)
        mine = oracle.knn(x, ctr, c["k"], mode)
        ok, msg = oracle.knn_tie_equivalent(mine, g[key].astype(np.int64), D, ulp=ulp)
        assert ok, msg
        assert oracle.sorted_by_distance(mine, D, 0)
    assert oracle.sorted_by_distance(g["knn_p4p"].astype(np.int64),
                                     oracle.pair_dist(x, ctr, oracle.KNN_P4P_CDIST), 1)
    codes, perm = oracle.morton(ctr)
    ref_perm = g["morton_perm"].astype(np.int64)
    assert np.array_equal(np.take_along_axis(codes, ref_perm, 1), np.take_along_axis(codes, perm, 1))


@pytest.mark.parametrize("name", list(cases.FPS_ND_CASES))
def test_fps_nd_cases(golden_dir, name):
    """General-D farthest_point_sampling (pix4point.py:8-53): the oracle reproduces the reference's picks for every D of
    the fixture, and for D = 3 the general restatement equals the xyz one."""
    c = cases.FPS_ND_CASES[name]
    g = _load(golden_dir, name)
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    for D in c["dims"]:
        pts = synth.make_points_nd(c["B"], c["N"], D, c["seed"])
        assert np.array_equal(oracle.fps_nd(pts, start, c["G"]), g[f"idx_D{D}"]), D
    p3 = synth.make_points_nd(c["B"], c["N"], 3, c["seed"])
    assert np.array_equal(oracle.fps_nd(p3, start, c["G"]), oracle.fps(p3, start, c["G"]))


def test_torch_row_sum_is_torchs_cpu_order():
    """The summation order the general-D FPS is held to (p3tok_oracle.c: torch_cpu_row_sum) IS torch.sum's on this host,
    bit for bit, for every D up to 32 - and it is NOT the left-to-right sum from D = 5 on (except D = 8), which is why the
    kernel spells the order out."""
    import torch
    if torch.backends.cpu.get_cpu_capability() not in ("AVX2", "AVX512"):
        pytest.skip("torch's CPU sum kernel has another vector width on this host")
    rng = np.random.default_rng(5)
    differs = []
    for D in range(1, 33):
        q = np.square(rng.standard_normal((4096, D)).astype(np.float32))
        mine = oracle.torch_row_sum(q)
        assert np.array_equal(mine, torch.sum(torch.from_numpy(q), -1).numpy()), D
        seq = q[:, 0].copy()
        for a in range(1, D):
            seq = (seq + q[:, a]).astype(np.float32)
        if not np.array_equal(seq, mine):
            differs.append(D)
    assert differs == [d for d in range(5, 33) if d != 8]


@pytest.mark.parametrize("name", list(cases.APF_CASES))
def test_apf_cases(golden_dir, name):
    c = cases.APF_CASES[name]
    g = _load(golden_dir, name)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], c["C"])
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    sd = synth.apf_encoder_state(c["E"], 2 * c["C"], c["seed"])
    tok, grp = oracle.pointnet_apf(sd, x, start, c["G"], c["k"])
    assert np.array_equal(grp["fps_idx"], g["fps_idx"])
    D = oracle.pair_dist(x, oracle.gather_points(x[..., :3], grp["fps_idx"]), oracle.KNN_APF_SQ)
    ok, msg = oracle.knn_tie_equivalent(grp["knn_idx"], g["knn_idx"].astype(np.int64), D, 0)
    assert ok, msg
    assert np.array_equal(grp["center"], g["center"])
    if g["neigh"].size:
        # same multiset of rows per group (reference order is topk(sorted=False)-arbitrary)
        a = np.sort(grp["neigh"].reshape(c["B"] * c["G"], c["k"], -1), axis=1)
        b = np.sort(g["neigh"].reshape(c["B"] * c["G"], c["k"], -1), axis=1)
        if "dups" not in name:
            assert np.array_equal(np.sort(a.sum(-1), 1), np.sort(b.sum(-1), 1))
    ref = g["tokens"].astype(np.float64)
    assert np.abs(tok - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.mark.parametrize("name", list(cases.P4P_CASES))
def test_p4p_cases(golden_dir, name):
    c = cases.P4P_CASES[name]
    g = _load(golden_dir, name)
    stages, dims = synth.p3embed_dims(3, c["sample_ratio"], 4, 4, c["embed_dim"])
    sd = synth.p3embed_state(3, c["sample_ratio"], 4, 4, c["embed_dim"], c["seed"])
    pts = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    feats = pts.copy()
    n = c["N"]
    for s in range(stages):
        start = synth.start_indices(c["B"], n, c["seed"], s)
        ctr, tok, fidx, kidx = oracle.p3embed_stage(sd, s, pts, feats, start, c["k"])
        assert np.array_equal(fidx, g[f"fps_idx{s}"])
        assert np.array_equal(ctr, g[f"centres{s}"])
        D = oracle.pair_dist(pts, ctr, oracle.KNN_P4P_CDIST)
        ok, msg = oracle.knn_tie_equivalent(kidx, g[f"knn_idx{s}"].astype(np.int64), D, 1)
        assert ok, msg
        ref = g[f"tokens{s}"].astype(np.float64)
        assert tok.shape == ref.shape == (c["B"], n // 4, dims[s][1])
        assert np.abs(tok - ref).max() <= 2e-5 * np.abs(ref).max()
        # next stage consumes the reference's fp32 outputs (as make_golden.py did)
        pts, feats = g[f"centres{s}"], g[f"tokens{s}"]
        n //= 4


@pytest.mark.parametrize("name", list(cases.HEAD_CASES))
def test_token_head_cases(golden_dir, name):
    """Pix4Point token head (SURVEY 8f next #1): oracle against the torch.nn evaluation stored by make_golden.py."""
    c = cases.HEAD_CASES[name]
    g = _load(golden_dir, name)
    sd = synth.token_head_state(c["W"], c["E"], c["seed"])
    tokens = synth.uniform01(c["seed"], c["B"] * c["G"] * c["W"], 9).reshape(c["B"], c["G"], c["W"])
    centres = synth.make_cloud("uniform", c["B"], c["G"], c["seed"], 3)
    feats, pos = oracle.token_head(sd, tokens, centres)
    assert feats.shape == g["feats"].shape == (c["B"], c["G"] + 1, c["E"])
    assert np.abs(feats - g["feats"]).max() <= 2e-6 * np.abs(g["feats"]).max()
    assert np.abs(pos - g["pos"]).max() <= 2e-6 * np.abs(g["pos"]).max()
    assert np.array_equal(feats[:, 0], np.broadcast_to(sd["cls_token"].reshape(1, -1), (c["B"], c["E"])).astype(np.float64))


@pytest.mark.parametrize("name", list(cases.VIT_CASES))
def test_vit_cases(golden_dir, name):
    """oracle.apf_vit against the reference's own APFViTLayer / LayerNorm / ClassificationHead outputs."""
    c = cases.VIT_CASES[name]
    g = _load(golden_dir, name)
    sd = synth.apf_vit_state(c["D"], c["depth"], c["classes"], c["seed"])
    tok = synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"])
    x, pooled, logits = oracle.apf_vit(sd, tok, c["depth"], c["heads"])
    for mine, key in ((x, "x"), (pooled, "pooled"), (logits, "logits")):
        ref = g[key].astype(np.float64)
        assert np.abs(mine - ref).max() <= 2e-5 * np.abs(ref).max(), key


@pytest.mark.parametrize("name", ["vit_small", "vit_hd64"])
def test_vit_port_matches_golden(golden_dir, name):
    """oracle/port.py's torch-CPU restatement of the block stack (the timed CPU baseline of bench.py --workload c2v)."""
    import torch
    from oracle import port
    c = cases.VIT_CASES[name]
    g = _load(golden_dir, name)
    sd = synth.to_torch_state(synth.apf_vit_state(c["D"], c["depth"], c["classes"], c["seed"]))
    tok = torch.from_numpy(synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"]))
    with torch.no_grad():
        pooled = port.apf_vit_features(sd, tok, c["depth"], c["heads"]).numpy()
    assert np.abs(pooled - g["pooled"]).max() <= 1e-5 * np.abs(g["pooled"]).max()


@pytest.mark.parametrize("name", list(cases.TRAIN_CASES))
def test_train_mode_oracle(golden_dir, name):
    """Groundwork for SURVEY 8f next #4: oracle/train.py (batch-statistics BN forward + backward through both max-pools)
    against what the reference Encoder's own autograd returned."""
    from oracle import train
    c = cases.TRAIN_CASES[name]
    g = _load(golden_dir, name)
    x = synth.make_cloud("uniform", c["B"], c["N"], c["seed"], c["C"])
    start = synth.start_indices(c["B"], c["N"], c["seed"])
    sd = synth.apf_encoder_state(c["E"], 2 * c["C"], c["seed"])
    neigh = oracle.group_apf(x, start, c["G"], c["k"])["neigh"].astype(np.float32)
    gt = (synth.uniform01(c["seed"], c["B"] * c["G"] * c["E"], 31).reshape(c["B"], c["G"], c["E"]) - 0.5).astype(np.float32)
    tokens, grads, running = train.apf_encoder_train(sd, neigh, gt)
    assert np.abs(tokens - g["tokens"]).max() <= 1e-5 * np.abs(g["tokens"]).max()
    scale = max(np.abs(g[k_]).max() for k_ in g.files if k_.startswith("grad.") and k_.endswith("weight"))
    for n, v in grads.items():                      # biases in front of a BatchNorm have (numerically) zero gradient
        if "grad." + n in g.files:
            ref = g["grad." + n]
            assert np.abs(v.reshape(ref.shape) - ref).max() <= 1e-5 * scale, n
        else:                                       # large matrices are stored as row sums and column sums
            m = v.reshape(v.shape[0], -1)
            for proj, mine in (("#rowsum", m.sum(1)), ("#colsum", m.sum(0))):
                ref = g["grad." + n + proj]
                assert np.abs(mine - ref).max() <= 1e-5 * max(np.abs(ref).max(), scale), n + proj
    for n, v in running.items():
        assert np.abs(v - g["running." + n]).max() <= 1e-5 * np.abs(g["running." + n]).max(), n


@pytest.mark.parametrize("name", list(cases.P4P_TRAIN_CASES))
def test_p3embed_train_mode_oracle(golden_dir, name):
    """oracle/train.py's P3Embed stage (train-mode BN, backward through both pools, the concat and the gather) against the
    reference P3Embed.forward + autograd."""
    from oracle import train
    c = cases.P4P_TRAIN_CASES[name]
    g = _load(golden_dir, name)
    x = synth.make_cloud("uniform", c["B"], c["N"], c["seed"], 3)
    start = synth.start_indices(c["B"], c["N"], c["seed"], 0)
    sd = synth.p3embed_state(3, 0.25, 4, 4, c["W"], c["seed"])
    G = c["N"] // 4
    go = (synth.uniform01(c["seed"], c["B"] * G * c["W"], 33).reshape(c["B"], G, c["W"]) - 0.5).astype(np.float32)
    _, _, _, kidx = oracle.p3embed_stage(sd, 0, x, x.copy(), start, c["k"])
    rows = np.concatenate([oracle.gather_points(x, kidx), oracle.gather_points(x, kidx)], -1)
    out, grads, running = train.p3embed_stage_train(sd, 0, rows, go)
    dp, df = train.scatter_rows_grad(grads["rows"], kidx, c["N"])
    for mine, key in ((out, "out"), (dp, "grad.p"), (df, "grad.f")):
        assert np.abs(mine - g[key]).max() <= 1e-5 * np.abs(g[key]).max(), key
    scale = max(np.abs(g[k_]).max() for k_ in g.files if k_.startswith("grad.convs") and k_.endswith("weight"))
    for n, v in grads.items():
        if n != "rows":
            assert np.abs(v.reshape(g["grad." + n].shape) - g["grad." + n]).max() <= 1e-5 * scale, n
    for n, v in running.items():
        assert np.abs(v - g["running." + n]).max() <= 1e-5 * np.abs(g["running." + n]).max(), n


@pytest.mark.parametrize("name", list(cases.VIT_TRAIN_CASES))
def test_vit_backward_oracle(golden_dir, name):
    """oracle/train.py::apf_vit_backward (dX through the frozen block stack, encoder_norm gradients) against the reference
    modules' autograd."""
    from oracle import train
    c = cases.VIT_TRAIN_CASES[name]
    g = _load(golden_dir, name)
    sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
    tok = synth.vit_tokens(c["B"], c["G"], c["D"], c["seed"])
    gp = (synth.uniform01(c["seed"], c["B"] * c["D"], 35).reshape(c["B"], c["D"]) - 0.5).astype(np.float32)
    pooled, dx, gn = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], gp)
    for mine, key in ((pooled, "pooled"), (dx, "grad_tokens"), (gn["encoder_norm.weight"], "grad_norm_w"),
                      (gn["encoder_norm.bias"], "grad_norm_b")):
        assert np.abs(mine - g[key]).max() <= 1e-5 * np.abs(g[key]).max(), key


@pytest.mark.parametrize("name", list(cases.VIT_FULL_TRAIN_CASES))
def test_full_consumer_train_oracle(golden_dir, name):
    """oracle/train.py - block stack with EVERY parameter gradient, forced dropout masks, encoder_norm, token max and the
    train-mode ClassificationHead (batch-statistics BatchNorm1d) - against the reference modules' autograd."""
    import make_golden
    from oracle import train
    c = cases.VIT_FULL_TRAIN_CASES[name]
    g = _load(golden_dir, name)
    sd, tok, gl, masks = make_golden.vit_full_train_inputs(c)
    lm = [(None, masks["adapter"][i], None) for i in range(c["depth"])]
    pm = 1.0 if masks["pool"] is None else masks["pool"]
    po, _, _ = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], np.zeros((c["B"], c["D"])), lm)
    lo, hg, run = train.head_train(sd, po * pm, gl, masks["head"])
    _, dx, bg = train.apf_vit_backward(sd, tok, c["depth"], c["heads"], hg.pop("input") * pm, lm, param_grads=True)
    rel = lambda a, b: np.abs(np.asarray(a).reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-30)
    assert rel(lo, g["logits"]) <= 1e-5 and rel(po, g["pooled"]) <= 1e-5 and rel(dx, g["grad.tokens"]) <= 1e-5
    scale = max(np.abs(g[k]).max() for k in g.files if k.startswith("grad.") and k.endswith("weight") and g[k].ndim == 2)
    for n, v in list(bg.items()) + list(hg.items()):
        key = "grad." + n
        if key in g.files:
            assert np.abs(v.reshape(g[key].shape) - g[key]).max() <= 1e-5 * scale, n
        else:
            m = v.reshape(v.shape[0], -1)
            assert np.abs(m.sum(1) - g[key + "#rowsum"]).max() <= 1e-5 * scale * m.shape[1] ** 0.5, n
            assert np.abs(m.sum(0) - g[key + "#colsum"]).max() <= 1e-5 * scale * m.shape[0] ** 0.5, n
    for n, v in run.items():
        assert rel(v, g["running." + n]) <= 1e-5, n


@pytest.mark.parametrize("name", list(cases.P4P_VIT_TRAIN_CASES))
def test_pointvit_backward_oracle(golden_dir, name):
    """oracle/train.py::pointvit_backward (Pix4Point's block loop under autograd: feats, pos, every parameter) against the
    torch.nn.TransformerEncoderLayer-autograd fixture."""
    import make_golden
    from oracle import train
    c = cases.P4P_VIT_TRAIN_CASES[name]
    g = _load(golden_dir, name)
    feats, pos, sd = make_golden.p4p_vit_inputs(c)
    gg = (synth.uniform01(c["seed"], c["B"] * 2 * c["D"], 39).reshape(c["B"], 2 * c["D"]) - 0.5).astype(np.float32)
    og, dx, dp, grads = train.pointvit_backward(sd, feats, pos, c["depth"], c["heads"], gg)
    rel = lambda a, b: np.abs(np.asarray(a).reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-30)
    assert rel(og, g["glob"]) <= 1e-5
    scale = max(np.abs(v).max() for k, v in grads.items() if k.endswith("weight") and v.ndim == 2)
    for n, v in list(grads.items()) + [("feats", dx), ("pos", dp)]:
        key = "grad." + n
        sc = scale if n not in ("feats", "pos") else np.abs(v).max()
        if key in g.files:
            assert np.abs(v.reshape(g[key].shape) - g[key]).max() <= 1e-5 * sc, n
        else:
            m = v.reshape(v.shape[0], -1)
            assert np.abs(m.sum(1) - g[key + "#rowsum"]).max() <= 1e-5 * sc * m.shape[1] ** 0.5, n
            assert np.abs(m.sum(0) - g[key + "#colsum"]).max() <= 1e-5 * sc * m.shape[0] ** 0.5, n


@pytest.mark.parametrize("name", list(cases.P4P_VIT_CASES))
def test_pointvit_block_oracle_matches_golden(golden_dir, name):
    """oracle.pointvit_blocks (timm Block restated, pix4point.py:254-271) against the fixture an independent implementation of the
    same block (torch.nn.TransformerEncoderLayer) produced in make_golden.py."""
    import make_golden
    c = cases.P4P_VIT_CASES[name]
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    feats, pos, sd = make_golden.p4p_vit_inputs(c)
    ox, og = oracle.pointvit_blocks(sd, feats, pos, c["depth"], c["heads"])
    assert np.abs(ox - g["feats"]).max() <= 2e-5 * np.abs(g["feats"]).max()
    assert np.abs(og - g["glob"]).max() <= 2e-5 * np.abs(g["glob"]).max()


@pytest.mark.parametrize("name", list(cases.INDEX_CASES))
def test_port_index_ops_match_golden(golden_dir, name):
    """oracle/port.py's FPS (both update forms) and kNN (both distance forms) against the reference's stored picks; the
    port's expanded squared distance equals the oracle's arithmetic spec."""
    import torch
    from oracle import port
    c = cases.INDEX_CASES[name]
    g = _load(golden_dir, name)
    x = synth.make_cloud(c["kind"], c["B"], c["N"], c["seed"], 3)
    st = torch.from_numpy(synth.start_indices(c["B"], c["N"], c["seed"]))
    xt = torch.from_numpy(x)
    f = torch.from_numpy(g["fps_idx"].astype(np.int64))
    assert torch.equal(port.fps_indices(xt, c["G"], st), f)
    assert torch.equal(port.fps_indices(xt, c["G"], st, masked_update=True), f)
    ctr = port.take(xt, f)
    d_sq = oracle.pair_dist(x, ctr.numpy(), oracle.KNN_APF_SQ)
    assert np.array_equal(d_sq, port.sq_dist_expanded(ctr, xt).numpy())
    ok, msg = oracle.knn_tie_equivalent(port.knn_apf(c["k"], xt, ctr).numpy(), g["knn_apf"].astype(np.int64), d_sq, ulp=0)
    assert ok, msg
    d_cd = oracle.pair_dist(x, ctr.numpy(), oracle.KNN_P4P_CDIST)
    ok, msg = oracle.knn_tie_equivalent(port.knn_p4p(c["k"], xt, ctr).numpy().astype(np.int64),
                                        g["knn_p4p"].astype(np.int64), d_cd, ulp=1)
    assert ok, msg


@pytest.mark.parametrize("D", cases.FPS_ND_CASES["fps_nd"]["dims"])
def test_port_fps_nd_matches_golden(golden_dir, D):
    """oracle/port.py's farthest_point_sampling loop on D-dimensional points against the reference's stored picks."""
    import torch
    from oracle import port
    c = cases.FPS_ND_CASES["fps_nd"]
    pts = synth.make_points_nd(c["B"], c["N"], D, c["seed"])
    st = synth.start_indices(c["B"], c["N"], c["seed"])
    with torch.no_grad():
        r = port.fps_indices(torch.from_numpy(pts), c["G"], torch.from_numpy(st), masked_update=True)
    assert np.array_equal(r.numpy(), _load(golden_dir, "fps_nd")[f"idx_D{D}"])


@pytest.mark.parametrize("name", ["p4p_2stage", "p4p_2stage_k32"])
def test_p3embed_port_matches_golden(golden_dir, name):
    """oracle/port.py's two-stage P3Embed against the reference's stored centres and tokens (both stages chained)."""
    import torch
    from oracle import port
    c = cases.P4P_CASES[name]
    g = _load(golden_dir, name)
    B, N = c["B"], c["N"]
    x = torch.from_numpy(synth.make_cloud(c["kind"], B, N, c["seed"], 3))
    sd = synth.to_torch_state(synth.p3embed_state(3, c["sample_ratio"], 4, 4, c["embed_dim"], c["seed"]))
    st = [torch.from_numpy(synth.start_indices(B, N, c["seed"], 0)), torch.from_numpy(synth.start_indices(B, N // 4, c["seed"], 1))]
    with torch.no_grad():
        pp, pf = port.p3embed(sd, x, x.transpose(1, 2).contiguous(), c["k"], 2, st)
    for s in range(2):
        assert np.array_equal(pp[s + 1].numpy(), g[f"centres{s}"])
        ref = g[f"tokens{s}"]
        assert np.abs(pf[s + 1].transpose(1, 2).numpy() - ref).max() <= 1e-6 * np.abs(ref).max()
