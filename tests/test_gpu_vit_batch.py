"""The ViT block stacks at serving batch sizes.

tests/test_gpu_vit.py checks the stacks on at most 3 clouds (M <= 392 rows, <= 24 attention items).  At serving batch sizes
two schedules take paths those shapes never reach:
  - attention_small_kernel (csrc/vit.cu, G <= 128) runs min(items, SMs x 3) CTAs (x 2 at head dim 64) that walk the
    (cloud, head) items, prefetching item i + grid into the other half of shared memory: items of the second and later
    passes depend on the prefetch, the buffer toggle and the item -> (cloud, head) mapping of later iterations;
  - tc_linear_kernel<PAIR, 16> (csrc/embed_tc.cu, every GEMM of the stack) gives a CTA pair more than one tile once the
    tiles outnumber the clusters: the second tile uses the second TMEM accumulator, its TMA reduce-add goes into the fp32
    residual stream, and with more M pairs than clusters the A-resident GEMMs walk a second M group.
Python mirrors of both launch schedules below tell each test which clouds land in those places (the sentinel clouds),
and every test asserts that its shape reaches the property it is there for, so that on another device it fails instead
of quietly testing less.  test_mirrors_match_the_launches ties the mirrors to the grids the library really launches.

Items of both kernels are computed independently: a cloud's outputs must not depend on which batch, pass or tile it
landed in, so the batch-invariance checks are bit for bit.  The float64 oracle runs only on the sentinel clouds.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import assert_tokens_close, dev, to_dev, vit_bf16_emulation
from oracle import oracle
from p3tok import ops, synth
from p3tok.apf_model import APFViTLayer, ClassificationHead, fold_vit_layer, run_blocks

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "adapting-2d-vits-for-3d-point-cloud-understanding_b200"


def cdiv(a, b):
    return -(-a // b)


def num_sms():
    """The SM count both schedules are sized by (num_sms_vit() / num_sms() in C)."""
    return torch.cuda.get_device_properties(dev()).multi_processor_count


# ------------------------------------------------------------------ the attention schedule, mirrored from csrc/vit.cu
AT_Q, AT_KV = 128, 64                      # query rows per CTA, keys per block


def attention_schedule(B, G, heads, hd, sms):
    """attention_bf16: the persistent form for G <= 128 (grid = min(items, slots), item i in pass i // grid), else one CTA
    per (128-query block, head, cloud)."""
    items = B * heads
    if G <= AT_Q:
        slots = sms * (3 if hd == 32 else 2)
        grid = min(items, slots)
        return dict(small=True, items=items, slots=slots, grid=[grid, 1, 1], passes=cdiv(items, grid))
    return dict(small=False, items=items, grid=[cdiv(G, AT_Q), heads, B], key_blocks=cdiv(G, AT_KV), passes=1)


def pass_clouds(att, heads):
    """The cloud holding the first item of every later pass (it straddles the boundary unless the pass starts at its head
    0) and, when it straddles, the first cloud wholly inside the pass."""
    out = set()
    if att["small"]:
        for p in range(1, att["passes"]):
            i = p * att["grid"][0]
            out.add(i // heads)
            if i % heads:
                out.add(i // heads + 1)
    return out


# ------------------------------------------------------------------ the GEMM schedule, mirrored from csrc/embed_tc.cu
TC_BM, TC_BK, TC_MAX_KB, TC_MAX_N = 128, 64, 8, 2048
TC_SMEM = 227 * 1024
TC_A_STAGE = TC_BM * TC_BK * 2
TC_SMEM_FIXED_EW16 = 16 * (32 * 128 + 256) + TC_MAX_N * 4 + 512 + 1024     # TcCfg<16>::SMEM_FIXED: one store box per warp
TC_THREADS_EW16 = 64 + 16 * 32 + 32


def pick_bn(N):
    best, waste = 64, 1 << 30
    for bn in range(256, 63, -64):
        w = cdiv(N, bn) * bn - N
        if w < waste:
            best, waste = bn, w
    return best


def wide_tile(n):
    return 256 if n > 1024 and n % 192 and n % 256 else 0


def gemm_schedule(M, K, N, bn, sms):
    """tc_linear with the ViT stack's options (16 epilogue warps, CTA pairs, A-resident mode when it fits)."""
    BN = bn or pick_bn(N)
    m_tiles, n_tiles, num_kb = cdiv(M, TC_BM), cdiv(N, BN), cdiv(K, TC_BK)
    pair = m_tiles >= 2
    CL = 2 if pair else 1
    ares = (pair and n_tiles >= 2 and num_kb <= TC_MAX_KB
            and (TC_SMEM - TC_SMEM_FIXED_EW16 - num_kb * TC_A_STAGE) // (BN // 2 * TC_BK * 2) >= 3)
    num_mg = cdiv(m_tiles, CL)
    items = num_mg if ares else num_mg * n_tiles
    return dict(M=M, K=K, N=N, BN=BN, m_tiles=m_tiles, n_tiles=n_tiles, pair=pair, CL=CL, ares=ares, num_mg=num_mg,
                items=items, clusters=min(items, sms // CL))


def work_list(s, cluster):
    """(M group, N tile) entries of one cluster, in order (`decode` in tc_linear_kernel)."""
    out, li = [], 0
    while True:
        if s["ares"]:
            g, nt = divmod(li, s["n_tiles"])
            mg = cluster + g * s["clusters"]
            if mg >= s["num_mg"]:
                return out
        else:
            item = cluster + li * s["clusters"]
            if item >= s["items"]:
                return out
            mg, nt = divmod(item, s["n_tiles"])
        out.append((mg, nt))
        li += 1


def later_groups(s):
    """M groups a cluster reaches after its first one: their tiles run in the cluster's second or later work item."""
    later = set()
    for c in range(s["clusters"]):
        w = work_list(s, c)
        later |= {mg for mg, _ in w if mg != w[0][0]}
    return sorted(later)


def vit_gemms(M, D, H, R, sms):
    """The GEMM launches of one layer of vit_forward, in order: linear_wide slices qkv and fc1d into <= 2048 columns."""
    out = []

    def wide(name, K, N):
        parts = cdiv(N, 2048)
        per = N if parts == 1 else cdiv(cdiv(N, parts), 256) * 256
        for n0 in range(0, N, per):
            n = min(per, N - n0)
            out.append((name if parts == 1 else f"{name}[{n0}:{n0 + n}]", gemm_schedule(M, K, n, wide_tile(n), sms)))

    wide("qkv", D, 3 * D)
    out.append(("proj", gemm_schedule(M, D, D, 0, sms)))
    wide("fc1d", D, H + R)
    out.append(("fc2u", gemm_schedule(M, H + R, D, 0, sms)))
    return out


def stack_schedule(B, G, D, heads, H, R):
    sms = num_sms()
    M = B * G
    att = attention_schedule(B, G, heads, D // heads, sms)
    gemms = vit_gemms(M, D, H, R, sms)
    print(f"[schedule] B={B} G={G} D={D} heads={heads}: M={M}, {sms} SMs; attention "
          + (f"persistent: {att['items']} items on {att['grid'][0]} CTAs, {att['passes']} passes" if att["small"]
             else f"general: grid {att['grid']}, {att['key_blocks']} key blocks"))
    for name, s in gemms:
        tiles = max(len(work_list(s, c)) for c in range(s["clusters"]))
        print(f"[schedule]   {name:<16} K={s['K']:<5} N={s['N']:<5} BN={s['BN']:<3} m_tiles={s['m_tiles']} "
              f"({'pairs' if s['pair'] else 'single CTAs'}, last tile {M - (s['m_tiles'] - 1) * TC_BM} rows) "
              f"{'A-resident ' if s['ares'] else ''}items={s['items']} clusters={s['clusters']} "
              f"tiles per cluster <= {tiles}, later M groups {len(later_groups(s))}")
    return att, gemms


def sentinel_clouds(B, G, heads, att, gemms):
    """Cloud 0 and the last; the clouds at the attention pass boundaries; the clouds of the first and the last M group a
    cluster reaches after its first one (both CTAs of the pair); the first cloud of the last, possibly ragged, M tile."""
    M = B * G
    s = {0, B - 1} | pass_clouds(att, heads)
    for _, g in gemms:
        later = later_groups(g)
        if later:
            r0 = later[0] * g["CL"] * TC_BM
            s |= {r0 // G, min(r0 + TC_BM, M - 1) // G, (min((later[-1] + 1) * g["CL"] * TC_BM, M) - 1) // G}
        s.add((g["m_tiles"] - 1) * TC_BM // G)
    return sorted(c for c in s if c < B)


def _differing(a, b):
    """Clouds (leading index) in which two equally shaped tensors differ."""
    d = (a != b).flatten(1).any(1)
    return torch.nonzero(d).flatten().tolist()


# ------------------------------------------------------------------ 1. the attention kernel alone
SMALL_G = (1, 63, 64, 65, 127, 128)
SMALL_CASES = ([(G, 32, 12) for G in SMALL_G] + [(G, 64, 6) for G in SMALL_G]
               + [(127, 32, 7), (65, 64, 5)])          # heads not dividing the slot count: a cloud straddles every pass boundary
GENERAL_CASES = [(G, hd, 384 // hd) for G in (129, 197, 513) for hd in (32, 64)]
GENERAL_B = 20


def _case_id(c):
    return "G{}-hd{}-h{}".format(*c)


def _small_batch(hd, heads):
    """Clouds for at least 2.5 passes of the persistent kernel on this device."""
    return cdiv(5 * num_sms() * (3 if hd == 32 else 2), 2 * heads) + 1


def _qkv(B, G, heads, hd):
    g = torch.Generator().manual_seed(100003 * G + 101 * hd + heads)     # CPU generator: the same values in every process
    return (torch.randn(B * G, 3 * heads * hd, generator=g) * 1.5).bfloat16().to(dev())


def _attention_ref(qkv, B, G, heads):
    """float64 softmax(q k^T / sqrt(hd)) v, (B, G, D)."""
    D = qkv.shape[1] // 3
    hd = D // heads
    t = qkv.double().reshape(B, G, 3, heads, hd).permute(2, 0, 3, 1, 4)
    att = ((t[0] @ t[1].transpose(-2, -1)) * hd ** -0.5).softmax(-1)
    return (att @ t[2]).transpose(1, 2).reshape(B, G, D)


def _check_attention(case, B):
    G, hd, heads = case
    sched = attention_schedule(B, G, heads, hd, num_sms())
    qkv = _qkv(B, G, heads, hd)
    got = ops.attention_bf16(qkv, B, G, heads).reshape(B, G, -1)
    ref = _attention_ref(qkv, B, G, heads)
    # the bounds of test_gpu_vit.py::test_attention_block, per cloud: bf16 probabilities and output (2^-9 relative each)
    d = got.double() - ref
    err = d.abs().flatten(1).amax(1) / ref.abs().flatten(1).amax(1)
    fro = d.flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1)
    print(f"[attention] {_case_id(case)} B={B}: items {sched['items']}, grid {sched['grid']}, passes {sched['passes']}; "
          f"worst cloud max|err|/max|ref| {float(err.max()):.2e}, fro {float(fro.max()):.2e}")
    bad = torch.nonzero((err > 1.5e-2) | (fro > 5e-3)).flatten().tolist()
    assert not bad, f"{_case_id(case)}: clouds {bad[:8]} outside the bf16 bounds (max err {float(err.max()):.2e}, fro {float(fro.max()):.2e})"
    # every item equals the same cloud run alone (B = 1: one CTA per head, one pass)
    alone = torch.stack([ops.attention_bf16(qkv[b * G:(b + 1) * G], 1, G, heads) for b in range(B)]).reshape(B, G, -1)
    diff = _differing(got, alone)
    where = [f"cloud {b} (items {b * heads}..{b * heads + heads - 1}, pass {b * heads // sched['grid'][0]})" for b in diff[:4]]
    assert not diff, f"{_case_id(case)}: {len(diff)} clouds differ from the cloud run alone: {where}"
    return sched, got


@pytest.mark.parametrize("case", SMALL_CASES, ids=_case_id)
def test_attention_persistent_form_past_one_pass(case, attention_general_form):
    G, hd, heads = case
    B = _small_batch(hd, heads)
    sched, got = _check_attention(case, B)
    assert sched["small"] and sched["items"] >= 2.5 * sched["slots"] and sched["passes"] >= 3, sched
    # P3TOK_ATTN_SMALL=0: the one-CTA-per-(cloud, head) form runs attention_block<HD> on the same key blocks in the same order
    other = attention_general_form[_case_id(case)]
    diff = _differing(got.cpu(), other.reshape(got.shape))
    assert not diff, f"{_case_id(case)}: clouds {diff[:8]} differ between the persistent and the general attention kernel"


@pytest.mark.parametrize("case", GENERAL_CASES, ids=_case_id)
def test_attention_general_form_at_batch(case):
    sched, _ = _check_attention(case, GENERAL_B)
    assert not sched["small"] and sched["grid"][2] == GENERAL_B >= 10, sched


def _run_general_form(path):
    """Entry point of the P3TOK_ATTN_SMALL=0 subprocess: the small cases through attention_kernel, saved to `path`."""
    out = {}
    for case in SMALL_CASES:
        G, hd, heads = case
        B = _small_batch(hd, heads)
        out[_case_id(case)] = ops.attention_bf16(_qkv(B, G, heads, hd), B, G, heads).cpu()
    torch.save(out, path)


_SUBPROCESS = ("import os, sys; r = os.getcwd(); sys.path[:0] = [r, os.path.join(r, %r), os.path.join(r, 'tests')];"
               "import test_gpu_vit_batch as t; t._run_general_form(sys.argv[1])" % PKG)


@pytest.fixture(scope="module")
def attention_general_form(tmp_path_factory):
    """{case: output of the general attention kernel} (P3TOK_ATTN_SMALL is read once per process: a subprocess)."""
    path = str(tmp_path_factory.mktemp("attn") / "general.pt")
    env = dict(os.environ, P3TOK_ATTN_SMALL="0")
    subprocess.run([sys.executable, "-c", _SUBPROCESS, path], check=True, env=env, cwd=ROOT, timeout=1200)
    return torch.load(path)


# ------------------------------------------------------------------ 2-4. the APF block stack at batch
APF_CASES = {
    # c2v of bench.py: B = 128 clouds x G = 128 tokens, ViT-S width, 12 layers, the bench's block weights
    "c2v": dict(D=384, heads=12, depth=12, B=128, G=128, seed=0, tok_seed=128, sub=4),
    # M = 20320: 159 M tiles (the last of 96 rows) in 80 pairs - the A-resident GEMMs walk a second M group, fc2u up to
    # 3 tiles per pair; G = 127: two key blocks, the second ragged
    "ragged_m20320": dict(D=384, heads=12, depth=3, B=160, G=127, seed=7, tok_seed=160, sub=4),
    # ViT-B width: qkv (2304) and fc1d (3136) column-sliced by linear_wide; head dim 64, G = 196: the general attention kernel
    "vit_b": dict(D=768, heads=12, depth=2, B=32, G=196, seed=8, tok_seed=32, sub=4),
}


def _require_apf(name, c, att, gemms):
    by = dict(gemms)
    fc2u = by["fc2u"]
    if name in ("c2v", "ragged_m20320"):
        assert att["small"] and att["passes"] >= 2, f"{name}: {att['passes']} attention pass(es) on this device"
        assert fc2u["items"] > fc2u["clusters"], f"{name}: fc2u has {fc2u['items']} items on {fc2u['clusters']} clusters"
    if name == "ragged_m20320":
        ares = [g for _, g in gemms if g["ares"]]
        assert len(ares) == 3 and all(g["num_mg"] > g["clusters"] for g in ares), \
            f"{name}: the A-resident GEMMs do not walk a second M group: {[(g['num_mg'], g['clusters']) for g in ares]}"
        assert fc2u["m_tiles"] % 2 and c["B"] * c["G"] % TC_BM, f"{name}: the last M tile is not ragged / not alone in its pair"
    if name == "vit_b":
        assert not att["small"], f"{name}: G = {c['G']} should take the general attention kernel"
        assert sum(n.startswith("qkv") for n in by) == 2 and sum(n.startswith("fc1d") for n in by) == 2, list(by)
        assert any(g["items"] > g["clusters"] for g in by.values()), f"{name}: no GEMM gives a pair a second tile"


def _apf_stack(D, heads, depth, sd):
    """The block stack, encoder_norm and head of AdaptPointFormer as modules, loaded from a synthetic state dict."""
    blocks = torch.nn.Sequential(*[APFViTLayer(D, heads) for _ in range(depth)]).eval().to(dev())
    norm = torch.nn.LayerNorm(D).eval().to(dev())
    head = ClassificationHead(D, 15).eval().to(dev())
    tsd = synth.to_torch_state(sd)
    for mod, prefix in ((blocks, "blocks."), (norm, "encoder_norm."), (head, "head.")):
        mod.load_state_dict({k[len(prefix):]: v for k, v in tsd.items() if k.startswith(prefix)}, strict=True)
    return blocks, norm, head


@pytest.fixture(scope="module")
def apf_model():
    """name -> (state dict, blocks, norm, head, tokens on the host, fold cache); built once per module."""
    built = {}

    def get(name):
        if name not in built:
            c = APF_CASES[name]
            sd = synth.apf_vit_state(c["D"], c["depth"], 15, c["seed"])
            blocks, norm, head = _apf_stack(c["D"], c["heads"], c["depth"], sd)
            built[name] = (sd, blocks, norm, head, synth.vit_tokens(c["B"], c["G"], c["D"], c["tok_seed"]), {})
        return built[name]
    return get


@pytest.mark.parametrize("name", list(APF_CASES))
def test_apf_stack_at_batch(name, apf_model):
    c = APF_CASES[name]
    B, G, D, heads, depth = c["B"], c["G"], c["D"], c["heads"], c["depth"]
    att, gemms = stack_schedule(B, G, D, heads, 4 * D, 64)
    _require_apf(name, c, att, gemms)
    sentinels = sentinel_clouds(B, G, heads, att, gemms)
    print(f"[{name}] sentinel clouds {sentinels}")
    sd, blocks, norm, head, tok, cache = apf_model(name)
    tokd = to_dev(tok)
    with torch.no_grad():
        x, pooled = run_blocks(blocks, tokd, norm, cache)
        logits = head(pooled)
        # every cloud against a torch model of the kernels' own arithmetic (bf16 operands, fp32 accumulation), on the GPU
        folded = [fold_vit_layer(blk) for blk in blocks]
        ex, ep = vit_bf16_emulation(folded, tokd, heads, 64, norm.weight, norm.bias)
    for got, emu, key in ((x, ex, "x"), (pooled, ep, "pooled")):
        d = (got.double() - emu.double()).abs().flatten(1).amax(1) / emu.double().abs().flatten(1).amax(1)
        print(f"[{name}] {key} vs bf16 emulation: worst cloud {int(d.argmax())} rel err {float(d.max()):.2e}")
        bad = torch.nonzero(d >= 4e-3).flatten().tolist()
        assert not bad, f"{name}: {key} of clouds {bad[:8]} off the bf16 emulation (worst {float(d.max()):.2e})"
    # the sentinels against the float64 oracle, each cloud alone (clouds are independent in eval mode)
    for j in sentinels:
        ox, op, ol = oracle.apf_vit(sd, tok[j:j + 1], depth, heads)
        for got, orc, key in ((x, ox, "x"), (pooled, op, "pooled"), (logits, ol, "logits")):
            assert_tokens_close(got[j:j + 1].cpu().numpy(), orc, 1e-2, f"{name} cloud {j} {key} vs oracle")
    _check_batch_invariance(name, lambda t: run_blocks(blocks, t, norm, cache), tokd, G, (x, pooled), c["sub"], sentinels)


def _check_batch_invariance(name, run, inp, G, outs, sub, sentinels):
    """outs = run(inp) must equal the same clouds run in sub-batches of `sub` and a second run of the whole batch, bit for
    bit; whether one cloud alone (B = 1: M = G rows, single-CTA GEMMs) is bit-identical too is reported."""
    B = inp.shape[0]
    assert sub * G > TC_BM, "the sub-batches must keep the CTA-pair GEMM route"
    with torch.no_grad():
        for i in range(0, B, sub):
            part = run(inp[i:i + sub])
            for k, (a, b) in enumerate(zip(part, outs)):
                diff = _differing(a, b[i:i + sub])
                assert not diff, f"{name}: output {k} of clouds {[i + d for d in diff]} differs between B = {B} and B = {len(a)}"
        again = run(inp)
        for k, (a, b) in enumerate(zip(again, outs)):
            diff = _differing(a, b)
            assert not diff, f"{name}: output {k} of clouds {diff[:8]} differs between two identical runs"
        same = {j: all(torch.equal(a[0], b[j]) for a, b in zip(run(inp[j:j + 1]), outs)) for j in sentinels}
    print(f"[{name}] B = 1 bit-identical to the batch (reported, not asserted): {same}")


# ------------------------------------------------------------------ 5. Pix4Point's block stack at batch
P4P_CASES = {
    # S = 1 + 64 (BASELINE C1 token count), head dim 64: 762 items, about 2.6 passes; M = 8255, a 63-row last M tile
    "s65_b127": dict(D=384, heads=6, depth=3, B=127, S=65, seed=65, sub=4),
    # S = 1 + 512 (the 8192-point P3Embed output): the general kernel with 5 query blocks x 9 key blocks
    "s513_b8": dict(D=384, heads=6, depth=3, B=8, S=513, seed=513, sub=2),
}


def _p4p_inputs(c):
    import make_golden
    from p3tok.p4p_model import TimmBlock
    feats, pos, sd = make_golden.p4p_vit_inputs(dict(B=c["B"], G=c["S"] - 1, D=c["D"], depth=c["depth"], seed=c["seed"]))
    tsd = synth.to_torch_state(sd)
    blocks = torch.nn.ModuleList([TimmBlock(c["D"], c["heads"]) for _ in range(c["depth"])]).eval().to(dev())
    blocks.load_state_dict({k[len("vit.blocks."):]: v for k, v in tsd.items() if k.startswith("vit.blocks.")}, strict=True)
    norm = torch.nn.LayerNorm(c["D"], eps=1e-6).eval().to(dev())
    norm.load_state_dict({k[len("vit.norm."):]: v for k, v in tsd.items() if k.startswith("vit.norm.")}, strict=True)
    return feats, pos, sd, blocks, norm


@pytest.mark.parametrize("name", list(P4P_CASES))
def test_pointvit_stack_at_batch(name):
    from p3tok.p4p_model import fold_timm_block
    c = P4P_CASES[name]
    B, S, D, heads, depth = c["B"], c["S"], c["D"], c["heads"], c["depth"]
    att, gemms = stack_schedule(B, S, D, heads, 4 * D, 0)
    if name == "s65_b127":
        assert att["small"] and att["passes"] >= 2, f"{name}: {att['passes']} attention pass(es) on this device"
        assert B * S % TC_BM, f"{name}: the last M tile is not ragged"
    else:
        assert not att["small"] and att["grid"][0] == 5 and att["key_blocks"] == 9, att
    sentinels = sentinel_clouds(B, S, heads, att, gemms)
    print(f"[{name}] sentinel clouds {sentinels}")
    feats, pos, sd, blocks, norm = _p4p_inputs(c)
    params = [t for blk in blocks for t in fold_timm_block(blk)]
    fw, fb = norm.weight.detach(), norm.bias.detach()

    def run(f, p):
        return ops.vit_blocks(f, p, params, heads, fw, fb, 1e-6, 1)
    fd, pd = to_dev(feats), to_dev(pos)
    out, pooled = run(fd, pd)
    for j in sentinels:
        ox, og = oracle.pointvit_blocks(sd, feats[j:j + 1], pos[j:j + 1], depth, heads)
        assert_tokens_close(out[j:j + 1].cpu().numpy(), ox, 1e-2, f"{name} cloud {j} normed feats vs oracle")
        assert_tokens_close(pooled[j:j + 1].cpu().numpy(), og[:, :D], 1e-2, f"{name} cloud {j} token max vs oracle")
    both = torch.stack([fd, pd], 1)      # (B, 2, S, D): feats and pos sliced together
    _check_batch_invariance(name, lambda t: run(t[:, 0].contiguous(), t[:, 1].contiguous()), both, S, (out, pooled), c["sub"],
                            sentinels)


# ------------------------------------------------------------------ 6. two steps in flight, as bench.py runs them
def test_two_graphed_steps_in_flight(apf_model):
    """run_blocks at the c2v shape captured into two GraphedTokenizer instances on two streams and replayed concurrently on
    two token batches (bench.py's device loop keeps two steps in flight): each output equals its eager result."""
    from p3tok.graph import GraphedTokenizer
    c = APF_CASES["c2v"]
    sd, blocks, norm, _, tok, cache = apf_model("c2v")
    toks = [to_dev(tok), to_dev(synth.vit_tokens(c["B"], c["G"], c["D"], c["tok_seed"] + 1))]
    fn = lambda t: run_blocks(blocks, t, norm, cache)       # noqa: E731
    with torch.no_grad():
        eager = [fn(t) for t in toks]
    assert not torch.equal(eager[0][1], eager[1][1])
    streams = [torch.cuda.Stream(device=dev()) for _ in range(2)]
    graphs = [GraphedTokenizer(fn, [toks[0]], stream=s) for s in streams]
    main = torch.cuda.current_stream(dev())
    for rnd in range(2):                     # round 1 feeds batch i to graph i, round 2 swaps them
        for s in streams:
            s.wait_stream(main)
        outs = [g(toks[(i + rnd) % 2]) for i, g in enumerate(graphs)]
        for s in streams:
            main.wait_stream(s)
        torch.cuda.synchronize()
        for i, (x, pooled) in enumerate(outs):
            ex, ep = eager[(i + rnd) % 2]
            assert torch.equal(x, ex) and torch.equal(pooled, ep), \
                f"round {rnd}: graph {i} on batch {(i + rnd) % 2}: clouds {_differing(pooled, ep)[:8]} differ from eager"


# ------------------------------------------------------------------ the mirrors against the launches
def _launched_kernels(fn, path):
    """(name, grid, block) of every kernel fn() launches, in launch order (torch.profiler's CUDA activity trace)."""
    from torch.profiler import ProfilerActivity, profile
    with torch.no_grad():
        fn()                                 # one-time kernel attributes outside the trace
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    assert kern, "the profiler recorded no kernels"
    return [(e["name"], list(e["args"]["grid"]), list(e["args"]["block"])) for e in kern]


@pytest.mark.parametrize("name", list(APF_CASES) + list(P4P_CASES))
def test_mirrors_match_the_launches(name, tmp_path):
    """One layer at each case's shape: the grids of its tc_linear_kernel and attention launches are what the mirrors say,
    and every GEMM is the 16-epilogue-warp form (as a CTA pair where the mirror says so)."""
    if name in APF_CASES:
        c = APF_CASES[name]
        B, G, D, heads, R = c["B"], c["G"], c["D"], c["heads"], 64
        blocks, norm, _ = _apf_stack(D, heads, 1, synth.apf_vit_state(D, 1, 15, c["seed"]))
        x, cache = to_dev(synth.vit_tokens(B, G, D, c["tok_seed"])), {}
        fn = lambda: run_blocks(blocks, x, norm, cache)       # noqa: E731  (the cache keeps the fold's torch ops out of the trace)
    else:
        from p3tok.p4p_model import fold_timm_block
        c = dict(P4P_CASES[name], depth=1)
        B, G, D, heads, R = c["B"], c["S"], c["D"], c["heads"], 0
        feats, pos, _, blocks, norm = _p4p_inputs(c)
        params = fold_timm_block(blocks[0])
        fd, pd = to_dev(feats), to_dev(pos)
        fn = lambda: ops.vit_blocks(fd, pd, params, heads, norm.weight.detach(), norm.bias.detach(), 1e-6, 1)   # noqa: E731
    att, gemms = stack_schedule(B, G, D, heads, 4 * D, R)
    kern = _launched_kernels(fn, str(tmp_path / "trace.json"))
    tc = [(n, g, b) for n, g, b in kern if "tc_linear_kernel" in n]
    at = [(n, g) for n, g, _ in kern if "attention" in n]
    assert len(tc) == len(gemms), f"{len(tc)} tc_linear_kernel launches, the mirror has {len(gemms)}: {[n for n, _, _ in kern]}"
    for (gname, s), (kname, grid, block) in zip(gemms, tc):
        m = re.search(r"tc_linear_kernel<(true|false), (\d+)>", kname)
        assert m, kname
        assert (m.group(1) == "true", int(m.group(2)), block) == (s["pair"], 16, [TC_THREADS_EW16, 1, 1]), (gname, kname, block)
        assert grid == [s["clusters"] * s["CL"], 1, 1], f"{gname}: launched grid {grid}, mirror {s['clusters']} x {s['CL']}"
    assert len(at) == 1, at
    assert ("attention_small_kernel" in at[0][0]) == att["small"] and at[0][1] == att["grid"], (at, att)
