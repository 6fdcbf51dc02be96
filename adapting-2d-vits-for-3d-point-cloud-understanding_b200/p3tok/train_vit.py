"""Training mode of the APF token consumer: the APFViTLayer stack, encoder_norm, the max over tokens and the
ClassificationHead as torch.autograd.Functions over the C ABI (csrc/train_vit.cu + csrc/train.cu).

Why it exists: the reference freezes the pre-trained blocks but keeps point_encoder.*, encoder_norm.* and head.* trainable
(reference src/models/apf.py:335-346), so the tokenizer's gradient arrives THROUGH the twelve layers
(src/models/apf_utils.py:268-293).  `BlocksTrainFn` carries dL/dpooled back to the tokens and produces the gradient of every
block / norm parameter that asks for one (`requires_grad`; the frozen ones cost nothing); `HeadTrainFn` is the head with
nn.BatchNorm1d in TRAIN mode (apf.py:219-252).  Stochastic regularisers - the adapter's dropout (apf_utils.py:223), the two
DropPath draws of a layer (apf_utils.py:277, 289), the dropout in front of and inside the head (apf.py:368, 237-242) - are keep
masks drawn with torch's generator (scaled by 1 / keep probability) and applied by the element-wise kernel; a caller may pass
the masks in (tests do, to compare against a reference evaluation under the same masks).

fp32 on CUDA cores (GEMMs: p3tok_linear_f32 / p3tok_linear_tn_f32); CUDA tensors only, no fallback.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import check
from .train import _L, _f32, _s, _t, deterministic, bn_backward, bn_forward, colstats, colsum, group_max_arg, group_max_bwd, linear, linear_tn

# parameter order of one APFViTLayer (state_dict names relative to the layer)
LAYER_PARAMS = ("norm1.weight", "norm1.bias", "attention.qkv.weight", "attention.qkv.bias", "attention.proj.weight",
                "attention.proj.bias", "adapter.adapter_norm.weight", "adapter.adapter_norm.bias", "adapter.scale",
                "adapter.down_proj.weight", "adapter.down_proj.bias", "adapter.up_proj.weight", "adapter.up_proj.bias",
                "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias")
NP = len(LAYER_PARAMS)


# ------------------------------------------------------------------------------------------------ kernel wrappers
def ln_fwd(x: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor], eps: float, want_y: bool = True):
    """x (M,D) -> (y or None, mean (M,), rstd (M,))  (p3tok_ln_fwd_f32)."""
    x = _f32(x)
    M, D = x.shape
    y = torch.empty_like(x) if want_y else None
    mean = torch.empty(M, dtype=torch.float32, device=x.device)
    rstd = torch.empty(M, dtype=torch.float32, device=x.device)
    wf = _f32(w) if w is not None else None
    bf = _f32(b) if b is not None else None
    with torch.cuda.device(x.device):
        check(_L().p3tok_ln_fwd_f32(x.data_ptr(), M, D, wf.data_ptr() if wf is not None else None,
                                    bf.data_ptr() if bf is not None else None, float(eps), y.data_ptr() if y is not None else None,
                                    mean.data_ptr(), rstd.data_ptr(), _s()), "ln_fwd_f32")
    return y, mean, rstd


def ln_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, w: Optional[torch.Tensor],
           into: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dx of LayerNorm; `into` (M,D) is accumulated into (and returned) when given."""
    dy, x = _f32(dy), _f32(x)
    M, D = x.shape
    dx = into if into is not None else torch.empty_like(x)
    wf = _f32(w) if w is not None else None
    with torch.cuda.device(x.device):
        check(_L().p3tok_ln_bwd_f32(dy.data_ptr(), x.data_ptr(), M, D, mean.data_ptr(), rstd.data_ptr(),
                                    wf.data_ptr() if wf is not None else None, 1 if into is not None else 0, dx.data_ptr(), _s()),
              "ln_bwd_f32")
    return dx


def ln_param_grad(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    dy, x = _f32(dy), _f32(x)
    M, D = x.shape
    g = torch.empty(2 * D, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        if deterministic():
            ws = torch.empty(int(_L().p3tok_colsum_det_workspace_bytes(M, D)), dtype=torch.uint8, device=x.device)
            check(_L().p3tok_ln_param_grad_det_f32(dy.data_ptr(), x.data_ptr(), M, D, mean.data_ptr(), rstd.data_ptr(), g.data_ptr(),
                                                   g.data_ptr() + 8 * D, ws.data_ptr(), ws.numel(), _s()), "ln_param_grad_det_f32")
        else:
            check(_L().p3tok_ln_param_grad_f32(dy.data_ptr(), x.data_ptr(), M, D, mean.data_ptr(), rstd.data_ptr(), g.data_ptr(),
                                               g.data_ptr() + 8 * D, _s()), "ln_param_grad_f32")
    return g[:D].float(), g[D:].float()


def attn_fwd(qkv: torch.Tensor, B: int, G: int, heads: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """qkv (B*G, 3D) -> (o (B*G, D), P (B*heads, G, G)); scale = head_dim ** -0.5 (apf_utils.py:126)."""
    qkv = _f32(qkv)
    D = qkv.shape[1] // 3
    hd = D // heads
    o = torch.empty((B * G, D), dtype=torch.float32, device=qkv.device)
    P = torch.empty((B * heads, G, G), dtype=torch.float32, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(_L().p3tok_attn_fwd_f32(qkv.data_ptr(), B, G, heads, hd, float(hd) ** -0.5, o.data_ptr(), P.data_ptr(), _s()), "attn_fwd_f32")
    return o, P


def attn_bwd(qkv: torch.Tensor, P: torch.Tensor, do: torch.Tensor, B: int, G: int, heads: int) -> torch.Tensor:
    qkv, do = _f32(qkv), _f32(do)
    D = qkv.shape[1] // 3
    hd = D // heads
    dqkv = torch.empty_like(qkv)
    scratch = torch.empty((2, B * heads, G, G), dtype=torch.float32, device=qkv.device)
    with torch.cuda.device(qkv.device):
        check(_L().p3tok_attn_bwd_f32(qkv.data_ptr(), P.data_ptr(), do.data_ptr(), B, G, heads, hd, float(hd) ** -0.5,
                                      scratch.data_ptr(), dqkv.data_ptr(), _s()), "attn_bwd_f32")
    return dqkv


def ew(op: int, a: torch.Tensor, b: Optional[torch.Tensor] = None, alpha: float = 1.0, beta: float = 1.0, bdiv: int = 1,
       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """p3tok_ew_f32: out = f(a, b) element-wise (out may be a or b)."""
    a = _f32(a)
    bb = _f32(b) if b is not None else None
    if out is None:
        out = torch.empty_like(a)
    with torch.cuda.device(a.device):
        check(_L().p3tok_ew_f32(int(op), a.data_ptr(), bb.data_ptr() if bb is not None else None, float(alpha), float(beta), a.numel(),
                                int(bdiv), out.data_ptr(), _s()), "ew_f32")
    return out


def axpby(alpha: float, a: torch.Tensor, beta: float, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    return ew(_lib.EW_AXPBY, a, b, alpha, beta, out=out)


def mask_mul(a: torch.Tensor, mask: Optional[torch.Tensor], per: int = 1, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """a * mask[e // per] (mask already scaled by 1 / keep probability); identity when mask is None."""
    if mask is None:
        return a
    return ew(_lib.EW_MUL, a, mask, 1.0, 0.0, per, out=out)


def keep_mask(shape: Sequence[int], p: float, device, generator: Optional[torch.Generator] = None) -> Optional[torch.Tensor]:
    """Bernoulli(1 - p) keep mask scaled by 1 / (1 - p) (nn.functional.dropout / timm DropPath); None when p == 0."""
    if p <= 0.0:
        return None
    if p >= 1.0:
        return torch.zeros(tuple(shape), dtype=torch.float32, device=device)
    keep = torch.rand(tuple(shape), dtype=torch.float32, device=device, generator=generator) >= p
    return keep.to(torch.float32) / (1.0 - p)


# ------------------------------------------------------------------------------------------------ the block stack
class BlocksTrainFn(torch.autograd.Function):
    """tokens (B,G,D) -> APFViTLayer x depth -> [final LayerNorm -> max over tokens].

    apply(tokens, heads, eps, masks, has_final, *params): params = depth x LAYER_PARAMS tensors (+ final norm weight, bias);
    eps = (per layer (norm1, adapter_norm, norm2) ..., final); masks = per layer (drop_path_attn (B,), adapter dropout (M,R),
    drop_path_mlp (B,)) entries or None.  Returns (x after the last layer (B,G,D), pooled (B,D)) - pooled is a zero-size
    tensor without a final norm."""

    @staticmethod
    def forward(ctx, tokens, heads, eps, masks, has_final, *params):
        B, G, D = tokens.shape
        M = B * G
        depth = (len(params) - (2 if has_final else 0)) // NP
        x = _f32(tokens).reshape(M, D)
        saved: List[torch.Tensor] = []
        meta = []
        for li in range(depth):
            (n1w, n1b, Wq, bq, Wp, bp, naw, nab, sc, Wd, bd, Wu, bu, n2w, n2b, W1, b1, W2, b2) = params[li * NP:(li + 1) * NP]
            e1, ea, e2 = eps[li]
            dp1, dmask, dp2 = masks[li] if masks is not None else (None, None, None)
            a, mu1, rs1 = ln_fwd(x, n1w, n1b, e1)                                   # apf_utils.py:275
            qkv = linear(a, Wq, bq)
            o, P = attn_fwd(qkv, B, G, heads)
            att = mask_mul(linear(o, Wp, bp), dp1, G * D)                           # attention + drop_path (276-277)
            x1 = axpby(1.0, x, 1.0, att, out=att)                                   # 278
            an, mua, rsa = ln_fwd(x1, naw, nab, ea)                                 # adapter (apf_utils.py:214-233)
            zd = linear(an, Wd, bd)
            dn = mask_mul(ew(_lib.EW_RELU, zd), dmask)
            up = linear(dn, Wu, bu)
            n2, mu2, rs2 = ln_fwd(x1, n2w, n2b, e2)                                 # MLP (286-289)
            z1 = linear(n2, W1, b1)
            m = mask_mul(linear(ew(_lib.EW_GELU, z1), W2, b2), dp2, G * D)
            scv = float(sc.detach().reshape(-1)[0].item()) if sc.numel() else 1.0
            y = axpby(1.0, m, scv, up, out=m)                                       # x_mlp + (up * scale + x1) + x1  (291)
            y = axpby(1.0, y, 2.0, x1, out=y)
            saved += [x, mu1, rs1, qkv, P, o, x1, mua, rsa, zd, mu2, rs2, z1]
            meta.append((scv, dp1, dmask, dp2))
            x = y
        if has_final:
            fw, fb = params[-2], params[-1]
            yn, muf, rsf = ln_fwd(x, fw, fb, eps[depth])                            # apf.py:364
            pooled, arg = group_max_arg(yn, G)                                      # apf.py:366 (first maximum)
            saved += [x, muf, rsf, arg]
        else:
            pooled = x.new_zeros((0,))
        ctx.save_for_backward(*saved, *[p for p in params])
        ctx.n_saved = len(saved)
        ctx.dims = (B, G, D, depth, heads, has_final)
        ctx.meta = meta
        ctx.eps = eps
        return x.reshape(B, G, D), pooled

    @staticmethod
    def backward(ctx, gx, gpooled):
        B, G, D, depth, heads, has_final = ctx.dims
        M = B * G
        saved, params = ctx.saved_tensors[:ctx.n_saved], ctx.saved_tensors[ctx.n_saved:]
        need = ctx.needs_input_grad[5:]
        grads: List[Optional[torch.Tensor]] = [None] * len(params)
        dx = _f32(gx).reshape(M, D).clone() if gx is not None else torch.zeros((M, D), dtype=torch.float32, device=params[0].device)
        if has_final and gpooled is not None and gpooled.numel():
            xl, muf, rsf, arg = saved[13 * depth:13 * depth + 4]
            dyn = group_max_bwd(gpooled, arg, G)
            if need[-2] or need[-1]:
                gw, gb = ln_param_grad(dyn, xl, muf, rsf)
                grads[-2], grads[-1] = (gw if need[-2] else None), (gb if need[-1] else None)
            ln_bwd(dyn, xl, muf, rsf, params[-2], into=dx)
        for li in reversed(range(depth)):
            (n1w, n1b, Wq, bq, Wp, bp, naw, nab, sc, Wd, bd, Wu, bu, n2w, n2b, W1, b1, W2, b2) = params[li * NP:(li + 1) * NP]
            nd = need[li * NP:(li + 1) * NP]
            x, mu1, rs1, qkv, P, o, x1, mua, rsa, zd, mu2, rs2, z1 = saved[13 * li:13 * li + 13]
            scv, dp1, dmask, dp2 = ctx.meta[li]
            e1, ea, e2 = ctx.eps[li]
            g = [None] * NP
            dy = dx
            # ---- MLP branch: y = drop_path(fc2(gelu(fc1(norm2(x1))))) + ...
            dm = mask_mul(dy, dp2, G * D)
            if nd[17] or nd[18]:
                h = ew(_lib.EW_GELU, z1)
                g[17], g[18] = (linear_tn(dm, h) if nd[17] else None), (colsum(dm) if nd[18] else None)
                del h
            dz1 = ew(_lib.EW_GELU_BWD, z1, linear(dm, _t(_f32(W2))))
            if nd[15] or nd[16]:
                n2 = ln_fwd(x1, n2w, n2b, e2)[0]
                g[15], g[16] = (linear_tn(dz1, n2) if nd[15] else None), (colsum(dz1) if nd[16] else None)
                del n2
            dn2 = linear(dz1, _t(_f32(W1)))
            del dz1
            if nd[13] or nd[14]:
                g[13], g[14] = ln_param_grad(dn2, x1, mu2, rs2)
            dx1 = axpby(2.0, dy, 0.0, dy)                                           # adapter's "+ residual" and the layer's
            ln_bwd(dn2, x1, mu2, rs2, n2w, into=dx1)
            del dn2
            # ---- adapter branch: (up_proj(dropout(relu(down_proj(adapter_norm(x1))))) * scale
            if nd[8] or nd[11] or nd[12] or nd[9] or nd[10] or nd[6] or nd[7]:
                an = ln_fwd(x1, naw, nab, ea)[0]
                dn = mask_mul(ew(_lib.EW_RELU, zd), dmask)
            if nd[8]:
                up = linear(dn, Wu, bu)
                g[8] = colstats(ew(_lib.EW_MUL, dy, up, 1.0, 0.0, 1))[0].sum().float().reshape(sc.shape)
            if nd[11]:
                g[11] = linear_tn(dy, dn) * scv
            if nd[12]:
                g[12] = colsum(dy) * scv
            ddn = mask_mul(linear(dy, _t(_f32(Wu)) * scv), dmask)
            dzd = ew(_lib.EW_RELU_BWD, zd, ddn, out=ddn)
            if nd[9] or nd[10]:
                g[9], g[10] = (linear_tn(dzd, an) if nd[9] else None), (colsum(dzd) if nd[10] else None)
            dan = linear(dzd, _t(_f32(Wd)))
            if nd[6] or nd[7]:
                g[6], g[7] = ln_param_grad(dan, x1, mua, rsa)
            ln_bwd(dan, x1, mua, rsa, naw, into=dx1)
            # ---- attention branch: x1 = x + drop_path(proj(attention(qkv(norm1(x)))))
            datt = mask_mul(dx1, dp1, G * D)
            if nd[4] or nd[5]:
                g[4], g[5] = (linear_tn(datt, o) if nd[4] else None), (colsum(datt) if nd[5] else None)
            dqkv = attn_bwd(qkv, P, linear(datt, _t(_f32(Wp))), B, G, heads)
            if nd[2] or nd[3]:
                a = ln_fwd(x, n1w, n1b, e1)[0]
                g[2], g[3] = (linear_tn(dqkv, a) if nd[2] else None), (colsum(dqkv) if nd[3] else None)
                del a
            da = linear(dqkv, _t(_f32(Wq)))
            if nd[0] or nd[1]:
                g[0], g[1] = ln_param_grad(da, x, mu1, rs1)
            dx = ln_bwd(da, x, mu1, rs1, n1w, into=dx1)
            for i in range(NP):
                if g[i] is not None and nd[i]:
                    grads[li * NP + i] = g[i].reshape(params[li * NP + i].shape)
        gtok = dx.reshape(B, G, D) if ctx.needs_input_grad[0] else None
        return (gtok, None, None, None, None, *grads)


def layer_params(layer) -> List[torch.Tensor]:
    sd = dict(layer.named_parameters())
    return [sd[n] for n in LAYER_PARAMS]


def draw_masks(layers, B: int, G: int, device, generator: Optional[torch.Generator] = None):
    """One (drop_path_attn, adapter dropout, drop_path_mlp) triple per layer, in the order the reference draws them
    (apf_utils.py:277 attention DropPath, 223 adapter dropout, 289 MLP DropPath); None when every rate is 0."""
    out = []
    any_mask = False
    for l in layers:
        dpr = float(getattr(l, "drop_path_rate", 0.0)) if l.training else 0.0
        pdrop = float(l.adapter.dropout) if l.training else 0.0
        t = (keep_mask((B,), dpr, device, generator), keep_mask((B * G, l.adapter.down_size), pdrop, device, generator),
             keep_mask((B,), dpr, device, generator))
        any_mask = any_mask or any(m is not None for m in t)
        out.append(t)
    return out if any_mask else None


def blocks_train(layers, x: torch.Tensor, final_norm=None, masks=None, generator: Optional[torch.Generator] = None):
    """Train-mode evaluation of a stack of APFViTLayers (+ encoder_norm and the max over tokens) under autograd:
    -> (x after the last layer (B,G,D), pooled (B,D) or None)."""
    layers = list(layers)
    if not x.is_cuda:
        raise RuntimeError("p3tok training path: CUDA tensors only (no CPU fallback)")
    B, G, _ = x.shape
    if masks is None:
        masks = draw_masks(layers, B, G, x.device, generator)
    params: List[torch.Tensor] = []
    eps = []
    for l in layers:
        params += layer_params(l)
        eps.append((float(l.norm1.eps), float(l.adapter.adapter_norm.eps), float(l.norm2.eps)))
    if final_norm is not None:
        params += [final_norm.weight, final_norm.bias]
        eps.append(float(final_norm.eps))
    y, pooled = BlocksTrainFn.apply(x, int(layers[0].attention.num_heads), tuple(eps), masks, final_norm is not None, *params)
    return y, (pooled if final_norm is not None else None)


# ------------------------------------------------------------------------------------------------ dropout on a tensor
class MaskMulFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mask):
        ctx.save_for_backward(mask)
        return mask_mul(x, mask).reshape(x.shape)

    @staticmethod
    def backward(ctx, g):
        (mask,) = ctx.saved_tensors
        return mask_mul(g, mask).reshape(g.shape), None


def dropout(x: torch.Tensor, p: float, training: bool, mask: Optional[torch.Tensor] = None,
            generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """nn.Dropout on a CUDA tensor (apf.py:368) through the element-wise kernel."""
    if mask is None:
        mask = keep_mask(x.shape, p if training else 0.0, x.device, generator)
    return x if mask is None else MaskMulFn.apply(x, mask)


# ------------------------------------------------------------------------------------------------ classification heads
class HeadTrainFn(torch.autograd.Function):
    """An MLP head in train mode: (Linear -> BatchNorm1d (batch statistics) -> ReLU -> Dropout) x n -> Linear - the reference's
    ClassificationHead (apf.py:230-252, n = 2) and ClsHead (pix4point.py:295-325).
    apply(x (B,E), eps (n), sync, masks (n entries or None), running (None, or n (running_mean, running_var) pairs: eval-mode
    BatchNorm), W1, b1, g1, be1, ..., Wn, bn, gn, ben, Wout, bout) -> (logits, batch mean / unbiased variance of every BatchNorm
    for the running-estimate update), or (logits,) in the running mode."""

    @staticmethod
    def forward(ctx, x, eps, sync, masks, running, *params):
        n = (len(params) - 2) // 4
        h = _f32(x)
        masks = tuple(masks) if masks is not None else (None,) * n
        saved, stats = [], []
        for i in range(n):
            W, b, g, be = params[4 * i:4 * i + 4]
            z = linear(h, W, b)
            y, st = bn_forward(z, g, be, eps[i], True, sync, None if running is None else running[i])
            saved += [h, z]
            stats.append(st)
            h = mask_mul(y, masks[i])
        out = linear(h, params[-2], params[-1])
        ctx.sync, ctx.stats, ctx.masks, ctx.n = sync, stats, masks, n
        ctx.save_for_backward(*saved, h, *params)
        outs = [out]
        for st in stats:
            if not st.running:
                outs += [st.mean64.float(), st.var_unbiased.float()]
        ctx.mark_non_differentiable(*outs[1:])
        return tuple(outs)

    @staticmethod
    def backward(ctx, g, *_unused):
        n = ctx.n
        saved, params = ctx.saved_tensors[:2 * n + 1], ctx.saved_tensors[2 * n + 1:]
        need = ctx.needs_input_grad[5:]
        grads = [None] * len(params)
        g = _f32(g)
        grads[-2] = linear_tn(g, saved[2 * n]) if need[-2] else None
        grads[-1] = colsum(g) if need[-1] else None
        d = linear(g, _t(_f32(params[-2])))
        for i in reversed(range(n)):
            W, b, gam, be = params[4 * i:4 * i + 4]
            hin, z = saved[2 * i], saved[2 * i + 1]
            nd = need[4 * i:4 * i + 4]
            dz, dgam, dbe = bn_backward(mask_mul(d, ctx.masks[i]), z, ctx.stats[i], gam, be, True, ctx.sync, nd[2] or nd[3])
            grads[4 * i:4 * i + 4] = [linear_tn(dz, hin) if nd[0] else None, colsum(dz) if nd[1] else None, dgam, dbe]
            if i > 0 or ctx.needs_input_grad[0]:
                d = linear(dz, _t(_f32(W)))
        return (d if ctx.needs_input_grad[0] else None, None, None, None, None, *grads)


def mlp_head_blocks(seq):
    """[(Linear, BatchNorm1d, Dropout), ...], final Linear of an nn.Sequential laid out (Linear, BN, ReLU, Dropout) x n, Linear."""
    mods = list(seq)
    n = (len(mods) - 1) // 4
    return [(mods[4 * i], mods[4 * i + 1], mods[4 * i + 3]) for i in range(n)], mods[-1]


def head_train(head, x: torch.Tensor, masks=None, sync: bool = False, generator: Optional[torch.Generator] = None,
               running: bool = False) -> torch.Tensor:
    """Forward of an MLP head module (attribute `mlp_head` or `head`) on x (B,E) under autograd.  Train mode: dropout keep masks,
    batch statistics, the BatchNorm buffers updated like nn.BatchNorm1d does.  running=True: the module in eval mode - dropout
    is the identity, BatchNorm uses the running estimates, no buffer changes, nothing all-reduced."""
    from .train import running_stats, update_running
    blocks, last = mlp_head_blocks(head.mlp_head if hasattr(head, "mlp_head") else head.head)
    if masks is None and not running:
        masks = tuple(keep_mask((x.shape[0], lin.out_features), float(dr.p), x.device, generator) for lin, _, dr in blocks)
        if all(m is None for m in masks):
            masks = None
    params = []
    for lin, bn, _ in blocks:
        params += [lin.weight, lin.bias, bn.weight, bn.bias]
    outs = HeadTrainFn.apply(x, tuple(float(bn.eps) for _, bn, _ in blocks), bool(sync) and not running, None if running else masks,
                             running_stats([bn for _, bn, _ in blocks]) if running else None, *params, last.weight, last.bias)
    if not running:
        for i, (_, bn, _) in enumerate(blocks):
            update_running(bn, outs[1 + 2 * i], outs[2 + 2 * i])
    return outs[0]


# ------------------------------------------------------------------------------------------------ Pix4Point (PointViT)
class LinearFn(torch.autograd.Function):
    """y = act(x W^T + b) on rows (nn.Linear, optionally followed by the exact GELU of pix4point.py:215-217); act: 0 none, 2 GELU."""

    @staticmethod
    def forward(ctx, x, W, b, act):
        shape = x.shape
        x2 = _f32(x).reshape(-1, shape[-1])
        z = linear(x2, W, b)
        ctx.save_for_backward(x2, _f32(W), z if act == 2 else x2.new_zeros(0))
        ctx.act, ctx.shape, ctx.has_bias = act, shape, b is not None
        y = ew(_lib.EW_GELU, z) if act == 2 else z
        return y.reshape(*shape[:-1], W.shape[0])

    @staticmethod
    def backward(ctx, g):
        x2, W, z = ctx.saved_tensors
        g2 = _f32(g).reshape(-1, W.shape[0])
        if ctx.act == 2:
            g2 = ew(_lib.EW_GELU_BWD, z, g2)
        dW = linear_tn(g2, x2) if ctx.needs_input_grad[1] else None
        db = colsum(g2) if ctx.has_bias and ctx.needs_input_grad[2] else None
        dx = linear(g2, _t(W)).reshape(ctx.shape) if ctx.needs_input_grad[0] else None
        return dx, dW, db, None


class TokenMaxFn(torch.autograd.Function):
    """torch.max over the tokens after the first `skip` rows of every cloud (pix4point.py:262-268): (B,S,D) -> (B,D)."""

    @staticmethod
    def forward(ctx, x, skip):
        B, S, D = x.shape
        body = _f32(x)[:, skip:, :].contiguous().reshape(B * (S - skip), D)
        out, arg = group_max_arg(body, S - skip)
        ctx.save_for_backward(arg)
        ctx.dims = (B, S, D, skip)
        return out

    @staticmethod
    def backward(ctx, g):
        (arg,) = ctx.saved_tensors
        B, S, D, skip = ctx.dims
        dx = torch.zeros((B, S, D), dtype=torch.float32, device=g.device)
        dx[:, skip:, :] = group_max_bwd(g, arg, S - skip).reshape(B, S - skip, D)
        return dx, None


TIMM_BLOCK_PARAMS = ("norm1.weight", "norm1.bias", "attn.qkv.weight", "attn.qkv.bias", "attn.proj.weight", "attn.proj.bias",
                     "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight", "mlp.fc2.bias")
NTP = len(TIMM_BLOCK_PARAMS)


class TimmBlocksTrainFn(torch.autograd.Function):
    """PointViT's block loop and final norm (pix4point.py:254-256): for blk: feats = blk(feats + pos_embed); feats = norm(feats),
    blk = timm's pre-norm Block (x + attn(norm1(x)), then x + mlp(norm2(x)); drop rates 0 as timm.create_model builds them).
    apply(feats (B,S,D), pos (B,S,D), heads, eps, *params): params = depth x TIMM_BLOCK_PARAMS + (norm.weight, norm.bias);
    eps = ((norm1, norm2) per block ..., final)."""

    @staticmethod
    def forward(ctx, feats, pos, heads, eps, *params):
        B, S, D = feats.shape
        M = B * S
        depth = (len(params) - 2) // NTP
        x = _f32(feats).reshape(M, D)
        pe = _f32(pos).reshape(M, D)
        saved: List[torch.Tensor] = []
        for li in range(depth):
            n1w, n1b, Wq, bq, Wp, bp, n2w, n2b, W1, b1, W2, b2 = params[li * NTP:(li + 1) * NTP]
            e1, e2 = eps[li]
            xin = axpby(1.0, x, 1.0, pe)
            a, mu1, rs1 = ln_fwd(xin, n1w, n1b, e1)
            qkv = linear(a, Wq, bq)
            o, P = attn_fwd(qkv, B, S, heads)
            att = linear(o, Wp, bp)
            x1 = axpby(1.0, xin, 1.0, att, out=att)
            n2, mu2, rs2 = ln_fwd(x1, n2w, n2b, e2)
            z1 = linear(n2, W1, b1)
            m = linear(ew(_lib.EW_GELU, z1), W2, b2)
            x = axpby(1.0, x1, 1.0, m, out=m)
            saved += [xin, mu1, rs1, qkv, P, o, x1, mu2, rs2, z1]
        yn, muf, rsf = ln_fwd(x, params[-2], params[-1], eps[depth])
        saved += [x, muf, rsf]
        ctx.save_for_backward(*saved, *params)
        ctx.n_saved = len(saved)
        ctx.dims = (B, S, D, depth, heads)
        ctx.eps = eps
        return yn.reshape(B, S, D)

    @staticmethod
    def backward(ctx, gout):
        B, S, D, depth, heads = ctx.dims
        M = B * S
        saved, params = ctx.saved_tensors[:ctx.n_saved], ctx.saved_tensors[ctx.n_saved:]
        need = ctx.needs_input_grad[4:]
        grads: List[Optional[torch.Tensor]] = [None] * len(params)
        g = _f32(gout).reshape(M, D)
        xl, muf, rsf = saved[10 * depth:10 * depth + 3]
        if need[-2] or need[-1]:
            gw, gb = ln_param_grad(g, xl, muf, rsf)
            grads[-2], grads[-1] = (gw if need[-2] else None), (gb if need[-1] else None)
        dx = ln_bwd(g, xl, muf, rsf, params[-2])
        dpos = torch.zeros((M, D), dtype=torch.float32, device=dx.device)
        for li in reversed(range(depth)):
            n1w, n1b, Wq, bq, Wp, bp, n2w, n2b, W1, b1, W2, b2 = params[li * NTP:(li + 1) * NTP]
            nd = need[li * NTP:(li + 1) * NTP]
            xin, mu1, rs1, qkv, P, o, x1, mu2, rs2, z1 = saved[10 * li:10 * li + 10]
            e1, e2 = ctx.eps[li]
            gp = [None] * NTP
            if nd[10] or nd[11]:
                h = ew(_lib.EW_GELU, z1)
                gp[10], gp[11] = (linear_tn(dx, h) if nd[10] else None), (colsum(dx) if nd[11] else None)
                del h
            dz1 = ew(_lib.EW_GELU_BWD, z1, linear(dx, _t(_f32(W2))))
            if nd[8] or nd[9]:
                n2 = ln_fwd(x1, n2w, n2b, e2)[0]
                gp[8], gp[9] = (linear_tn(dz1, n2) if nd[8] else None), (colsum(dz1) if nd[9] else None)
                del n2
            dn2 = linear(dz1, _t(_f32(W1)))
            del dz1
            if nd[6] or nd[7]:
                gp[6], gp[7] = ln_param_grad(dn2, x1, mu2, rs2)
            dx1 = ln_bwd(dn2, x1, mu2, rs2, n2w, into=dx)          # dx (the block's output gradient) + the MLP branch
            if nd[4] or nd[5]:
                gp[4], gp[5] = (linear_tn(dx1, o) if nd[4] else None), (colsum(dx1) if nd[5] else None)
            dqkv = attn_bwd(qkv, P, linear(dx1, _t(_f32(Wp))), B, S, heads)
            if nd[2] or nd[3]:
                a = ln_fwd(xin, n1w, n1b, e1)[0]
                gp[2], gp[3] = (linear_tn(dqkv, a) if nd[2] else None), (colsum(dqkv) if nd[3] else None)
                del a
            da = linear(dqkv, _t(_f32(Wq)))
            if nd[0] or nd[1]:
                gp[0], gp[1] = ln_param_grad(da, xin, mu1, rs1)
            dx = ln_bwd(da, xin, mu1, rs1, n1w, into=dx1)          # = d(feats + pos_embed) of this block
            axpby(1.0, dpos, 1.0, dx, out=dpos)
            for i in range(NTP):
                if gp[i] is not None and nd[i]:
                    grads[li * NTP + i] = gp[i].reshape(params[li * NTP + i].shape)
        return (dx.reshape(B, S, D) if ctx.needs_input_grad[0] else None, dpos.reshape(B, S, D) if ctx.needs_input_grad[1] else None,
                None, None, *grads)


def timm_blocks_train(blocks, norm, feats: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """Train-mode / gradient-carrying evaluation of PointViT's block loop + final norm: -> (B,S,D)."""
    blocks = list(blocks)
    if not feats.is_cuda:
        raise RuntimeError("p3tok training path: CUDA tensors only (no CPU fallback)")
    params: List[torch.Tensor] = []
    eps = []
    for blk in blocks:
        sd = dict(blk.named_parameters())
        params += [sd[n] for n in TIMM_BLOCK_PARAMS]
        eps.append((float(blk.norm1.eps), float(blk.norm2.eps)))
    params += [norm.weight, norm.bias]
    eps.append(float(norm.eps))
    return TimmBlocksTrainFn.apply(feats, pos, int(blocks[0].attn.num_heads), tuple(eps), *params)


def token_head_train(tok_mod, tokens: torch.Tensor, centers: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """proj / pos_embed / cls concat of PointViT.forward (pix4point.py:245-252) under autograd: tokens (B,G,W), centers (B,G,3)
    -> (feats (B,1+G,E), pos (B,1+G,E))."""
    B = tokens.shape[0]
    x = LinearFn.apply(tokens, tok_mod.proj.weight, tok_mod.proj.bias, 0)
    pe = LinearFn.apply(centers, tok_mod.pos_embed[0].weight, tok_mod.pos_embed[0].bias, 2)
    pe = LinearFn.apply(pe, tok_mod.pos_embed[2].weight, tok_mod.pos_embed[2].bias, 0)
    feats = torch.cat([tok_mod.cls_token.float().expand(B, -1, -1), x], dim=1)
    pos = torch.cat([tok_mod.cls_pos.float().expand(B, -1, -1), pe], dim=1)
    return feats, pos
