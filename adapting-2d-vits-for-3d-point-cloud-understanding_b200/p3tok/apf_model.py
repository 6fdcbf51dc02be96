"""Drop-ins for the consumer of the APF tokens (SURVEY.md 8f "next" #3): the reference's ViT block stack.

  AttentionLayer / AdapterLayer / APFViTLayer  <- reference src/models/apf_utils.py:106-293
  ClassificationHead / AdaptPointFormer        <- reference src/models/apf.py:219-373

Same constructor arguments, attribute names and state_dict keys (`blocks.{i}.norm1`, `.attention.qkv`, `.mlp.fc1`,
`.adapter.down_proj`, `encoder_norm`, `point_encoder.encoder.first_conv.0`, `head.mlp_head.0`, ...), so a reference
checkpoint loads with strict=True.  The torch submodules are parameter containers.  Serving (eval mode, no gradient
wanted): forward runs `p3tok::apf_vit` - LayerNorm -> tcgen05 GEMMs with GELU / residual epilogues -> attention, fp32
residual stream, the head's BatchNorms folded - or, with block_precision="fp32tc", `p3tok::apf_vit_x3`, the same kernels on
bf16x3 split operands (fp32-accurate).  Training (`.train()`, or a gradient is wanted through eval-mode blocks):
the fp32 autograd path of p3tok/train_vit.py - dropout / DropPath as keep masks, BatchNorm batch statistics, gradients
for the tokens and for every parameter that requires one (the reference keeps point_encoder / encoder_norm / head
trainable, apf.py:335-346).  Differences from the reference constructor: no timm / no network here, so
`pretrained=True` raises - load a state_dict instead.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch
from torch import nn

from . import fold, ops
from .modules import PointNet, wants_input_grad


class _Mlp(nn.Module):
    """timm.models.layers.Mlp's parameter layout (fc1 -> GELU -> fc2); container only."""

    def __init__(self, in_features: int, hidden_features: int):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.fc2 = nn.Linear(hidden_features, in_features)


class AttentionLayer(nn.Module):
    """apf_utils.py:106-160 (container; evaluated inside p3tok::apf_vit)."""

    def __init__(self, dim: int, num_heads: int):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)


class AdapterLayer(nn.Module):
    """apf_utils.py:162-233 (container).  Same initialisation: kaiming down_proj, zero up_proj / biases."""

    def __init__(self, model_dimension: int = 768, bottleneck: int = 64, dropout: float = 0.0):
        super().__init__()
        self.n_embd, self.down_size, self.dropout = model_dimension, bottleneck, dropout
        self.adapter_norm = nn.LayerNorm(self.n_embd)
        self.scale = nn.Parameter(torch.ones(1))
        self.down_proj = nn.Linear(self.n_embd, self.down_size)
        self.relu = nn.ReLU()
        self.up_proj = nn.Linear(self.down_size, self.n_embd)
        with torch.no_grad():
            nn.init.kaiming_uniform_(self.down_proj.weight, a=math.sqrt(5))
            nn.init.zeros_(self.up_proj.weight)
            nn.init.zeros_(self.down_proj.bias)
            nn.init.zeros_(self.up_proj.bias)


class APFViTLayer(nn.Module):
    """apf_utils.py:236-293.  forward(x (B,G,D)) -> (B,G,D); a single layer is a 1-layer stack."""

    def __init__(self, dim: int = 768, num_heads: int = 12, drop_path: float = 0.0, dropout: float = 0.1):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(dim)
        self.drop_path = nn.Identity()                     # parameter-free; the rate below drives the train-mode keep masks
        self.drop_path_rate = float(drop_path)             # apf_utils.py:258 (timm DropPath, scale_by_keep)
        self.mlp = _Mlp(dim, dim * 4)
        self.attention = AttentionLayer(dim=dim, num_heads=num_heads)
        self.adapter = AdapterLayer(model_dimension=dim, dropout=dropout)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return run_blocks([self], x, None)[0]


def fold_vit_layer64(layer: "APFViTLayer") -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """One APFViTLayer folded into the four GEMMs of struct p3tok_vit_layer (include/p3tok.h) in float64: (matrix, bias) for
    qkv, proj, fc1d, fc2u:
      LayerNorm affines move into the weights that consume the normalised rows (W diag(g), b + W beta);
      norm2 and adapter_norm share their statistics, so [fc1 ; down_proj] is one GEMM on one normalised matrix;
      [fc2 | scale * up_proj] consumes [gelu(fc1) | relu(down)] whole (apf_utils.py:217-233, 284-292)."""
    d = lambda t: t.detach().double()
    g1, b1 = d(layer.norm1.weight), d(layer.norm1.bias)
    g2, b2 = d(layer.norm2.weight), d(layer.norm2.bias)
    ga, ba = d(layer.adapter.adapter_norm.weight), d(layer.adapter.adapter_norm.bias)
    sc = d(layer.adapter.scale).reshape(())
    qw, qb = d(layer.attention.qkv.weight), d(layer.attention.qkv.bias)
    f1w, f1b = d(layer.mlp.fc1.weight), d(layer.mlp.fc1.bias)
    dw, db = d(layer.adapter.down_proj.weight), d(layer.adapter.down_proj.bias)
    f2w, f2b = d(layer.mlp.fc2.weight), d(layer.mlp.fc2.bias)
    uw, ub = d(layer.adapter.up_proj.weight), d(layer.adapter.up_proj.bias)
    return [
        (qw * g1[None, :], qb + qw @ b1),
        (d(layer.attention.proj.weight), d(layer.attention.proj.bias)),
        (torch.cat([f1w * g2[None, :], dw * ga[None, :]], 0), torch.cat([f1b + f1w @ b2, db + dw @ ba], 0)),
        (torch.cat([f2w, sc * uw], 1), f2b + sc * ub),
    ]


def bf16_layer(mats) -> List[torch.Tensor]:
    """float64 (matrix, bias) pairs -> bf16 matrices / f32 biases in ops.VIT_LAYER_TENSORS order (the bf16 stack)."""
    out: List[torch.Tensor] = []
    for w, b in mats:
        out += [w.to(torch.bfloat16).contiguous(), b.float().contiguous()]
    return out


def x3_layer(mats) -> List[torch.Tensor]:
    """float64 (matrix, bias) pairs -> the x3 form of the fp32-accurate stack (include/p3tok.h p3tok_apf_vit_forward_x3): every
    matrix fold.split_x3 [W_hi | W_hi | W_lo] over its input padded to a multiple of 64, fc1d's rows and bias padded with zeros
    to pad64(H + R) (so fc2u's reduction length matches), f32 biases, in ops.VIT_LAYER_TENSORS order."""
    (qw, qb), (pw, pb), (f1w, f1b), (f2w, f2b) = mats
    hrp = fold.pad64(f1w.shape[0])
    f1bp = f1b.new_zeros(hrp)
    f1bp[:f1b.shape[0]] = f1b
    out: List[torch.Tensor] = []
    for w, b, rows in ((qw, qb, None), (pw, pb, None), (f1w, f1bp, hrp), (f2w, f2b, None)):
        out += [fold.split_x3(w, rows), b.float().contiguous()]
    return out


def fold_vit_layer(layer: "APFViTLayer") -> List[torch.Tensor]:
    """fold_vit_layer64 as bf16 matrices / f32 biases in ops.VIT_LAYER_TENSORS order (the bf16 stack, ops.apf_vit)."""
    return bf16_layer(fold_vit_layer64(layer))


def fold_vit_layer_x3(layer: "APFViTLayer") -> List[torch.Tensor]:
    """fold_vit_layer64 in the x3 form of the fp32-accurate stack (ops.apf_vit_x3)."""
    return x3_layer(fold_vit_layer64(layer))


BLOCK_PRECISIONS = ("bf16", "fp32tc")


def check_block_precision(p: str) -> bool:
    """True for the fp32-accurate block stack ("fp32tc": bf16x3 on the tensor cores), False for "bf16"."""
    if p not in BLOCK_PRECISIONS:
        raise ValueError(f"block_precision must be 'bf16' or 'fp32tc', got {p!r}")
    return p == "fp32tc"


def _layer_params(layer: "APFViTLayer", cache: dict, precision: str = "bf16") -> List[torch.Tensor]:
    """fold_vit_layer (fold_vit_layer_x3 for "fp32tc"), cached per parameter version and precision (no host synchronisation
    on the steady-state path)."""
    ver = tuple((t._version, t.data_ptr()) for t in layer.parameters())
    key = (id(layer), precision)
    hit = cache.get(key)
    if hit is None or hit[0] != ver:
        hit = (ver, fold_vit_layer_x3(layer) if precision == "fp32tc" else fold_vit_layer(layer))
        cache[key] = hit
    return hit[1]


def _wants_autograd(layers, x: torch.Tensor, final_norm: Optional[nn.LayerNorm]) -> bool:
    """The fp32 autograd path (train_vit) instead of the serving kernels: any layer in train mode, or a gradient is wanted
    for the input (frozen eval-mode blocks still pass the tokenizer's gradient through, apf.py:335-346).  Eval-mode modules on
    an input without gradient always take the serving path, whatever `requires_grad` their parameters carry."""
    if any(l.training for l in layers) or (final_norm is not None and final_norm.training):
        return True
    return torch.is_grad_enabled() and x.requires_grad


def run_blocks(layers, x: torch.Tensor, final_norm: Optional[nn.LayerNorm], cache: Optional[dict] = None,
               precision: str = "bf16"):
    """(x after the last layer, pooled = max over tokens of final_norm(x) or None).  precision: "bf16" (ops.apf_vit, rtol 1e-2)
    or "fp32tc" (ops.apf_vit_x3: the same kernels on bf16x3 split operands, rtol 1e-4); train mode and gradient-wanted calls
    take the fp32 autograd path whatever it says."""
    x3 = check_block_precision(precision)
    layers = list(layers)
    if _wants_autograd(layers, x, final_norm):
        from . import train_vit
        return train_vit.blocks_train(layers, x, final_norm)
    cache = {} if cache is None else cache
    params: List[torch.Tensor] = []
    for l in layers:
        params += _layer_params(l, cache, precision)
    heads = layers[0].attention.num_heads
    D = x.shape[-1]
    # one eps for every normalisation of the stack (norm2 and adapter_norm share their statistics in the folded layer)
    norms = [n for l in layers for n in (l.norm1, l.norm2, l.adapter.adapter_norm)] + ([final_norm] if final_norm is not None else [])
    eps = {float(n.eps) for n in norms}
    if len(eps) != 1:
        raise RuntimeError(f"APFViTLayer stack: all LayerNorms must share one eps, got {sorted(eps)}")
    ln_eps = eps.pop()
    if final_norm is None:
        fw, fb = torch.ones(D, device=x.device), torch.zeros(D, device=x.device)
    else:
        fw, fb = final_norm.weight.detach().float(), final_norm.bias.detach().float()
    y, pooled = (ops.apf_vit_x3 if x3 else ops.apf_vit)(x.float(), params, heads, layers[0].adapter.down_size, fw, fb, ln_eps)
    return y, (pooled if final_norm is not None else None)


class ClassificationHead(nn.Module):
    """apf.py:219-252.  Linear -> BN -> ReLU -> Dropout -> Linear -> BN -> ReLU -> Dropout -> Linear; eval mode: the
    BatchNorms fold into the linears (p3tok::linear_f32, fp32 on CUDA cores - a (B,E) problem)."""

    def __init__(self, in_channels: int, num_classes: int):
        super().__init__()
        self.mlp_head = nn.Sequential(
            nn.Linear(in_channels, 512), nn.BatchNorm1d(512), nn.ReLU(inplace=True), nn.Dropout(p=0.4),
            nn.Linear(512, 256), nn.BatchNorm1d(256), nn.ReLU(inplace=True), nn.Dropout(p=0.4),
            nn.Linear(256, num_classes))

    def _fold(self, lin: nn.Linear, bn: Optional[nn.BatchNorm1d]):
        w, b = lin.weight.detach().double(), lin.bias.detach().double()
        if bn is not None:
            s = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + bn.eps)
            w = w * s[:, None]
            b = (b - bn.running_mean.double()) * s + bn.bias.detach().double()
        return w.float().contiguous(), b.float().contiguous()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.training or wants_input_grad(x):         # eval mode + gradient wanted: running statistics, dropout off
            from . import train_vit
            return train_vit.head_train(self, x, sync=bool(getattr(self, "sync_bn", False)), running=not self.training)
        m = self.mlp_head
        x = x.float().contiguous()
        for lin, bn, relu in ((m[0], m[1], True), (m[4], m[5], True), (m[8], None, False)):
            w, b = self._fold(lin, bn)
            x = ops.linear_f32(x, w, b, relu)
        return x


class AdaptPointFormer(nn.Module):
    """apf.py:254-373.  forward(x (B,N,C)) -> (B,num_classes) logits: PointNet tokenizer -> 12 APFViTLayers ->
    encoder_norm -> max over tokens -> classification head.  `precision` selects the tokenizer's embed path,
    `block_precision` the block stack's: "bf16" (default) runs bf16 GEMMs on tcgen05 with an fp32 residual stream (rtol
    1e-2), "fp32tc" the same kernels on bf16x3 split operands (rtol 1e-4, the fp32 contract; about 3x the tensor work)."""

    def __init__(self, num_classes: int = 15, embedding_dim: int = 768, vit_name: str = "vit_base_patch16_224",
                 pretrained: bool = False, npoint: int = 196, nsample: int = 32, in_channels: int = 3,
                 dropout_rate: float = 0.1, dropout_path_rate: float = 0.1, precision: str = "bf16",
                 block_precision: str = "bf16"):
        super().__init__()
        check_block_precision(block_precision)
        self.block_precision = block_precision
        if pretrained:
            raise RuntimeError("AdaptPointFormer: no timm / network in this build - construct with pretrained=False and "
                               "load_state_dict() a reference checkpoint (keys are identical)")
        in_channels = in_channels * 2                      # apf.py:293: [rel || centre] concat
        depth = 12
        dpr = [v.item() for v in torch.linspace(0, dropout_path_rate, depth)]      # apf.py:298: deeper layers drop more
        self.dropout = nn.Dropout(dropout_rate)
        self.encoder_norm = nn.LayerNorm(embedding_dim)
        self.point_encoder = PointNet(embedding_dim, npoint, nsample, in_channels, precision=precision)
        self.head = ClassificationHead(in_channels=embedding_dim, num_classes=num_classes)
        self.blocks = nn.Sequential(*[APFViTLayer(dim=embedding_dim, num_heads=12, drop_path=dpr[i], dropout=dropout_rate)
                                      for i in range(depth)])

    def features(self, x: torch.Tensor, start_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
        """(B,D) pooled features: everything before the classification head (apf.py:358-366)."""
        tok = self.point_encoder(x, start_idx)
        cache = self.__dict__.setdefault("_vit_cache", {})
        return run_blocks(self.blocks, tok, self.encoder_norm, cache, self.block_precision)[1]

    def _freeze(self) -> None:
        """apf.py:335-346 verbatim in effect: everything frozen except parameters whose name contains 'adaptmlp', 'head',
        'enc_norm' or 'encoder' (point_encoder.*, encoder_norm.*, head.*; the adapters are named `adapter` and stay frozen)."""
        for param in self.parameters():
            param.requires_grad_(False)
        for name, param in self.named_parameters():
            if "adaptmlp" in name or "head" in name or "enc_norm" in name or "encoder" in name:
                param.requires_grad = True

    def forward(self, x: torch.Tensor, start_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
        feats = self.features(x, start_idx)
        if self.dropout.training and self.dropout.p > 0:                          # apf.py:368
            from . import train_vit
            feats = train_vit.dropout(feats, float(self.dropout.p), True)
        return self.head(feats)
