"""Drop-in for the reference's PointViT (src/models/pix4point.py:194-271): P3Embed tokenizer -> proj / pos_embed / cls concat
-> the ViT blocks with `feats + pos_embed` re-added in front of every block -> final norm -> 'max,cls' global features.

The reference takes its blocks from `timm.create_model(...)` (pix4point.py:221-228); timm is not part of the reference tree
(pinned timm==1.0.16, requirements.txt) and is not installed here, so the block containers below carry timm's `Block`
parameter layout (`vit.blocks.{i}.norm1 / attn.qkv / attn.proj / norm2 / mlp.fc1 / mlp.fc2`, `vit.norm`, `vit.cls_token`,
`vit.pos_embed`) - a PointViT checkpoint loads with strict=False (timm's own unused patch embedding / head are skipped).
forward runs the sm_100a kernels (`p3tok::vit_blocks`: the APF block-stack kernels without the adapter columns, the
positional add fused into each block's first normalisation pass; `p3tok::vit_blocks_x3` with block_precision="fp32tc") in
eval mode; `.train()` - or a gradient wanted through
eval-mode blocks - takes the fp32 autograd path of p3tok/train_vit.py (Pix4Point trains everything, or everything but `vit.*`
with frozen=True, pix4point.py:229-233).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import nn

from . import ops
from .apf_model import bf16_layer, check_block_precision, x3_layer
from .modules import PointViTTokens, wants_input_grad


class _Attn(nn.Module):
    def __init__(self, dim: int, num_heads: int):
        super().__init__()
        self.num_heads = num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)


class _Mlp(nn.Module):
    def __init__(self, dim: int, hidden: int):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class TimmBlock(nn.Module):
    """Parameter container with timm.models.vision_transformer.Block's names (norm eps 1e-6 as timm builds ViTs)."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, eps: float = 1e-6):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=eps)
        self.attn = _Attn(dim, num_heads)
        self.norm2 = nn.LayerNorm(dim, eps=eps)
        self.mlp = _Mlp(dim, int(dim * mlp_ratio))


def fold_timm_block64(blk: TimmBlock) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """A block folded into the four GEMMs of struct p3tok_vit_layer (LayerNorm affines moved into the consuming weights) in
    float64: (matrix, bias) for qkv, proj, fc1, fc2."""
    d = lambda t: t.detach().double()
    g1, b1, g2, b2 = d(blk.norm1.weight), d(blk.norm1.bias), d(blk.norm2.weight), d(blk.norm2.bias)
    qw, qb = d(blk.attn.qkv.weight), d(blk.attn.qkv.bias)
    f1w, f1b = d(blk.mlp.fc1.weight), d(blk.mlp.fc1.bias)
    return [(qw * g1[None, :], qb + qw @ b1), (d(blk.attn.proj.weight), d(blk.attn.proj.bias)),
            (f1w * g2[None, :], f1b + f1w @ b2), (d(blk.mlp.fc2.weight), d(blk.mlp.fc2.bias))]


def fold_timm_block(blk: TimmBlock) -> List[torch.Tensor]:
    """fold_timm_block64 as bf16 matrices / f32 biases in ops.VIT_LAYER_TENSORS order (ops.vit_blocks)."""
    return bf16_layer(fold_timm_block64(blk))


def fold_timm_block_x3(blk: TimmBlock) -> List[torch.Tensor]:
    """fold_timm_block64 in the x3 form of the fp32-accurate stack (ops.vit_blocks_x3, apf_model.x3_layer)."""
    return x3_layer(fold_timm_block64(blk))


class _Vit(nn.Module):
    """The slice of timm's VisionTransformer PointViT uses: blocks, norm, cls_token, pos_embed (only its first row, as cls_pos)."""

    def __init__(self, dim: int, depth: int, num_heads: int, mlp_ratio: float, seq: int = 577):
        super().__init__()
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, seq, dim))
        self.blocks = nn.ModuleList([TimmBlock(dim, num_heads, mlp_ratio) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)


class PointViT(nn.Module):
    """pix4point.py:194-271.  forward(p, x=None) -> (p_list, x_list, feats (B,1+G,E) after the final norm);
    forward_cls_feat(p, x=None) -> (B, E * len(global_features)).  Defaults = vit_small_patch16_384 (E 384, depth 12, 6 heads).
    `precision` selects the tokenizer's embed path, `block_precision` the block stack's: "bf16" (default, rtol 1e-2) or
    "fp32tc" (bf16x3 split operands on the same kernels, rtol 1e-4)."""

    def __init__(self, in_channels: int = 3, embed_dim: int = 384, pretrained_model: str = "vit_small_patch16_384.augreg_in21k_ft_in1k",
                 pretrained: bool = False, frozen: bool = False, k_neighbors: int = 16, global_features: str = "max,cls",
                 depth: int = 12, num_heads: int = 6, mlp_ratio: float = 4.0, precision: str = "bf16", block_precision: str = "bf16",
                 **p3embed_kwargs):
        super().__init__()
        check_block_precision(block_precision)
        self.block_precision = block_precision
        if pretrained:
            raise RuntimeError("PointViT: no timm / network in this build - construct with pretrained=False and load_state_dict() "
                               "a reference checkpoint (strict=False: timm's unused patch embedding / head keys are skipped)")
        self.num_features = self.embed_dim = embed_dim
        self.global_features = global_features.split(",")
        tok = PointViTTokens(in_channels=in_channels, embed_dim=embed_dim, k_neighbors=k_neighbors, precision=precision, **p3embed_kwargs)
        self.patch_embed, self.proj, self.pos_embed = tok.patch_embed, tok.proj, tok.pos_embed
        self.vit = _Vit(embed_dim, depth, num_heads, mlp_ratio)
        self.vit_blocks = self.vit.blocks                    # aliases, as in the reference (pix4point.py:224-228)
        self.norm = self.vit.norm
        self.cls_token = self.vit.cls_token
        self.cls_pos = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.__dict__["_tok"] = tok                          # not a registered submodule: its parameters are the ones above
        tok.cls_token, tok.cls_pos = self.cls_token, self.cls_pos
        if frozen:                                           # pix4point.py:229-233
            for name, param in self.named_parameters():
                if "vit" in name:
                    param.requires_grad = False

    def _folded(self) -> List[torch.Tensor]:
        ver = tuple((t._version, t.data_ptr()) for t in self.vit.blocks.parameters())
        cache = self.__dict__.setdefault("_fold_cache", {})
        hit = cache.get(self.block_precision)
        if hit is None or hit[0] != ver:
            fold_block = fold_timm_block_x3 if self.block_precision == "fp32tc" else fold_timm_block
            hit = (ver, [t for blk in self.vit.blocks for t in fold_block(blk)])
            cache[self.block_precision] = hit
        return hit[1]

    def _run(self, p: torch.Tensor, x: Optional[torch.Tensor], start_idx=None):
        tok = self.__dict__["_tok"]
        tok.train(self.training)                             # not a registered submodule: follow the owner's mode
        p_list, x_list, feats, pos = tok(p, x, start_idx)
        if self.training or (torch.is_grad_enabled() and (feats.requires_grad or pos.requires_grad)):
            from . import train_vit
            out = train_vit.timm_blocks_train(self.vit.blocks, self.norm, feats, pos)
            return p_list, x_list, out, train_vit.TokenMaxFn.apply(out, 1)
        eps = {float(n.eps) for blk in self.vit.blocks for n in (blk.norm1, blk.norm2)} | {float(self.norm.eps)}
        if len(eps) != 1:
            raise RuntimeError(f"PointViT: all LayerNorms must share one eps, got {sorted(eps)}")
        heads = self.vit.blocks[0].attn.num_heads
        blocks = ops.vit_blocks_x3 if self.block_precision == "fp32tc" else ops.vit_blocks
        out, pooled = blocks(feats, pos, self._folded(), heads, self.norm.weight.detach().float(), self.norm.bias.detach().float(),
                             eps.pop(), 1)
        return p_list, x_list, out, pooled

    def forward(self, p: torch.Tensor, x: Optional[torch.Tensor] = None, start_idx=None) -> Tuple[list, list, torch.Tensor]:
        p_list, x_list, out, _ = self._run(p, x, start_idx)
        return p_list, x_list, out

    def forward_cls_feat(self, p: torch.Tensor, x: Optional[torch.Tensor] = None, start_idx=None) -> torch.Tensor:
        _, _, out, pooled = self._run(p, x, start_idx)
        feats = []
        for token_type in self.global_features:              # pix4point.py:264-269
            if "cls" in token_type:
                feats.append(out[:, 0, :])
            if "max" in token_type:
                feats.append(pooled)
        return torch.cat(feats, dim=1)


class ClsHead(nn.Module):
    """pix4point.py:295-325: (Linear -> BatchNorm1d -> ReLU -> Dropout) per hidden width, then Linear; attribute `head`, same
    state_dict keys.  eval: BatchNorm folded into the linears (p3tok::linear_f32); train: p3tok/train_vit.py (batch statistics,
    dropout keep masks, gradients)."""

    def __init__(self, in_channels: int = 768, num_classes: int = 15, mlps: Optional[List[int]] = None, dropout: float = 0.5,
                 point_dim: int = 2):
        super().__init__()
        self.point_dim = point_dim
        widths = [in_channels] + list(mlps if mlps is not None else [256, 256]) + [num_classes]
        layers: List[nn.Module] = []
        for i in range(len(widths) - 2):
            layers += [nn.Linear(widths[i], widths[i + 1], True), nn.BatchNorm1d(widths[i + 1]), nn.ReLU(), nn.Dropout(dropout)]
        layers += [nn.Linear(widths[-2], widths[-1], True)]
        self.head = nn.Sequential(*layers)

    def forward(self, end_points: torch.Tensor) -> torch.Tensor:
        from . import train_vit
        if self.training or wants_input_grad(end_points):   # eval mode + gradient wanted: running statistics, dropout off
            return train_vit.head_train(self, end_points, running=not self.training)
        blocks, last = train_vit.mlp_head_blocks(self.head)
        x = end_points.float().contiguous()
        for lin, bn, _ in blocks:
            s = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + bn.eps)
            w = (lin.weight.detach().double() * s[:, None]).float().contiguous()
            b = ((lin.bias.detach().double() - bn.running_mean.double()) * s + bn.bias.detach().double()).float().contiguous()
            x = ops.linear_f32(x, w, b, True)
        return ops.linear_f32(x, last.weight.detach().float().contiguous(), last.bias.detach().float().contiguous(), False)


class Pix4Point(nn.Module):
    """pix4point.py:328-437: PointViT encoder (`model`) + ClsHead on its 'max,cls' global features (`cls_head`, 2 * embed_dim
    inputs).  Same constructor arguments (plus the PointViT geometry, since timm cannot supply it here), same initialisation
    (xavier linears, zero biases, unit BatchNorm; cls token / position ~ N(0, 0.02) when not pretrained), same helpers.
    pointvit_kwargs go to PointViT (precision, block_precision, depth, num_heads, ...)."""

    def __init__(self, num_classes: int = 15, embed_dim: int = 768, pretrained_model: str = "vit_small_patch16_384.augreg_in21k_ft_in1k",
                 pretrained: bool = False, frozen: bool = False, k_neighbors: int = 16, **pointvit_kwargs):
        super().__init__()
        self.pretrained = pretrained
        self.model = PointViT(pretrained_model=pretrained_model, pretrained=pretrained, embed_dim=embed_dim, k_neighbors=k_neighbors,
                              frozen=frozen, **pointvit_kwargs)
        self.cls_head = ClsHead(in_channels=2 * embed_dim, num_classes=num_classes)
        self.initialize_weights()

    def initialize_weights(self):
        if not self.pretrained:
            torch.nn.init.normal_(self.model.cls_token, std=.02)
            torch.nn.init.normal_(self.model.cls_pos, std=.02)
        for name, module in self.named_modules():
            if name.startswith("vit") and self.pretrained:
                continue
            self._init_weights(module)

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            torch.nn.init.xavier_uniform_(m.weight)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    def get_param_groups(self):
        """pix4point.py:388-401: weight decay for everything but cls token / position, biases and norms."""
        decay, no_decay = [], []
        for name, param in self.named_parameters():
            if not param.requires_grad:
                continue
            if "cls_token" in name or "cls_pos" in name or name.endswith(".bias") or "norm" in name:
                no_decay.append(param)
            else:
                decay.append(param)
        return [{"params": decay}, {"params": no_decay, "weight_decay": 0.0}]

    def get_trainable_params(self):
        return filter(lambda p: p.requires_grad, self.model.parameters())

    def forward(self, points: torch.Tensor, start_idx=None) -> torch.Tensor:
        return self.cls_head(self.model.forward_cls_feat(points, None, start_idx))
