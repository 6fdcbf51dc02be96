"""nn.Module drop-ins for the reference's tokenizer modules, same constructor and forward
signatures and the same state_dict keys, running on the sm_100a kernels.

  Group / Encoder / PointNet  <- reference src/models/apf.py:12-217
  P3Embed                     <- reference src/models/pix4point.py:105-191

The parameter containers (Conv1d/BatchNorm1d/... inside nn.Sequential at the reference's
indices) exist so reference checkpoints load with strict=True; forward never calls them.
eval():  BatchNorm uses the running statistics, folded into the weights (p3tok/fold.py); `precision` selects
         "fp32" (CUDA-core FFMA, rtol 1e-4 contract) or "bf16" (tcgen05 tensor cores, rtol 1e-2 contract).
eval() with a gradient wanted for the input (grad mode on and the input requires grad, `wants_input_grad`): the fp32
         autograd path of train() with running-statistics BatchNorm - buffers untouched, nothing all-reduced - so x.grad
         (and the gradient of every parameter that requires one) is filled as with the reference; fp32 tokens whatever
         `precision` / `token_dtype` say.  Every other eval-mode call runs the serving kernels above.
train(): batch-statistics BatchNorm (running estimates updated like nn.BatchNorm) and autograd through both
         max-pools, the concat and the gather to the input points - p3tok/train.py over csrc/train.cu, fp32 (SURVEY.md 8f
         "next" #4); `sync_bn=True` all-reduces the BatchNorm sums when the batch is sharded over ranks.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import torch
from torch import nn

from . import _lib, fold, ops, train
from .functional import _start


def _check_precision(p: str) -> bool:
    """True for the plain bf16 tensor-core path.  "fp32" = CUDA-core FFMA, "fp32tc" = the same rtol-1e-4 contract on the
    tensor cores (bf16x3 split operands, csrc/embed_tc.cu patch_embed_x3)."""
    if p not in ("fp32", "bf16", "fp32tc"):
        raise ValueError(f"precision must be 'fp32', 'fp32tc' or 'bf16', got {p!r}")
    return p == "bf16"


def _check_token_dtype(token_dtype, precision: str) -> bool:
    """True when the tokens leave as bfloat16 (bf16 path only); default float32 like the reference."""
    if token_dtype in (None, torch.float32):
        return False
    if token_dtype != torch.bfloat16:
        raise ValueError(f"token_dtype must be torch.float32 or torch.bfloat16, got {token_dtype!r}")
    if precision != "bf16":
        raise ValueError("token_dtype=torch.bfloat16 needs precision='bf16'")
    return True


def wants_input_grad(*inputs: Optional[torch.Tensor]) -> bool:
    """An eval-mode module takes the fp32 autograd path (running-statistics BatchNorm) only when a gradient is wanted for one of
    its inputs - grad mode on and the input requires grad (the rule of apf_model._wants_autograd).  Any other eval-mode call,
    whatever `requires_grad` the parameters carry, runs the serving kernels."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in inputs)


def _bn_eps(module: nn.Module):
    """{prefix of each BatchNorm in `module`: its eps} - the folding uses the module's eps, not a constant."""
    return {name: float(m.eps) for name, m in module.named_modules()
            if isinstance(m, (nn.BatchNorm1d, nn.BatchNorm2d))}


class _FoldedMixin:
    """Caches the folded weights per (device, dtype); refolds when any parameter changes."""

    def _folded(self, build, device, bf16: bool) -> fold.PatchMLP:
        ver = tuple((t._version, t.data_ptr()) for t in list(self.parameters()) + list(self.buffers()))
        cache = self.__dict__.setdefault("_fold_cache", {})
        if cache.get("ver") != ver:
            cache.clear()
            cache["ver"] = ver
            cache["host"] = build()
        if getattr(self, "precision", None) == "fp32tc":
            return cache["host"].to_x3(device)
        return cache["host"].to(device, torch.bfloat16 if bf16 else torch.float32)

    def _require_eval(self):
        if self.training:
            raise RuntimeError(
                f"{type(self).__name__}: p3tok implements the eval-mode (folded BatchNorm) forward only; "
                "call .eval() first (training-mode batch statistics are out of scope, SURVEY.md 8f)")


class Group(nn.Module):
    """apf.py:12-112.  forward(x (B,N,C), xyz (B,N,3)) -> (neighborhood (B,G,k,2C), center (B,G,3)),
    groups in Morton order of their centres.  The reference's dead cdist(center,center) work
    (apf.py:38-39) is not reproduced."""

    def __init__(self, num_group: int, group_size: int):
        super().__init__()
        self.num_group = num_group
        self.group_size = group_size

    def indices(self, x: torch.Tensor, start_idx: Optional[torch.Tensor] = None):
        """(fps_idx (B,G), center (B,G,3), knn_idx (B,G,k), perm (B,G)) - the index half of forward, computed on the
        coordinates x[..., :3] (read in place when x has 3 or 4 channels)."""
        fps_idx, ws = ops.fps_with_knn_prepare(x, _start(x, start_idx), self.num_group)   # kNN preparation overlaps FPS
        center = ops.gather_points(x, fps_idx)[..., :3].contiguous() if x.shape[-1] != 3 else ops.gather_points(x, fps_idx)
        knn_idx = ops.knn_query(x, ws, center, self.group_size, _lib.KNN_APF_SQ, False)
        perm = ops.morton_order(center)[0]
        return fps_idx, center, knn_idx, perm

    @staticmethod
    def _xyz_is_prefix_of(x: torch.Tensor, xyz: torch.Tensor) -> bool:
        """xyz is x[:, :, :3] itself (the reference's only call site, apf.py:212-214): same storage, same strides."""
        return (xyz.shape[-1] == 3 and xyz.dtype == x.dtype and xyz.device == x.device and xyz.data_ptr() == x.data_ptr()
                and xyz.stride() == x.stride())

    def forward(self, x: torch.Tensor, xyz: torch.Tensor, start_idx: Optional[torch.Tensor] = None):
        """FPS, kNN and the Morton order run on `xyz`, the gather / centre-subtraction on `x` (apf.py:64-95).  When xyz
        is the x[:, :, :3] view (apf.py:212-214) the kernels read it in place; any other xyz (normalised, augmented)
        is honoured through a contiguous copy, and the returned centres are xyz rows as in the reference (apf.py:70)."""
        if xyz.shape[:2] != x.shape[:2] or xyz.shape[-1] != 3:
            raise RuntimeError("Group.forward: xyz must be (B,N,3) with x's B and N")
        if x.dtype == torch.float32 and x.is_contiguous() and self._xyz_is_prefix_of(x, xyz):
            fps_idx, _, knn_idx, perm = self.indices(x, start_idx)
            return ops.apf_group(x, fps_idx, knn_idx, perm)
        x = x.float().contiguous()
        pts = xyz.float().contiguous()
        fps_idx, center, knn_idx, perm = self.indices(pts, start_idx)
        neigh, _ = ops.apf_group(x, fps_idx, knn_idx, perm)
        center = torch.gather(center, 1, perm.unsqueeze(-1).expand(-1, -1, 3))      # Morton order of the xyz centres
        return neigh, center


class Encoder(nn.Module, _FoldedMixin):
    """apf.py:114-181.  forward(point_groups (B,G,k,Cin)) -> (B,G,E)."""

    def __init__(self, encoder_channel: int, in_channel: int, precision: str = "fp32", token_dtype=None, sync_bn: bool = False):
        super().__init__()
        self.encoder_channel = encoder_channel
        self.precision = precision
        self.token_dtype = token_dtype
        self.sync_bn = sync_bn                  # train mode: all-reduce the BatchNorm sums over torch.distributed ranks
        E = encoder_channel
        self.first_conv = nn.Sequential(
            nn.Conv1d(in_channel, 256, 1), nn.BatchNorm1d(256), nn.ReLU(inplace=True),
            nn.Conv1d(256, 512, 1), nn.BatchNorm1d(512), nn.ReLU(inplace=True),
            nn.Conv1d(512, E, 1))
        self.second_conv = nn.Sequential(
            nn.Conv1d(2 * E, 2 * E, 1), nn.BatchNorm1d(2 * E), nn.ReLU(inplace=True),
            nn.Conv1d(2 * E, E, 1))

    def folded(self, device) -> fold.PatchMLP:
        return self._folded(lambda: fold.fold_apf_encoder(self.state_dict(), _bn_eps(self)), device,
                            _check_precision(self.precision))

    def forward(self, point_groups: torch.Tensor) -> torch.Tensor:
        B, G, k, cin = point_groups.shape
        if self.training or wants_input_grad(point_groups):   # autograd (p3tok/train.py), fp32; eval: running statistics
            rows = point_groups.float().reshape(B * G * k, cin)
            return train.encoder_train(self, rows, k, self.sync_bn, not self.training).view(B, G, self.encoder_channel)
        m = self.folded(point_groups.device)
        rows = point_groups.float().reshape(B * G * k, cin)
        tok = ops.patch_embed(_lib.ROWS_DIRECT, rows, None, None, None, None, B * G, k, m.tensors(), m.meta(),
                              _check_precision(self.precision), _check_token_dtype(self.token_dtype, self.precision),
                              self.precision == "fp32tc")
        return tok.view(B, G, self.encoder_channel)

    get_features = forward


class PointNet(nn.Module):
    """apf.py:183-217.  forward(x (B,N,C)) -> (B,G,E).  Fused: the (B,G,k,2C) neighbourhood tensor
    is never written - the embed kernels gather, centre-subtract and apply the Morton order as the
    output row."""

    def __init__(self, embed_dim: int, num_group: int, group_size: int, in_channel: int, precision: str = "fp32",
                 token_dtype=None, sync_bn: bool = False):
        super().__init__()
        self.group = Group(num_group, group_size)
        self.encoder = Encoder(embed_dim, in_channel, precision, token_dtype, sync_bn)

    def forward(self, x: torch.Tensor, start_idx: Optional[torch.Tensor] = None) -> torch.Tensor:
        x = x.float().contiguous()
        B, N, C = x.shape
        G, k = self.group.num_group, self.group.group_size
        with torch.no_grad():
            fps_idx, _, knn_idx, perm = self.group.indices(x, start_idx)
        if self.encoder.training or wants_input_grad(x):
            # autograd: the gathered rows (differentiable with respect to x) feed the Encoder - batch statistics in train mode,
            # running statistics in eval mode (p3tok/train.py)
            rows = train.apf_rows(x, fps_idx, knn_idx, perm)
            return train.encoder_train(self.encoder, rows, k, self.encoder.sync_bn, not self.encoder.training).view(B, G, -1)
        m = self.encoder.folded(x.device)
        if m.cin != 2 * C:
            raise RuntimeError(f"PointNet: in_channel={m.cin} but input has C={C} (expects in_channel == 2*C)")
        tok = ops.patch_embed(_lib.ROWS_APF, x, None, fps_idx, knn_idx, perm, B * G, k, m.tensors(), m.meta(),
                              _check_precision(self.encoder.precision),
                              _check_token_dtype(self.encoder.token_dtype, self.encoder.precision), self.encoder.precision == "fp32tc")
        return tok.view(B, G, -1)


class P3Embed(nn.Module, _FoldedMixin):
    """pix4point.py:105-191.  forward(p (B,N,3), f (B,D,N)) -> ([p, (B,N/4,3), ...], [f, (B,W0,N/4), ...]).
    Features are kept channel-last internally; the returned feature tensors are (B,W,G) views."""

    def __init__(self, in_channels: int = 3, sample_ratio: float = 0.25, scale: int = 4, k: int = 32,
                 layers: int = 4, embed_dim: int = 256, precision: str = "fp32", token_dtype=None, sync_bn: bool = False,
                 **kwargs):
        super().__init__()
        if layers != 4:
            raise ValueError("p3tok P3Embed supports the reference's layers=4 layout only")
        self.sample_ratio = sample_ratio
        self.k = k
        self.precision = precision
        self.token_dtype = token_dtype          # dtype of the LAST stage's tokens (earlier stages feed the next gather in f32)
        self.sync_bn = sync_bn                  # train mode: all-reduce the BatchNorm sums over torch.distributed ranks
        stages = int(math.log(1 / sample_ratio, scale))
        embed_dim = int(embed_dim // 2 ** (stages - 1))
        self.convs = nn.ModuleList()
        self.channel_list = [in_channels]
        for _ in range(stages):
            W = embed_dim
            conv1 = nn.Sequential(nn.Conv2d(in_channels + 3, W, 1, bias=False), nn.Conv2d(W, W, 1, bias=True),
                                  nn.BatchNorm2d(W), nn.ReLU())
            conv2 = nn.Sequential(nn.Conv2d(2 * W, 2 * W, 1, bias=False), nn.BatchNorm2d(2 * W), nn.ReLU(),
                                  nn.Conv2d(2 * W, W, 1, bias=False), nn.BatchNorm2d(W), nn.ReLU())
            self.convs.append(nn.ModuleList([conv1, conv2]))
            self.channel_list.append(W)
            in_channels = W
            embed_dim *= 2
        self.out_channels = self.channel_list[-1]

    def folded(self, device) -> List[fold.PatchMLP]:
        bf16 = _check_precision(self.precision)
        ver = tuple((t._version, t.data_ptr()) for t in list(self.parameters()) + list(self.buffers()))
        cache = self.__dict__.setdefault("_fold_cache", {})
        if cache.get("ver") != ver:
            cache.clear()
            cache["ver"] = ver
            sd = self.state_dict()
            eps = _bn_eps(self)
            cache["host"] = [fold.fold_p3embed_stage(sd, s, eps) for s in range(len(self.convs))]
        if self.precision == "fp32tc":
            return [m.to_x3(device) for m in cache["host"]]
        return [m.to(device, torch.bfloat16 if bf16 else torch.float32) for m in cache["host"]]

    def forward(self, p: torch.Tensor, f: torch.Tensor, start_idx: Optional[List[torch.Tensor]] = None
                ) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        if self.training or wants_input_grad(p, f):
            return self._forward_train(p, f, start_idx, running=not self.training)
        bf16 = _check_precision(self.precision)
        B, N = int(p.shape[0]), int(p.shape[1])
        out_p, out_f = [p], [f]
        pts = p.float().contiguous()
        feat = f.float().transpose(1, 2).contiguous()            # channel-last (B,N,D)
        folded = self.folded(p.device)
        bf16_last = _check_token_dtype(self.token_dtype, self.precision)
        for s, m in enumerate(folded):
            N = N // 4                                           # pix4point.py:174
            G = min(N, int(pts.shape[1]))                        # clamp of farthest_point_sampling (line 23)
            st = None if start_idx is None else start_idx[s]
            cidx, ws = ops.fps_with_knn_prepare(pts, _start(pts, st, device_draw=True), G)   # kNN preparation overlaps FPS
            ctr = ops.gather_points(pts, cidx)
            kidx = ops.knn_query(pts, ws, ctr, self.k, _lib.KNN_P4P_CDIST, True)
            tok = ops.patch_embed(_lib.ROWS_P4P, pts, feat, None, kidx, None, B * G, self.k, m.tensors(), m.meta(), bf16,
                                  bf16_last and s == len(folded) - 1, self.precision == "fp32tc")
            feat = tok.view(B, G, -1)
            pts = ctr
            out_p.append(ctr)
            out_f.append(feat.transpose(1, 2))
        return out_p, out_f


def _p3embed_forward_train(self, p, f, start_idx=None, running=False):
    """P3Embed.forward under autograd (pix4point.py:166-191): index ops without gradient, differentiable gather of the rows
    (points and features collect the gradients of every neighbourhood they appear in), stage MLP with batch-statistics
    BatchNorm (train mode) or, running=True, the running estimates (eval mode with a gradient wanted for p or f)."""
    B, N = int(p.shape[0]), int(p.shape[1])
    out_p, out_f = [p], [f]
    pts = p.float()
    feat = f.float().transpose(1, 2)                             # channel-last (B,N,D)
    for s, (conv1, conv2) in enumerate(self.convs):
        N = N // 4
        G = min(N, int(pts.shape[1]))
        st = None if start_idx is None else start_idx[s]
        with torch.no_grad():
            pd = pts.detach().contiguous()
            cidx, ws = ops.fps_with_knn_prepare(pd, _start(pd, st, device_draw=True), G)
            ctr_nd = ops.gather_points(pd, cidx)
            kidx = ops.knn_query(pd, ws, ctr_nd, self.k, _lib.KNN_P4P_CDIST, True)
        ctr = torch.gather(pts, 1, cidx.unsqueeze(-1).expand(-1, -1, 3))     # pix4point.py:176 (differentiable like the reference)
        rows = train.GatherRowsFn.apply(pts.contiguous(), feat.contiguous(), kidx)
        tok = train.p3stage_train(conv1, conv2, rows, self.k, self.sync_bn, running)
        feat = tok.view(B, G, -1)
        pts = ctr
        out_p.append(ctr)
        out_f.append(feat.transpose(1, 2))
    return out_p, out_f


P3Embed._forward_train = _p3embed_forward_train


class PointViTTokens(nn.Module):
    """The tokenizer half of the reference's PointViT (pix4point.py:194-258) - everything `PointViT.forward` does
    before the timm blocks: P3Embed, `proj`, `pos_embed`, cls token / cls position concat.  Same attribute names and
    state_dict keys (`patch_embed.*`, `proj.*`, `pos_embed.{0,2}.*`, `cls_token`, `cls_pos`), so the tokenizer part of
    a PointViT checkpoint loads with strict=False.  forward(p, x=None) -> (p_list, x_list, feats (B,1+G,E),
    pos_embed (B,1+G,E)); the ViT blocks (out of scope) consume `feats + pos_embed`."""

    def __init__(self, in_channels: int = 3, embed_dim: int = 384, k_neighbors: int = 16, precision: str = "fp32",
                 **p3embed_kwargs):
        super().__init__()
        self.num_features = self.embed_dim = embed_dim
        self.patch_embed = P3Embed(in_channels=in_channels, k=k_neighbors, precision=precision, **p3embed_kwargs)
        self.proj = nn.Linear(self.patch_embed.out_channels, embed_dim)
        self.pos_embed = nn.Sequential(nn.Linear(3, 128, bias=True), nn.GELU(), nn.Linear(128, embed_dim))
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.cls_pos = nn.Parameter(torch.zeros(1, 1, embed_dim))

    def forward(self, p: torch.Tensor, x: Optional[torch.Tensor] = None, start_idx: Optional[List[torch.Tensor]] = None):
        if x is None:
            x = p.transpose(1, 2)                          # pix4point.py:237-238: features := coordinates
        p_list, x_list = self.patch_embed(p, x, start_idx)
        tokens = x_list[-1].transpose(1, 2)                # channel-last view of the kernel's native layout
        if self.training or (torch.is_grad_enabled() and tokens.requires_grad):
            from . import train_vit                        # autograd path: gradients for proj / pos_embed / cls and the tokens
            feats, pos = train_vit.token_head_train(self, tokens, p_list[-1])
            return p_list, x_list, feats, pos
        d = lambda t: t.detach()                           # serving op: parameters enter as plain tensors
        feats, pos = ops.token_head(tokens, p_list[-1], d(self.proj.weight), d(self.proj.bias),
                                    d(self.pos_embed[0].weight), d(self.pos_embed[0].bias), d(self.pos_embed[2].weight),
                                    d(self.pos_embed[2].bias), d(self.cls_token), d(self.cls_pos))
        return p_list, x_list, feats, pos
