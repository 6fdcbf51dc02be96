"""Host-side weight preparation: fold eval-mode BatchNorm (and P3Embed's activation-free conv
pair) into the per-layer matrices the kernels consume (struct p3tok_mlp).

  BN(eval):  y = (x - mean) / sqrt(var + eps) * gamma + beta     (eps 1e-5, running stats)
  conv+BN :  W' = diag(s) W,  b' = (b - mean) * s + beta,  s = gamma / sqrt(var + eps)

APF Encoder (reference src/models/apf.py:129-143): first_conv.{0+1, 3+4, 6}, second_conv.{0+1, 3};
the concat layer second_conv.0 acts on [global || local] (apf.py:162-163), so its matrix is split
column-wise into the half applied once per group and the half applied per point.
P3Embed stage (src/models/pix4point.py:135-156): conv1 = Conv(Cin->W, no bias) then
Conv(W->W, bias)+BN+ReLU with nothing in between, so the two matrices multiply into one
(W x Cin); conv2 = [Conv(2W->2W)+BN+ReLU, Conv(2W->W)+BN+ReLU] with input [pooled || local]
(pix4point.py:184-186).  All folding is done in float64 and rounded once.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import torch

BN_EPS = 1e-5


@dataclass
class PatchMLP:
    """Folded weights of one patch-embedding block, on one device, in one dtype."""
    cin: int
    pre_dims: List[int]
    pre_relu: List[int]
    mid_dim: int
    out_dim: int
    out_relu: int
    w_pre: List[torch.Tensor]
    b_pre: List[torch.Tensor]
    w_mid_g: torch.Tensor
    w_mid_f: torch.Tensor
    b_mid: torch.Tensor
    w_out: torch.Tensor
    b_out: torch.Tensor
    _cast: Dict = field(default_factory=dict, repr=False)

    def tensors(self) -> List[torch.Tensor]:
        out: List[torch.Tensor] = []
        for w, b in zip(self.w_pre, self.b_pre):
            out += [w, b]
        return out + [self.w_mid_g, self.w_mid_f, self.b_mid, self.w_out, self.b_out]

    def meta(self) -> List[int]:
        return [self.cin, len(self.pre_dims)] + list(self.pre_dims) + list(self.pre_relu) + [
            self.mid_dim, self.out_dim, self.out_relu]

    def to_x3(self, device) -> "PatchMLP":
        """The bf16x3 (fp32-accurate tensor-core) form: a first layer with cin <= 16 stays float32 [out, cin] (CUDA cores, fp32
        coordinates); every other matrix W [out, in] becomes bfloat16 [out, 3 * pad64(in)] = [W_hi | W_hi | W_lo] with
        W_hi = bf16(W), W_lo = bf16(W - W_hi), matching activations stored as [hi | lo]: one GEMM over the tripled reduction
        length evaluates a_hi.w_hi + a_lo.w_hi + a_hi.w_lo (csrc/embed_tc.cu).  Biases float32."""
        key = (str(device), "x3")
        if key not in self._cast:
            def x3(w):
                return split_x3(w.cpu()).to(device)

            def b(t):
                return t.to(device=device, dtype=torch.float32).contiguous()
            w_pre = [(b(w) if (i == 0 and self.cin <= 16) else x3(w)) for i, w in enumerate(self.w_pre)]
            self._cast[key] = PatchMLP(
                self.cin, list(self.pre_dims), list(self.pre_relu), self.mid_dim, self.out_dim, self.out_relu,
                w_pre, [b(x) for x in self.b_pre], x3(self.w_mid_g), x3(self.w_mid_f), b(self.b_mid), x3(self.w_out), b(self.b_out))
        return self._cast[key]

    def to(self, device, wdtype: torch.dtype = torch.float32) -> "PatchMLP":
        """Matrices in `wdtype` (float32 or bfloat16), biases always float32, contiguous on device."""
        key = (str(device), wdtype)
        if key not in self._cast:
            def m(t):
                return t.to(device=device, dtype=wdtype).contiguous()

            def b(t):
                return t.to(device=device, dtype=torch.float32).contiguous()
            self._cast[key] = PatchMLP(
                self.cin, list(self.pre_dims), list(self.pre_relu), self.mid_dim, self.out_dim, self.out_relu,
                [m(w) for w in self.w_pre], [b(x) for x in self.b_pre], m(self.w_mid_g), m(self.w_mid_f),
                b(self.b_mid), m(self.w_out), b(self.b_out))
        return self._cast[key]


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def split_x3(w: torch.Tensor, rows: Optional[int] = None) -> torch.Tensor:
    """The weight operand of a bf16x3 (fp32-accurate tensor-core) GEMM: W [out, in] -> bfloat16 [rows, 3 * pad64(in)] =
    [W_hi | W_hi | W_lo] with W_hi = bf16(W), W_lo = bf16(W - W_hi), both taken from W in float64 and zero padded to
    pad64(in) columns and `rows` (default out) rows, on W's device.  Against activations stored as [hi | lo] one GEMM over
    the tripled reduction length evaluates a_hi.w_hi + a_lo.w_hi + a_hi.w_lo (csrc/embed_tc.cu tc_linear x3)."""
    w = w.detach().double()
    n, k = w.shape
    wp = w.new_zeros((n if rows is None else rows, pad64(k)))
    wp[:n, :k] = w
    hi = wp.bfloat16()
    lo = (wp - hi.double()).bfloat16()
    return torch.cat([hi, hi, lo], 1).contiguous()


def _mat(sd, name) -> torch.Tensor:
    w = sd[name + ".weight"].detach().double().cpu()
    return w.reshape(w.shape[0], w.shape[1])


def _bias(sd, name, n) -> torch.Tensor:
    b = sd.get(name + ".bias")
    return b.detach().double().cpu() if b is not None else torch.zeros(n, dtype=torch.float64)


def _bn_affine(sd, name, eps=None):
    """eps: {BatchNorm module name: eps} from the module (modules._bn_eps); the nn default 1e-5 when absent."""
    g = sd[name + ".weight"].detach().double().cpu()
    b = sd[name + ".bias"].detach().double().cpu()
    m = sd[name + ".running_mean"].detach().double().cpu()
    v = sd[name + ".running_var"].detach().double().cpu()
    s = g / torch.sqrt(v + (eps or {}).get(name, BN_EPS))
    return s, b - m * s


def _conv_bn(sd, conv, bn, eps=None):
    W = _mat(sd, conv)
    b = _bias(sd, conv, W.shape[0])
    s, t = _bn_affine(sd, bn, eps)
    return W * s[:, None], b * s + t


def fold_apf_encoder(sd: Dict[str, torch.Tensor], eps: Optional[Dict[str, float]] = None) -> PatchMLP:
    W1, b1 = _conv_bn(sd, "first_conv.0", "first_conv.1", eps)
    W2, b2 = _conv_bn(sd, "first_conv.3", "first_conv.4", eps)
    W3, b3 = _mat(sd, "first_conv.6"), _bias(sd, "first_conv.6", 0)
    Wm, bm = _conv_bn(sd, "second_conv.0", "second_conv.1", eps)
    Wo = _mat(sd, "second_conv.3")
    bo = _bias(sd, "second_conv.3", Wo.shape[0])
    E = W3.shape[0]
    assert Wm.shape == (2 * E, 2 * E) and Wo.shape == (E, 2 * E)
    # first_conv.6 has no BN / activation behind it (apf.py:136), so its bias passes linearly through the max over k and the
    # concat (apf.py:160-163) into second_conv.0:  Wm [g + b3 || f + b3] + bm = Wm [g || f] + (bm + (Wm_g + Wm_f) b3).  Folding
    # it there (float64) leaves the layer that WRITES the rows x E feature tensor without a bias: its epilogue is the critical
    # path between two row tiles of the pair kernel (csrc/embed_fused.cu), and a bias costs it 8 LDS + 32 FADD per 32 columns.
    bm = bm + (Wm[:, :E] + Wm[:, E:]) @ b3
    b3 = torch.zeros_like(b3)
    f = lambda t: t.float().contiguous()
    return PatchMLP(cin=W1.shape[1], pre_dims=[W1.shape[0], W2.shape[0], E], pre_relu=[1, 1, 0],
                    mid_dim=2 * E, out_dim=E, out_relu=0,
                    w_pre=[f(W1), f(W2), f(W3)], b_pre=[f(b1), f(b2), f(b3)],
                    w_mid_g=f(Wm[:, :E]), w_mid_f=f(Wm[:, E:]), b_mid=f(bm), w_out=f(Wo), b_out=f(bo))


def fold_p3embed_stage(sd: Dict[str, torch.Tensor], s: int, eps: Optional[Dict[str, float]] = None) -> PatchMLP:
    p = f"convs.{s}"
    A = _mat(sd, f"{p}.0.0")                       # (W, Cin), no bias, no BN, no activation
    Bm = _mat(sd, f"{p}.0.1")                      # (W, W) + bias, then BN + ReLU
    bb = _bias(sd, f"{p}.0.1", Bm.shape[0])
    s1, t1 = _bn_affine(sd, f"{p}.0.2", eps)
    W1 = (Bm @ A) * s1[:, None]
    b1 = bb * s1 + t1
    Wm, bm = _conv_bn(sd, f"{p}.1.0", f"{p}.1.1", eps)
    Wo, bo = _conv_bn(sd, f"{p}.1.3", f"{p}.1.4", eps)
    W = W1.shape[0]
    assert Wm.shape == (2 * W, 2 * W) and Wo.shape == (W, 2 * W)
    f = lambda t: t.float().contiguous()
    return PatchMLP(cin=W1.shape[1], pre_dims=[W], pre_relu=[1], mid_dim=2 * W, out_dim=W, out_relu=1,
                    w_pre=[f(W1)], b_pre=[f(b1)], w_mid_g=f(Wm[:, :W]), w_mid_f=f(Wm[:, W:]), b_mid=f(bm),
                    w_out=f(Wo), b_out=f(bo))
