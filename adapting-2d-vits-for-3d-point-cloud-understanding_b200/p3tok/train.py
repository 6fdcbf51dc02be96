"""Training mode of the tokenizer's mini-PointNets (SURVEY.md 8f "next" #4): batch-statistics BatchNorm forward and the
backward through both max-pools, the concat and the gather, as torch.autograd.Functions over the C ABI (csrc/train.cu).

What the reference trains: AdaptPointFormer keeps every parameter whose name contains "encoder" trainable
(reference src/models/apf.py:335-346), Pix4Point trains everything - so `Encoder.forward` (apf.py:145-181) and
`P3Embed.forward` (src/models/pix4point.py:171-189) run with nn.BatchNorm in TRAIN mode (batch statistics, biased variance
for the normalisation; running estimates updated with momentum and the unbiased variance) and autograd differentiates
them.  The drop-in modules (p3tok/modules.py) call these Functions when `module.training` is set; parameters receive
`.grad` exactly as with the reference modules, and the BatchNorm buffers are updated the way nn.BatchNorm updates them.

Sharded batches: BatchNorm couples the clouds of a batch, so with the batch split over ranks the per-channel sums (forward:
sum x, sum x^2, row count; backward: sum dy, sum dy*xhat) are all-reduced - the ONE collective the path has (`sync_bn=True`
on the module, torch.distributed initialised).  Weight gradients are per-rank partial sums, reduced by the caller (DDP).

Running-statistics mode (`running` on the Functions, `running=True` on encoder_train / p3stage_train): the same Functions for
eval-mode modules whose input wants a gradient (adversarial attacks, saliency) - nn.BatchNorm's eval semantics (running mean /
variance, no update, no all-reduce), and the weight-gradient products of parameters that do not require grad are skipped.
ApfRowsFn builds the APF rows and sends their gradient back to the input points.

fp32 on CUDA cores; per-channel sums in fp64.  The eval-mode (serving) path is the tensor-core one; this path exists so that
the kernels can replace the reference inside its trainers and wherever the reference is differentiated.  Opt-in:
P3TOK_TRAIN_TC=1 (or `set_tensor_core_gemms(1)`) sends the forward and dX products through the fp32-accurate bf16x3 tensor-core GEMM (`p3tok_linear_x3_f32`: operands split into bf16
hi + lo, three partial products in one tcgen05 GEMM, fp32 accumulate, ~1e-5 of max); the weight-gradient products stay on CUDA
cores.  The fp32 CUDA-core SGEMMs stay the default: they are what the 1e-4 parity tests pin.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Tuple

import torch

from . import _lib, ops
from ._lib import check


def _L():
    return _lib.lib()


def _s() -> int:
    return torch.cuda.current_stream().cuda_stream


def _f32(t: torch.Tensor) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError("p3tok training path: CUDA tensors only (no CPU fallback)")
    return t.detach().float().contiguous()


_TC_LEVEL = int(os.environ.get("P3TOK_TRAIN_TC", "0") or 0)
_TC_MIN_ROWS = 1024          # below this the split + ramp of the tensor-core GEMM costs more than the SGEMM


def set_tensor_core_gemms(level: int) -> int:
    """0: fp32 SGEMMs on CUDA cores (default); 1: forward / dX products (a w^T with >= 1024 rows) on the tensor cores
    (bf16x3, fp32-accurate).  The weight-gradient products dY^T X stay on CUDA cores: their output is a small matrix and their
    reduction axis is the row count, so without a split-K schedule a tensor-core tile walk keeps only a handful of SMs busy.
    Returns the previous level."""
    global _TC_LEVEL
    prev, _TC_LEVEL = _TC_LEVEL, int(level)
    return prev


def _linear_x3(a: torch.Tensor, w: torch.Tensor, b, g, rows_per_group: int) -> torch.Tensor:
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    L = _L()
    ws = torch.empty(int(L.p3tok_linear_x3_workspace_bytes(M, K, N)), dtype=torch.uint8, device=a.device)
    with torch.cuda.device(a.device):
        check(L.p3tok_linear_x3_f32(a.data_ptr(), M, K, w.data_ptr(), N, b.data_ptr() if b is not None else None,
                                    g.data_ptr() if g is not None else None, int(rows_per_group), 0, out.data_ptr(), ws.data_ptr(),
                                    ws.numel(), _s()), "linear_x3_f32")
    return out


# ------------------------------------------------------------------------------------------------ kernel wrappers
def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, gbias: Optional[torch.Tensor] = None,
           rows_per_group: int = 1) -> torch.Tensor:
    """a (M,K) w (N,K) -> a w^T + bias + gbias[m // rows_per_group]  (p3tok_linear_f32; P3TOK_TRAIN_TC: p3tok_linear_x3_f32)."""
    a, w = _f32(a), _f32(w)
    M, K = a.shape
    N = w.shape[0]
    b = _f32(bias) if bias is not None else None
    g = _f32(gbias) if gbias is not None else None
    if _TC_LEVEL >= 1 and M >= _TC_MIN_ROWS and N % 8 == 0 and N <= 2048 and K >= 16:
        return _linear_x3(a, w, b, g, rows_per_group)
    out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        check(_L().p3tok_linear_f32(a.data_ptr(), M, K, w.data_ptr(), N, b.data_ptr() if b is not None else None,
                                    g.data_ptr() if g is not None else None, int(rows_per_group), 0, out.data_ptr(), _s()), "linear_f32")
    return out


def linear_tn(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dy (M,N), x (M,K) -> dy^T x (N,K): the weight gradient of y = x w^T (p3tok_linear_tn_f32)."""
    dy, x = _f32(dy), _f32(x)
    M, N = dy.shape
    K = x.shape[1]
    out = torch.empty((N, K), dtype=torch.float32, device=dy.device)
    with torch.cuda.device(dy.device):
        check(_L().p3tok_linear_tn_f32(dy.data_ptr(), x.data_ptr(), M, N, K, out.data_ptr(), 0, _s()), "linear_tn_f32")
    return out


def colstats(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    x = _f32(x)
    M, N = x.shape
    s = torch.empty(N, dtype=torch.float64, device=x.device)
    q = torch.empty(N, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        check(_L().p3tok_colstats_f32(x.data_ptr(), M, N, s.data_ptr(), q.data_ptr(), _s()), "colstats_f32")
    return s, q


def colsum(x: torch.Tensor) -> torch.Tensor:
    return colstats(x)[0].float()


def group_max_arg(x: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    x = _f32(x)
    M, C = x.shape
    G = M // k
    out = torch.empty((G, C), dtype=torch.float32, device=x.device)
    arg = torch.empty((G, C), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device):
        check(_L().p3tok_group_max_arg_f32(x.data_ptr(), G, k, C, out.data_ptr(), arg.data_ptr(), _s()), "group_max_arg_f32")
    return out, arg


def group_max_bwd(dout: torch.Tensor, arg: torch.Tensor, k: int, into: Optional[torch.Tensor] = None) -> torch.Tensor:
    dout = _f32(dout)
    G, C = dout.shape
    dx = into if into is not None else torch.empty((G * k, C), dtype=torch.float32, device=dout.device)
    with torch.cuda.device(dout.device):
        check(_L().p3tok_group_max_bwd_f32(dout.data_ptr(), arg.data_ptr(), G, k, C, 1 if into is not None else 0, dx.data_ptr(), _s()),
              "group_max_bwd_f32")
    return dx


def group_sum(x: torch.Tensor, k: int) -> torch.Tensor:
    x = _f32(x)
    M, C = x.shape
    out = torch.empty((M // k, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        check(_L().p3tok_group_sum_f32(x.data_ptr(), M // k, k, C, out.data_ptr(), _s()), "group_sum_f32")
    return out


class BNState:
    """Statistics of one BatchNorm application: what forward normalised with and what backward needs.  count is None in the
    running-statistics mode (eval-mode BatchNorm: the statistics are constants, not functions of the batch)."""

    def __init__(self, mean, rstd, count, var_unbiased, mean64):
        self.mean, self.rstd, self.count, self.var_unbiased, self.mean64 = mean, rstd, count, var_unbiased, mean64

    @property
    def running(self) -> bool:
        return self.count is None


def _all_reduce(t: torch.Tensor, sync: bool) -> torch.Tensor:
    if sync:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(t)
    return t


def combine_stats(s: torch.Tensor, q: torch.Tensor, count: float, eps: float):
    """(sum, sum of squares, rows) -> (mean, rstd, unbiased variance), fp64: nn.BatchNorm's train-mode statistics."""
    mean = s / count
    var = torch.clamp(q / count - mean * mean, min=0.0)
    rstd = 1.0 / torch.sqrt(var + eps)
    return mean, rstd, var * (count / max(count - 1.0, 1.0))


def bn_forward(z: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, relu: bool, sync: bool,
               running: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, BNState]:
    """act(BatchNorm(z)) on rows.  running=None: batch statistics (train mode, all-reduced with sync); running=(running_mean,
    running_var): eval-mode BatchNorm - normalise with the module's running estimates, no reduction, nothing all-reduced."""
    M, N = z.shape
    if running is not None:
        mean64 = _f32(running[0]).double()
        mean, rstd = mean64.float(), (1.0 / torch.sqrt(_f32(running[1]).double() + eps)).float()
        st = BNState(mean, rstd, None, None, mean64)
    else:
        s, q = colstats(z)
        packed = _all_reduce(torch.cat([s, q, torch.tensor([float(M)], dtype=torch.float64, device=z.device)]), sync)
        s, q = packed[:N], packed[N:2 * N]
        count = float(packed[2 * N].item()) if sync else float(M)
        mean64, rstd64, var_unb = combine_stats(s, q, count, eps)
        st = BNState(mean64.float(), rstd64.float(), count, var_unb, mean64)
    y = torch.empty_like(z)
    g, b = _f32(gamma), _f32(beta)
    with torch.cuda.device(z.device):
        check(_L().p3tok_bn_act_f32(z.data_ptr(), M, N, st.mean.data_ptr(), st.rstd.data_ptr(), g.data_ptr(), b.data_ptr(), int(relu),
                                    y.data_ptr(), _s()), "bn_act_f32")
    return y, st


def bn_backward(dy: torch.Tensor, z: torch.Tensor, st: BNState, gamma: torch.Tensor, beta: torch.Tensor, relu: bool, sync: bool,
                want_params: bool = True):
    """-> (dz, dgamma, dbeta) for dy = dL/d(act(BN(z))).  In the running-statistics mode dz = gamma rstd dy' (the apply kernel
    with both sums zero), and dgamma / dbeta (the sums of dy' xhat and dy') are computed only when want_params."""
    dy = _f32(dy)
    M, N = z.shape
    g, b = _f32(gamma), _f32(beta)
    stats = not st.running or want_params
    s12 = (torch.empty if stats else torch.zeros)(2 * N, dtype=torch.float64, device=z.device)
    local = None
    with torch.cuda.device(z.device):
        if stats:
            check(_L().p3tok_bn_bwd_stats_f32(dy.data_ptr(), z.data_ptr(), M, N, st.mean.data_ptr(), st.rstd.data_ptr(), g.data_ptr(),
                                              b.data_ptr(), int(relu), s12.data_ptr(), s12.data_ptr() + 8 * N, _s()), "bn_bwd_stats_f32")
            local = s12.clone()
            if st.running:
                s12.zero_()
        if not st.running:
            _all_reduce(s12, sync)
        dz = torch.empty_like(z)
        check(_L().p3tok_bn_bwd_apply_f32(dy.data_ptr(), z.data_ptr(), M, N, 1 if st.running else int(round(st.count)), st.mean.data_ptr(),
                                          st.rstd.data_ptr(), g.data_ptr(), b.data_ptr(), int(relu), s12.data_ptr(), s12.data_ptr() + 8 * N,
                                          dz.data_ptr(), _s()), "bn_bwd_apply_f32")
    if local is None:
        return dz, None, None
    # parameter gradients stay per-rank partial sums (the caller's gradient all-reduce, e.g. DDP, sums them)
    return dz, local[N:].float(), local[:N].float()


def _w2(w: torch.Tensor) -> torch.Tensor:
    return _f32(w).reshape(w.shape[0], -1)


def _t(w: torch.Tensor) -> torch.Tensor:
    return w.t().contiguous()


# ------------------------------------------------------------------------------------------------ APF Encoder
def _running(i: int, running):
    return None if running is None else running[i]


def _with_stats(ctx, out: torch.Tensor, stats) -> tuple:
    """(out, mean, unbiased variance per BatchNorm) in train mode; (out,) in the running-statistics mode."""
    outs = [out]
    for st in stats:
        if not st.running:
            outs += [st.mean64.float(), st.var_unbiased.float()]
    ctx.mark_non_differentiable(*outs[1:])
    return tuple(outs)


def running_stats(bns) -> tuple:
    """((running_mean, running_var), ...) of eval-mode BatchNorm modules (the running-statistics mode of the Functions)."""
    return tuple((bn.running_mean, bn.running_var) for bn in bns)


def _grad_if(need: bool, fn):
    """fn() when the gradient is wanted: the weight-gradient products of frozen parameters are never computed."""
    return fn() if need else None


class EncoderTrainFn(torch.autograd.Function):
    """Encoder.get_features under autograd (apf.py:145-169).  inputs: rows (M, cin) with M = groups * k, k, the three BatchNorm
    eps, sync, running, then the 16 parameter tensors in state_dict order of first_conv.{0,1,3,4,6}, second_conv.{0,1,3}.
    running=None: train mode (batch statistics); running = ((running_mean, running_var) x 3): eval-mode BatchNorm.
    Returns (tokens (groups, E), batch mean / unbiased variance of the three BatchNorms for the running-estimate update); in the
    running mode, where nothing is updated, (tokens,)."""

    @staticmethod
    def forward(ctx, rows, k, eps, sync, running, W1, b1, g1, be1, W2, b2, g2, be2, W3, b3, W4, b4, g4, be4, W5, b5):
        rows = _f32(rows)
        W1m, W2m, W3m, W4m, W5m = (_w2(w) for w in (W1, W2, W3, W4, W5))
        E = W3m.shape[0]
        z1 = linear(rows, W1m, b1)
        h1, s1 = bn_forward(z1, g1, be1, eps[0], True, sync, _running(0, running))
        z2 = linear(h1, W2m, b2)
        h2, s2 = bn_forward(z2, g2, be2, eps[1], True, sync, _running(1, running))
        ft = linear(h2, W3m, b3)
        gl, arg_g = group_max_arg(ft, k)                           # apf.py:160
        W4g, W4f = W4m[:, :E].contiguous(), W4m[:, E:].contiguous()
        gb = linear(gl, W4g, b4)                                   # the expanded global half of the concat, once per group
        z4 = linear(ft, W4f, None, gb, k)                          # apf.py:162-163 without the (M, 2E) concat tensor
        h4, s4 = bn_forward(z4, g4, be4, eps[2], True, sync, _running(2, running))
        o = linear(h4, W5m, b5)
        tok, arg_o = group_max_arg(o, k)                           # apf.py:167
        ctx.k, ctx.sync, ctx.E = k, sync, E
        ctx.stats = (s1, s2, s4)
        ctx.save_for_backward(rows, z1, h1, z2, h2, ft, gl, z4, h4, arg_g, arg_o, W1m, W2m, W3m, W4g, W4f, W5m, g1, be1, g2, be2, g4, be4)
        ctx.shapes = [w.shape for w in (W1, W2, W3, W4, W5)]
        return _with_stats(ctx, tok, (s1, s2, s4))

    @staticmethod
    def backward(ctx, gtok, *_unused):
        (rows, z1, h1, z2, h2, ft, gl, z4, h4, arg_g, arg_o, W1m, W2m, W3m, W4g, W4f, W5m, g1, be1, g2, be2, g4, be4) = ctx.saved_tensors
        k, sync, E = ctx.k, ctx.sync, ctx.E
        s1, s2, s4 = ctx.stats
        need = ctx.needs_input_grad[5:]        # W1 b1 g1 be1 W2 b2 g2 be2 W3 b3 W4 b4 g4 be4 W5 b5
        do = group_max_bwd(gtok, arg_o, k)
        dW5, db5 = _grad_if(need[14], lambda: linear_tn(do, h4)), _grad_if(need[15], lambda: colsum(do))
        dz4, dg4, dbe4 = bn_backward(linear(do, _t(W5m)), z4, s4, g4, be4, True, sync, need[12] or need[13])
        dzg = group_sum(dz4, k)                                    # the global feature collects its k copies
        dW4 = _grad_if(need[10], lambda: torch.cat([linear_tn(dzg, gl), linear_tn(dz4, ft)], 1))
        db4 = _grad_if(need[11], lambda: colsum(dz4))
        dft = linear(dz4, _t(W4f))
        group_max_bwd(linear(dzg, _t(W4g)), arg_g, k, into=dft)
        dW3, db3 = _grad_if(need[8], lambda: linear_tn(dft, h2)), _grad_if(need[9], lambda: colsum(dft))
        dz2, dg2, dbe2 = bn_backward(linear(dft, _t(W3m)), z2, s2, g2, be2, True, sync, need[6] or need[7])
        dW2, db2 = _grad_if(need[4], lambda: linear_tn(dz2, h1)), _grad_if(need[5], lambda: colsum(dz2))
        dz1, dg1, dbe1 = bn_backward(linear(dz2, _t(W2m)), z1, s1, g1, be1, True, sync, need[2] or need[3])
        dW1, db1 = _grad_if(need[0], lambda: linear_tn(dz1, rows)), _grad_if(need[1], lambda: colsum(dz1))
        drows = linear(dz1, _t(W1m)) if ctx.needs_input_grad[0] else None
        sh = ctx.shapes
        rs = lambda t, s: None if t is None else t.reshape(s)
        return (drows, None, None, None, None, rs(dW1, sh[0]), db1, dg1, dbe1, rs(dW2, sh[1]), db2, dg2, dbe2, rs(dW3, sh[2]), db3,
                rs(dW4, sh[3]), db4, dg4, dbe4, rs(dW5, sh[4]), db5)


# ------------------------------------------------------------------------------------------------ P3Embed stage
class P3StageTrainFn(torch.autograd.Function):
    """One P3Embed stage under autograd on its gathered rows (pix4point.py:179-188): rows (M, 3+D), k, eps, sync, running (None:
    train mode; three (running_mean, running_var) pairs: eval-mode BatchNorm), parameters of convs.s.{0.0, 0.1, 0.2, 1.0, 1.1,
    1.3, 1.4}.  Returns (out (groups, W), batch statistics of the three BatchNorms), or (out,) in the running mode."""

    @staticmethod
    def forward(ctx, rows, k, eps, sync, running, Wa, Wb, bb, g1, be1, Wc, g2, be2, Wd, g3, be3):
        rows = _f32(rows)
        Wam, Wbm, Wcm, Wdm = (_w2(w) for w in (Wa, Wb, Wc, Wd))
        W = Wbm.shape[0]
        a = linear(rows, Wam)                                      # no bias, no activation (pix4point.py:139)
        z1 = linear(a, Wbm, bb)
        f1, s1 = bn_forward(z1, g1, be1, eps[0], True, sync, _running(0, running))
        gl, arg_g = group_max_arg(f1, k)                           # pix4point.py:185
        Wcg, Wcf = Wcm[:, :W].contiguous(), Wcm[:, W:].contiguous()
        z2 = linear(f1, Wcf, None, linear(gl, Wcg), k)             # [pooled || local] concat, pooled half once per group
        h2, s2 = bn_forward(z2, g2, be2, eps[1], True, sync, _running(1, running))
        z3 = linear(h2, Wdm)
        h3, s3 = bn_forward(z3, g3, be3, eps[2], True, sync, _running(2, running))
        out, arg_o = group_max_arg(h3, k)                          # pix4point.py:188
        ctx.k, ctx.sync = k, sync
        ctx.stats = (s1, s2, s3)
        ctx.save_for_backward(rows, a, z1, f1, gl, z2, h2, z3, arg_g, arg_o, Wam, Wbm, Wcg, Wcf, Wdm, g1, be1, g2, be2, g3, be3)
        ctx.shapes = [w.shape for w in (Wa, Wb, Wc, Wd)]
        return _with_stats(ctx, out, (s1, s2, s3))

    @staticmethod
    def backward(ctx, gout, *_unused):
        (rows, a, z1, f1, gl, z2, h2, z3, arg_g, arg_o, Wam, Wbm, Wcg, Wcf, Wdm, g1, be1, g2, be2, g3, be3) = ctx.saved_tensors
        k, sync = ctx.k, ctx.sync
        s1, s2, s3 = ctx.stats
        need = ctx.needs_input_grad[5:]        # Wa Wb bb g1 be1 Wc g2 be2 Wd g3 be3
        dh3 = group_max_bwd(gout, arg_o, k)
        dz3, dg3, dbe3 = bn_backward(dh3, z3, s3, g3, be3, True, sync, need[9] or need[10])
        dWd = _grad_if(need[8], lambda: linear_tn(dz3, h2))
        dz2, dg2, dbe2 = bn_backward(linear(dz3, _t(Wdm)), z2, s2, g2, be2, True, sync, need[6] or need[7])
        dzg = group_sum(dz2, k)
        dWc = _grad_if(need[5], lambda: torch.cat([linear_tn(dzg, gl), linear_tn(dz2, f1)], 1))
        df1 = linear(dz2, _t(Wcf))
        group_max_bwd(linear(dzg, _t(Wcg)), arg_g, k, into=df1)
        dz1, dg1, dbe1 = bn_backward(df1, z1, s1, g1, be1, True, sync, need[3] or need[4])
        dWb, dbb = _grad_if(need[1], lambda: linear_tn(dz1, a)), _grad_if(need[2], lambda: colsum(dz1))
        da = linear(dz1, _t(Wbm))
        dWa = _grad_if(need[0], lambda: linear_tn(da, rows))
        drows = linear(da, _t(Wam)) if ctx.needs_input_grad[0] else None
        sh = ctx.shapes
        rs = lambda t, s: None if t is None else t.reshape(s)
        return (drows, None, None, None, None, rs(dWa, sh[0]), rs(dWb, sh[1]), dbb, dg1, dbe1, rs(dWc, sh[2]), dg2, dbe2,
                rs(dWd, sh[3]), dg3, dbe3)


class GatherRowsFn(torch.autograd.Function):
    """rows (B*G*k, 3+D) = [pnts[b, idx] || feats[b, idx]] (group_knn's gather, pix4point.py:92-102, + the concat of 179-182);
    backward scatters the row gradients back to the points and features they were gathered from."""

    @staticmethod
    def forward(ctx, pnts, feats, idx):
        p, f = _f32(pnts), _f32(feats)
        B, N, _ = p.shape
        D = f.shape[-1]
        G, k = idx.shape[1], idx.shape[2]
        i32 = idx.to(torch.int32).contiguous()
        r = _lib.RowsStruct()
        r.kind, r.C, r.D, r.idx_dtype = _lib.ROWS_P4P, 3, D, _lib.I32
        r.B, r.N, r.G, r.k = B, N, G, k
        r.x, r.feats, r.knn_idx = p.data_ptr(), f.data_ptr(), i32.data_ptr()
        rows = torch.empty((B * G * k, 3 + D), dtype=torch.float32, device=p.device)
        with torch.cuda.device(p.device):
            check(_L().p3tok_build_rows_f32(ctypes.byref(r), rows.data_ptr(), _s()), "build_rows_f32")
        ctx.save_for_backward(i32)
        ctx.dims = (B, N, G, k, D)
        return rows

    @staticmethod
    def backward(ctx, drows):
        (i32,) = ctx.saved_tensors
        B, N, G, k, D = ctx.dims
        drows = _f32(drows)
        dp = torch.zeros((B, N, 3), dtype=torch.float32, device=drows.device) if ctx.needs_input_grad[0] else None
        df = torch.zeros((B, N, D), dtype=torch.float32, device=drows.device) if ctx.needs_input_grad[1] else None
        if dp is not None or df is not None:
            with torch.cuda.device(drows.device):
                check(_L().p3tok_scatter_rows_add_f32(drows.data_ptr(), i32.data_ptr(), B, N, G, k, D,
                                                      dp.data_ptr() if dp is not None else None,
                                                      df.data_ptr() if df is not None else None, _s()), "scatter_rows_add_f32")
        return dp, df, None


class ApfRowsFn(torch.autograd.Function):
    """The (B*G*k, 2C) rows [x[nbr] - x[ctr] || x[ctr]] of Group.forward (apf.py:74-110) in Morton group order; backward sends
    the row gradients to the points (p3tok_apf_rows_bwd_f32): every neighbour collects d rel, every centre sum_k (d ctr - d rel)."""

    @staticmethod
    def forward(ctx, x, fps_idx, knn_idx, perm):
        x = _f32(x)
        B, N, C = x.shape
        r, keep = ops.apf_rows_descriptor(B, N, C, fps_idx, knn_idx.to(torch.int64), perm)
        r.x = x.data_ptr()
        rows = torch.empty((B * r.G * r.k, 2 * C), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            check(_L().p3tok_build_rows_f32(ctypes.byref(r), rows.data_ptr(), _s()), "build_rows_f32")
        ctx.save_for_backward(*keep[:2], perm)
        ctx.dims = (N, C)
        return rows

    @staticmethod
    def backward(ctx, drows):
        fps_idx, knn_idx, perm = ctx.saved_tensors
        N, C = ctx.dims
        dx = ops.apf_group_bwd(drows, None, fps_idx, knn_idx, perm, N, C) if ctx.needs_input_grad[0] else None
        return dx, None, None, None


def apf_rows(x: torch.Tensor, fps_idx: torch.Tensor, knn_idx: torch.Tensor, perm: Optional[torch.Tensor]) -> torch.Tensor:
    """The APF rows of x under autograd (ApfRowsFn): the gradient reaches x when x requires one."""
    return ApfRowsFn.apply(x, fps_idx, knn_idx, perm)


@torch.no_grad()
def update_running(bn: torch.nn.modules.batchnorm._BatchNorm, mean: torch.Tensor, var_unbiased: torch.Tensor) -> None:
    """nn.BatchNorm's running-estimate update in train mode (momentum; None = cumulative average)."""
    if not bn.track_running_stats or bn.running_mean is None:
        return
    bn.num_batches_tracked += 1
    m = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
    bn.running_mean.mul_(1.0 - m).add_(mean.to(bn.running_mean.dtype), alpha=m)
    bn.running_var.mul_(1.0 - m).add_(var_unbiased.to(bn.running_var.dtype), alpha=m)


def encoder_train(enc, rows: torch.Tensor, k: int, sync: bool, running: bool = False) -> torch.Tensor:
    """Encoder.forward under autograd on rows (M, cin) -> tokens (groups, E).  running=False: train mode, updates the module's
    BatchNorm buffers; running=True: eval-mode BatchNorm on the running estimates, buffers untouched, nothing all-reduced."""
    fc, sc = enc.first_conv, enc.second_conv
    bns = (fc[1], fc[4], sc[1])
    eps = tuple(float(bn.eps) for bn in bns)
    outs = EncoderTrainFn.apply(rows, int(k), eps, bool(sync) and not running, running_stats(bns) if running else None,
                                fc[0].weight, fc[0].bias, fc[1].weight, fc[1].bias, fc[3].weight, fc[3].bias, fc[4].weight, fc[4].bias,
                                fc[6].weight, fc[6].bias, sc[0].weight, sc[0].bias, sc[1].weight, sc[1].bias, sc[3].weight, sc[3].bias)
    if not running:
        for bn, i in zip(bns, (1, 3, 5)):
            update_running(bn, outs[i], outs[i + 1])
    return outs[0]


def p3stage_train(conv1, conv2, rows: torch.Tensor, k: int, sync: bool, running: bool = False) -> torch.Tensor:
    """One P3Embed stage under autograd on its rows; running as in encoder_train."""
    bns = (conv1[2], conv2[1], conv2[4])
    eps = tuple(float(bn.eps) for bn in bns)
    outs = P3StageTrainFn.apply(rows, int(k), eps, bool(sync) and not running, running_stats(bns) if running else None,
                                conv1[0].weight, conv1[1].weight, conv1[1].bias, conv1[2].weight, conv1[2].bias, conv2[0].weight,
                                conv2[1].weight, conv2[1].bias, conv2[3].weight, conv2[4].weight, conv2[4].bias)
    if not running:
        for bn, i in zip(bns, (1, 3, 5)):
            update_running(bn, outs[i], outs[i + 1])
    return outs[0]
