"""torch custom ops (`torch.ops.p3tok.*`) over the C ABI of libp3tok.so.

Each op validates its tensors (CUDA, dtype, contiguity), allocates the outputs with torch (the
library owns no memory), and enqueues the kernels on torch's current stream.  Shape-only "fake"
implementations are registered so the ops trace under torch.export / FakeTensor.  The three gathers
(gather_points, apf_group, group_gather) are differentiable with respect to their point / feature
inputs through adjoint ops of their own; every other op is a forward / inference op (indices are not
differentiable).  There is no implementation for any device but CUDA.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import check

_lib_handle = None


def _L():
    global _lib_handle
    if _lib_handle is None:
        _lib_handle = _lib.lib()
    return _lib_handle


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# Optional per-op device timing (bench.py's roofline leg): when a list is installed, every C-ABI call
# is bracketed by CUDA events recorded on the launching stream.
_PROFILE = None


def set_profile(sink):
    """sink: None (off) or a list that receives (op_name, start_event, end_event)."""
    global _PROFILE
    _PROFILE = sink


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if _PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream())

    def __exit__(self, *a):
        if _PROFILE is not None:
            self.e1.record(torch.cuda.current_stream())
            _PROFILE.append((self.name, self.e0, self.e1))
        return False


def kernel_launches() -> int:
    """Kernels launched by libp3tok.so in this process so far."""
    return int(_L().p3tok_kernel_launches())


def _need_cuda(name: str, *tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(f"p3tok::{name}: CUDA tensors only (got {t.device}); p3tok has no CPU fallback")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"p3tok::{name}: tensors on different devices ({dev} vs {t.device})")
    return dev


def _f32c(name: str, t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise RuntimeError(f"p3tok::{name}: expected float32, got {t.dtype}")
    return t.contiguous()


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _point_stride(x: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Accept (B,N,C) rows with C in {3,4} in place (xyz are channels 0..2); anything else is
    first reduced to a contiguous (B,N,3) copy like the reference's `.contiguous()` (apf.py:65)."""
    if x.dim() != 3 or x.shape[-1] < 3:
        raise RuntimeError(f"expected (B,N,C>=3) points, got {tuple(x.shape)}")
    if x.is_contiguous() and x.shape[-1] in (3, 4):
        return x, int(x.shape[-1])
    # a [:, :, :3] view of a contiguous (B,N,4) tensor: read the parent rows in place
    if x.shape[-1] == 3 and x.stride(-1) == 1 and x.stride(1) == 4 and x.stride(0) == 4 * x.shape[1]:
        return x, 4
    return x[..., :3].contiguous(), 3


# --------------------------------------------------------------------------------------------- fps
@torch.library.custom_op("p3tok::fps", mutates_args=(), device_types="cuda")
def fps(x: torch.Tensor, start_idx: torch.Tensor, npoint: int) -> torch.Tensor:
    """(B,npoint) int64 FPS indices (p3tok_fps): every iteration updates every point; one CTA per cloud, a
    thread-block cluster per cloud beyond 8192 points."""
    _need_cuda("fps", x, start_idx)
    B, N = int(x.shape[0]), int(x.shape[1])
    x = x if x.dtype == torch.float32 else x.float()
    x, stride = _point_stride(x)
    start = start_idx.to(torch.int64).contiguous()
    if start.shape != (B,):
        raise RuntimeError(f"p3tok::fps: start_idx must have shape ({B},)")
    out = torch.empty((B, npoint), dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device), _timed("fps"):
        check(_L().p3tok_fps(x.data_ptr(), B, N, stride, start.data_ptr(), npoint, out.data_ptr(), _stream()), "fps")
    return out


@fps.register_fake
def _(x, start_idx, npoint):
    return x.new_empty((x.shape[0], npoint), dtype=torch.int64)


@torch.library.custom_op("p3tok::fps_nd", mutates_args=(), device_types="cuda")
def fps_nd(points: torch.Tensor, start_idx: torch.Tensor, npoint: int) -> torch.Tensor:
    """(B,npoint) int64 FPS indices of D-dimensional points (B,N,D), 1 <= D <= 16: farthest_point_sampling's distance over
    ALL coordinates (pix4point.py:44), summed in torch's CPU order (csrc/fps_nd.cu).  The xyz case runs on p3tok::fps."""
    _need_cuda("fps_nd", points, start_idx)
    if points.dim() != 3:
        raise RuntimeError(f"p3tok::fps_nd: expected (B,N,D) points, got {tuple(points.shape)}")
    x = (points if points.dtype == torch.float32 else points.float()).contiguous()
    B, N, D = (int(v) for v in x.shape)
    start = start_idx.to(torch.int64).contiguous()
    if start.shape != (B,):
        raise RuntimeError(f"p3tok::fps_nd: start_idx must have shape ({B},)")
    out = torch.empty((B, npoint), dtype=torch.int64, device=x.device)
    ws = torch.empty((B, N), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed("fps"):
        check(_L().p3tok_fps_nd(x.data_ptr(), B, N, D, D, start.data_ptr(), npoint, out.data_ptr(), ws.data_ptr(), _stream()),
              "fps_nd")
    return out


@fps_nd.register_fake
def _(points, start_idx, npoint):
    return points.new_empty((points.shape[0], npoint), dtype=torch.int64)


@torch.library.custom_op("p3tok::square_distance", mutates_args=(), device_types="cuda")
def square_distance(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """_square_distance (sampler.py:47-62): src (B,S,3), dst (B,N,3) -> (B,S,N) f32, the kNN kernels' APF arithmetic."""
    _need_cuda("square_distance", src, dst)
    if src.dim() != 3 or dst.dim() != 3 or src.shape[0] != dst.shape[0] or src.shape[-1] != 3 or dst.shape[-1] != 3:
        raise RuntimeError(f"p3tok::square_distance: expected (B,S,3) and (B,N,3), got {tuple(src.shape)} and {tuple(dst.shape)}")
    if dst.dtype != torch.float32:
        raise RuntimeError(f"p3tok::square_distance: expected float32, got {dst.dtype}")
    c = _f32c("square_distance", src)
    d, stride = _point_stride(dst)          # a [:, :, :3] view of (B,N,4) rows is read in place
    B, S, N = int(c.shape[0]), int(c.shape[1]), int(d.shape[1])
    out = torch.empty((B, S, N), dtype=torch.float32, device=c.device)
    with torch.cuda.device(c.device), _timed("sqdist"):
        check(_L().p3tok_square_distance(c.data_ptr(), B, S, d.data_ptr(), N, stride, out.data_ptr(), _stream()),
              "square_distance")
    return out


@square_distance.register_fake
def _(src, dst):
    return src.new_empty((src.shape[0], src.shape[1], dst.shape[1]), dtype=torch.float32)


# ------------------------------------------------------------------------------------------- gather
@torch.library.custom_op("p3tok::gather_points", mutates_args=(), device_types="cuda")
def gather_points(x: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _need_cuda("gather_points", x, idx)
    x = _f32c("gather_points", x)
    B, N, C = (int(v) for v in x.shape)
    flat = idx.to(torch.int64).reshape(B, -1).contiguous()
    S = int(flat.shape[1])
    out = torch.empty((B, S, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed("gather"):
        check(_L().p3tok_gather_points(x.data_ptr(), B, N, C, flat.data_ptr(), S, out.data_ptr(), _stream()),
              "gather_points")
    return out.view(*idx.shape, C)


@gather_points.register_fake
def _(x, idx):
    return x.new_empty((*idx.shape, x.shape[-1]))


# --------------------------------------------------------------------------------------------- knn
@torch.library.custom_op("p3tok::knn", mutates_args=(), device_types="cuda")
def knn(x: torch.Tensor, centres: torch.Tensor, k: int, mode: int, int32_out: bool,
        return_dist: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    _need_cuda("knn", x, centres)
    x = x if x.dtype == torch.float32 else x.float()
    x, stride = _point_stride(x)
    c = _f32c("knn", centres[..., :3])
    B, N = int(x.shape[0]), int(x.shape[1])
    if c.dim() != 3 or c.shape[0] != B:
        raise RuntimeError("p3tok::knn: centres must be (B,G,3)")
    G = int(c.shape[1])
    if k > N:
        # same failure the reference hits in torch.topk (sampler.py:74)
        raise RuntimeError(f"p3tok::knn: selected index k out of range (k={k} > N={N})")
    idx = torch.empty((B, G, k), dtype=torch.int32 if int32_out else torch.int64, device=x.device)
    dist = torch.empty((B, G, k) if return_dist else (0,), dtype=torch.float32, device=x.device)
    # Z-order sorted blocks + bounding-box culling (same results bit for bit; clouds beyond 8192 points as segments of
    # 8192, up to 131072); the plain sweep beyond that
    ws_bytes = int(_L().p3tok_knn_workspace_bytes(B, N)) if B * G > 0 else 0
    with torch.cuda.device(x.device), _timed("knn"):
        if ws_bytes > 0:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            check(_L().p3tok_knn_sorted(x.data_ptr(), B, N, stride, c.data_ptr(), G, k, mode, idx.data_ptr(),
                                        _lib.I32 if int32_out else _lib.I64, dist.data_ptr() if return_dist else None,
                                        ws.data_ptr(), ws_bytes, _stream()), "knn_sorted")
        else:
            check(_L().p3tok_knn(x.data_ptr(), B, N, stride, c.data_ptr(), G, k, mode, idx.data_ptr(),
                                 _lib.I32 if int32_out else _lib.I64, dist.data_ptr() if return_dist else None,
                                 _stream()), "knn")
    return idx, dist


@knn.register_fake
def _(x, centres, k, mode, int32_out, return_dist):
    B, G = x.shape[0], centres.shape[1]
    return (x.new_empty((B, G, k), dtype=torch.int32 if int32_out else torch.int64),
            x.new_empty((B, G, k) if return_dist else (0,), dtype=torch.float32))


@torch.library.custom_op("p3tok::knn_prepare", mutates_args=(), device_types="cuda")
def knn_prepare(x: torch.Tensor) -> torch.Tensor:
    """The centre-independent half of the sorted kNN (Z-order sort + block boxes of every cloud) -> workspace bytes;
    empty when the sorted variant does not apply (N > 131072).  Enqueued on the CURRENT stream:
    modules run it on a side stream next to FPS."""
    _need_cuda("knn_prepare", x)
    x_in = x
    x = x if x.dtype == torch.float32 else x.float()
    x, stride = _point_stride(x)
    B, N = int(x.shape[0]), int(x.shape[1])
    ws_bytes = int(_L().p3tok_knn_workspace_bytes(B, N)) if B > 0 else 0
    ws = torch.empty(max(ws_bytes, 0), dtype=torch.uint8, device=x.device)
    if ws_bytes > 0:
        with torch.cuda.device(x.device), _timed("knn"):
            check(_L().p3tok_knn_prepare(x.data_ptr(), B, N, stride, ws.data_ptr(), ws_bytes, _stream()), "knn_prepare")
        _ws_bind(ws, x_in)
    return ws


@knn_prepare.register_fake
def _(x):
    return x.new_empty((0,), dtype=torch.uint8)


@torch.library.custom_op("p3tok::knn_query", mutates_args=(), device_types="cuda")
def knn_query(x: torch.Tensor, ws: torch.Tensor, centres: torch.Tensor, k: int, mode: int, int32_out: bool) -> torch.Tensor:
    """kNN indices (B,G,k) from a workspace knn_prepare(x) filled (falls back to the plain sweep when it is empty)."""
    if ws.numel() == 0:
        return knn(x, centres, k, mode, int32_out, False)[0]
    _need_cuda("knn_query", x, ws, centres)
    _ws_check(ws, x)
    c = _f32c("knn_query", centres[..., :3])
    B, N, G = int(x.shape[0]), int(x.shape[1]), int(c.shape[1])
    if c.dim() != 3 or c.shape[0] != B:
        raise RuntimeError("p3tok::knn_query: centres must be (B,G,3)")
    if k > N:
        raise RuntimeError(f"p3tok::knn: selected index k out of range (k={k} > N={N})")
    idx = torch.empty((B, G, k), dtype=torch.int32 if int32_out else torch.int64, device=x.device)
    with torch.cuda.device(x.device), _timed("knn"):
        check(_L().p3tok_knn_query(ws.data_ptr(), int(ws.numel()), B, N, c.data_ptr(), G, k, mode, idx.data_ptr(),
                                   _lib.I32 if int32_out else _lib.I64, None, _stream()), "knn_query")
    return idx


@knn_query.register_fake
def _(x, ws, centres, k, mode, int32_out):
    return x.new_empty((x.shape[0], centres.shape[1], k), dtype=torch.int32 if int32_out else torch.int64)


# A prepared workspace answers queries for the clouds it was sorted from and nothing else; the C side can only check its
# size.  knn_prepare records which tensor (storage address, shape, version counter) a workspace belongs to and knn_query
# refuses a workspace prepared from other clouds or from an `x` that was modified in place since.
_WS_OWNER = {}


def _ws_key(x: torch.Tensor):
    return (x.data_ptr(), tuple(x.shape), tuple(x.stride()), x._version)


def _ws_bind(ws: torch.Tensor, x: torch.Tensor) -> None:
    if len(_WS_OWNER) > 64:                           # stale entries of freed workspaces
        _WS_OWNER.clear()
    _WS_OWNER[ws.data_ptr()] = _ws_key(x)


def _ws_check(ws: torch.Tensor, x: torch.Tensor) -> None:
    owner = _WS_OWNER.get(ws.data_ptr())
    if owner is not None and owner != _ws_key(x):
        raise RuntimeError("p3tok::knn_query: this workspace was prepared from a different (or since modified) point tensor; "
                           "call knn_prepare(x) again")


def fps_with_knn_prepare(x: torch.Tensor, start_idx: torch.Tensor, npoint: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(fps_idx, knn workspace): FPS on the current stream with the kNN preparation of the same clouds on a side stream
    (both are one-CTA-per-cloud kernels that leave most of every SM idle; the preparation does not need the centres).
    Fork / join by events, so the pair is capturable into a CUDA graph.  Measured (B200, same box): with one CTA per cloud
    in each kernel the pair helps only while the two grids fit side by side - c1 (B = 32) 0.319 -> 0.293 ms per step; at
    c2 (B = 128) the preparation's 1024-thread sort shares SMs with FPS, whose dependent iterations are the critical
    path, and the step gets slower (0.972 -> 1.012 ms; c5 2.34 -> 2.38) - so the pair overlaps only when 2 B <= #SMs."""
    _need_cuda("fps_with_knn_prepare", x)         # before the stream calls below, which reject CPU devices
    if 2 * int(x.shape[0]) > _sm_count(x.device):
        return fps(x, start_idx, npoint), knn_prepare(x)
    cur = torch.cuda.current_stream(x.device)
    side = _side_stream(x.device)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        ws = knn_prepare(x)
    idx = fps(x, start_idx, npoint)
    cur.wait_stream(side)
    ws.record_stream(cur)
    return idx, ws


_SIDE = {}
_SMS = {}


def _sm_count(device) -> int:
    key = device.index if device.index is not None else torch.cuda.current_device()
    if key not in _SMS:
        _SMS[key] = torch.cuda.get_device_properties(key).multi_processor_count
    return _SMS[key]


def _side_stream(device) -> torch.cuda.Stream:
    key = (device.index if device.index is not None else torch.cuda.current_device())
    s = _SIDE.get(key)
    if s is None:
        s = _SIDE[key] = torch.cuda.Stream(device=device)
    return s


# ------------------------------------------------------------------------------------------ morton
@torch.library.custom_op("p3tok::morton_order", mutates_args=(), device_types="cuda")
def morton_order(centres: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    _need_cuda("morton_order", centres)
    c = _f32c("morton_order", centres)
    B, G = int(c.shape[0]), int(c.shape[1])
    perm = torch.empty((B, G), dtype=torch.int64, device=c.device)
    codes = torch.empty((B, G), dtype=torch.int64, device=c.device)
    with torch.cuda.device(c.device), _timed("morton"):
        check(_L().p3tok_morton_order(c.data_ptr(), B, G, perm.data_ptr(), codes.data_ptr(), _stream()), "morton_order")
    return perm, codes


@morton_order.register_fake
def _(centres):
    s = (centres.shape[0], centres.shape[1])
    return centres.new_empty(s, dtype=torch.int64), centres.new_empty(s, dtype=torch.int64)


# --------------------------------------------------------------------------------------- apf group
@torch.library.custom_op("p3tok::apf_group", mutates_args=(), device_types="cuda")
def apf_group(x: torch.Tensor, fps_idx: torch.Tensor, knn_idx: torch.Tensor,
              perm: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
    _need_cuda("apf_group", x, fps_idx, knn_idx, perm)
    x = _f32c("apf_group", x)
    B, N, C = (int(v) for v in x.shape)
    G, k = int(knn_idx.shape[1]), int(knn_idx.shape[2])
    f = fps_idx.to(torch.int64).contiguous()
    kn = knn_idx.to(torch.int64).contiguous()
    pm = perm.to(torch.int64).contiguous() if perm is not None else None
    neigh = torch.empty((B, G, k, 2 * C), dtype=torch.float32, device=x.device)
    center = torch.empty((B, G, 3), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed("apf_group"):
        check(_L().p3tok_apf_group(x.data_ptr(), B, N, C, f.data_ptr(), kn.data_ptr(), _ptr(pm), G, k,
                                   neigh.data_ptr(), center.data_ptr(), _stream()), "apf_group")
    return neigh, center


@apf_group.register_fake
def _(x, fps_idx, knn_idx, perm):
    B, G, k = knn_idx.shape
    return x.new_empty((B, G, k, 2 * x.shape[-1])), x.new_empty((B, G, 3))


# ------------------------------------------------------------------------------------ group gather
@torch.library.custom_op("p3tok::group_gather", mutates_args=(), device_types="cuda")
def group_gather(pnts: torch.Tensor, feats: torch.Tensor, idx: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    _need_cuda("group_gather", pnts, feats, idx)
    p = _f32c("group_gather", pnts)
    f = _f32c("group_gather", feats)
    B, N, _ = (int(v) for v in p.shape)
    D = int(f.shape[-1])
    G, k = int(idx.shape[1]), int(idx.shape[2])
    i32 = idx.to(torch.int32).contiguous()
    gp = torch.empty((B, G, k, 3), dtype=torch.float32, device=p.device)
    gf = torch.empty((B, G, k, D), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device), _timed("group_gather"):
        check(_L().p3tok_group_gather(p.data_ptr(), f.data_ptr(), B, N, D, i32.data_ptr(), G, k, gp.data_ptr(),
                                      gf.data_ptr(), _stream()), "group_gather")
    return gp, gf


@group_gather.register_fake
def _(pnts, feats, idx):
    B, G, k = idx.shape
    return pnts.new_empty((B, G, k, 3)), pnts.new_empty((B, G, k, feats.shape[-1]))


# ------------------------------------------------------------------------------- gradients of the gathers
# gather_points, apf_group and group_gather are differentiable with respect to their point / feature inputs, as the
# reference's index_points and advanced-index gathers are (sampler.py:77-94, apf.py:70-95, pix4point.py:92-102); index inputs
# get no gradient.  Each adjoint is an op of its own over csrc/train.cu.  By default it scatters with fp32 atomic adds, so the
# gradient is reproducible to rounding, not bit for bit.  Under torch.use_deterministic_algorithms (deterministic(), read when
# the adjoint runs) it calls the *_det_f32 kernels instead: fixed-point integer sums with a per-cloud power-of-two scale,
# converted to fp32 once per call - bit-identical from run to run, and each cloud's gradient independent of the rest of the batch.
def deterministic() -> bool:
    """True while torch.use_deterministic_algorithms is on (warn_only included).  The wrappers of the kernels that finish their
    sums with floating-point atomics (these adjoints; train.linear_tn, colstats, bn_backward, GatherRowsFn;
    train_vit.ln_param_grad) then launch their deterministic versions.  Read at call time, as torch's own ops do."""
    return torch.are_deterministic_algorithms_enabled()


def _scatter_ws(B: int, N: int, C: int, device) -> torch.Tensor:
    """Scratch of a fixed-point scatter, on the current stream's allocator (the library allocates nothing)."""
    return torch.empty(int(_L().p3tok_scatter_det_workspace_bytes(B, N, C)), dtype=torch.uint8, device=device)


@torch.library.custom_op("p3tok::gather_points_bwd", mutates_args=(), device_types="cuda")
def gather_points_bwd(grad: torch.Tensor, idx: torch.Tensor, N: int) -> torch.Tensor:
    """grad (*idx.shape, C) -> dX (B,N,C): the adjoint of gather_points (p3tok_gather_points_bwd_f32)."""
    _need_cuda("gather_points_bwd", grad, idx)
    g = grad.float().contiguous()
    B, C = int(idx.shape[0]), int(g.shape[-1])
    flat = idx.to(torch.int64).reshape(B, -1).contiguous()
    dx = torch.zeros((B, N, C), dtype=torch.float32, device=g.device)
    with torch.cuda.device(g.device), _timed("gather_bwd"):
        if deterministic():
            ws = _scatter_ws(B, N, C, g.device)
            check(_L().p3tok_gather_points_bwd_det_f32(g.data_ptr(), B, N, C, flat.data_ptr(), int(flat.shape[1]), dx.data_ptr(),
                                                       ws.data_ptr(), ws.numel(), _stream()), "gather_points_bwd_det")
        else:
            check(_L().p3tok_gather_points_bwd_f32(g.data_ptr(), B, N, C, flat.data_ptr(), int(flat.shape[1]), dx.data_ptr(), _stream()),
                  "gather_points_bwd")
    return dx


@gather_points_bwd.register_fake
def _(grad, idx, N):
    return grad.new_empty((idx.shape[0], N, grad.shape[-1]), dtype=torch.float32)


def _gather_points_setup(ctx, inputs, output):
    x, idx = inputs
    ctx.save_for_backward(idx)
    ctx.N = int(x.shape[1])


def _gather_points_backward(ctx, grad):
    (idx,) = ctx.saved_tensors
    return gather_points_bwd(grad, idx, ctx.N), None


gather_points.register_autograd(_gather_points_backward, setup_context=_gather_points_setup)


def apf_rows_descriptor(B: int, N: int, C: int, fps_idx: torch.Tensor, knn_idx: torch.Tensor, perm: Optional[torch.Tensor]):
    """(p3tok_rows of kind 0 over these indices, the index tensors it points into).  knn_idx stays int32 or int64."""
    ci = fps_idx.to(torch.int64).contiguous()
    kn = (knn_idx if knn_idx.dtype in (torch.int32, torch.int64) else knn_idx.to(torch.int64)).contiguous()
    pm = perm.to(torch.int64).contiguous() if perm is not None else None
    r = _lib.RowsStruct()
    r.kind, r.C, r.D, r.idx_dtype = _lib.ROWS_APF, C, 0, _lib.I32 if kn.dtype == torch.int32 else _lib.I64
    r.B, r.N, r.G, r.k = B, N, int(kn.shape[1]), int(kn.shape[2])
    r.ctr_idx, r.knn_idx, r.perm = ci.data_ptr(), kn.data_ptr(), _ptr(pm)
    return r, (ci, kn, pm)


@torch.library.custom_op("p3tok::apf_group_bwd", mutates_args=(), device_types="cuda")
def apf_group_bwd(grad_neigh: Optional[torch.Tensor], grad_center: Optional[torch.Tensor], fps_idx: torch.Tensor,
                  knn_idx: torch.Tensor, perm: Optional[torch.Tensor], N: int, C: int) -> torch.Tensor:
    """The adjoint of apf_group -> dX (B,N,C): the neighbourhood rows through p3tok_apf_rows_bwd_f32, the centres (xyz of
    x[b, fps_idx[b, perm[b,j]]]) through p3tok_gather_points_bwd_f32.  Either gradient may be None.  Deterministic mode: the
    *_det_f32 versions, the neighbourhood part converted and added to dX first, then the centre part."""
    _need_cuda("apf_group_bwd", grad_neigh, grad_center, fps_idx, knn_idx, perm)
    B, G = int(knn_idx.shape[0]), int(knn_idx.shape[1])
    dx = torch.zeros((B, N, C), dtype=torch.float32, device=fps_idx.device)
    L = _L()
    det = deterministic()
    ws = _scatter_ws(B, N, C, dx.device) if det else None
    with torch.cuda.device(dx.device), _timed("apf_group_bwd"):
        if grad_neigh is not None:
            g = grad_neigh.float().contiguous()
            r, keep = apf_rows_descriptor(B, N, C, fps_idx, knn_idx, perm)
            if det:
                check(L.p3tok_apf_rows_bwd_det_f32(ctypes.byref(r), g.data_ptr(), dx.data_ptr(), ws.data_ptr(), ws.numel(), _stream()),
                      "apf_rows_bwd_det_f32")
            else:
                check(L.p3tok_apf_rows_bwd_f32(ctypes.byref(r), g.data_ptr(), dx.data_ptr(), _stream()), "apf_rows_bwd_f32")
            del keep
        if grad_center is not None:
            src = fps_idx.to(torch.int64)
            src = (torch.gather(src, 1, perm.to(torch.int64)) if perm is not None else src).contiguous()
            gc = grad_center.float()
            if C != 3:                                     # the centres are channels 0..2 of the gathered rows
                gc = torch.nn.functional.pad(gc, (0, C - 3))
            gc = gc.contiguous()
            if det:
                check(L.p3tok_gather_points_bwd_det_f32(gc.data_ptr(), B, N, C, src.data_ptr(), G, dx.data_ptr(), ws.data_ptr(),
                                                        ws.numel(), _stream()), "gather_points_bwd_det")
            else:
                check(L.p3tok_gather_points_bwd_f32(gc.data_ptr(), B, N, C, src.data_ptr(), G, dx.data_ptr(), _stream()),
                      "gather_points_bwd")
    return dx


@apf_group_bwd.register_fake
def _(grad_neigh, grad_center, fps_idx, knn_idx, perm, N, C):
    return fps_idx.new_empty((knn_idx.shape[0], N, C), dtype=torch.float32)


def _apf_group_setup(ctx, inputs, output):
    x, fps_idx, knn_idx, perm = inputs
    ctx.set_materialize_grads(False)                       # an unused output (often `center`) costs no scatter
    ctx.save_for_backward(fps_idx, knn_idx, perm)
    ctx.N, ctx.C = int(x.shape[1]), int(x.shape[2])


def _apf_group_backward(ctx, grad_neigh, grad_center):
    fps_idx, knn_idx, perm = ctx.saved_tensors
    if grad_neigh is None and grad_center is None:
        return None, None, None, None
    return apf_group_bwd(grad_neigh, grad_center, fps_idx, knn_idx, perm, ctx.N, ctx.C), None, None, None


apf_group.register_autograd(_apf_group_backward, setup_context=_apf_group_setup)


@torch.library.custom_op("p3tok::group_gather_bwd", mutates_args=(), device_types="cuda")
def group_gather_bwd(grad_p: Optional[torch.Tensor], grad_f: Optional[torch.Tensor], idx: torch.Tensor, N: int, D: int,
                     need_p: bool, need_f: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    """The adjoint of group_gather through p3tok_scatter_rows_add_f32 -> (dP (B,N,3), dF (B,N,D)); an output not asked for
    (need_p / need_f False) is returned empty."""
    _need_cuda("group_gather_bwd", grad_p, grad_f, idx)
    B, G, k = (int(v) for v in idx.shape)
    dev = idx.device
    gp = grad_p.float() if grad_p is not None else torch.zeros((B, G, k, 3), dtype=torch.float32, device=dev)
    gf = grad_f.float() if grad_f is not None else torch.zeros((B, G, k, D), dtype=torch.float32, device=dev)
    drows = torch.cat([gp, gf], -1).contiguous()           # the (B,G,k,3+D) row layout of the scatter
    i32 = idx.to(torch.int32).contiguous()
    dp = torch.zeros((B, N, 3) if need_p else (0,), dtype=torch.float32, device=dev)
    df = torch.zeros((B, N, D) if need_f else (0,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), _timed("group_gather_bwd"):
        if deterministic():
            ws = _scatter_ws(B, N, 3 + D, dev)
            check(_L().p3tok_scatter_rows_add_det_f32(drows.data_ptr(), i32.data_ptr(), B, N, G, k, D, dp.data_ptr() if need_p else None,
                                                      df.data_ptr() if need_f else None, ws.data_ptr(), ws.numel(), _stream()),
                  "scatter_rows_add_det_f32")
        else:
            check(_L().p3tok_scatter_rows_add_f32(drows.data_ptr(), i32.data_ptr(), B, N, G, k, D, dp.data_ptr() if need_p else None,
                                                  df.data_ptr() if need_f else None, _stream()), "scatter_rows_add_f32")
    return dp, df


@group_gather_bwd.register_fake
def _(grad_p, grad_f, idx, N, D, need_p, need_f):
    B = idx.shape[0]
    return (idx.new_empty((B, N, 3) if need_p else (0,), dtype=torch.float32),
            idx.new_empty((B, N, D) if need_f else (0,), dtype=torch.float32))


def _group_gather_setup(ctx, inputs, output):
    pnts, feats, idx = inputs
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(idx)
    ctx.N, ctx.D = int(pnts.shape[1]), int(feats.shape[-1])


def _group_gather_backward(ctx, grad_p, grad_f):
    (idx,) = ctx.saved_tensors
    need_p, need_f = bool(ctx.needs_input_grad[0]), bool(ctx.needs_input_grad[1])
    if (grad_p is None and grad_f is None) or not (need_p or need_f):
        return None, None, None
    dp, df = group_gather_bwd(grad_p, grad_f, idx, ctx.N, ctx.D, need_p, need_f)
    return (dp if need_p else None), (df if need_f else None), None


group_gather.register_autograd(_group_gather_backward, setup_context=_group_gather_setup)


# ------------------------------------------------------------------------------------- patch embed
def _mlp_struct(weights: Sequence[torch.Tensor], meta: Sequence[int], wdtype: int) -> _lib.MlpStruct:
    m = _lib.MlpStruct()
    cin, n_pre = int(meta[0]), int(meta[1])
    m.cin, m.n_pre = cin, n_pre
    dims = [int(v) for v in meta[2:2 + n_pre]]
    relu = [int(v) for v in meta[2 + n_pre:2 + 2 * n_pre]]
    m.mid_dim, m.out_dim, m.out_relu = (int(v) for v in meta[2 + 2 * n_pre:5 + 2 * n_pre])
    m.wdtype = wdtype
    x3 = wdtype == _lib.BF16X3
    want = torch.float32 if wdtype == _lib.F32 else torch.bfloat16
    kw = (lambda k_: 3 * ((k_ + 63) // 64 * 64)) if x3 else (lambda k_: k_)     # bf16x3: [W_hi | W_hi | W_lo] over the padded width
    kin = cin
    for i in range(n_pre):
        w, b = weights[2 * i], weights[2 * i + 1]
        if x3 and i == 0 and cin <= 16:          # the narrow first layer stays float32 (CUDA cores)
            if w.dtype != torch.float32 or tuple(w.shape) != (dims[i], kin) or not w.is_contiguous():
                raise RuntimeError(f"p3tok::patch_embed: bf16x3 layer 0 weight must be contiguous float32 ({dims[i]},{kin})")
        elif w.dtype != want or tuple(w.shape) != (dims[i], kw(kin)) or not w.is_contiguous():
            raise RuntimeError(f"p3tok::patch_embed: layer {i} weight must be contiguous {want} ({dims[i]},{kw(kin)})")
        if b.dtype != torch.float32 or tuple(b.shape) != (dims[i],):
            raise RuntimeError(f"p3tok::patch_embed: layer {i} bias must be float32 ({dims[i]},)")
        m.pre_dim[i], m.pre_relu[i] = dims[i], relu[i]
        m.w_pre[i], m.b_pre[i] = w.data_ptr(), b.data_ptr()
        kin = dims[i]
    wg, wf, bm, wo, bo = weights[2 * n_pre:2 * n_pre + 5]
    for t, shp, dt, nm in ((wg, (m.mid_dim, kw(kin)), want, "w_mid_g"), (wf, (m.mid_dim, kw(kin)), want, "w_mid_f"),
                           (bm, (m.mid_dim,), torch.float32, "b_mid"), (wo, (m.out_dim, kw(m.mid_dim)), want, "w_out"),
                           (bo, (m.out_dim,), torch.float32, "b_out")):
        if t.dtype != dt or tuple(t.shape) != shp or not t.is_contiguous():
            raise RuntimeError(f"p3tok::patch_embed: {nm} must be contiguous {dt} {shp}, got {t.dtype} {tuple(t.shape)}")
    m.w_mid_g, m.w_mid_f, m.b_mid, m.w_out, m.b_out = (t.data_ptr() for t in (wg, wf, bm, wo, bo))
    return m


@torch.library.custom_op("p3tok::patch_embed", mutates_args=(), device_types="cuda")
def patch_embed(kind: int, x: torch.Tensor, feats: Optional[torch.Tensor], ctr_idx: Optional[torch.Tensor],
                knn_idx: Optional[torch.Tensor], perm: Optional[torch.Tensor], ngroups: int, k: int,
                weights: Sequence[torch.Tensor], meta: Sequence[int], bf16: bool, bf16_tokens: bool = False,
                x3: bool = False) -> torch.Tensor:
    """kind 0: APF rows from x (B,N,C) + ctr_idx (B,G) + knn_idx (B,G,k) [+ perm];
    kind 1: P4P rows from x=pnts (B,N,3) + feats (B,N,D) + knn_idx (B,G,k);
    kind 2: x is the row matrix (ngroups*k, cin).  Returns tokens (ngroups, out_dim) float32, or bfloat16 with
    bf16_tokens (bf16 path only: the patch max is rounded once by the epilogue that produces it)."""
    _need_cuda("patch_embed", x, feats, ctr_idx, knn_idx, perm, *weights)
    x = _f32c("patch_embed", x)
    prec = _lib.BF16X3 if x3 else (_lib.BF16 if bf16 else _lib.F32)     # x3: fp32-accurate tensor-core mode (weights from PatchMLP.to_x3)
    m = _mlp_struct(weights, meta, prec)
    r = _lib.RowsStruct()
    r.kind = kind
    keep = [x]
    if kind == _lib.ROWS_DIRECT:
        if x.dim() != 2 or x.shape[0] != ngroups * k or x.shape[1] != m.cin:
            raise RuntimeError(f"p3tok::patch_embed: rows must be ({ngroups * k},{m.cin}), got {tuple(x.shape)}")
        r.B, r.G, r.N, r.k, r.C, r.D = 1, ngroups, 0, k, 0, 0
    else:
        B, N, C = (int(v) for v in x.shape)
        kn = knn_idx if knn_idx.dtype in (torch.int32, torch.int64) else knn_idx.to(torch.int64)
        kn = kn.contiguous()
        G = int(kn.shape[1])
        if B * G != ngroups or int(kn.shape[2]) != k:
            raise RuntimeError("p3tok::patch_embed: knn_idx shape does not match ngroups/k")
        r.B, r.G, r.N, r.k, r.C = B, G, N, k, C
        r.idx_dtype = _lib.I32 if kn.dtype == torch.int32 else _lib.I64
        r.knn_idx = kn.data_ptr()
        keep.append(kn)
        if kind == _lib.ROWS_APF:
            ci = ctr_idx.to(torch.int64).contiguous()
            r.ctr_idx = ci.data_ptr()
            keep.append(ci)
            if perm is not None:
                pm = perm.to(torch.int64).contiguous()
                r.perm = pm.data_ptr()
                keep.append(pm)
        else:
            f = _f32c("patch_embed", feats)
            r.D = int(f.shape[-1])
            r.feats = f.data_ptr()
            keep.append(f)
    r.x = x.data_ptr()
    L = _L()
    ws_bytes = L.p3tok_patch_embed_workspace_bytes(ctypes.byref(m), ngroups, k, prec)
    if ws_bytes < 0:
        raise RuntimeError("p3tok::patch_embed: bad descriptor")
    ws = torch.empty((max(int(ws_bytes), 256),), dtype=torch.uint8, device=x.device)
    if bf16_tokens and not bf16:
        raise RuntimeError("p3tok::patch_embed: bfloat16 tokens are emitted by the bf16 path only")
    tokens = torch.empty((ngroups, m.out_dim), dtype=torch.bfloat16 if bf16_tokens else torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed("embed"):
        check(L.p3tok_patch_embed(ctypes.byref(r), ctypes.byref(m), prec, _lib.BF16 if bf16_tokens else _lib.F32, ws.data_ptr(),
                                  int(ws.numel()), tokens.data_ptr(), _stream()), "patch_embed")
    del keep
    return tokens


@patch_embed.register_fake
def _(kind, x, feats, ctr_idx, knn_idx, perm, ngroups, k, weights, meta, bf16, bf16_tokens=False, x3=False):
    n_pre = meta[1]
    return x.new_empty((ngroups, meta[3 + 2 * n_pre]), dtype=torch.bfloat16 if bf16_tokens else torch.float32)


# ------------------------------------------------------------------------------ exported building blocks
@torch.library.custom_op("p3tok::linear_f32", mutates_args=(), device_types="cuda")
def linear_f32(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], relu: bool) -> torch.Tensor:
    _need_cuda("linear_f32", a, w, bias)
    a2 = _f32c("linear_f32", a).reshape(-1, a.shape[-1])
    w = _f32c("linear_f32", w)
    b = _f32c("linear_f32", bias) if bias is not None else None
    M, K = (int(v) for v in a2.shape)
    N = int(w.shape[0])
    out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device), _timed("linear_f32"):
        check(_L().p3tok_linear_f32(a2.data_ptr(), M, K, w.data_ptr(), N, _ptr(b), None, 1, int(relu), out.data_ptr(),
                                    _stream()), "linear_f32")
    return out.view(*a.shape[:-1], N)


@linear_f32.register_fake
def _(a, w, bias, relu):
    return a.new_empty((*a.shape[:-1], w.shape[0]))


@torch.library.custom_op("p3tok::linear_bf16", mutates_args=(), device_types="cuda")
def linear_bf16(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], relu: bool,
                want_max32: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """tcgen05 GEMM building block: a (M,K) bf16, w (N,K) bf16 -> (bf16 out, f32 out, f32 max over 32-row blocks)."""
    _need_cuda("linear_bf16", a, w, bias)
    if a.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise RuntimeError("p3tok::linear_bf16: operands must be bfloat16")
    a, w = a.contiguous(), w.contiguous()
    b = _f32c("linear_bf16", bias) if bias is not None else None
    M, K = (int(v) for v in a.shape)
    N = int(w.shape[0])
    ob = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
    of = torch.empty((M, N), dtype=torch.float32, device=a.device)
    om = torch.empty(((M + 31) // 32 if want_max32 else 0, N), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device), _timed("linear_bf16"):
        check(_L().p3tok_linear_bf16(a.data_ptr(), M, K, w.data_ptr(), N, _ptr(b), None, 1, int(relu), ob.data_ptr(),
                                     of.data_ptr(), om.data_ptr() if want_max32 else None, _stream()), "linear_bf16")
    return ob, of, om


@linear_bf16.register_fake
def _(a, w, bias, relu, want_max32):
    M, N = a.shape[0], w.shape[0]
    return (a.new_empty((M, N)), a.new_empty((M, N), dtype=torch.float32),
            a.new_empty(((M + 31) // 32 if want_max32 else 0, N), dtype=torch.float32))


@torch.library.custom_op("p3tok::token_head", mutates_args=(), device_types="cuda")
def token_head(tokens: torch.Tensor, centres: torch.Tensor, proj_w: torch.Tensor, proj_b: torch.Tensor,
               pos_w1: torch.Tensor, pos_b1: torch.Tensor, pos_w2: torch.Tensor, pos_b2: torch.Tensor,
               cls_token: torch.Tensor, cls_pos: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Pix4Point token head (pix4point.py:245-252): tokens (B,G,W), centres (B,G,3) -> feats, pos_embed (B,1+G,E)."""
    ts = [_f32c("token_head", t) for t in (tokens, centres, proj_w, proj_b, pos_w1, pos_b1, pos_w2, pos_b2,
                                           cls_token.reshape(-1), cls_pos.reshape(-1))]
    _need_cuda("token_head", *ts)
    tk, ct, pw, pb, w1, b1, w2, b2, cl, cp = ts
    B, G, W = (int(v) for v in tk.shape)
    E, H = int(pw.shape[0]), int(w1.shape[0])
    if tuple(pw.shape) != (E, W) or tuple(w1.shape) != (H, 3) or tuple(w2.shape) != (E, H) or cl.numel() != E or cp.numel() != E:
        raise RuntimeError("p3tok::token_head: weight shapes do not match tokens/centres")
    feats = torch.empty((B, G + 1, E), dtype=torch.float32, device=tk.device)
    pos = torch.empty((B, G + 1, E), dtype=torch.float32, device=tk.device)
    hidden = torch.empty((B * G, H), dtype=torch.float32, device=tk.device)
    with torch.cuda.device(tk.device), _timed("token_head"):
        check(_L().p3tok_token_head_f32(tk.data_ptr(), ct.data_ptr(), B, G, W, E, H, pw.data_ptr(), pb.data_ptr(),
                                        w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(), cl.data_ptr(),
                                        cp.data_ptr(), hidden.data_ptr(), feats.data_ptr(), pos.data_ptr(), _stream()),
              "token_head")
    return feats, pos


@token_head.register_fake
def _(tokens, centres, proj_w, proj_b, pos_w1, pos_b1, pos_w2, pos_b2, cls_token, cls_pos):
    B, G = tokens.shape[0], tokens.shape[1]
    E = proj_w.shape[0]
    return tokens.new_empty((B, G + 1, E)), tokens.new_empty((B, G + 1, E))


@torch.library.custom_op("p3tok::group_max", mutates_args=(), device_types="cuda")
def group_max(x: torch.Tensor, k: int) -> torch.Tensor:
    _need_cuda("group_max", x)
    x = _f32c("group_max", x)
    C = int(x.shape[-1])
    ng = x.numel() // (C * k)
    out = torch.empty((ng, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _timed("group_max"):
        check(_L().p3tok_group_max(x.data_ptr(), ng, k, C, out.data_ptr(), _stream()), "group_max")
    return out


@group_max.register_fake
def _(x, k):
    return x.new_empty((x.numel() // (x.shape[-1] * k), x.shape[-1]))


# --------------------------------------------------------------------------------------------- ViT block stack
# ("next" row 3, SURVEY.md 8f): APFViTLayer stack + encoder_norm + token max of AdaptPointFormer.forward
VIT_LAYER_TENSORS = ("qkv_w", "qkv_b", "proj_w", "proj_b", "fc1d_w", "fc1d_b", "fc2u_w", "fc2u_b")   # struct p3tok_vit_layer
_NVT = len(VIT_LAYER_TENSORS)


def vit_layer_shapes(D: int, HR: int, x3: bool) -> dict:
    """Shapes of one p3tok_vit_layer's tensors (include/p3tok.h) for token width D and fc1d width HR (= H + R; x3: the padded
    width pad64(H + R)): the bf16 layout, or the x3 layout in which every matrix W [out, in] is [W_hi | W_hi | W_lo] over
    pad64(in) columns (fold.split_x3)."""
    k = (lambda n: 3 * ((n + 63) // 64 * 64)) if x3 else (lambda n: n)
    return dict(qkv_w=(3 * D, k(D)), qkv_b=(3 * D,), proj_w=(D, k(D)), proj_b=(D,), fc1d_w=(HR, k(D)), fc1d_b=(HR,),
                fc2u_w=(D, k(HR)), fc2u_b=(D,))


def _vit_layers(name: str, params: Sequence[torch.Tensor], D: int, R: int, x3: bool):
    """Validate the folded layers against the token width and fill the host array of p3tok_vit_layer descriptors.
    Returns (descriptors, layer count, H, tensors to keep alive during the call)."""
    if len(params) % _NVT:
        raise RuntimeError(f"p3tok::{name}: expected {_NVT} tensors per layer")
    nl = len(params) // _NVT
    keep = []
    layers = (_lib.VitLayerStruct * max(nl, 1))()
    H = 64
    for li in range(nl):
        for j, tname in enumerate(VIT_LAYER_TENSORS):
            t = params[li * _NVT + j]
            want = torch.bfloat16 if tname.endswith("_w") else torch.float32
            if t.dtype != want:
                raise RuntimeError(f"p3tok::{name}: layer {li} {tname} must be {want}, got {t.dtype}")
            t = t.contiguous()
            keep.append(t)
            setattr(layers[li], tname, t.data_ptr())
        HR = int(params[li * _NVT + 4].shape[0])
        want = vit_layer_shapes(D, HR, x3)
        if any(tuple(params[li * _NVT + j].shape) != want[n] for j, n in enumerate(VIT_LAYER_TENSORS) if n.endswith("_w")):
            raise RuntimeError(f"p3tok::{name}: weight shapes do not match the token width")
        if any(params[li * _NVT + j].numel() != want[n][0] for j, n in enumerate(VIT_LAYER_TENSORS) if n.endswith("_b")):
            raise RuntimeError(f"p3tok::{name}: bias length does not match its matrix")
        if x3 and (HR % 64 or HR <= R):
            raise RuntimeError(f"p3tok::{name}: fc1d has {HR} rows, expected pad64(H + R)")
        H = (HR - R) // 64 * 64 if x3 else HR - R   # x3: H is a multiple of 64 and H + R <= HR < H + R + 64
    return layers, nl, H, keep


def _apf_vit(name: str, x3: bool, tokens, params, heads, bottleneck, final_w, final_b, ln_eps):
    _need_cuda(name, tokens, final_w, final_b, *params)
    x = _f32c(name, tokens).clone()                        # the residual stream is updated in place
    B, G, D = (int(v) for v in x.shape)
    fw, fb = _f32c(name, final_w), _f32c(name, final_b)
    R = int(bottleneck)
    layers, nl, H, keep = _vit_layers(name, params, D, R, x3)
    pooled = torch.empty((B, D), dtype=torch.float32, device=x.device)
    L = _L()
    ws_bytes, forward = ((L.p3tok_vit_x3_workspace_bytes, L.p3tok_apf_vit_forward_x3) if x3
                         else (L.p3tok_apf_vit_workspace_bytes, L.p3tok_apf_vit_forward))
    with torch.cuda.device(x.device):
        nbytes = int(ws_bytes(B, G, D, H, R))
        ws = torch.empty((max(nbytes, 1024),), dtype=torch.uint8, device=x.device)
        with _timed(name):
            check(forward(x.data_ptr(), B, G, D, int(heads), H, R, layers, nl, fw.data_ptr(), fb.data_ptr(), float(ln_eps),
                          pooled.data_ptr(), ws.data_ptr(), nbytes, _stream()), name)
    del keep
    return x, pooled


@torch.library.custom_op("p3tok::apf_vit", mutates_args=(), device_types="cuda")
def apf_vit(tokens: torch.Tensor, params: Sequence[torch.Tensor], heads: int, bottleneck: int, final_w: torch.Tensor,
            final_b: torch.Tensor, ln_eps: float = 1e-5) -> Tuple[torch.Tensor, torch.Tensor]:
    """tokens (B,G,D) f32 -> (x (B,G,D) f32 after the last block, pooled (B,D) f32 = max_G encoder_norm(x)).
    params: 8 tensors per layer in VIT_LAYER_TENSORS order - the layer as folded by apf_model.fold_vit_layer
    (matrices bf16 [out,in], biases f32)."""
    return _apf_vit("apf_vit", False, tokens, params, heads, bottleneck, final_w, final_b, ln_eps)


@apf_vit.register_fake
def _(tokens, params, heads, bottleneck, final_w, final_b, ln_eps=1e-5):
    return tokens.new_empty(tokens.shape), tokens.new_empty((tokens.shape[0], tokens.shape[2]))


@torch.library.custom_op("p3tok::apf_vit_x3", mutates_args=(), device_types="cuda")
def apf_vit_x3(tokens: torch.Tensor, params: Sequence[torch.Tensor], heads: int, bottleneck: int, final_w: torch.Tensor,
               final_b: torch.Tensor, ln_eps: float = 1e-5) -> Tuple[torch.Tensor, torch.Tensor]:
    """apf_vit, fp32-accurate (bf16x3 split operands on the same kernels, rtol 1e-4): params are the layers as folded by
    apf_model.fold_vit_layer_x3 (vit_layer_shapes(D, pad64(H + R), True)); D must be a multiple of 64."""
    return _apf_vit("apf_vit_x3", True, tokens, params, heads, bottleneck, final_w, final_b, ln_eps)


@apf_vit_x3.register_fake
def _(tokens, params, heads, bottleneck, final_w, final_b, ln_eps=1e-5):
    return tokens.new_empty(tokens.shape), tokens.new_empty((tokens.shape[0], tokens.shape[2]))


def _vit_blocks(name: str, x3: bool, feats, pos, params, heads, final_w, final_b, ln_eps, pool_skip):
    _need_cuda(name, feats, pos, final_w, final_b, *params)
    x = _f32c(name, feats).clone()
    B, S, D = (int(v) for v in x.shape)
    p = _f32c(name, pos) if pos is not None else None
    if p is not None and tuple(p.shape) != (B, S, D):
        raise RuntimeError(f"p3tok::{name}: pos must have the shape of feats")
    fw, fb = _f32c(name, final_w), _f32c(name, final_b)
    layers, nl, H, keep = _vit_layers(name, params, D, 0, x3)
    out = torch.empty((B, S, D), dtype=torch.float32, device=x.device)
    pooled = torch.empty((B, D), dtype=torch.float32, device=x.device)
    L = _L()
    ws_bytes, forward = ((L.p3tok_vit_x3_workspace_bytes, L.p3tok_vit_forward_x3) if x3
                         else (L.p3tok_apf_vit_workspace_bytes, L.p3tok_vit_forward))
    with torch.cuda.device(x.device):
        nbytes = int(ws_bytes(B, S, D, H, 0))
        ws = torch.empty((max(nbytes, 1024),), dtype=torch.uint8, device=x.device)
        with _timed(name):
            check(forward(x.data_ptr(), B, S, D, int(heads), H, layers, nl, _ptr(p), fw.data_ptr(), fb.data_ptr(), float(ln_eps),
                          out.data_ptr(), pooled.data_ptr(), int(pool_skip), ws.data_ptr(), nbytes, _stream()), name)
    del keep
    return out, pooled


@torch.library.custom_op("p3tok::vit_blocks", mutates_args=(), device_types="cuda")
def vit_blocks(feats: torch.Tensor, pos: Optional[torch.Tensor], params: Sequence[torch.Tensor], heads: int, final_w: torch.Tensor,
               final_b: torch.Tensor, ln_eps: float, pool_skip: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Plain pre-norm ViT blocks (timm `Block`, what Pix4Point runs): feats (B,S,D) f32 = [cls ; tokens], pos (B,S,D) or None
    re-added in front of every block -> (LayerNorm(x) (B,S,D) f32, max over rows >= pool_skip (B,D) f32).  params: 8 tensors
    per layer in VIT_LAYER_TENSORS order, folded by p4p_model.fold_timm_block (no adapter columns)."""
    return _vit_blocks("vit_blocks", False, feats, pos, params, heads, final_w, final_b, ln_eps, pool_skip)


@vit_blocks.register_fake
def _(feats, pos, params, heads, final_w, final_b, ln_eps, pool_skip):
    return feats.new_empty(feats.shape), feats.new_empty((feats.shape[0], feats.shape[2]))


@torch.library.custom_op("p3tok::vit_blocks_x3", mutates_args=(), device_types="cuda")
def vit_blocks_x3(feats: torch.Tensor, pos: Optional[torch.Tensor], params: Sequence[torch.Tensor], heads: int,
                  final_w: torch.Tensor, final_b: torch.Tensor, ln_eps: float, pool_skip: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """vit_blocks, fp32-accurate (bf16x3 split operands, rtol 1e-4): params folded by p4p_model.fold_timm_block_x3
    (vit_layer_shapes(D, pad64(H), True)); D must be a multiple of 64."""
    return _vit_blocks("vit_blocks_x3", True, feats, pos, params, heads, final_w, final_b, ln_eps, pool_skip)


@vit_blocks_x3.register_fake
def _(feats, pos, params, heads, final_w, final_b, ln_eps, pool_skip):
    return feats.new_empty(feats.shape), feats.new_empty((feats.shape[0], feats.shape[2]))


@torch.library.custom_op("p3tok::layernorm_bf16", mutates_args=(), device_types="cuda")
def layernorm_bf16(x: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor], eps: float) -> torch.Tensor:
    """bf16(LayerNorm(x)) over the last dimension of x (M,D) f32; w = b = None: normalisation without affine."""
    _need_cuda("layernorm_bf16", x, w, b)
    x = _f32c("layernorm_bf16", x)
    w = None if w is None else _f32c("layernorm_bf16", w)
    b = None if b is None else _f32c("layernorm_bf16", b)
    M, D = int(x.shape[0]), int(x.shape[1])
    out = torch.empty((M, D), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device), _timed("layernorm_bf16"):
        check(_L().p3tok_layernorm_bf16(x.data_ptr(), M, D, float(eps), _ptr(w), _ptr(b), out.data_ptr(), _stream()),
              "layernorm_bf16")
    return out


@layernorm_bf16.register_fake
def _(x, w, b, eps):
    return x.new_empty(x.shape, dtype=torch.bfloat16)


@torch.library.custom_op("p3tok::attention_bf16", mutates_args=(), device_types="cuda")
def attention_bf16(qkv: torch.Tensor, B: int, G: int, heads: int) -> torch.Tensor:
    """qkv (B*G, 3D) bf16 in AttentionLayer's column order -> softmax(q k^T / sqrt(hd)) v as (B*G, D) bf16."""
    _need_cuda("attention_bf16", qkv)
    if qkv.dtype != torch.bfloat16 or qkv.dim() != 2 or qkv.shape[0] != B * G or qkv.shape[1] % 3:
        raise RuntimeError("p3tok::attention_bf16: expected (B*G, 3D) bf16")
    qkv = qkv.contiguous()
    D = int(qkv.shape[1]) // 3
    out = torch.empty((B * G, D), dtype=torch.bfloat16, device=qkv.device)
    with torch.cuda.device(qkv.device), _timed("attention_bf16"):
        check(_L().p3tok_attention_bf16(qkv.data_ptr(), B, G, D, int(heads), out.data_ptr(), _stream()), "attention_bf16")
    return out


@attention_bf16.register_fake
def _(qkv, B, G, heads):
    return qkv.new_empty((qkv.shape[0], qkv.shape[1] // 3))


@torch.library.custom_op("p3tok::layernorm_split", mutates_args=(), device_types="cuda")
def layernorm_split(x: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor], eps: float) -> torch.Tensor:
    """LayerNorm(x) of x (M,D) f32 as the split operand of the x3 stack: (M, 2D) bf16 = [hi | lo], hi + lo = the fp32 value
    to 16 mantissa bits."""
    _need_cuda("layernorm_split", x, w, b)
    x = _f32c("layernorm_split", x)
    w = None if w is None else _f32c("layernorm_split", w)
    b = None if b is None else _f32c("layernorm_split", b)
    M, D = int(x.shape[0]), int(x.shape[1])
    out = torch.empty((M, 2 * D), dtype=torch.bfloat16, device=x.device)
    with torch.cuda.device(x.device), _timed("layernorm_split"):
        check(_L().p3tok_layernorm_split(x.data_ptr(), M, D, float(eps), _ptr(w), _ptr(b), out.data_ptr(), _stream()),
              "layernorm_split")
    return out


@layernorm_split.register_fake
def _(x, w, b, eps):
    return x.new_empty((x.shape[0], 2 * x.shape[1]), dtype=torch.bfloat16)


@torch.library.custom_op("p3tok::attention_x3", mutates_args=(), device_types="cuda")
def attention_x3(qkv: torch.Tensor, B: int, G: int, heads: int) -> torch.Tensor:
    """qkv (B*G, 6D) bf16 = [hi | lo] of the qkv matrix of attention_bf16 -> [hi | lo] of softmax(q k^T / sqrt(hd)) v as
    (B*G, 2D) bf16, fp32-accurate (bf16x3 products, fp32 softmax)."""
    _need_cuda("attention_x3", qkv)
    if qkv.dtype != torch.bfloat16 or qkv.dim() != 2 or qkv.shape[0] != B * G or qkv.shape[1] % 6:
        raise RuntimeError("p3tok::attention_x3: expected (B*G, 6D) bf16")
    qkv = qkv.contiguous()
    D = int(qkv.shape[1]) // 6
    out = torch.empty((B * G, 2 * D), dtype=torch.bfloat16, device=qkv.device)
    with torch.cuda.device(qkv.device), _timed("attention_x3"):
        check(_L().p3tok_attention_x3(qkv.data_ptr(), B, G, D, int(heads), out.data_ptr(), _stream()), "attention_x3")
    return out


@attention_x3.register_fake
def _(qkv, B, G, heads):
    return qkv.new_empty((qkv.shape[0], qkv.shape[1] // 3))


@torch.library.custom_op("p3tok::linear_bf16_ex", mutates_args=(), device_types="cuda")
def linear_bf16_ex(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, act: int, gelu_cols: int,
                   residual: Optional[torch.Tensor], res_mul: float, out_scale: float) -> torch.Tensor:
    """act(a w^T + bias) on tcgen05 with the ViT epilogues: act 0/1/2 = none/ReLU/exact GELU, 3 = GELU on columns
    < gelu_cols and ReLU on the rest -> bf16 (M,N); with a residual (M,N) f32 the result is
    res_mul * residual + out_scale * (a w^T + bias) as f32."""
    _need_cuda("linear_bf16_ex", a, w, bias, residual)
    if a.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise RuntimeError("p3tok::linear_bf16_ex: bf16 operands expected")
    a, w, bias = a.contiguous(), w.contiguous(), _f32c("linear_bf16_ex", bias)
    M, K, N = int(a.shape[0]), int(a.shape[1]), int(w.shape[0])
    with torch.cuda.device(a.device), _timed("linear_bf16_ex"):
        if residual is None:
            out = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
            check(_L().p3tok_linear_bf16_ex(a.data_ptr(), M, K, w.data_ptr(), N, bias.data_ptr(), int(act), int(gelu_cols), None,
                                            0.0, 1.0, out.data_ptr(), None, _stream()), "linear_bf16_ex")
        else:
            res = _f32c("linear_bf16_ex", residual)
            if float(res_mul) == 1.0:
                # the in-place form the ViT stack uses: residual aliases the output, the kernel ADDS into it (TMA reduce)
                out = res.clone()
                res = out
            else:
                out = torch.empty((M, N), dtype=torch.float32, device=a.device)
            check(_L().p3tok_linear_bf16_ex(a.data_ptr(), M, K, w.data_ptr(), N, bias.data_ptr(), int(act), int(gelu_cols),
                                            res.data_ptr(), float(res_mul), float(out_scale), None, out.data_ptr(), _stream()),
                  "linear_bf16_ex")
    return out


@linear_bf16_ex.register_fake
def _(a, w, bias, act, gelu_cols, residual, res_mul, out_scale):
    return a.new_empty((a.shape[0], w.shape[0]), dtype=torch.bfloat16 if residual is None else torch.float32)
