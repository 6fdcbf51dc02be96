"""float64 references for the input-point gradients (test infrastructure).

oracle/port.py's eval-mode tokenizer with the point indices injected instead of recomputed: torch autograd then differentiates
the reference's own arithmetic on exactly the picks the kernels made.  Indices must come from the fp32 index path (the kernels,
or port.py on the float32 cloud): recomputing FPS / kNN in float64 can move picks, and the gradient would land on other points.
tests/test_grad_reference.py pins these functions to port.py's tokens when they are fed port.py's own indices."""
import numpy as np
import torch

from oracle import port


def state64(sd, requires_grad: bool = True):
    """numpy / torch state_dict -> float64 CPU tensors; every floating entry except the BatchNorm running estimates requires
    grad (they are the module's parameters)."""
    out = {}
    for k, v in sd.items():
        t = torch.as_tensor(np.asarray(v.detach().cpu() if torch.is_tensor(v) else v)).clone()
        if t.is_floating_point():
            t = t.double()
            if requires_grad and "running_" not in k:
                t.requires_grad_(True)
        out[k] = t
    return out


def apf_group_idx(x: torch.Tensor, fps_idx: torch.Tensor, knn_idx: torch.Tensor, perm: torch.Tensor):
    """Group.forward (apf.py:64-110, port.apf_group) on given indices -> (neigh (B,G,k,2C), center (B,G,3)), Morton order."""
    B, N, _ = x.shape
    G, k = int(knn_idx.shape[1]), int(knn_idx.shape[2])
    fps_idx, knn_idx, perm = fps_idx.long().cpu(), knn_idx.long().cpu(), perm.long().cpu()
    center = port.take(x[:, :, :3], fps_idx)
    cfeat = port.take(x, fps_idx)
    flat = (knn_idx + torch.arange(B).view(-1, 1, 1) * N).view(-1)
    neigh = x.reshape(B * N, -1)[flat, :].view(B, G, k, -1)
    neigh = neigh - cfeat.unsqueeze(-2)
    neigh = torch.cat([neigh, cfeat.unsqueeze(2).repeat(1, 1, k, 1)], dim=-1)
    order = (perm + (torch.arange(B) * G).unsqueeze(1)).view(-1)
    return neigh.view(B * G, k, -1)[order].view(B, G, k, -1), center.reshape(B * G, -1)[order].view(B, G, -1)


def pointnet_idx(sd, x: torch.Tensor, fps_idx, knn_idx, perm) -> torch.Tensor:
    """PointNet.forward in eval mode (apf.py:202-217) on given indices: port.apf_encode of the grouped rows."""
    return port.apf_encode(sd, apf_group_idx(x, fps_idx, knn_idx, perm)[0])


def p3embed_idx(sd, p: torch.Tensor, f: torch.Tensor, k: int, idx):
    """port.p3embed (pix4point.py:166-191, eval) with the stage indices given: idx = [(centre idx (B,G), kNN idx (B,G,k)), ...].
    f is channel-first (B,D,N).  -> (centres per stage, features per stage (B,W,G))."""
    B = p.shape[0]
    ps, fs = [p], [f]
    for s, (cidx, nidx) in enumerate(idx):
        pts, feat = ps[-1], fs[-1].transpose(1, 2)
        cidx, nidx = cidx.long().cpu(), nidx.long().cpu()
        ctr = torch.gather(pts, 1, cidx.unsqueeze(-1).expand(-1, -1, 3))
        bi = torch.arange(B).view(B, 1, 1).expand(-1, ctr.shape[1], k)
        dp = pts[bi, nidx].permute(0, 3, 1, 2).contiguous()
        fj = feat[bi, nidx].permute(0, 3, 1, 2).contiguous()
        h = torch.cat([dp, fj], dim=1)
        pre = f"convs.{s}"
        h = torch.nn.functional.conv2d(h, sd[f"{pre}.0.0.weight"])
        h = torch.relu(port._bn2(sd, f"{pre}.0.2", torch.nn.functional.conv2d(h, sd[f"{pre}.0.1.weight"], sd[f"{pre}.0.1.bias"])))
        h = torch.cat([torch.max(h, dim=-1, keepdim=True)[0].expand(-1, -1, -1, k), h], dim=1)
        h = torch.relu(port._bn2(sd, f"{pre}.1.1", torch.nn.functional.conv2d(h, sd[f"{pre}.1.0.weight"])))
        h = torch.relu(port._bn2(sd, f"{pre}.1.4", torch.nn.functional.conv2d(h, sd[f"{pre}.1.3.weight"])))
        fs.append(torch.max(h, dim=-1, keepdim=True)[0].squeeze(-1))
        ps.append(ctr)
    return ps, fs
