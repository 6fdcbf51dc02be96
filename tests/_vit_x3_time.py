"""Time the ViT block stacks in their two serving precisions and the fp32 autograd forward.

For c2v (B = 128 clouds x G = 128 tokens, ViT-S width D = 384, 12 heads) and ViT-B (B = 32, G = 196, D = 768, 12 heads),
12 APF layers each, prints ms per forward (CUDA events around `--iters` back-to-back forwards after `--warmup` untimed
ones), clouds/s and kernel launches of libp3tok.so per forward for:
  bf16     run_blocks(..., precision="bf16")        p3tok::apf_vit
  fp32tc   run_blocks(..., precision="fp32tc")      p3tok::apf_vit_x3 (bf16x3 split operands)
  autograd the fp32 autograd forward (train_vit.blocks_train; the input requires grad; forward only)
and the max error of each against the float64 oracle on the first cloud.  The GPU's name and power limit are read in the
same run.  Usage: python tests/_vit_x3_time.py [--iters 20] [--warmup 3]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import oracle  # noqa: E402
from p3tok import ops, synth  # noqa: E402
from p3tok.apf_model import APFViTLayer, run_blocks  # noqa: E402

SHAPES = {"c2v": dict(B=128, G=128, D=384, heads=12), "vit_b": dict(B=32, G=196, D=768, heads=12)}
DEPTH = 12


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    print(f"GPU: {gpu_info()}  (name, power limit, max SM clock)")
    print(f"{DEPTH} APF layers, {a.iters} timed forwards after {a.warmup} warm-up forwards, CUDA events")
    for name, c in SHAPES.items():
        B, G, D, heads = c["B"], c["G"], c["D"], c["heads"]
        sd = synth.apf_vit_state(D, DEPTH, 15, 0)
        tsd = synth.to_torch_state(sd)
        blocks = torch.nn.Sequential(*[APFViTLayer(D, heads) for _ in range(DEPTH)]).eval().to(dev)
        blocks.load_state_dict({k[7:]: v for k, v in tsd.items() if k.startswith("blocks.")})
        norm = torch.nn.LayerNorm(D).eval().to(dev)
        norm.load_state_dict({"weight": tsd["encoder_norm.weight"], "bias": tsd["encoder_norm.bias"]})
        tok_np = synth.vit_tokens(B, G, D, B)
        tok = torch.from_numpy(tok_np).to(dev)
        _, op, _ = oracle.apf_vit(sd, tok_np[:1], DEPTH, heads)
        cache = {}
        tg = tok.clone().requires_grad_(True)
        runs = {
            "bf16": lambda: run_blocks(blocks, tok, norm, cache, "bf16"),
            "fp32tc": lambda: run_blocks(blocks, tok, norm, cache, "fp32tc"),
            "autograd": lambda: run_blocks(blocks, tg, norm),
        }
        times = {}
        for kind, fn in runs.items():
            ctx = torch.enable_grad() if kind == "autograd" else torch.no_grad()
            with ctx:
                for _ in range(a.warmup):
                    out = fn()
                torch.cuda.synchronize()
                n0 = ops.kernel_launches()
                out = fn()
                torch.cuda.synchronize()
                launches = ops.kernel_launches() - n0
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    out = fn()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.iters
            times[kind] = ms
            pooled = out[1].detach()[:1].cpu().numpy().astype(np.float64)
            err = float(np.abs(pooled - op).max() / np.abs(op).max())
            print(f"[{name}] B={B} G={G} D={D}  {kind:8s}  {ms:8.3f} ms/forward  {B / ms * 1e3:10.0f} clouds/s  "
                  f"{launches:4d} launches  pooled max|err|/max|ref| vs float64 (cloud 0) {err:.2e}")
        print(f"[{name}] fp32tc / bf16 = {times['fp32tc'] / times['bf16']:.2f}x   autograd / fp32tc = {times['autograd'] / times['fp32tc']:.2f}x")


if __name__ == "__main__":
    main()
