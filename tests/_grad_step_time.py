"""Timing of one input-gradient step on the kernels - what an adversarial attack (PGD) or a saliency map pays per iteration:
eval mode, every parameter frozen, forward + backward() to the input points - next to the bf16 serving forward of the same
model.  AdaptPointFormer at BASELINE config 2 shapes (B 128, N 2048, G 128, k 32, E 384, 12 layers) and Pix4Point at config 1
shapes (B 32, N 1024, k 32, P3Embed width 256 over two stages, ViT-S blocks: E 384, depth 12, 6 heads).  The gradient step runs
with the default fp32 CUDA-core GEMMs and with the bf16x3 tensor-core GEMMs (P3TOK_TRAIN_TC=1 / set_tensor_core_gemms(1)).
CUDA events after warm-up; prints the GPU name and power limit of the same run.   python tests/_grad_step_time.py [iters]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200")]
import torch
from p3tok import synth, train
from p3tok.apf_model import AdaptPointFormer
from p3tok.p4p_model import Pix4Point

ITERS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
dev = torch.device("cuda:0")
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
print(f"GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {smi.stdout.strip() or smi.stderr.strip()}")


def timed(fn, iters=ITERS, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def frozen(m):
    for p in m.parameters():
        p.requires_grad_(False)
    return m.to(dev).eval()


def report(name, B, model, x, call):
    y = torch.arange(B, device=dev) % 15

    def serve():
        with torch.no_grad():
            return call(x)

    def grad_step():
        xg = x.detach().requires_grad_(True)
        torch.nn.functional.cross_entropy(call(xg), y).backward()
        return xg.grad

    ms_serve = timed(serve)
    line = f"{name}: bf16 serving forward {ms_serve:.2f} ms"
    for level in (0, 1):
        prev = train.set_tensor_core_gemms(level)
        try:
            ms = timed(grad_step)
        finally:
            train.set_tensor_core_gemms(prev)
        line += f"; input-gradient step P3TOK_TRAIN_TC={level} {ms:.1f} ms ({ms / ms_serve:.1f}x serving)"
    print(line + f"; peak memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB", flush=True)


B, N, G, k, E = 128, 2048, 128, 32, 384
apf = frozen(AdaptPointFormer(num_classes=15, embedding_dim=E, npoint=G, nsample=k, in_channels=3))
x = torch.from_numpy(synth.make_cloud("uniform", B, N, 3, 3)).to(dev)
st = torch.from_numpy(synth.start_indices(B, N, 3)).to(dev)
report(f"AdaptPointFormer B={B} N={N} G={G} k={k} E={E} depth=12", B, apf, x, lambda t: apf(t, st))
del apf
torch.cuda.empty_cache()
torch.cuda.reset_peak_memory_stats()

B, N = 32, 1024
p4p = frozen(Pix4Point(num_classes=15, embed_dim=384, k_neighbors=32, depth=12, num_heads=6, sample_ratio=1 / 16))
x = torch.from_numpy(synth.make_cloud("uniform", B, N, 5, 3)).to(dev)
sts = [torch.from_numpy(synth.start_indices(B, N // 4 ** s, 5, s)).to(dev) for s in range(2)]
report(f"Pix4Point B={B} N={N} k=32 W=256 (2 stages) E=384 depth=12", B, p4p, x, lambda t: p4p(t, sts))
