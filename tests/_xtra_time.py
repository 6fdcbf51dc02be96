"""Timing of the general-D FPS and the squared-distance matrix (scratch driver, not a test):
python tests/_xtra_time.py      ->  one line per case, CUDA events, after a clock warm-up (profiles/r02_xtra_time.txt)
python tests/_xtra_time.py ncu  ->  one launch of each kernel, for `ncu --set full` (profiles/r02_xtra_ncu_full.txt)"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200"))
from p3tok import ops, synth  # noqa: E402


def timed(fn, reps=5):
    for _ in range(2):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


dev = torch.device("cuda:0")
if len(sys.argv) > 1 and sys.argv[1] == "ncu":     # one launch of each kernel for `ncu --set full` (no timing)
    x = torch.from_numpy(synth.make_cloud("uniform", 16, 65536, 2, 3)).to(dev)
    ops.square_distance(x[:, :512].contiguous(), x)
    p = torch.from_numpy(synth.make_points_nd(32, 8192, 8, 1)).to(dev)
    ops.fps_nd(p, torch.zeros(32, dtype=torch.long, device=dev), 512)
    torch.cuda.synchronize()
    sys.exit(0)
a = torch.randn(8192, 8192, device=dev, dtype=torch.bfloat16)
for _ in range(200):                       # ~0.3 s of tensor work: clocks up before anything is timed
    a @ a
torch.cuda.synchronize()
for B, N, D, G in ((32, 1024, 4, 256), (128, 2048, 6, 128), (32, 8192, 8, 512), (256, 512, 5, 128), (128, 2048, 3, 128)):
    x = torch.from_numpy(synth.make_points_nd(B, N, D, 1)).to(dev)
    st = torch.zeros(B, dtype=torch.long, device=dev)
    ms = timed(lambda: ops.fps_nd(x, st, G), reps=20)
    line = f"fps_nd B={B} N={N} D={D} G={G}: {ms:.3f} ms ({ms * 1e3 / G:.2f} us/iteration)"
    if D == 3:
        line += f"; fps_kernel (xyz path) {timed(lambda: ops.fps(x, st, G), reps=20):.3f} ms"
    print(line)
for B, S, N in ((128, 128, 2048), (16, 2048, 65536)):
    x = torch.from_numpy(synth.make_cloud("uniform", B, N, 2, 3)).to(dev)
    c = x[:, :S].contiguous()
    ms = timed(lambda: ops.square_distance(c, x), reps=10)
    print(f"square_distance B={B} S={S} N={N}: {ms:.3f} ms, {B * S * N * 4 / ms / 1e6:.0f} GB/s written")
