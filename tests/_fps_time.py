"""Scratch driver (not a test): device time of p3tok_fps alone.  usage: python tests/_fps_time.py"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200"))
from p3tok import ops, synth  # noqa: E402

dev = torch.device("cuda:0")
for (B, N, G) in ((256, 8192, 2048), (148, 8192, 2048), (256, 4096, 1024), (128, 2048, 128), (512, 1024, 256), (2309, 2048, 1024), (16, 65536, 2048)):
    x = torch.from_numpy(synth.make_cloud("uniform", B, N, 5, 3)).to(dev)
    st = torch.from_numpy(synth.start_indices(B, N, 5)).to(dev)
    ref = None
    ts = []
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = ops.fps(x, st, G)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    print(f"B={B:5d} N={N:6d} G={G:5d}: {min(ts):8.3f} ms  ({1e3 * min(ts) / G:.3f} us/iter)  checksum {int(out.sum())}")
