"""Cost of the deterministic reductions (torch.use_deterministic_algorithms): step times with the flag off and on, alternated,
CUDA events after warm-up, and per-kernel times of the atomic and deterministic kernels from a separate torch.profiler run.
  - the APF training step at BASELINE config 2 shapes (B 128, N 2048, G 128, k 32, E 384, 12 layers; the reference's _freeze
    rule, loss (logits * w).sum(), backward, AdamW step)
  - the frozen-weight input-gradient step (eval mode, every parameter frozen, backward to the points) of the same model
  - the Pix4Point training step at config 1 shapes (B 32, N 1024, k 32, P3Embed width 256 over two stages, E 384, depth 12)
  - each of these with the bf16x3 tensor-core GEMMs (P3TOK_TRAIN_TC=1 / set_tensor_core_gemms(1))
  - one eval serving forward with the flag off and on (under the flag torch's fill_uninitialized_memory fills every
    torch.empty, the serving path's buffers included)
Writes the report (GPU name and power limit read in the same run) to the path given (default profiles/det_step_time.txt).
    python tests/_det_step_time.py [out_path] [runs]"""
import os
import subprocess
import sys
from collections import defaultdict

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")   # torch refuses cuBLAS calls under the flag without it
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200")]
import torch
from p3tok import synth, train
from p3tok.apf_model import AdaptPointFormer
from p3tok.p4p_model import Pix4Point

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "det_step_time.txt")
RUNS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
ITERS = 5
dev = torch.device("cuda:0")
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def set_flag(on):
    torch.use_deterministic_algorithms(bool(on))


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


def compare(name, fn):
    """RUNS alternating off / on measurements of fn; median of each, overhead of on over off."""
    res = {0: [], 1: []}
    for _ in range(RUNS):
        for flag in (0, 1):
            set_flag(flag)
            try:
                res[flag].append(timed(fn))
            finally:
                set_flag(0)
    med = {f: sorted(v)[len(v) // 2] for f, v in res.items()}
    fmt = lambda v: ", ".join(f"{t:.2f}" for t in v)
    say(f"{name}: flag off {med[0]:.2f} ms (runs {fmt(res[0])}), flag on {med[1]:.2f} ms (runs {fmt(res[1])}), "
        f"overhead {100 * (med[1] / med[0] - 1):+.1f} %")


def kernel_table(name, fn, pats):
    """Per-kernel CUDA time (sum over one step, from torch.profiler) of the kernels whose names contain one of pats."""
    for flag in (0, 1):
        set_flag(flag)
        try:
            fn()
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
        finally:
            set_flag(0)
        acc = defaultdict(lambda: [0.0, 0])
        for e in prof.events():
            if e.device_type == torch.autograd.DeviceType.CUDA and any(p in e.name for p in pats):
                key = e.name.split("(")[0].replace("void ", "").replace("p3tok::", "")
                acc[key][0] += e.device_time if hasattr(e, "device_time") else e.cuda_time
                acc[key][1] += 1
        say(f"  {name}, flag {'on' if flag else 'off'}: " + ("; ".join(f"{k} {v[0] / 1e3:.3f} ms / {v[1]} launches"
                                                                   for k, v in sorted(acc.items())) or "none"))


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
say(f"# deterministic reductions: step time with torch.use_deterministic_algorithms off / on (tests/_det_step_time.py)")
say(f"# GPU: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {smi.stdout.strip() or smi.stderr.strip()}")
say(f"# {RUNS} alternating runs per mode, each {ITERS} steps after 2 warm-up steps, CUDA events; medians; torch {torch.__version__}")
say()

B, N, G, k, E = 128, 2048, 128, 32, 384
x = torch.from_numpy(synth.make_cloud("uniform", B, N, 3, 3)).to(dev)
st = torch.from_numpy(synth.start_indices(B, N, 3)).to(dev)
torch.manual_seed(0)
apf = AdaptPointFormer(num_classes=15, embedding_dim=E, npoint=G, nsample=k, in_channels=3, precision="fp32").to(dev).train()
apf._freeze()
opt = torch.optim.AdamW([p for p in apf.parameters() if p.requires_grad], lr=1e-4)
w = torch.randn(B, 15, device=dev)


def apf_step():
    opt.zero_grad(set_to_none=True)
    (apf(x, st) * w).sum().backward()
    opt.step()


apf_eval = AdaptPointFormer(num_classes=15, embedding_dim=E, npoint=G, nsample=k, in_channels=3).to(dev).eval()
for p in apf_eval.parameters():
    p.requires_grad_(False)


def apf_grad_step():
    xg = x.detach().requires_grad_(True)
    (apf_eval(xg, st) * w).sum().backward()


def apf_serve():
    with torch.no_grad():
        apf_eval(x, st)


B1, N1 = 32, 1024
x1 = torch.from_numpy(synth.make_cloud("uniform", B1, N1, 5, 3)).to(dev)
sts1 = [torch.from_numpy(synth.start_indices(B1, N1 // 4 ** s, 5, s)).to(dev) for s in range(2)]
p4p = Pix4Point(num_classes=15, embed_dim=384, k_neighbors=32, depth=12, num_heads=6, sample_ratio=1 / 16,
                precision="fp32").to(dev).train()
opt1 = torch.optim.AdamW(p4p.parameters(), lr=1e-4)
w1 = torch.randn(B1, 15, device=dev)


def p4p_step():
    opt1.zero_grad(set_to_none=True)
    (p4p(x1, sts1) * w1).sum().backward()
    opt1.step()


for level in (0, 1):
    prev = train.set_tensor_core_gemms(level)
    try:
        say(f"## P3TOK_TRAIN_TC={level}")
        compare(f"APF training step B={B} N={N} G={G} k={k} E={E} depth=12 (_freeze)", apf_step)
        compare(f"APF frozen-weight input-gradient step B={B} N={N} (eval, bf16 blocks)", apf_grad_step)
        compare(f"Pix4Point training step B={B1} N={N1} k=32 W=256 (2 stages) E=384 depth=12", p4p_step)
    finally:
        train.set_tensor_core_gemms(prev)
say()
say("## eval serving forward (no gradient): the flag only adds torch's fill of uninitialised memory")
compare(f"APF bf16 serving forward B={B} N={N}", apf_serve)
say()
say("## per-kernel time in one APF training step at config 2 (torch.profiler, separate run): atomic vs deterministic kernels")
kernel_table("APF training step", apf_step, ("sgemm_tn_kernel", "colstats_kernel", "bn_bwd_stats_kernel", "ln_param_grad_kernel",
                                             "slice_sum_kernel", "strip_sum_kernel"))
say("## per-kernel time in one APF input-gradient step at config 2: the scatter adjoints")
kernel_table("APF input-gradient step", apf_grad_step, ("apf_rows_bwd_kernel", "gather_points_bwd_kernel", "fixed_to_f32_kernel",
                                                        "sgemm_tn_kernel", "colstats_kernel", "bn_bwd_stats_kernel"))
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, "w") as f:
    f.write("\n".join(lines) + "\n")
print(f"wrote {OUT}")
