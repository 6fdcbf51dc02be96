#!/usr/bin/env python
"""bench.py - tokenized clouds/sec of the point-patch tokenizer (FPS + kNN + gather/normalise + embed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl p3tok|reference] [--workload c2|c2v|c1|c3|c4|c5|c5w]
                    [--clouds uniform|clustered|both] [--token-dtype bf16|f32] [--precision bf16|fp32] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic clouds.  Default workload = BASELINE.json
configs[1] ("c2"): APF tokenizer PointNet(E=384, G=128, k=32, in_channel=6), B=128 clouds of N=2048 points
per GPU (batch sharding, weak scaling: every rank tokenizes its own B clouds, no collective on the path).
`--workload c5` is BASELINE configs[4] as written: 4096 clouds per step split 4096/N per GPU (STRONG scaling) with the
final token all-gather over NVLink timed inside `e2e_with_gather`; a short run of it is attached to the default line
as `c5_strong` so the driver's 1/2/4/8-GPU sweep records the curve.

Printed JSON line (rank 0):
  value     whole-job clouds/s with inputs resident in HBM: one timed window of exactly K steps, device-timed (CUDA events
            on the launching stream), max over ranks.
  e2e       the same metric through the public serving call with HOST buffers: pinned H2D copy of the clouds and start
            indices and D2H read of the tokens inside the timed region, every step (again exactly K steps).
  roofline  the dominant kernel family (patch embedding) against the measured bf16 peak of MEASURED_PEAKS.json - the
            burst figure when the clock record shows burst conditions (no power cap), else the sustained one; both
            fractions are printed.  `traffic` = measured DRAM bytes of those kernels (ncu), from profiles/r02_traffic.json.
  cpu_baseline  the reference tokenizer's torch-CPU port (oracle/port.py) timed on this box's host cores.
`--impl reference` times that port alone (the reference is pure Python; see DESIGN.md) and prints the same line with
"impl": "reference".
`--dump-outputs DIR` writes what the timed path returned in its last step as DIR/<name>.npy (float32; an output above
64 MB is cut to a fixed, seeded sample of whole clouds).  The inputs depend on the arguments only, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "adapting-2d-vits-for-3d-point-cloud-understanding_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "tokenized clouds/sec (FPS+kNN+embed)"
UNIT = "clouds/s"
DUMP_MAX_BYTES = 64 * 10**6     # --dump-outputs: total size of the written arrays


def dump_outputs(directory, outputs):
    """Writes every tensor of `outputs` ({name: tensor}) as float32 <directory>/<name>.npy.  Each output gets an equal
    share of DUMP_MAX_BYTES; one above its share is cut to a fixed sample of whole clouds (dim 0, seed 0), so the dump
    stays comparable between runs with the same arguments."""
    os.makedirs(directory, exist_ok=True)
    arrays = {n: t.detach().float().cpu().numpy() for n, t in outputs.items()}
    budget = (DUMP_MAX_BYTES - 4096 * len(arrays)) // len(arrays)           # 4 KB per file for the .npy header
    for name, a in arrays.items():
        if a.nbytes > budget:
            keep = max(1, budget * a.shape[0] // a.nbytes)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)

# name -> family, clouds per GPU (weak) or per job (strong), N, centres G, k, embed E, description
WORKLOADS = {
    "c1": dict(family="p4p", B=32, N=1024, k=32, embed_dim=256, sample_ratio=1 / 16,
               desc="Pix4Point P3Embed 2-stage 1024->256->64, k=32 (BASELINE configs[0])"),
    "c2": dict(family="apf", B=128, N=2048, G=128, k=32, E=384, C=3,
               desc="APF PointNet tokenizer E=384 G=128 k=32 (BASELINE configs[1])"),
    "c2v": dict(family="apf", vit=True, B=128, N=2048, G=128, k=32, E=384, C=3,
                desc="APF tokenizer + ViT-S forward: PointNet E=384 G=128 k=32 -> 12 APFViTLayers (12 heads) -> encoder_norm -> "
                     "token max (BASELINE configs[1] with its ViT tail, SURVEY 8f next #3)"),
    "c3": dict(family="p4p", B=256, N=8192, k=32, embed_dim=256, sample_ratio=1 / 16,
               desc="Pix4Point P3Embed 2-stage 8192->2048->512, k=32 (BASELINE configs[2])"),
    "c4": dict(family="apf", B=16, N=65536, G=2048, k=64, E=384, C=3,
               desc="large-scene APF Group(2048,64)+Encoder(384) (BASELINE configs[3])"),
    "c5": dict(family="p4p", B=4096, strong=True, N=1024, k=32, embed_dim=256, sample_ratio=1 / 16,
               desc="batch-sharded sweep: 4096 clouds per step split 4096/N per GPU, C1 shapes, final token all-gather "
                    "(BASELINE configs[4], strong scaling)"),
    "c5w": dict(family="p4p", B=512, N=1024, k=32, embed_dim=256, sample_ratio=1 / 16,
                desc="C1 shapes at 512 clouds per GPU (weak-scaling form of BASELINE configs[4]; per-GPU roofline)"),
}


def algorithmic_work(w):
    """Per-cloud work (SURVEY.md 8d): minimal / as-written / executed embed FLOPs, FPS / kNN pairs, compulsory bytes.
    executed = what the kernels really multiply: the minimal form (pooled half of the concat applied once per group,
    P3Embed's activation-free conv pair folded) with the padded reduction widths the tensor-core path uses (P3Embed stage 1:
    131 -> 136 input columns) - so a dense-as-written implementation could not borrow the minimal denominator."""
    k = w["k"]
    if w["family"] == "apf":
        E, G, N, C = w["E"], w["G"], w["N"], w["C"]
        per_pt = 2 * C * 256 + 256 * 512 + 512 * E + 4 * E * E      # minimal: global half applied once/group
        per_grp = 2 * E * E
        macs = G * k * per_pt + G * per_grp
        as_written = G * k * (2 * C * 256 + 256 * 512 + 512 * E + 6 * E * E)
        executed = G * k * (C * 256 + 256 * 512 + 512 * E + 4 * E * E) + G * (C * 256 + per_grp)   # centre half of layer 1 once per group
        pairs = G * N
        out = dict(embed_flops=2 * macs, embed_flops_as_written=2 * as_written, embed_flops_executed=2 * executed,
                   fps_pairs=pairs, knn_pairs=pairs, compulsory_bytes=4 * C * N + 4 * G * E)
        if w.get("vit"):      # 12 x (qkv + proj + fc1 + fc2 + adapter down/up) per token + the two attention products per head
            vit_macs = 12 * (G * (3 * E * E + E * E + 8 * E * E + 2 * E * 64) + 2 * G * G * E)
            out.update(compulsory_bytes=4 * C * N + 4 * E, vit_flops=2 * vit_macs)
        return out
    n, cin, wd = w["N"], 6, int(w["embed_dim"] // 2)
    macs = aw = ex = pairs = 0
    byts = 12 * n
    for _ in range(2):
        g = n // 4
        macs += g * k * (cin * wd + 4 * wd * wd) + g * 2 * wd * wd
        aw += g * k * (cin * wd + 7 * wd * wd)
        cpad = cin if cin <= 16 else (cin + 7) // 8 * 8
        ex += g * k * (cpad * wd + 4 * wd * wd) + g * 2 * wd * wd
        pairs += g * n
        n, cin, wd = g, wd + 3, wd * 2
    byts += 4 * n * (wd // 2)
    return dict(embed_flops=2 * macs, embed_flops_as_written=2 * aw, embed_flops_executed=2 * ex, fps_pairs=pairs,
                knn_pairs=pairs, compulsory_bytes=byts)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measured_traffic(workload, precision, clouds):
    """DRAM bytes (read + write) of the patch-embedding launches of ONE step, from the committed ncu capture
    (profiles/r02_traffic.json, written by profiles/summarize.py traffic).  None + the reason when there is no capture."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.isfile(p):
        return None, "no profiles/r02_traffic.json"
    d = json.load(open(p))
    key = f"{workload}:{precision}:{clouds}"
    if key not in d:
        return None, f"no ncu capture for {key} in profiles/r02_traffic.json"
    return d[key]["embed_dram_bytes_per_step"], d[key].get("source", "profiles/r02_traffic.json")


# ------------------------------------------------------------------------------------------ inputs / models
def per_gpu_clouds(w, world):
    if w.get("strong"):
        if w["B"] % world:
            raise SystemExit(f"strong-scaling workload: {w['B']} clouds do not split over {world} GPUs")
        return w["B"] // world
    return w["B"]


def make_inputs(w, B, seed, kind):
    from p3tok import synth
    x = synth.make_cloud(kind, B, w["N"], seed, w.get("C", 3))
    if w["family"] == "apf":
        starts = [synth.start_indices(B, w["N"], seed)]
    else:
        starts = [synth.start_indices(B, w["N"], seed, 0), synth.start_indices(B, w["N"] // 4, seed, 1)]
    return x, starts


def make_vit_state(w):
    from p3tok import synth
    return synth.apf_vit_state(w["E"], 12, 15, 0)


def make_state(w):
    from p3tok import synth
    if w["family"] == "apf":
        return synth.apf_encoder_state(w["E"], 2 * w["C"], 0)
    return synth.p3embed_state(3, w["sample_ratio"], 4, 4, w["embed_dim"], 0)


def build_gpu_model(w, precision, device, token_dtype):
    """(module, run(x, starts) -> tokens).  P3Embed: the returned tokens are the channel-last (B,G,W) tensor the kernels
    write (the module's (B,W,G) return value is a transposed view of it - what PointViT transposes back, pix4point.py:245)."""
    from p3tok import synth
    from p3tok.modules import P3Embed, PointNet
    sd = synth.to_torch_state(make_state(w))
    if w.get("vit"):
        from p3tok.apf_model import AdaptPointFormer
        net = AdaptPointFormer(num_classes=15, embedding_dim=w["E"], npoint=w["G"], nsample=w["k"], in_channels=w["C"],
                               precision=precision).eval().to(device)
        net.point_encoder.encoder.load_state_dict(sd, strict=True)
        net.load_state_dict(synth.to_torch_state(make_vit_state(w)), strict=False)
        return net, (lambda x, st: net.features(x, st[0]))
    if w["family"] == "apf":
        net = PointNet(w["E"], w["G"], w["k"], 2 * w["C"], precision=precision, token_dtype=token_dtype).eval().to(device)
        net.encoder.load_state_dict(sd, strict=True)
        return net, (lambda x, st: net(x, st[0]))
    net = P3Embed(sample_ratio=w["sample_ratio"], k=w["k"], embed_dim=w["embed_dim"], precision=precision,
                  token_dtype=token_dtype).eval().to(device)
    net.load_state_dict(sd, strict=True)

    def run(x, st):
        ps, fs = net(x, x.transpose(1, 2), st)
        return fs[-1].transpose(1, 2)
    return net, run


def cpu_port_runner(w):
    """The reference's tokenizer on CPU (oracle/port.py), all host threads."""
    from oracle import port
    from p3tok import synth
    sd = synth.to_torch_state(make_state(w))
    if w.get("vit"):
        vsd = synth.to_torch_state(make_vit_state(w))
        return lambda x, st: port.apf_vit_features(vsd, port.apf_pointnet(sd, x, w["G"], w["k"], st[0]), 12, 12)
    if w["family"] == "apf":
        return lambda x, st: port.apf_pointnet(sd, x, w["G"], w["k"], st[0])
    return lambda x, st: port.p3embed(sd, x, x.transpose(1, 2).contiguous(), w["k"], 2, st)[1][-1]


CPU_SAMPLE = {"c2": 32, "c2v": 32, "c1": 32, "c5": 32, "c5w": 32, "c3": 4, "c4": 1}     # clouds per CPU pass (~1-10 s each)


def time_cpu_port(w, clouds, repeats, seed=4321):
    torch.set_num_threads(os.cpu_count() or 1)
    x, st = make_inputs(w, clouds, seed, "uniform")
    xt, stt = torch.from_numpy(x), [torch.from_numpy(s) for s in st]
    run = cpu_port_runner(w)
    with torch.no_grad():
        run(xt, stt)                                   # warm-up
        best = float("inf")
        for _ in range(repeats):
            t0 = time.perf_counter()
            run(xt, stt)
            best = min(best, time.perf_counter() - t0)
    return clouds / best, best


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.th = index, [], threading.Event(), None

    def _loop(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def start(self):
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(s[0]) for s in self.samples]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons, "samples": len(sm)}
        try:
            out["power_w_max"] = max(float(s[6]) for s in self.samples if len(s) > 6)
        except Exception:
            pass
        return out


def pin_rank_to_cores(local_rank, local_world):
    """Give every rank of the box its own slice of the host cores (the launcher leaves all ranks on the full mask, so the
    graph-launch threads, the pinned-buffer first touch and the NCCL proxy threads of 8 ranks migrate over each other)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if local_world <= 1 or len(cores) < 2 * local_world:
            return None
        per = len(cores) // local_world
        mine = cores[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, mine)
        return [mine[0], mine[-1]]
    except Exception:
        return None


# ------------------------------------------------------------------------------------------ arms
def run_reference(args, w, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (torch-CPU port), rank 0 only."""
    if rank != 0:
        return
    sample = min(per_gpu_clouds(w, 1), {"c2": 16, "c2v": 16, "c1": 16, "c5": 16, "c5w": 16, "c3": 2, "c4": 1}[args.workload])
    torch.set_num_threads(os.cpu_count() or 1)
    x, st = make_inputs(w, sample, 4321, "uniform")
    xt, stt = torch.from_numpy(x), [torch.from_numpy(s) for s in st]
    run = cpu_port_runner(w)
    with torch.no_grad():
        for _ in range(max(args.warmup, 1)):
            run(xt, stt)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = run(xt, stt)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"tokens": out})
    v = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong" if w.get("strong") else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {w['desc']}", "clouds_per_step": sample,
                   "note": "CPU port of the reference tokenizer (oracle/port.py), same torch calls in the same order"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{sample} clouds per step x {args.steps} steps of the {args.workload} workload"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Harness:
    """One workload on this rank's GPU: builds the model, the L2-defeating input pool and the graphs, and times steps."""

    def __init__(self, w, B, precision, token_dtype, device, rank, world, kind, eager=False, streams=2):
        import torch.distributed as dist
        self.dist, self.w, self.B, self.device, self.rank, self.world, self.eager = dist, w, B, device, rank, world, eager
        self.streams = streams
        self.net, self.run = build_gpu_model(w, precision, device, token_dtype)
        x_np, st_np = make_inputs(w, B, 1234 + rank, kind)
        self.x_host = torch.from_numpy(x_np).pin_memory()
        self.st_host = [torch.from_numpy(s).pin_memory() for s in st_np]
        # rotating pool of distinct input batches, total footprint > 2x L2 (126 MB), so every timed step reads its clouds
        # from HBM ("inputs larger than L2")
        self.in_bytes = self.x_host.numel() * 4
        self.pool_n = max(2, min(256, int(2.2 * 126e6 / self.in_bytes) + 1))
        base = self.x_host.to(device)
        self.base = base
        self.pool = [torch.roll(base, shifts=i, dims=1).contiguous() for i in range(self.pool_n)]
        self.st_pool = [[(s.to(device) + i) % (w["N"] if j == 0 else w["N"] // 4) for j, s in enumerate(self.st_host)]
                        for i in range(self.pool_n)]
        self.gdev = None
        self.graphs = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def step_dev(self, i):
        j = i % self.pool_n
        if self.gdev is not None:
            return self.gdev[i % len(self.gdev)](self.pool[j], *self.st_pool[j])
        return self.run(self.pool[j], self.st_pool[j])

    def prepare_device_loop(self, warmup):
        from p3tok import ops
        from p3tok.graph import GraphedTokenizer
        with torch.no_grad():
            for i in range(max(warmup, 3)):
                self.out = self.run(self.pool[i % self.pool_n], self.st_pool[i % self.pool_n])
            torch.cuda.synchronize()
            l0 = ops.kernel_launches()
            self.out = self.run(self.pool[0], self.st_pool[0])
            self.launches_per_step = ops.kernel_launches() - l0
            # Device-resident loop: the step is the module call captured once into a CUDA graph (p3tok.graph, the serving
            # wrapper); every step first copies its clouds and start indices from the HBM-resident pool into the graph's
            # input buffers (device-to-device, inside the timed region), then replays.  --eager times the Python-dispatched
            # module call instead (launch-bound for the small workloads).
            # `streams` instances on as many streams keep that many steps in flight (default 2, like the e2e path): the index
            # kernels of one step (FPS is a latency chain on <= 1 CTA per SM) overlap the embedding of the other.
            if not self.eager:
                self.dev_streams = [torch.cuda.Stream(device=self.device) for _ in range(self.streams)] if self.streams > 1 else [None]
                self.gdev = [GraphedTokenizer(lambda x, *st: self.run(x, list(st)), [self.base] + self.st_pool[0], stream=s_)
                             for s_ in self.dev_streams]
                for i in range(2 * len(self.gdev)):
                    self.step_dev(i)
            torch.cuda.synchronize()

    def time_device(self, steps):
        """ms of EXACTLY `steps` steps, barrier + synchronize on both sides, CUDA events on the launching stream, max over
        ranks.  `self.last_out` is what the last step returned."""
        with torch.no_grad():
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            main = torch.cuda.current_stream(self.device)
            e0.record()
            multi = self.gdev is not None and self.dev_streams[0] is not None
            if multi:
                for s_ in self.dev_streams:
                    s_.wait_stream(main)           # the step streams start after the start event ...
            for i in range(steps):
                self.last_out = self.step_dev(i)
            if multi:
                for s_ in self.dev_streams:
                    main.wait_stream(s_)           # ... and the end event is recorded after both have drained
            e1.record()
            self.barrier()
            return self.reduce_max(e0.elapsed_time(e1))

    def reduce_max(self, v):
        if self.world == 1:
            return float(v)
        t = torch.tensor([v], dtype=torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    # ---- e2e: host buffers in, host tokens out, through the public serving API (p3tok.graph.GraphedHostTokenizer):
    # one CUDA graph per step = pinned-host -> device copies of the clouds and start indices, the captured module call,
    # device -> pinned-host copy of the tokens.  As many instances as the device-resident loop has steps in flight (>= 3) are
    # replayed round-robin on their own streams, so the copies of step i+1 overlap the kernels of step i; the host pays one
    # graph launch per step.
    def prepare_e2e(self):
        from p3tok.graph import GraphedHostTokenizer
        with torch.no_grad():
            self.graphs = [GraphedHostTokenizer(lambda x, *st: self.run(x, list(st)), [self.x_host] + self.st_host, self.device)
                           for _ in range(max(3, self.streams))]       # a third instance hides the copies of copy-heavy steps (c3: e2e +4.7 %; neutral elsewhere)
            for i in range(2 * len(self.graphs)):
                self.graphs[i % len(self.graphs)].replay()
            for g in self.graphs:
                g.synchronize()
        self.h2d_bytes = self.in_bytes + sum(s.numel() * 8 for s in self.st_host)
        ho = self.graphs[0].host_output
        self.d2h_bytes = ho.numel() * ho.element_size()

    def time_e2e(self, steps, gather=None):
        """ms of EXACTLY `steps` steps, wall clock (the host is part of this number), barrier + synchronize on both sides.
        gather: optional callable(graph) enqueued after each step on the step's stream (the token all-gather)."""
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            g = self.graphs[i % len(self.graphs)]
            g.replay()
            if gather is not None:
                gather(g)
        for g in self.graphs:
            g.synchronize()
        self.barrier()
        return self.reduce_max(1e3 * (time.perf_counter() - t0))

    def copy_bandwidth(self):
        """Pinned H2D and D2H GB/s of this rank while every rank copies at once (names the e2e limiter at N > 1)."""
        n = 64 << 20
        h = torch.empty(n, dtype=torch.uint8).pin_memory()
        d = torch.empty(n, dtype=torch.uint8, device=self.device)
        res = {}
        for name, (dst, src) in (("h2d", (d, h)), ("d2h", (h, d))):
            dst.copy_(src, non_blocking=True)
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e1.record()
            self.barrier()
            res[name] = 4 * n / (self.reduce_max(e0.elapsed_time(e1)) * 1e-3) / 1e9
        return res


def run_p3tok(args, w, rank, world, local_rank):
    import torch.distributed as dist
    from p3tok import ops
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    cores = pin_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    precision = args.precision
    tok_dtype = torch.bfloat16 if (args.token_dtype == "bf16" and precision == "bf16" and not w.get("vit")) else None
    B = per_gpu_clouds(w, world)
    kinds = ["uniform", "clustered"] if args.clouds == "both" else [args.clouds]

    if args.streams <= 0:
        # auto: FPS / kNN are one CTA (or cluster) per cloud, so a batch of B clouds leaves SMs idle during the index half of a
        # step when B is well below the SM count; up to 4 steps in flight fill them (c1, B = 32: 152 k -> 194 k clouds/s on the
        # same box with 4; c2 / c5w, B >= 128: no gain beyond 2)
        # (c4, B = 16 x 65536 points, runs FPS as one CLUSTER per cloud and fills the device: 2 stays best, 3052 vs 3018)
        sms = torch.cuda.get_device_properties(device).multi_processor_count
        ctas = B * max(1, -(-int(w["N"]) // 8192))          # index-kernel CTAs of one step: one per cloud, a cluster beyond 8192 points
        args.streams = 2 if 2 * ctas > sms else min(4, max(2, sms // ctas))
    H = Harness(w, B, precision, tok_dtype, device, rank, world, kinds[0], args.eager, args.streams)
    if args.ncu > 0:
        # profiling aid, not a measurement: `ncu --profile-from-start off ... bench.py --ncu 1` sees exactly N eager steps
        with torch.no_grad():
            for i in range(3):
                H.run(H.pool[i % H.pool_n], H.st_pool[i % H.pool_n])
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            for i in range(args.ncu):
                H.run(H.pool[i % H.pool_n], H.st_pool[i % H.pool_n])
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"ncu_steps": args.ncu, "workload": args.workload, "clouds_per_gpu_per_step": B, "precision": precision,
                              "note": "profiling run - no timing"}))
        return
    H.prepare_device_loop(args.warmup)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms = H.time_device(args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tokens": H.last_out})
    H.prepare_e2e()
    e2e_ms = H.time_e2e(args.steps)
    clocks = sampler.stop() if rank == 0 else None
    with torch.no_grad():
        # the host-to-host graph and the device graph return the same tokens as the eager module call on the same clouds
        ref_out = H.run(H.x_host.to(device), [s.to(device) for s in H.st_host])
        assert torch.equal(H.graphs[0].host_output.to(device), ref_out), "e2e graph != eager"
        if H.gdev is not None:
            got = H.gdev[0](H.pool[0], *H.st_pool[0])
            torch.cuda.synchronize()
            assert torch.equal(got, H.run(H.pool[0], H.st_pool[0])), "graph replay != eager"
    copy_bw = H.copy_bandwidth()

    # ---- e2e with the reference's token dtype (f32) when the headline moved bf16 tokens, and with the token all-gather
    e2e_f32 = None
    if tok_dtype is not None:
        H32 = Harness(w, B, precision, None, device, rank, world, kinds[0], False, args.streams)
        with torch.no_grad():
            for i in range(3):
                H32.run(H32.pool[0], H32.st_pool[0])
        H32.prepare_e2e()
        ms = H32.time_e2e(args.steps)
        e2e_f32 = {"value": B * world * args.steps / (ms / 1e3), "unit": UNIT,
                   "d2h_bytes_per_step": H32.d2h_bytes, "ms_per_step": ms / args.steps}
        del H32
    gather_info = None
    if world > 1:
        out0 = H.graphs[0].output
        gbuf = [torch.empty((world,) + tuple(out0.shape), dtype=out0.dtype, device=device) for _ in range(2)]

        def gather(g):
            with torch.cuda.stream(g.stream):
                dist.all_gather_into_tensor(gbuf[0 if g is H.graphs[0] else 1], g.output)
        ms = H.time_e2e(args.steps, gather=gather)
        H.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            dist.all_gather_into_tensor(gbuf[0], out0)
        g1.record()
        H.barrier()
        gather_info = {"e2e_with_gather": B * world * args.steps / (ms / 1e3),
                       "ms_per_step": ms / args.steps,
                       "allgather_alone_ms": H.reduce_max(g0.elapsed_time(g1) / 5),
                       "gathered_bytes_per_rank": gbuf[0].numel() * gbuf[0].element_size()}

    # ---- the other input kind (north star: uniform AND clustered clouds)
    other = None
    if len(kinds) > 1:
        H2 = Harness(w, B, precision, tok_dtype, device, rank, world, kinds[1], args.eager, args.streams)
        H2.prepare_device_loop(3)
        ms = H2.time_device(args.steps)
        H2.prepare_e2e()
        ems = H2.time_e2e(args.steps)
        other = {"clouds": kinds[1], "value": B * world * args.steps / (ms / 1e3), "ms_per_step": ms / args.steps,
                 "e2e": B * world * args.steps / (ems / 1e3)}
        del H2

    # ---- per-stage device times (separate pass, CUDA events on the launching stream around every C-ABI call)
    with torch.no_grad():
        sink = []
        for i in range(2):
            H.run(H.pool[i % H.pool_n], H.st_pool[i % H.pool_n])
        torch.cuda.synchronize()
        ops.set_profile(sink)
        reps = 8
        for i in range(reps):
            H.run(H.pool[i % H.pool_n], H.st_pool[i % H.pool_n])
        torch.cuda.synchronize()
        ops.set_profile(None)
        stage_ms = {}
        for name, a, b in sink:
            stage_ms[name] = stage_ms.get(name, 0.0) + a.elapsed_time(b) / reps

    # ---- BASELINE configs[4] as written, attached to the default line so the driver's N = 1/2/4/8 sweep records it
    c5s = None
    if args.workload == "c2" and not args.no_extra:
        try:
            c5s = c5_strong_probe(args, rank, world, device, precision, tok_dtype)
        except Exception as ex:                                     # never lose the headline line to the side measurement
            c5s = {"error": f"{type(ex).__name__}: {ex}"[:300]}

    if rank != 0:
        return
    clouds = B * world * args.steps
    value = clouds / (dev_ms / 1e3)
    work = algorithmic_work(w)
    pk = peaks()
    embed_ms = stage_ms.get("embed", 0.0)
    ach_tf = (work["embed_flops"] * B / (embed_ms / 1e3) / 1e12) if embed_ms > 0 else None
    # Which measured peak applies: the sustained figure is cuBLAS back to back for seconds under the power cap; a run whose
    # clock record shows no power cap and SM clocks at their maximum ran under burst conditions and is held to the burst peak.
    capped = bool(clocks and ("sw_power_cap" in clocks["reasons"]))
    at_max = bool(clocks and clocks["sm_mhz"] and clocks["sm_max_mhz"] and clocks["sm_mhz"] >= 0.97 * clocks["sm_max_mhz"])
    peak_kind = "sustained" if (capped or not at_max) else "burst"
    peak_tf = pk["bf16_tflops_sustained"] if peak_kind == "sustained" else pk["bf16_tflops"]
    traffic, traffic_src = measured_traffic(args.workload, precision, B)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if w.get("strong") else "weak", "vs_baseline": None,
        "dtype": {"bf16": "bf16", "fp32": "f32", "fp32tc": "bf16x3 (fp32-accurate split operands on the tensor cores)"}[precision],
        "data": "synthetic",
        "config": {"workload": f"{args.workload}: {w['desc']}", "clouds": kinds[0], "clouds_per_gpu_per_step": B,
                   "global_clouds_per_step": B * world, "points": w["N"], "k": w["k"],
                   "parallelism": f"batch-shard x{world}, no collective on the path",
                   "l2": f"rotating pool of {H.pool_n} distinct input batches ({H.pool_n * H.in_bytes / 1e6:.0f} MB > L2)",
                   "embed_precision": precision, "token_dtype": "bf16" if tok_dtype is not None else "f32",
                   "step": "eager module call" if args.eager else
                           f"CUDA-graph replay of the module call, {args.streams} step(s) in flight on as many streams",
                   "host_cores_of_rank0": cores},
        "timing": {"timed_steps": args.steps, "timed_device_s": dev_ms / 1e3, "timed_e2e_s": e2e_ms / 1e3,
                   "statistic": "one timed run of --steps steps"},
        "e2e": {"value": clouds / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": H.h2d_bytes,
                "d2h_bytes_per_step": H.d2h_bytes, "ms_per_step": e2e_ms / args.steps,
                "copy_GBps_per_rank_all_ranks_busy": {k: round(v, 1) for k, v in copy_bw.items()}},
        "gpu_launches": int(H.launches_per_step * args.steps),
        "gpu_launches_per_step": int(H.launches_per_step),
        "clocks": clocks,
        "stage_ms_per_step": {k: round(v, 4) for k, v in sorted(stage_ms.items())},
        "roofline": {"bound": "tensor", "kernel": "patch embedding (p3tok_patch_embed)",
                     "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": (ach_tf / peak_tf) if ach_tf else None,
                     "peak_kind": peak_kind, "peak_source": pk["source"],
                     "frac_of_burst_peak": (ach_tf / pk["bf16_tflops"]) if ach_tf else None,
                     "frac_of_sustained_peak": (ach_tf / pk["bf16_tflops_sustained"]) if ach_tf else None,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_flops_per_launch_group": work["embed_flops"] * B,
                     "executed_flops": work["embed_flops_executed"] * B,
                     "as_written_flops": work["embed_flops_as_written"] * B, "duration_ms": embed_ms},
        "roofline_hbm": {
            "fps_onchip_streaming_equiv_GBps": (16 * work["fps_pairs"] * B / (stage_ms["fps"] / 1e3) / 1e9) if stage_ms.get("fps") else None,
            "fps_note": "16 B per (centre, point) pair served from registers / shared memory - an on-chip equivalent (SURVEY 8d), "
                        "NOT HBM traffic; the cloud is read from HBM once",
            "knn_pairs_per_s": (work["knn_pairs"] * B / (stage_ms["knn"] / 1e3)) if stage_ms.get("knn") else None,
            "compulsory_bytes_per_step": work["compulsory_bytes"] * B, "peak_GBps": pk["hbm_gbs"],
            "whole_path_roof_ms": max(work["compulsory_bytes"] * B / (pk["hbm_gbs"] * 1e9),
                                      work["embed_flops"] * B / (peak_tf * 1e12)) * 1e3},
    }
    line["roofline_hbm"]["whole_path_frac"] = line["roofline_hbm"]["whole_path_roof_ms"] / line["ms_per_step"]
    if e2e_f32 is not None:
        line["e2e_f32_tokens"] = e2e_f32
    if gather_info is not None:
        line["e2e_with_gather"] = gather_info
    if other is not None:
        line["other_clouds"] = other
    if c5s is not None:
        line["c5_strong"] = c5s
    if w.get("vit") and stage_ms.get("apf_vit"):
        line["vit"] = {"ms_per_step": stage_ms["apf_vit"], "algorithmic_flops": work["vit_flops"] * B,
                       "achieved_tflops": work["vit_flops"] * B / (stage_ms["apf_vit"] / 1e3) / 1e12,
                       "frac_of_bf16_peak": work["vit_flops"] * B / (stage_ms["apf_vit"] / 1e3) / 1e12 / peak_tf}
    if world == 1 and not args.no_cpu_baseline:
        sample = CPU_SAMPLE[args.workload]
        v, secs = time_cpu_port(w, sample, 2)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"{sample} clouds of the {args.workload} workload, best of 2 after 1 warm-up ({secs:.2f} s per pass)"}
    print(json.dumps(line), flush=True)


def c5_strong_probe(args, rank, world, device, precision, tok_dtype):
    """BASELINE configs[4]: B = 4096 clouds per step split 4096/world per GPU, final all-gather of the (4096/world, 64, 256)
    token shards inside the e2e step, timed over --steps steps; strong scaling: value = 4096 clouds / max-over-ranks step
    time."""
    import torch.distributed as dist
    w = dict(WORKLOADS["c5"])
    B = per_gpu_clouds(w, world)
    H = Harness(w, B, precision, tok_dtype, device, rank, world, "uniform")
    H.prepare_device_loop(3)
    steps = args.steps
    ms = H.time_device(steps)
    H.prepare_e2e()
    ems = H.time_e2e(steps)
    res = {"workload": w["desc"], "scaling": "strong", "clouds_per_step": w["B"], "clouds_per_gpu": B,
           "value": w["B"] * steps / (ms / 1e3), "ms_per_step": ms / steps,
           "e2e": w["B"] * steps / (ems / 1e3), "e2e_ms_per_step": ems / steps,
           "h2d_bytes_per_step": H.h2d_bytes, "d2h_bytes_per_step": H.d2h_bytes}
    if world > 1:
        out0 = H.graphs[0].output
        gbuf = [torch.empty((world,) + tuple(out0.shape), dtype=out0.dtype, device=device) for _ in range(2)]

        def gather(g):
            with torch.cuda.stream(g.stream):
                dist.all_gather_into_tensor(gbuf[0 if g is H.graphs[0] else 1], g.output)
        gms = H.time_e2e(steps, gather=gather)
        res["e2e_with_gather"] = w["B"] * steps / (gms / 1e3)
        res["e2e_with_gather_ms_per_step"] = gms / steps
        res["gathered_bytes_per_rank"] = gbuf[0].numel() * gbuf[0].element_size()
    return res


def main():
    sys.dont_write_bytecode = True      # the project modules are imported from here on; the source tree may be read-only
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="p3tok", choices=["p3tok", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("P3TOK_BENCH_PRECISION", "bf16"), choices=["fp32", "bf16", "fp32tc"])
    ap.add_argument("--token-dtype", default="bf16", choices=["bf16", "f32"],
                    help="dtype of the tokens the serving step returns (bf16 path: rounded once in the producing epilogue; f32 = the reference's dtype)")
    ap.add_argument("--clouds", default="both", choices=["uniform", "clustered", "both"],
                    help="input kind of the headline numbers; 'both' = uniform headline + a short clustered run attached as other_clouds")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the c5 strong-scaling probe attached to the default c2 line")
    ap.add_argument("--streams", type=int, default=0, help="steps in flight (graphs replayed round-robin on as many streams) in the device-resident and e2e loops; 0 = auto: 2, up to 4 when the batch is well below the SM count")
    ap.add_argument("--ncu", type=int, default=0, help="profiling aid: run N eager steps between cudaProfilerStart/Stop and exit (no timing)")
    ap.add_argument("--eager", action="store_true", help="time the Python-dispatched module call instead of the CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.gpus > 1:
        print(json.dumps({"error": "launch with torch.distributed.run for --gpus > 1"}))
        sys.exit(2)
    try:
        run_p3tok(args, w, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
