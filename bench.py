#!/usr/bin/env python
"""bench.py -- images/sec of GANsformer synthesis (BASELINE.json configs, default configs[1]: 256x256, K=16, batch 32/GPU)
+ attention roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one generator forward over one batch of synthetic latents (weak scaling: every rank runs its own slice of a
globally seeded batch, no data-path collective -- SURVEY 8e).  Rank 0 prints ONE JSON line.

  value            images/s with latents resident in HBM (CUDA events, max over ranks); value_fp32_convs: the same steps with
                   fp32 (not TF32) cuDNN convolutions
  e2e              images/s through the public ``Generator.run``-shaped call: pinned host latents -> H2D -> forward ->
                   D2H of the images, every step
  roofline         the WHOLE attention path of the step (batched stage I + every layer call): ALGORITHMIC bytes (read X once +
                   write X' once per layer, SURVEY 8d) / CUDA-event time, vs MEASURED_PEAKS.json hbm_gbs; stage_T = the
                   dominant kernel alone; traffic = DRAM bytes of the largest stage-T launch parsed from the tracked
                   profiles/r02/traffic_config<N>.csv (tools/traffic_capture.sh, ncu on the current build)
  roofline_conv    row f1: the library's own 3x3 convolution kernel against the tensor roofline (TFLOP/s, measured bf16 peak / 2)
  roofline_duplex  BASELINE's second named metric: the 12 duplex layer calls of configs[2] (K=32, batch 64), same formula
  train_step       BASELINE configs[3]: G+D training step, data-parallel with the NCCL gradient all-reduce, at every N
  cpu_baseline     the CPU oracle (oracle/generator.py, fp32, pinned thread count, median of 3) on a bounded sample, N = 1 only

--dump-outputs DIR writes DIR/images.npy: the float32 images [B, 3, R, R] the last timed step returned (rank 0's slice).
Weights (seed 0) and latents (seed 1) are fixed, so two builds run with the same arguments can be compared image for image.
The comparison needs a tolerance: cuDNN picks its TF32 algorithms per process, and two runs of one build differed by
2.6e-4 relative RMS (NVIDIA B200, 1000 W power limit).

--impl reference times the reference arm: the reference's own implementation cannot be installed (no source in
/root/reference, TensorFlow 1.14 unavailable -- DESIGN.md), so per the tier contract the arm is the CPU oracle port.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# BASELINE.json configs, numbered as in SURVEY.md 8d (config N = configs[N-1]).  The default (and the driver's) line is config 2.
CONFIGS = {
    1: dict(res=64, k=8, batch=4, duplex=False, layers=8, label="BASELINE configs[0]: GANsformer generator forward, 64x64, K=8 latents, batch 4 (the reference's CPU-runnable case)"),
    2: dict(res=256, k=16, batch=32, duplex=False, layers=12, label="BASELINE configs[1]: 256x256 synthesis, K=16 latents, 12 attention layers, batch 32 per GPU, simplex"),
    3: dict(res=256, k=32, batch=64, duplex=True, layers=12, label="BASELINE configs[2]: 256x256 duplex-attention variant, K=32 latents, batch 64 per GPU"),
    5: dict(res=512, k=32, batch=16, duplex=False, layers=14, label="BASELINE configs[4]: 512x512 synthesis, K=32 latents, batch 16 per GPU (128 over 8 GPUs), 14 attention layers"),
}
RES, K_LATENTS, LATENT_DIM, B_PER_GPU, DUPLEX = 256, 16, 32, 32, False
METRIC = "images/sec @256^2 synth (GANsformer generator forward, K=16 latents, 12 attention layers, batch 32/GPU)"
UNIT = "images/s"
CPU_THREADS_CAP = 32          # MKL-DNN convolutions collapse beyond ~32 threads on the 64/128-thread hosts of this pool


def select_config(n: int):
    global RES, K_LATENTS, B_PER_GPU, DUPLEX, METRIC
    c = CONFIGS[n]
    RES, K_LATENTS, B_PER_GPU, DUPLEX = c["res"], c["k"], c["batch"], c["duplex"]
    METRIC = (f"images/sec @{RES}^2 synth (GANsformer generator forward, K={K_LATENTS} latents, {c['layers']} attention layers, "
              f"batch {B_PER_GPU}/GPU{', duplex' if DUPLEX else ''})")
    return c


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each array as out_dir/<name>.npy (float32)."""
    import numpy as np
    arrays = {n: a.detach().float().cpu().numpy() for n, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def conv_roofline_probe(device, iters: int = 5):
    """Row f1 kernel against the tensor roofline: the five stride-1 3x3 convolutions of the 256x256 generator (batch 32) on the library's
    own tcgen05 implicit-GEMM kernel, each layer timed on its own with CUDA events after warm-up (inputs 67 MB ... 1.07 GB, alternating
    between two buffers).  FLOPs = 2 * 9 * B * H * W * Cin * Cout.  Peak = measured cuBLAS bf16 throughput / 2 (kind::tf32 runs at half
    the bf16 rate)."""
    from importlib import import_module
    ops = import_module("gansformer-reproducibility-challenge_b200.ops")
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        peak, src = float(pk["bf16_tflops"]) / 2, "measured cuBLAS bf16 burst (MEASURED_PEAKS.json) / 2"
    except Exception:
        peak, src = 1125.0, "nominal dense TF32 (2250 bf16 / 2)"
    B = 32
    layers, tot_flop, tot_ms = [], 0.0, 0.0
    for res, C in [(16, 512), (32, 512), (64, 512), (128, 256), (256, 128)]:
        xs = [torch.randn(B, C, res, res, device=device).contiguous(memory_format=torch.channels_last) for _ in range(2)]
        wt = ops.conv3x3_pack(torch.randn(C, C, 3, 3, device=device) / (3.0 * C ** 0.5))
        for i in range(3):
            ops.conv3x3_native(xs[i & 1], wt)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            ops.conv3x3_native(xs[i & 1], wt)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        fl = 2.0 * 9 * B * res * res * C * C
        layers.append({"res": res, "channels": C, "ms": ms, "tflops": fl / ms / 1e9})
        tot_flop += fl
        tot_ms += ms
        del xs, wt
    torch.cuda.empty_cache()
    ach = tot_flop / tot_ms / 1e9
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "peak_source": src,
            "kernel": "conv3x3_tc_kernel / conv3x3_tc_kernel_v2 (gf_conv3x3_nhwc_tf32): the five stride-1 3x3 convolutions of the step, "
                      "timed layer by layer outside the step", "ms_total": tot_ms, "layers": layers}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (recipe in B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def build_generator(device):
    import gansformer_b200 as gf
    torch.manual_seed(0)                                   # SURVEY 8d: weights seed 0, N(0,1), biases 0
    G = gf.Generator(resolution=RES, components_num=K_LATENTS, latent_dim=LATENT_DIM, kmeans=DUPLEX)
    return G.to(device).eval()


def global_latents(world: int):
    g = torch.Generator().manual_seed(1)                   # SURVEY 8d: latents seed 1, generated on CPU
    return torch.randn(B_PER_GPU * world, K_LATENTS + 1, LATENT_DIM, generator=g)


def cpu_threads() -> int:
    """Thread count of the CPU arm: pinned (no per-run search -- the r01 picker made the same work move 0.9 -> 1.7 img/s)."""
    return max(1, min(os.cpu_count() or 1, CPU_THREADS_CAP))


def cpu_oracle_run(G_state, steps: int, warmup: int, sample_b: int, duplex: bool = None):
    """Times the CPU oracle generator (fp32, NCHW, direct op order) on `sample_b` images per step: median of `steps` (>= 3)."""
    from oracle import generator as og
    threads = cpu_threads()
    torch.set_num_threads(threads)
    z = global_latents(1)[:sample_b]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        og.generator_forward(G_state, z, resolution=RES, components_num=K_LATENTS, latent_dim=LATENT_DIM,
                             duplex=DUPLEX if duplex is None else duplex, dtype=torch.float32)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    return sample_b / t, t, threads


def duplex_attention_probe(device, peak_gbs: float, iters: int = 6):
    """BASELINE configs[2] attention path: the 12 duplex attention layers of the 256x256 generator (K=32, batch 64) exactly as the
    synthesis network issues them -- ONE batched stage-I launch for all 12 layers (gf_attn_prologue_batch), then per layer pass A +
    key products + stage T -- captured in one CUDA graph and replayed; CUDA-event timed.  Every layer has its own input tensor
    (15.7 GB of activations in total: nothing is L2-resident between replays).  ALG bytes as for simplex (2 * 4 * B * n * C per layer)."""
    import gansformer_b200 as gf
    from importlib import import_module
    am = import_module("gansformer-reproducibility-challenge_b200.attention")
    B, k, D = 64, 32, 32
    shapes = [(8, 512), (8, 512), (16, 512), (16, 512), (32, 512), (32, 512), (64, 512), (64, 512), (128, 256), (128, 256), (256, 128), (256, 128)]
    y = torch.randn(B, k, D, device=device)
    layers, xs, tot_bytes = [], [], 0
    out = torch.empty(B * 256 * 256 * 128, device=device)             # one output buffer, viewed per layer
    for res, C in shapes:
        layers.append(gf.BipartiteAttention(C, D, k, kmeans=True).to(device))
        xs.append(torch.randn(B, res, res, C, device=device))
        tot_bytes += 2 * 4 * B * res * res * C

    def run_all():
        am.prologue_batch([(m, y, tuple(x.shape), None) for m, x in zip(layers, xs)])
        for m, x in zip(layers, xs):
            m(x, y, out=out[:x.numel()].view_as(x), stage="token", need_centroids=False)

    with torch.no_grad():
        for _ in range(2):
            run_all()
        torch.cuda.synchronize()
        gph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gph):
            run_all()
        gph.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            gph.replay()
        e1.record()
        torch.cuda.synchronize()
    tot_ms = e0.elapsed_time(e1) / iters
    cen_path = gf._lib.last_centroid_path()
    del gph, xs, out, layers
    torch.cuda.empty_cache()
    achieved = tot_bytes / (tot_ms * 1e-3) / 1e9
    return {"workload": "BASELINE configs[2] attention path: the 12 duplex layers of the 256x256 generator, K=32, batch 64, as the synthesis "
                        "network issues them (one batched stage-I launch, then pass A + key products + stage T per layer), one CUDA graph",
            "ms": tot_ms, "alg_bytes": tot_bytes, "achieved": achieved,
            "unit": "GB/s", "frac": achieved / peak_gbs, "pass_a_path": cen_path,
            "dram_note": "three passes over X by construction (pass A reads it, stage T reads it again and writes X'): 1.5x the algorithmic "
                         "bytes; the B200 L2 keeps ~50 MB of a streamed tensor (tools/probes/l2_reuse_probe.cu), less than one 256^2 image + the "
                         "pipeline depth, so the second read cannot be an L2 hit (DESIGN.md 9.1)"}


def duplex_generator_probe(device, steps: int = 5, warmup: int = 2, B: int = 64, k: int = 32, with_cpu: bool = True):
    """BASELINE configs[2] end to end: the 256x256 generator with duplex attention (kmeans=True), K = 32 latents, batch 64,
    CUDA-graph replay with the latents resident; next to the CPU oracle on a 2-image sample of the same network."""
    import gansformer_b200 as gf
    torch.manual_seed(0)
    G = gf.Generator(resolution=256, components_num=k, latent_dim=32, kmeans=True).to(device).eval()
    g = torch.Generator().manual_seed(1)
    z = torch.randn(B, k + 1, 32, generator=g).to(device)
    with torch.no_grad():
        for _ in range(2):
            G(z)
        replay = G.graphed(B)
        for _ in range(warmup):
            replay(z)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            replay(z)
        e1.record()
        torch.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3
    out = {"workload": f"BASELINE configs[2]: 256x256 generator, duplex attention (kmeans), K={k} latents, batch {B}, 12 attention layers",
           "images_per_s": B * steps / t, "ms_per_step": t / steps * 1e3, "steps": steps, "warmup": warmup,
           "attention_path": gf._lib.last_path(), "pass_a_path": gf._lib.last_centroid_path()}
    if with_cpu:
        from oracle import generator as og
        sd = {n: v.detach().cpu() for n, v in G.state_dict().items()}
        zc = z[:2].cpu()
        torch.set_num_threads(cpu_threads())
        dts = []
        for _ in range(3):
            t0 = time.perf_counter()
            og.generator_forward(sd, zc, resolution=256, components_num=k, latent_dim=32, duplex=True, dtype=torch.float32)
            dts.append(time.perf_counter() - t0)
        out["cpu_baseline"] = {"value": 2 / statistics.median(dts), "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                               "sample": "median of 3 steps x 2 images of the same duplex generator, oracle/generator.py fp32"}
    del replay, G
    torch.cuda.empty_cache()
    return out


def train_probe(device, rank, world, steps: int = 3, warmup: int = 1, B: int = 32, graphed: bool = True):
    """BASELINE configs[3]: one D + one G update of the 256x256 GANsformer (K = 16, simplex) on synthetic reals, batch 32 per
    GPU, gradients averaged over ranks through one flat all-reduce per network (NCCL).  Attention forward = the CUDA
    kernels, attention backward = the stage-T backward kernel + batched GEMMs (autograd.py); convolutions and the discriminator = cuDNN."""
    import gansformer_b200 as gf
    from importlib import import_module
    tr = import_module("gansformer-reproducibility-challenge_b200.training")
    dist_mod = import_module("gansformer-reproducibility-challenge_b200.dist")
    torch.manual_seed(0)
    TR_RES, TR_K = 256, 16                           # configs[3] is quoted on the 256x256 K=16 simplex network
    G = gf.Generator(resolution=TR_RES, components_num=TR_K, latent_dim=LATENT_DIM, att_dp=0.12).to(device)    # attention dropout as upstream
    D = tr.Discriminator(TR_RES).to(device)
    trainer = tr.Trainer(G, D, world=world)
    g = torch.Generator().manual_seed(4)
    z = dist_mod.shard_batch(torch.randn(world * B, TR_K + 1, G.latent_dim, generator=g), rank, world).to(device)
    reals = dist_mod.shard_batch(torch.rand(world * B, 3, TR_RES, TR_RES, generator=g) * 2 - 1, rank, world).to(device)
    do_step = trainer.step_graphed if graphed else trainer.step
    trainer.it = 1                                   # timed steps are the common case (no lazy R1 term: 15 of 16 steps)
    for _ in range(warmup):
        do_step(z, reals)
        trainer.it = 1
    dist_mod.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for _ in range(steps):
        last = do_step(z, reals)
        trainer.it = 1
    e1.record()
    torch.cuda.synchronize()
    dist_mod.barrier()
    t = dist_mod.max_over_ranks(e0.elapsed_time(e1) * 1e-3, device=device)
    # the collective on its own (inside a replayed graph it cannot be bracketed by events): every bucket of both networks' flat
    # gradient buffers, back to back on the communication stream -- in the step these overlap the backward pass
    ar_ms, ar_bytes, n_buckets = 0.0, 0.0, 0
    if world > 1:
        bks = [trainer.buckets_d, trainer.buckets_g]
        n_buckets = sum(len(b.buckets) for b in bks)
        for rep in range(2):                          # first pass warms NCCL up for these message sizes
            dist_mod.barrier()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            ar_bytes = 0.0
            for b in bks:
                b._active = True
                b._pending = [1] * len(b.buckets)     # nothing pending from hooks: finish() reduces every bucket
                ar_bytes += b.finish()
            a1.record()
            torch.cuda.synchronize()
            ar_ms = a0.elapsed_time(a1)
    out = {"workload": "BASELINE configs[3]: 256x256 G+D training step (logistic NS + lazy R1, Adam, EMA), synthetic reals, "
                       f"batch {B}/GPU, data-parallel dp{world}", "images_per_s": world * B * steps / t, "ms_per_step": t / steps * 1e3,
           "global_batch": world * B, "steps": steps, "warmup": warmup, "allreduce_ms_per_step": ar_ms,
           "allreduce_bytes_per_step": ar_bytes, "allreduce_buckets": n_buckets,
           "allreduce_note": "bucketed NCCL all-reduce (ReduceOp.AVG) of both networks' flat gradient buffers, timed back to back on its own; "
                             "inside the step the buckets are launched from backward hooks on a communication stream and overlap backward", "loss_g": last.loss_g, "loss_d": last.loss_d,
           "peak_mem_gb": torch.cuda.max_memory_allocated(device) / 2 ** 30,
           "cuda_graph": bool(graphed),
           "attention_dropout": 0.12,
           "backward": "attention: CUDA forward (tcgen05 kernel with Philox attention dropout p = 0.12 on the probabilities) + hand-written stage-T backward kernel "
                       "(gf_attn_simplex_bwd_ex, same mask) + batched GEMMs for the token reductions; FIR filters: native (self-adjoint) "
                       "kernel; convolutions / discriminator: cuDNN; gradients: bucketed NCCL all-reduce overlapped with backward"}
    del trainer, G, D
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    """The reference arm: the reference's own implementation cannot be installed or run (its source is not available and
    it needs TensorFlow 1.14), so this times the CPU oracle port on the host cores: pinned thread count, median of --steps
    steps of a bounded sample (2 images per step; config 1: its exact batch of 4)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    cfg = select_config(args.config)
    torch.manual_seed(0)
    import gansformer_b200 as gf
    G = gf.Generator(resolution=RES, components_num=K_LATENTS, latent_dim=LATENT_DIM, kmeans=DUPLEX)
    sample_b = B_PER_GPU if args.config == 1 else (1 if RES >= 512 else 2)
    steps, warmup = args.steps, 1
    ips, t, cores = cpu_oracle_run(G.state_dict(), steps, warmup, sample_b)
    line = {"impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["label"], "batch_per_step": sample_b,
                       "note": "reference source absent from /root/reference and TF1.14 unavailable: CPU oracle port (parity unpinned); "
                               f"{cores} pinned threads, median of {steps} steps"},
            "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"median of {steps} steps x {sample_b} images of the same generator forward (oracle/generator.py, fp32)"},
            "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


def parse_traffic(config_n: int):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch, read from the TRACKED csv that
    tools/traffic_capture.sh produced with ncu on the current build (profiles/r02/traffic_config<N>.csv); None if absent."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02", f"traffic_config{config_n}.csv")
    if not os.path.exists(path):
        return None, None
    best = None
    try:
        with open(path) as f:
            rows = list(csv.DictReader(l for l in f if not l.startswith("==")))
        per = {}
        for r in rows:
            if not r["Metric Name"].startswith("dram__bytes"):
                continue
            v = float(r["Metric Value"].replace(",", "")) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[r["Metric Unit"]]
            e = per.setdefault(r["ID"], {"name": r["Kernel Name"], "bytes": 0.0})
            e["bytes"] += v
        for e in per.values():
            if ("token_tc_kernel" in e["name"] or "token_simt" in e["name"]) and (best is None or e["bytes"] > best["bytes"]):
                best = e
    except Exception:
        return None, None
    if best is None:
        return None, None
    return best["bytes"], f"profiles/r02/traffic_config{config_n}.csv ({best['name'][:60]}: largest stage-T launch of one eager step)"


def run_ours(args):
    import gansformer_b200 as gf
    from importlib import import_module
    dist_mod = import_module("gansformer-reproducibility-challenge_b200.dist")
    attn_mod = import_module("gansformer-reproducibility-challenge_b200.attention")
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device: the product has no CPU path")
    cfg = select_config(args.config)
    rank, world, local = dist_mod.init_distributed("nccl")
    if world != args.gpus:
        raise RuntimeError(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    # surrounding cuDNN convolutions (plumbing, SURVEY row f1 is "next"): TF32 tensor-core math, fp32 storage; the same steps are
    # also timed with true-fp32 convolutions (value_fp32_convs) -- the reference's precision for them
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True

    G = build_generator(device)
    z_host = dist_mod.shard_batch(global_latents(world), rank, world).contiguous().pin_memory()
    z_dev = z_host.to(device)
    B = z_host.shape[0]
    img_host = torch.empty((B, 3, RES, RES), dtype=torch.float32).pin_memory()
    timer = attn_mod.StageTimer()

    use_graph = not args.no_cuda_graph
    with torch.no_grad():
        for _ in range(2):
            G(z_dev)                                  # eager warm-up: cuDNN autotune, weight folding, workspaces
    replay = G.graphed(B) if use_graph else None

    def step_eager():
        with torch.no_grad():
            return G(z_dev)

    def step_resident():
        if replay is not None:
            return replay(z_dev)
        return step_eager()

    # the public Gs.run-shaped call: host latents in, host images out.  ONE call over steps x B latents with minibatch B: every
    # step (= minibatch) copies its latents host->device and its images device->host inside the timed region; run() overlaps
    # the device->host copy of a minibatch with the next minibatch's compute.
    e2e_chunk = min(args.steps, 10)                  # minibatches per run() call (bounds the pinned host buffers)
    z_host_all = z_host.repeat(e2e_chunk, 1, 1).pin_memory()
    img_host_all = torch.empty((e2e_chunk * B, 3, RES, RES), dtype=torch.float32).pin_memory()

    def step_e2e():                                   # warm-up form: one minibatch
        return G.run(z_host, minibatch_size=B, cuda_graph=use_graph, out=img_host)

    for _ in range(args.warmup):
        step_resident()
        step_e2e()
    torch.cuda.synchronize()

    # ---- attention timing (eager: CUDA events around the launches cannot live inside a graph replay; the kernels and their
    #      inputs are the same ones the graph replays).  Whole attention = the batched stage-I launch of the step + every
    #      layer call (pass A + key products for duplex, stage T); stage T alone is reported next to it. -------------------
    attn_mod.STAGE_TIMER = timer
    timer.reset()
    launches0 = gf._lib.launch_count()
    torch.cuda.synchronize()
    for _ in range(args.steps):
        step_eager()
    torch.cuda.synchronize()
    launches = (gf._lib.launch_count() - launches0) // max(args.steps, 1)   # our kernels per step (same in the graph)
    attn_mod.STAGE_TIMER = None

    # ---- timed region 1: latents resident in HBM -------------------------------------------------------------
    sampler = ClockSampler(local)
    dist_mod.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()              # ncu --profile-from-start off captures exactly the timed steps
    ev0.record()
    for _ in range(args.steps):
        img = step_resident()
    ev1.record()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    if args.dump_outputs and rank == 0:              # before the next replay overwrites the graph's static output
        dump_outputs(args.dump_outputs, {"images": img})
    dist_mod.barrier()
    clocks = sampler.stop() if rank == 0 else None
    t_total = dist_mod.max_over_ranks(ev0.elapsed_time(ev1) * 1e-3, device)
    stage_t_s = sum(r[0].elapsed_time(r[1]) for r in timer.records) * 1e-3
    call_s = sum(r[3].elapsed_time(r[1]) for r in timer.records) * 1e-3 + sum(a.elapsed_time(b) for a, b in timer.batch_records) * 1e-3
    attn_bytes = sum(r[2] for r in timer.records)
    n_attn_calls = len(timer.records)
    path = gf._lib.last_path()

    # ---- timed region 2: end to end through the public call (H2D + forward + D2H every step) -----------------
    dist_mod.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    done = 0
    while done < args.steps:                         # K steps = K minibatches, in calls of up to 10 minibatches
        m = min(e2e_chunk, args.steps - done)
        G.run(z_host_all[:m * B], minibatch_size=B, cuda_graph=use_graph, out=img_host_all[:m * B])
        done += m
    e1.record()
    torch.cuda.synchronize()
    dist_mod.barrier()
    t_e2e = dist_mod.max_over_ranks(e0.elapsed_time(e1) * 1e-3, device)

    # ---- the same resident steps with true-fp32 cuDNN convolutions (the reference's convolution precision) ----
    t_fp32 = None
    if not args.no_fp32_convs:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        with torch.no_grad():
            G(z_dev)
        replay32 = G.graphed(B) if use_graph else None          # graph key includes the TF32 switches: a new capture
        n32 = max(3, min(args.steps, 10))
        for _ in range(2):
            replay32(z_dev) if replay32 is not None else step_eager()
        dist_mod.barrier()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(n32):
            replay32(z_dev) if replay32 is not None else step_eager()
        f1.record()
        torch.cuda.synchronize()
        dist_mod.barrier()
        t_fp32 = dist_mod.max_over_ranks(f0.elapsed_time(f1) * 1e-3, device) / n32
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cuda.matmul.allow_tf32 = True
        del replay32

    # ---- the same resident steps with cuDNN's TF32 stride-1 convolutions instead of the library's own implicit-GEMM kernel (row f1) ----
    t_cudnn = None
    if not args.no_fp32_convs:
        os.environ["GF_CUDNN_CONV"] = "1"
        try:
            with torch.no_grad():
                G(z_dev)
            replay_c = G.graphed(B) if use_graph else None      # graph key includes the switch: a new capture
            nc = max(3, min(args.steps, 10))
            for _ in range(2):
                replay_c(z_dev) if replay_c is not None else step_eager()
            dist_mod.barrier()
            torch.cuda.synchronize()
            c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0_.record()
            for _ in range(nc):
                replay_c(z_dev) if replay_c is not None else step_eager()
            c1_.record()
            torch.cuda.synchronize()
            dist_mod.barrier()
            t_cudnn = dist_mod.max_over_ranks(c0_.elapsed_time(c1_) * 1e-3, device) / nc
            del replay_c
        finally:
            del os.environ["GF_CUDNN_CONV"]

    # ---- BASELINE configs[3]: the training step (the only collective of the system: the gradient all-reduce).  Runs at every N
    #      (SCALE carries it); a watchdog prints the headline line without it if a rank hangs inside the probe.
    tp = None
    want_train = (not args.no_train_probe) and args.config == 2
    state = {"line": None}

    def finish(tp_obj):
        if rank != 0:
            return
        line = state["line"]
        if tp_obj is not None:
            line["train_step"] = tp_obj
        print(json.dumps(line), flush=True)

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = attn_bytes / call_s / 1e9 if call_s > 0 else 0.0
        achieved_t = attn_bytes / stage_t_s / 1e9 if stage_t_s > 0 else 0.0
        traffic, traffic_src = parse_traffic(args.config)
        line = {
            "metric": METRIC, "value": world * B * args.steps / t_total, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "tf32 (fp32 storage; tcgen05 kind::tf32 attention and stride-1 3x3 convolutions (own kernels), TF32 cuDNN up-convolutions; value_fp32_convs = the same with fp32 cuDNN convolutions)" if path == "tcgen05_tf32" else "f32 (CUDA-core attention; TF32 cuDNN convs)",
            "data": "synthetic",
            "config": {"workload": cfg["label"] + ", integration=mul, norm=layer, random-init weights (seed 0), latents seed 1",
                       "global_batch": world * B, "parallelism": f"dp{world} (images sharded, no data-path collective)",
                       "l2_policy": "activations per layer (up to 1.07 GB) exceed the 126 MB L2; no flush needed",
                       "attention_path": path, "cuda_graph": bool(use_graph)},
            "gpu_launches": int(launches) * args.steps,
            "e2e": {"value": world * B * args.steps / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(z_host.numel() * 4 * world),
                    "d2h_bytes_per_step": int(img_host.numel() * 4 * world), "ms_per_step": t_e2e / args.steps * 1e3,
                    "call": "Generator.run(latents[m*B], minibatch_size=B, cuda_graph=True, out=pinned) over the K steps in calls of m <= 10 minibatches; per minibatch: H2D latents, "
                            "graph replay, D2H images on a copy stream overlapping the next minibatch"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": f"whole attention path of the step: stage I (one batched launch) + {'pass A + key products + ' if DUPLEX else ''}stage T ({path})",
                         "calls_timed": n_attn_calls, "alg_bytes_per_step": attn_bytes // max(args.steps, 1),
                         "attention_ms_per_step": call_s / args.steps * 1e3,
                         "attention_share_of_step": call_s / (ev0.elapsed_time(ev1) * 1e-3),
                         "stage_T": {"achieved": achieved_t, "frac": achieved_t / peak, "ms_per_step": stage_t_s / args.steps * 1e3,
                                     "note": "the dominant kernel alone (token_tc_kernel launches of the step)"},
                         "note": "timed in an eager pass of the same K steps (CUDA events on the launch stream); the step itself replays a "
                                 "CUDA graph. Each stage-T launch also carries the fused demodulation scale, noise, bias, leaky-ReLU and "
                                 "next-layer style scale (SURVEY row f3), which are not counted in the algorithmic bytes"},
            "clocks": clocks,
        }
        if t_fp32 is not None:
            line["value_fp32_convs"] = {"value": world * B / t_fp32, "unit": UNIT, "ms_per_step": t_fp32 * 1e3,
                                        "note": "same step, torch.backends.cudnn.allow_tf32 = False (fp32 cuDNN convolutions); attention unchanged"}
        if t_cudnn is not None:
            line["value_cudnn_convs"] = {"value": world * B / t_cudnn, "unit": UNIT, "ms_per_step": t_cudnn * 1e3,
                                         "note": "same step with GF_CUDNN_CONV=1: cuDNN TF32 for the five stride-1 3x3 convolutions that otherwise run on "
                                                 "the library's own tcgen05 implicit-GEMM kernel (gf_conv3x3_nhwc_tf32, SURVEY row f1)"}
        state["line"] = line
    if world == 1 and not args.no_duplex_probe and args.config == 2:
        peak, _ = measured_peak_gbs()
        for key, fn in (("duplex_attention", lambda: duplex_attention_probe(device, peak)),
                        ("duplex_generator", lambda: duplex_generator_probe(device, with_cpu=not args.no_cpu_baseline))):
            try:
                state["line"][key] = fn()
            except Exception as exc:
                state["line"][key] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        da = state["line"].get("duplex_attention", {})
        if "frac" in da:      # BASELINE's second named metric ("duplex-attn %HBM-peak") in roofline form
            state["line"]["roofline_duplex"] = {"bound": "hbm", "achieved": da["achieved"], "peak": peak, "unit": "GB/s", "frac": da["frac"],
                                                "traffic": None, "kernel": "12 duplex layer calls of configs[2] (stage I + pass A + key products + stage T)"}
    if world == 1 and not args.no_duplex_probe and args.config == 2:
        try:
            state["line"]["roofline_conv"] = conv_roofline_probe(device)
        except Exception as exc:
            state["line"]["roofline_conv"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if world == 1 and not args.no_cpu_baseline:
        ips, t, cores = cpu_oracle_run(G.state_dict(), steps=3, warmup=1, sample_b=B_PER_GPU if args.config == 1 else (1 if RES >= 512 else 2))
        state["line"]["cpu_baseline"] = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port",
                                         "sample": f"median of 3 steps (+1 warm-up) x {B_PER_GPU if args.config == 1 else (1 if RES >= 512 else 2)} images of the same generator forward, "
                                                   f"oracle/generator.py fp32 on {cores} pinned host threads; oracle = in-repo restatement, "
                                                   "reference source unavailable, parity unpinned"}
    if want_train:
        done_evt = threading.Event()

        def watchdog():
            if not done_evt.wait(args.train_timeout):
                finish({"error": f"training probe did not finish within {args.train_timeout} s (rank {rank}); headline line printed without it"})
                os._exit(0)
        threading.Thread(target=watchdog, daemon=True).start()
        try:
            tp = train_probe(device, rank, world, graphed=not args.no_cuda_graph)
        except Exception as exc:                     # the probe must never take the headline line down with it
            tp = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        done_evt.set()
    finish(tp)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE.json config (SURVEY 8d numbering): 1 = 64^2 K=8 B=4, 2 = 256^2 K=16 B=32 (default, the driver's line), "
                         "3 = 256^2 duplex K=32 B=64, 5 = 512^2 K=32 B=16/GPU; config 4 (training step) is the train_step object of config 2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-duplex-probe", action="store_true")
    ap.add_argument("--no-fp32-convs", action="store_true", help="skip the value_fp32_convs variant")
    ap.add_argument("--no-train-probe", action="store_true", help="skip the BASELINE configs[3] probe (G+D training step, train_step object)")
    ap.add_argument("--train-probe", action="store_true", help="(kept for compatibility: the probe now runs at every N by default)")
    ap.add_argument("--train-timeout", type=float, default=240.0, help="watchdog of the training probe in seconds")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the images of the last timed step to DIR/images.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "ours":
        args.warmup = max(args.warmup, 3)
    rc = run_reference(args) if args.impl == "reference" else run_ours(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
