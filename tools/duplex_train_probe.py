"""Duplex training with attention dropout, measured: one GPU call, one JSON file under profiles/r03/ (default
profiles/r03/duplex_train_probe.json; DTP_OUT overrides it).

Layer level, at the config-3 duplex shapes (K = 32, B = 64; res 256 / C 128, res 128 / C 256, res 64 / C 512):
  * forward + backward of one layer with att_dp = 0.12 (stage-T backward kernel + pass-A recompute / backward kernels) and with
    att_dp = 0 (the torch composite backward), alternated in the same run;
  * the two pass-A kernels alone (gf_attn_centroid_recompute, gf_attn_centroid_bwd): CUDA events around each launch after a
    warm-up, median of DTP_REPS (>= 20) launches; achieved bytes/s and FLOP/s from shape-computed algorithmic counts.
Step level: Trainer.step_graphed of the 256x256 duplex generator (K = 16, B = 32, att_dp = 0.12), the simplex step with att_dp = 0.12,
and the duplex step at att_dp = 0 (composite backward); an out-of-memory or other failure is recorded as the result.
The card name, its power limit and max SM clock (nvidia-smi, read-only query) and a device-to-device copy bandwidth measured in the
same run are recorded beside the numbers."""
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time
from importlib import import_module

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import gansformer_b200 as gf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.environ.get("DTP_OUT", os.path.join(ROOT, "profiles", "r03", "duplex_train_probe.json"))
REPS = max(20, int(os.environ.get("DTP_REPS", 30)))
LAYER_SHAPES = [(256, 128), (128, 256), (64, 512)]          # (resolution, C) of the config-3 duplex layers
LAYER_B, LAYER_K, LATENT_DIM = 64, 32, 32
HBM_PEAK = 7.7e12                                          # B200 data sheet, one GPU (bytes/s)


def card_info(dev):
    info = {"device": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[dev.index or 0] if q.returncode == 0 else f"rc {q.returncode}: {q.stderr.strip()}"
    except Exception as e:  # the query is informational; a missing tool is recorded, not fatal
        info["nvidia_smi"] = f"unavailable: {e}"
    # CUDA-core FP32 FMA rate of this card: SMs x 128 lanes x 2 FLOP x max SM clock (nvidia-smi); a ceiling, not a measured rate
    try:
        mhz = float(info["nvidia_smi"].split(",")[1].strip().split()[0])
        info["fp32_fma_peak_flop_per_s"] = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 2 * mhz * 1e6
    except Exception:
        info["fp32_fma_peak_flop_per_s"] = None
    return info


def copy_bandwidth(dev, nbytes=2 << 30, reps=10):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    for _ in range(2):
        b.copy_(a)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    return {"bytes_moved": 2 * nbytes, "median_s": statistics.median(ts), "GB_per_s": 2 * nbytes / statistics.median(ts) / 1e9}


def _events(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def layer_level(dev, fp32_peak):
    ag = import_module("gansformer-reproducibility-challenge_b200.autograd")
    L = gf._lib
    lib = L.load()
    rows = []
    for res, C in LAYER_SHAPES:
        B, k, n = LAYER_B, LAYER_K, res * res
        row = {"res": res, "C": C, "B": B, "k": k}
        torch.manual_seed(0)
        attn = gf.BipartiteAttention(C, LATENT_DIM, k, kmeans=True, att_dp=0.12).to(dev).train()
        x = torch.randn(B, res, res, C, device=dev, requires_grad=True)
        y = torch.randn(B, k, LATENT_DIM, device=dev, requires_grad=True)
        gout = torch.randn(B, res, res, C, device=dev)

        def fwd_bwd():
            out, _, _ = attn(x, y)
            out.backward(gout)
            x.grad = y.grad = None
            attn.zero_grad(set_to_none=True)
        # alternate the two routes in the same run: dropout on (kernel route) / off (composite)
        ts = {"att_dp_0.12_kernel_route_ms": [], "att_dp_0_composite_ms": []}
        try:
            for rnd in range(4):
                for key, p in (("att_dp_0.12_kernel_route_ms", 0.12), ("att_dp_0_composite_ms", 0.0)):
                    attn.att_dp = p
                    t = _events(fwd_bwd, 1 if rnd == 0 else 3)
                    if rnd > 0:                                # round 0 warms both routes up
                        ts[key] += t
            for key, v in ts.items():
                row[key] = statistics.median(v)
        except torch.cuda.OutOfMemoryError as e:
            row["layer_error"] = f"out of memory: {str(e).splitlines()[0]}"
        torch.cuda.empty_cache()

        # the two pass-A kernels alone, on tables of the layer's own size
        KP = 16 if k <= 16 else 32
        X = torch.randn(B, n, C, device=dev)
        qy = torch.randn(B, k, C, device=dev)
        with torch.no_grad():
            M, Rt2, Ct2 = ag.duplex_query_tables(qy, {n_: p_.detach() for n_, p_ in attn.named_parameters()}, H=res, W=res, C=C, use_pos=True)
        desc = L.make_desc(B, res, res, C, k, LATENT_DIM, pos_dim=attn.pos_dim, duplex=1)
        ws = torch.empty(L.workspace_bytes(desc), dtype=torch.uint8, device=dev)
        Xbar, lse = torch.empty(B, k, C, device=dev), torch.empty(B, k, device=dev)
        dXbar = torch.randn(B, k, C, device=dev)
        dX = torch.zeros(B, n, C, device=dev)
        dSa = torch.empty(B, n, KP, device=dev)
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        rec = lambda: L.check(lib.gf_attn_centroid_recompute(ctypes.byref(desc), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(),
                                                              Xbar.data_ptr(), lse.data_ptr(), ws.data_ptr(), st), "recompute")
        bwd = lambda: L.check(lib.gf_attn_centroid_bwd(ctypes.byref(desc), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(), lse.data_ptr(),
                                                        Xbar.data_ptr(), dXbar.data_ptr(), dX.data_ptr(), dSa.data_ptr(), st), "bwd")
        for fn in (rec, bwd):
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        t_rec = statistics.median(_events(rec, REPS)) * 1e-3
        t_bwd = statistics.median(_events(bwd, REPS)) * 1e-3
        # algorithmic counts from the shapes (the working set, 4 B * B * n * C per [B,n,C] tensor, is >= 268 MB: larger than L2)
        by_rec = 4 * B * n * C                                   # X read once
        fl_rec = 2 * B * n * KP * C * 2                          # logits (x.M) + weighted sums (A x), FMA = 2 FLOP
        by_bwd = 4 * B * n * C * 3 + 4 * B * n * KP              # X read, dX read + written, dSa written
        fl_bwd = 2 * B * n * KP * C * 4                          # x.M, x.dXbar, dSa.M, A.dXbar
        for name, t, by, fl in (("recompute", t_rec, by_rec, fl_rec), ("centroid_bwd", t_bwd, by_bwd, fl_bwd)):
            row[name] = {"median_ms": t * 1e3, "reps": REPS, "alg_bytes": by, "alg_flop": fl, "GB_per_s": by / t / 1e9,
                         "TFLOP_per_s": fl / t / 1e12}
            if fp32_peak:
                t_by, t_fl = by / HBM_PEAK, fl / fp32_peak
                row[name].update(bound_by="HBM bytes" if t_by >= t_fl else "FP32 FMA", share_of_bound=max(t_by, t_fl) / t)
        rows.append(row)
        del attn, x, y, gout, X, dX, dSa
        torch.cuda.empty_cache()
    return rows


def step_level(dev, B=32, steps=3, warmup=2):
    tr = import_module("gansformer-reproducibility-challenge_b200.training")
    out = []
    for name, kw in (("duplex_att_dp_0.12", dict(kmeans=True, att_dp=0.12)), ("simplex_att_dp_0.12", dict(att_dp=0.12)),
                     ("duplex_att_dp_0_composite", dict(kmeans=True, att_dp=0.0))):
        rec = {"config": name, "res": 256, "k": 16, "B": B}
        try:
            torch.manual_seed(0)
            G = gf.Generator(resolution=256, components_num=16, latent_dim=LATENT_DIM, **kw).to(dev)
            D = tr.Discriminator(256).to(dev)
            trainer = tr.Trainer(G, D)
            g = torch.Generator().manual_seed(4)
            z = torch.randn(B, 17, LATENT_DIM, generator=g).to(dev)
            reals = (torch.rand(B, 3, 256, 256, generator=g) * 2 - 1).to(dev)
            trainer.it = 1
            for _ in range(warmup):
                trainer.step_graphed(z, reals)
                trainer.it = 1
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                st = trainer.step_graphed(z, reals)
                trainer.it = 1
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            rec.update(ms_per_step=ms, images_per_s=B / ms * 1e3, loss_g=st.loss_g, loss_d=st.loss_d,
                       peak_mem_GB=torch.cuda.max_memory_allocated(dev) / 1e9)
        except torch.cuda.OutOfMemoryError as e:
            rec["error"] = f"out of memory: {str(e).splitlines()[0]}"
        except Exception as e:  # a failing configuration is a finding of the probe, recorded as such
            rec["error"] = f"{type(e).__name__}: {str(e).splitlines()[0] if str(e) else ''}"
        out.append(rec)
        G = D = trainer = None
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit("duplex_train_probe: no CUDA device (this probe measures on the GPU only)")
    dev = torch.device("cuda:0")
    t0 = time.time()
    res = {"card": card_info(dev), "copy_bandwidth": copy_bandwidth(dev)}
    res["layers"] = layer_level(dev, res["card"]["fp32_fma_peak_flop_per_s"])
    if not os.environ.get("DTP_NO_STEPS"):
        res["steps"] = step_level(dev)
    res["copy_bandwidth_after"] = copy_bandwidth(dev)
    res["wall_s"] = time.time() - t0
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
