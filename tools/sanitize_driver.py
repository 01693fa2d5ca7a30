"""Small-shape driver for compute-sanitizer (tools/sanitize.sh): one launch of every tensor-path kernel family --
token_tc_kernel single-pass (C = 128, fused post-op with both scales), two-pass (C = 512), short tiles (8x8 grid),
centroid_tc_kernel (+ gemm_tc_kernel, merge) via duplex layers incl. the C = 512 channel-split -- plus the CUDA-core kernels
(fp32 mode), the stage-T backward, and every instantiation of the 3x3 convolution kernel (SAN_ONLY=conv for those alone).  Checks every output against the fp64 oracle so a sanitizer-clean run is also a
correct one."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gansformer_b200 as gf
from oracle import bipartite as ob

dev = torch.device("cuda:0")
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
only = os.environ.get("SAN_ONLY")
cases = [
    # name, C, H, W, k, B, integration, duplex, exact, postop
    ("token_tc/single-pass", 128, 16, 16, 16, 3, "both", False, False, True),
    ("token_tc/two-pass", 512, 16, 16, 16, 2, "mul", False, False, False),
    ("token_tc/short-tiles", 512, 8, 8, 8, 3, "mul", False, False, False),
    ("token_tc/KP32", 256, 16, 16, 32, 2, "add", False, False, False),
    ("centroid_tc/C128-K32", 128, 32, 32, 32, 2, "mul", True, False, True),
    ("centroid_tc/C512-split", 512, 16, 16, 16, 2, "mul", True, False, False),
    ("centroid_tc/short", 512, 8, 8, 32, 3, "mul", True, False, False),
    ("simt/fp32-duplex", 96, 10, 13, 7, 2, "both", True, True, False),
    ("token_tc/rgb-epilogue", 128, 16, 16, 16, 2, "mul", False, False, "rgb"),
]
D = p = 32
bad = 0
for name, C, H, W, k, B, integ, duplex, exact, post in cases:
    if only and only not in name:
        continue
    g = torch.Generator().manual_seed(C + k)
    x64 = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    y64 = torch.randn(B, k, D, generator=g, dtype=torch.float64)
    w = ob.init_params(C, D, k, p, integ, duplex, seed=3, bias_std=0.3)
    din = torch.rand(B, C, generator=g, dtype=torch.float64) + 0.5 if post else None
    ps = torch.rand(B, C, generator=g, dtype=torch.float64) + 0.5 if post else None
    bias = torch.randn(C, generator=g, dtype=torch.float64) * 0.3
    ref, _, _ = ob.transformer_layer(x64 * din[:, :, None, None] if post else x64, y64, w, integration=integ, duplex=duplex)
    if post:
        ref = torch.nn.functional.leaky_relu(ref + bias[None, :, None, None], 0.2) * 1.4 * ps[:, :, None, None]
    attn = gf.BipartiteAttention(C, D, k, pos_dim=p, integration=integ, kmeans=duplex, exact_fp32=exact).to(dev)
    with torch.no_grad():
        for n, prm in attn.named_parameters():
            prm.copy_(w[n].float())
        po = dict(bias=bias.float().to(dev), act="lrelu", gain=1.4, in_scale=din.float().to(dev), post_scale=ps.float().to(dev)) if post else None
        if post == "rgb":
            po.update(rgb_w=torch.randn(B, 3, C, device=dev) / C ** 0.5, rgb_bias=torch.zeros(3, device=dev), rgb_out=torch.empty(B, 3, H, W, device=dev))
        out, _, _ = attn(x64.permute(0, 2, 3, 1).contiguous().float().to(dev), y64.float().to(dev), postop=po)
    torch.cuda.synchronize()
    err = (out.double().cpu() - ref.permute(0, 2, 3, 1)).abs()
    atol, rtol = (4e-5, 4e-4) if exact else (1.6e-2, 1.6e-2)
    ratio = (err / (atol + rtol * ref.permute(0, 2, 3, 1).abs())).max().item()
    print(f"{name:28s} path={gf._lib.last_path()} cen={gf._lib.last_centroid_path() if duplex else '-'} max_err={err.max().item():.3e} ratio={ratio:.3f}", flush=True)
    bad += ratio > 1.0
# row f1: the implicit-GEMM convolution, both versions (small grids take version 1, H % 16 == 0 with enough tiles version 2)
if not only or "conv" in only:
    from importlib import import_module
    ops = import_module("gansformer-reproducibility-challenge_b200.ops")
    for (B, H, W, ci, co) in [(2, 8, 16, 64, 64), (10, 32, 32, 64, 128), (6, 32, 32, 32, 256)]:
        x = torch.randn(B, ci, H, W, device=dev).contiguous(memory_format=torch.channels_last)
        w = torch.randn(co, ci, 3, 3, device=dev) / (ci * 9) ** 0.5
        got = ops.conv3x3_native(x, ops.conv3x3_pack(w))
        ref = torch.nn.functional.conv2d(x, w, padding=1)
        torch.cuda.synchronize()
        r = ((got - ref).abs().max() / ref.abs().max()).item()
        print(f"conv3x3 B={B} {H}x{W} {ci}->{co} max rel err {r:.3e}", flush=True)
        bad += r > 3e-3
    # each of the twelve instantiations once, forced through gf_conv3x3_nhwc_tf32_ex, on a grid of 2 x SMs + 2 tiles (every CTA
    # runs two or three tiles: accumulator sets reused, barrier phases flipped)
    nsm = torch.cuda.get_device_properties(dev).multi_processor_count
    for v in (1, 2):
        for bn in (256, 128, 64):
            for mt in (2, 1):
                B, H, W, ci, co = nsm + 1, 8 * mt, 32, 32, bn
                x = torch.randn(B, ci, H, W, device=dev).contiguous(memory_format=torch.channels_last)
                w = torch.randn(co, ci, 3, 3, device=dev) / (ci * 9) ** 0.5
                got = ops.conv3x3_native(x, ops.conv3x3_pack(w), variant=(v, bn, mt))
                ref = torch.nn.functional.conv2d(x, w, padding=1)
                torch.cuda.synchronize()
                r = ((got - ref).abs().max() / ref.abs().max()).item()
                print(f"conv3x3 v{v} bn={bn} mt={mt} B={B} {H}x{W} {ci}->{co} tiles={2 * B} max rel err {r:.3e}", flush=True)
                bad += r > 3e-3 or gf._lib.conv3x3_last_variant() != (v, bn, mt)
# attention dropout (CUDA-core forward + backward with the Philox mask)
if not only or "dropout" in only:
    attn = gf.BipartiteAttention(64, 16, 4, pos_dim=16, att_dp=0.2).to(dev).train()
    x = torch.randn(2, 8, 16, 64, device=dev, requires_grad=True)
    y = torch.randn(2, 4, 16, device=dev, requires_grad=True)
    out, _, _ = attn(x, y)
    out.square().mean().backward()
    torch.cuda.synchronize()
    print("dropout fwd/bwd ok", bool(torch.isfinite(x.grad).all()), flush=True)
# duplex attention dropout: forward on both kernel families (stage T reads the constants the duplex prologue writes), and the backward
# through the pass-A recompute / backward kernels (KP = 16 and 32, ragged grid, two k-means iterations)
if not only or "duplex-dropout" in only:
    for exact, C, H, W, k, iters in ((False, 128, 16, 16, 16, 1), (True, 96, 10, 13, 20, 2)):
        attn = gf.BipartiteAttention(C, 16, k, pos_dim=16, kmeans=True, kmeans_iters=iters, att_dp=0.2, exact_fp32=exact).to(dev).train()
        x = torch.randn(2, H, W, C, device=dev, requires_grad=True)
        y = torch.randn(2, k, 16, device=dev, requires_grad=True)
        with torch.no_grad():
            o0, _, _ = attn(x, y)
        out, _, _ = attn(x, y)
        out.square().mean().backward()
        torch.cuda.synchronize()
        ok = bool(torch.isfinite(x.grad).all()) and torch.equal(o0, out.detach())
        print(f"duplex-dropout C={C} k={k} iters={iters} path={gf._lib.last_path()} fwd/bwd ok", ok, flush=True)
        bad += not ok
# backward kernel
if not only or "bwd" in only:
    attn = gf.BipartiteAttention(64, 16, 4, pos_dim=16, integration="both").to(dev)
    x = torch.randn(2, 8, 16, 64, device=dev, requires_grad=True)
    y = torch.randn(2, 4, 16, device=dev, requires_grad=True)
    out, _, _ = attn(x, y)
    out.square().mean().backward()
    torch.cuda.synchronize()
    print("bwd/simplex ok", bool(torch.isfinite(x.grad).all()), flush=True)
sys.exit(1 if bad else 0)
