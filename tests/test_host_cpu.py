"""CPU tests of the host side: the C-ABI library loads and exports what include/gf_attn.h declares, descriptor
validation, the generator plumbing against the oracle, and the world_size-2 (gloo) data-parallel helpers.
No kernel is launched here (no GPU in this container)."""
import ctypes
import os
import re

import pytest
import torch
import torch.multiprocessing as mp

from oracle import bipartite as ob
from oracle import generator as og

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols(header):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gf_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported(gf):
    lib = gf._lib.load()
    for header, exports in (("gf_attn.h", gf._lib.EXPORTS), ("gf_ops.h", gf._lib.OPS_EXPORTS)):
        declared = _declared_symbols(header)
        assert declared == sorted(exports), (header, declared, exports)
        for name in declared:
            assert hasattr(lib, name), f"{name} declared in include/{header} but not exported by libgf_attn.so"
    assert lib.gf_attn_abi_version() == 2


def test_struct_layouts_match_c(gf):
    assert ctypes.sizeof(gf._lib.GfAttnDesc) == 12 * 4
    assert ctypes.sizeof(gf._lib.GfAttnWeights) == 23 * ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(gf._lib.GfAttnPostop) == 3 * 8 + 8 + 4 + 4 + 2 * 8 + 2 * 4 + 3 * 8 + 4 + 4 + 8
    assert ctypes.sizeof(gf._lib.GfDemodJob) == 3 * 8 + 4 * 4                      # gf_demod_job of include/gf_ops.h
    assert gf._lib.GfDemodJob.O.offset == 28 and gf._lib.GfDemodJob.I.offset == 32
    header = open(os.path.join(ROOT, "include", "gf_ops.h")).read()
    assert f"#define GF_DEMOD_MAX_JOBS {gf._lib.DEMOD_MAX_JOBS}" in header


def test_native_op_entry_points_validate_before_touching_the_device(gf):
    """gf_ops.h entry points added in round 2: argument errors come back as gf_status + message (no GPU needed to see them)."""
    lib = gf._lib.load()
    err = lambda: lib.gf_last_error().decode()
    assert lib.gf_conv3x3_nhwc_tf32(1, 1, 1, 2, 7, 16, 32, 64, None) == -2 and "H % 8 == 0" in err()       # GF_ERR_UNSUPPORTED
    assert lib.gf_conv3x3_nhwc_tf32(1, 1, 1, 2, 8, 16, 48, 64, None) == -2 and "Cin % 32" in err()
    assert lib.gf_conv3x3_nhwc_tf32(None, 1, 1, 2, 8, 16, 32, 64, None) == -1 and "null pointer" in err()    # GF_ERR_INVALID
    assert lib.gf_conv3x3_pack_weights(None, None, 4, 4, 1.0, None) == -1
    jobs = (gf._lib.GfDemodJob * 1)()
    as_ptr = ctypes.cast(jobs, ctypes.c_void_p)
    assert lib.gf_demod_coef_batch(None, 0, 4, 1e-8, None) == -1 and "1 <= n <= 32" in err()
    assert lib.gf_demod_coef_batch(as_ptr, gf._lib.DEMOD_MAX_JOBS + 1, 4, 1e-8, None) == -1
    assert lib.gf_demod_coef_batch(as_ptr, 1, 4, 1e-8, None) == -1 and "job 0" in err()


def test_integration_stub_matches_the_abi(gf):
    """The ctypes stub shown in INTEGRATION.md declares the same descriptor / weight members as the binding the tests run through."""
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"class gf_attn_weights\(C\.Structure\):.*?\((\"wq\".*?)\)\]", doc, re.S)
    assert m, "weights stub not found"
    assert tuple(re.findall(r'"(\w+)"', m.group(1))) == tuple(gf._lib.WEIGHT_FIELDS)
    m = re.search(r"class gf_attn_desc\(C\.Structure\):.*?\((\"B\".*?)\)\]", doc, re.S)
    assert m and tuple(re.findall(r'"(\w+)"', m.group(1))) == tuple(n for n, _ in gf._lib.GfAttnDesc._fields_)


def test_batched_demodulation_falls_back_per_layer_on_cpu():
    """ops.demod_coef_batch without CUDA tensors = the per-layer definition (the batched launch is a CUDA-only fast path)."""
    from importlib import import_module
    ops = import_module("gansformer-reproducibility-challenge_b200.ops")
    g = torch.Generator().manual_seed(3)
    pairs = [(torch.rand(3, 20, generator=g) + 0.5, torch.rand(7, 20, generator=g)), (torch.rand(3, 12, generator=g), torch.rand(5, 12, generator=g))]
    got = ops.demod_coef_batch(pairs)
    for d, (s_, w_) in zip(got, pairs):
        assert torch.allclose(d, torch.rsqrt(s_.square() @ w_.t() + 1e-8))
    assert ops.demod_coef_batch([]) == []


def test_sizes_and_validation(gf):
    L = gf._lib
    d = L.make_desc(4, 16, 16, 128, 16, 32, pos_dim=32)
    f1, w1 = L.folded_floats(d), L.workspace_bytes(d)
    assert f1 > 32 * (128 + 36) and w1 > 4 * 16 * 128 * 4
    d2 = L.make_desc(8, 16, 16, 128, 16, 32, pos_dim=32)
    assert L.workspace_bytes(d2) > w1 and L.folded_floats(d2) == f1          # folded weights do not depend on B
    dd = L.make_desc(4, 16, 16, 128, 16, 32, pos_dim=32, duplex=True)
    assert L.folded_floats(dd) > f1 and L.workspace_bytes(dd) > w1
    for bad, msg in [(dict(C=100), "C=100"), (dict(k=33), "k=33"), (dict(heads=8), "num_heads"), (dict(pos_dim=6), "pos_dim")]:
        kw = dict(B=1, H=8, W=8, C=64, k=4, D=16, heads=1, pos_dim=16)
        kw.update(bad)
        desc = L.make_desc(kw["B"], kw["H"], kw["W"], kw["C"], kw["k"], kw["D"], heads=kw["heads"], pos_dim=kw["pos_dim"])
        with pytest.raises(RuntimeError, match=msg):
            L.workspace_bytes(desc)


def test_no_cpu_path(gf):
    """The product must fail loudly on CPU tensors: there is no CPU fallback."""
    attn = gf.BipartiteAttention(64, 16, 4)
    x = torch.randn(1, 8, 16, 64)
    y = torch.randn(1, 4, 16)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU path"):
        attn(x, y)


def _small_generator(gf, **kw):
    torch.manual_seed(0)
    G = gf.Generator(resolution=32, components_num=4, latent_dim=16, fmap_base=512, fmap_max=64, mapping_layers=2, **kw)
    with torch.no_grad():  # make every term live: biases, noise strengths, w_avg
        for n, p in G.named_parameters():
            if n.endswith("bias") or n.endswith(".bq") or n.endswith(".bk") or n.endswith(".bv") or n.endswith(".bo"):
                p.normal_(0, 0.3)
            if n.endswith("noise_strength"):
                p.fill_(0.1)
        G.mapping.w_avg.normal_(0, 0.2)
    return G.double()


def test_generator_plumbing_matches_oracle_without_attention(gf):
    G = _small_generator(gf, transformer=False)
    z = torch.randn(2, 5, 16, dtype=torch.float64)
    with torch.no_grad():
        img = G(z, truncation_psi=0.7)
    ref = og.generator_forward(G.state_dict(), z, resolution=32, components_num=4, latent_dim=16, truncation_psi=0.7, mapping_layers=2)
    assert img.shape == (2, 3, 32, 32)
    assert (img - ref).abs().max() < 1e-9 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("duplex", [False, True, "extensions"])
def test_generator_plumbing_matches_oracle_with_patched_attention(gf, monkeypatch, duplex):
    """Host plumbing (layout, layer order, skip connections, the `iterative` centroid carry) checked on CPU by swapping the CUDA
    op for the oracle.  "extensions" = duplex with iterative carry, two k-means iterations and g_img2ltnt."""
    ext = duplex == "extensions"
    duplex = bool(duplex)
    G = _small_generator(gf, kmeans=duplex, integration="both", **(dict(iterative=True, kmeans_iters=2, g_img2ltnt=True) if ext else {}))
    carried = []

    def fake_forward(self, x, y, centroids=None, return_att=False, out=None, centroids_init=None):
        w = {n: p.detach() for n, p in self.named_parameters(recurse=False)}
        carried.append(centroids_init is not None)
        o, att, cen = ob.transformer_layer(x.permute(0, 3, 1, 2), y, w, integration=self.integration, norm=self.norm,
                                           duplex=self.duplex, use_pos=self.use_pos, return_att=return_att,
                                           kmeans_iters=self.kmeans_iters, img2ltnt=self.img2ltnt, centroids_init=centroids_init)
        return o.permute(0, 2, 3, 1).contiguous(), att, cen

    monkeypatch.setattr(gf.BipartiteAttention, "forward", fake_forward)
    z = torch.randn(2, 5, 16, dtype=torch.float64)
    with torch.no_grad():
        img, atts = G(z, return_att=True)
    ref, ratts = og.generator_forward(G.state_dict(), z, resolution=32, components_num=4, latent_dim=16, integration="both",
                                      duplex=duplex, mapping_layers=2, return_att=True,
                                      **(dict(iterative=True, kmeans_iters=2, img2ltnt=True) if ext else {}))
    assert len(atts) == len(ratts) == G.synthesis.num_attention_layers == 6
    assert any(carried) == ext                         # widths: 64 (res 8), 64 (res 16), 32 (res 32): carries inside and across blocks
    assert (img - ref).abs().max() < 1e-9 * max(1.0, ref.abs().max().item())
    for a, r in zip(atts, ratts):
        assert (a - r).abs().max() < 1e-10


def test_attention_layer_count_at_256(gf):
    """BASELINE config 2: 256x256, attention on both conv layers of every resolution 8..256 -> 12 layers."""
    from importlib import import_module
    nets = import_module("gansformer-reproducibility-challenge_b200.networks")
    assert [nets.nf(r) for r in (4, 8, 16, 32, 64, 128, 256, 512)] == [512, 512, 512, 512, 512, 256, 128, 64]
    with torch.device("meta"):
        G = gf.Generator(resolution=256, components_num=16, latent_size=512)
    assert G.latent_dim == 32 and G.synthesis.num_attention_layers == 12
    per_image = sum(l.resolution ** 2 * l.weight.shape[0] for l in G.synthesis.layers if l.attention is not None)
    assert per_image == 30736384          # SURVEY 8a: feature elements per image per pass


def _dist_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import gansformer_b200  # noqa: F401
    from importlib import import_module
    d = import_module("gansformer-reproducibility-challenge_b200.dist")
    r, w, _ = d.init_distributed("gloo")
    g = torch.Generator().manual_seed(1)
    glob = torch.randn(7, 3, generator=g)
    mine = d.shard_batch(glob, r, w)
    gathered = [None] * w
    dist.all_gather_object(gathered, mine)
    ok_union = torch.equal(torch.cat(gathered), glob)
    lin = torch.nn.Linear(3, 2)
    with torch.no_grad():
        lin.weight.fill_(0.5)
        lin.bias.zero_()
    lin(mine).square().sum().backward()
    nbytes = d.allreduce_gradients(lin.parameters(), w)
    mx = d.max_over_ranks(float(r + 1))
    q.put((r, ok_union, lin.weight.grad.clone(), nbytes, mx))
    d.barrier()
    dist.destroy_process_group()


def test_data_parallel_helpers_world2():
    """world_size-2 gloo: shards tile the global batch; the all-reduced gradient equals the mean of per-rank gradients."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dist_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    g = torch.Generator().manual_seed(1)
    glob = torch.randn(7, 3, generator=g)
    lin = torch.nn.Linear(3, 2)
    with torch.no_grad():
        lin.weight.fill_(0.5)
        lin.bias.zero_()
    grads = []
    for lo, hi in ((0, 4), (4, 7)):
        lin.zero_grad()
        lin(glob[lo:hi]).square().sum().backward()
        grads.append(lin.weight.grad.clone())
    expect = (grads[0] + grads[1]) / 2
    for r, ok_union, grad, nbytes, mx in res:
        assert ok_union
        assert torch.allclose(grad, expect, atol=1e-6)
        assert nbytes == (6 + 2) * 4 and mx == 2.0


def _bucket_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import gansformer_b200  # noqa: F401
    from importlib import import_module
    d = import_module("gansformer-reproducibility-challenge_b200.dist")
    r, w, _ = d.init_distributed("gloo")
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(6, 32), torch.nn.Tanh(), torch.nn.Linear(32, 16), torch.nn.Tanh(), torch.nn.Linear(16, 1))
    unused = torch.nn.Parameter(torch.ones(5))                      # a parameter that never receives a gradient
    params = list(net.parameters()) + [unused]
    buckets = d.GradBuckets(params, w, bucket_mb=0.0005)            # ~130 floats per bucket: several buckets
    x = torch.randn(8, 6, generator=torch.Generator().manual_seed(2))
    outs = []
    for step in range(2):                                           # second step: the views survive, the buffer is re-zeroed
        buckets.begin()
        net(d.shard_batch(x, r, w)).square().mean().backward()
        nbytes = buckets.finish()
        outs.append(torch.cat([p.grad.reshape(-1) for p in params]).clone())
    inside = all(p.grad.data_ptr() >= buckets.flat.data_ptr() and p.grad.data_ptr() < buckets.flat.data_ptr() + buckets.flat.numel() * 4 for p in params)
    q.put((r, outs[0].numpy(), outs[1].numpy(), nbytes, len(buckets.buckets), inside))
    d.barrier()
    dist.destroy_process_group()


def test_grad_buckets_world2_equal_full_batch_gradients():
    """GradBuckets (flat gradient buffer, reverse-order buckets reduced from post-accumulate hooks): the averaged gradients of
    two ranks on disjoint shards equal the single-process gradients of the full batch; parameters without a gradient stay 0."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_bucket_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=180) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(6, 32), torch.nn.Tanh(), torch.nn.Linear(32, 16), torch.nn.Tanh(), torch.nn.Linear(16, 1))
    x = torch.randn(8, 6, generator=torch.Generator().manual_seed(2))
    net(x).square().mean().backward()                                # shards of 4 + 4: mean of the shard means == full mean
    want = torch.cat([p.grad.reshape(-1) for p in net.parameters()] + [torch.zeros(5)])
    for r, g1, g2, nbytes, nb, inside in res:
        assert inside and nb >= 2
        assert nbytes == want.numel() * 4
        assert torch.allclose(torch.from_numpy(g1), want, atol=1e-6) and torch.allclose(torch.from_numpy(g2), want, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------
# G/D training step (SURVEY row f2): plumbing on CPU without attention layers (the attention op has no CPU form)
# ---------------------------------------------------------------------------------------------------------
def _tiny_gan(gf, seed=0):
    from importlib import import_module
    tr = import_module("gansformer-reproducibility-challenge_b200.training")
    torch.manual_seed(seed)
    G = gf.Generator(resolution=16, components_num=4, latent_dim=16, fmap_base=256, fmap_max=32, mapping_layers=2, transformer=False)
    D = tr.Discriminator(16, fmap_base=256, fmap_max=32)
    return tr, G, D


def test_training_step_plumbing(gf):
    tr, G, D = _tiny_gan(gf)
    trainer = tr.Trainer(G, D, tr.TrainConfig(noise_mode="const"))
    g = torch.Generator().manual_seed(3)
    z, reals = torch.randn(4, 5, 16, generator=g), torch.rand(4, 3, 16, 16, generator=g) * 2 - 1
    g0 = [p.detach().clone() for p in G.parameters()]
    d0 = [p.detach().clone() for p in D.parameters()]
    e0 = [p.detach().clone() for p in trainer.G_ema.parameters()]
    s1 = trainer.step(z, reals)                    # iteration 0: includes the lazy R1 term
    s2 = trainer.step(z, reals)
    for s in (s1, s2):
        assert all(map(lambda v: v == v and abs(v) < 1e6, (s.loss_g, s.loss_d, s.r1)))
    assert s1.r1 > 0 and s2.r1 == 0
    assert any((a - b.detach()).abs().max() > 0 for a, b in zip(g0, G.parameters()))
    assert any((a - b.detach()).abs().max() > 0 for a, b in zip(d0, D.parameters()))
    assert any((a - b).abs().max() > 0 for a, b in zip(e0, trainer.G_ema.parameters()))
    assert D(reals).shape == (4,)


def _train_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import gansformer_b200 as gf
    from importlib import import_module
    d = import_module("gansformer-reproducibility-challenge_b200.dist")
    r, w, _ = d.init_distributed("gloo")
    torch.set_num_threads(2)
    tr, G, D = _tiny_gan(gf)
    trainer = tr.Trainer(G, D, tr.TrainConfig(noise_mode="const", r1_gamma=0.0), world=w)
    g = torch.Generator().manual_seed(3)
    z, reals = torch.randn(4, 5, 16, generator=g), torch.rand(4, 3, 16, 16, generator=g) * 2 - 1
    st = trainer.step(d.shard_batch(z, r, w), d.shard_batch(reals, r, w))
    flat = lambda m: torch.cat([p.detach().reshape(-1) for p in m.parameters()]).numpy()      # by value: the worker exits first
    q.put((r, flat(D), flat(G), st.allreduce_bytes))
    d.barrier()
    dist.destroy_process_group()


def test_training_step_world2_keeps_replicas_identical(gf):
    """world_size-2 gloo: after one step on disjoint shards both ranks hold identical G and D weights, and the flat-buffer
    all-reduce moved every gradient once per network."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_train_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    (_, d0, g0, nb0), (_, d1, g1, nb1) = res
    assert (d0 == d1).all() and (g0 == g1).all()
    tr, G, D = _tiny_gan(gf)
    nparams = sum(p.numel() for p in D.parameters()) + sum(p.numel() for p in G.parameters() if p.requires_grad)
    assert nb0 == nb1 and 0 < nb0 <= 4 * nparams
    assert (torch.from_numpy(d0) - torch.cat([p.detach().reshape(-1) for p in D.parameters()])).abs().max() > 0   # and they did move


# ---------------------------------------------------------------------------------------------------------
# training path: the differentiable per-image tables (stages W + I in torch) equal the oracle's folded prologue
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,H,W,k,D,p,integration,use_pos", [(64, 8, 16, 4, 16, 16, "both", True), (96, 10, 13, 20, 12, 8, "mul", True),
                                                              (32, 4, 4, 3, 8, 4, "add", False)])
def test_folded_tables_match_oracle_prologue(gf, C, H, W, k, D, p, integration, use_pos):
    from importlib import import_module
    from oracle import folded as of
    ag = import_module("gansformer-reproducibility-challenge_b200.autograd")
    w = ob.init_params(C, D, k, p, integration, False, seed=3, bias_std=0.4)
    y = torch.randn(2, k, D, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    f = of.fold_weights(w, C=C, k=k, integration=integration, duplex=False, use_pos=use_pos)
    Kp, Vt, Rt, Ct = of.prologue(y, f, C=C, H=H, W=W, p=p, use_pos=use_pos)
    gKp, gVt, gRt, gCt, gcb = ag.folded_tables(y, w, H=H, W=W, C=C, integration=integration, use_pos=use_pos)
    for got, want in ((gKp, Kp), (gVt, Vt), (gCt, Ct)):
        assert got.shape == want.shape and (got - want).abs().max() < 1e-11 * max(1.0, want.abs().max().item())
    fin = torch.isfinite(Rt)
    assert torch.equal(torch.isfinite(gRt), fin) and (gRt[fin] - Rt[fin]).abs().max() < 1e-11 * max(1.0, Rt[fin].abs().max().item())
    # and they are differentiable end to end (padded -inf columns carry no gradient)
    ys = y.clone().requires_grad_(True)
    ws = {n: t.clone().requires_grad_(True) for n, t in w.items()}
    tabs = ag.folded_tables(ys, ws, H=H, W=W, C=C, integration=integration, use_pos=use_pos)
    loss = sum((t[torch.isfinite(t)] ** 2).sum() for t in tabs)
    loss.backward()
    assert torch.isfinite(ys.grad).all() and all(torch.isfinite(t.grad).all() for t in ws.values() if t.grad is not None)


def test_upconv_polyphase_decomposition_cpu(gf):
    """The four stride-1 convolutions of ops.upconv_phase_weights are the polyphase components of the stride-2 transposed 3x3
    convolution (what the inference path feeds the polyphase blur kernel with)."""
    from importlib import import_module
    ops = import_module("gansformer-reproducibility-challenge_b200.ops")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 8, 5, 7, generator=g, dtype=torch.float64)
    w = torch.randn(12, 8, 3, 3, generator=g, dtype=torch.float64)
    T = torch.nn.functional.conv_transpose2d(x, w.transpose(0, 1), stride=2)                 # [2, 12, 11, 15]
    for (a, b), (wk, pad) in zip(((0, 0), (0, 1), (1, 0), (1, 1)), ops.upconv_phase_weights(w)):
        ph = torch.nn.functional.conv2d(x, wk, padding=pad)
        assert ph.shape == T[:, :, a::2, b::2].shape
        assert (ph - T[:, :, a::2, b::2]).abs().max() < 1e-12
    # tRGB definition with the fused second output (torch form)
    wr, st, s2 = torch.randn(3, 8, 1, 1, generator=g, dtype=torch.float64), torch.rand(2, 8, generator=g, dtype=torch.float64), torch.rand(2, 8, generator=g, dtype=torch.float64)
    rgb, xs = ops.torgb(x, wr, st, None, next_styles=s2)
    assert torch.equal(xs, x * s2[:, :, None, None]) and torch.equal(rgb, ops.torgb(x, wr, st, None))


def test_bench_configs_follow_baseline_json():
    """bench.py's --config table carries the resolution / K / batch figures BASELINE.json names (configs[3] is the train probe)."""
    import importlib.util, json
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))["configs"]
    for n, c in bench.CONFIGS.items():
        txt = base[n - 1].replace("\u00d7", "x")
        assert f"{c['res']}x{c['res']}" in txt and f"K={c['k']}" in txt, (n, txt)
        per_gpu = c["batch"] * (8 if n == 5 else 1)                     # configs[4] names the 8-GPU global batch
        assert f"batch={per_gpu}" in txt, (n, txt)
        assert ("duplex" in txt) == c["duplex"]
    c = bench.select_config(3)
    assert bench.RES == 256 and bench.K_LATENTS == 32 and bench.DUPLEX and "duplex" in bench.METRIC
    bench.select_config(2)
    assert "256^2" in bench.METRIC and "K=16" in bench.METRIC and bench.UNIT == "images/s"


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (the CPU oracle port timed on the host cores) runs without a GPU and prints ONE JSON line
    carrying the keys of the bench contract."""
    import json
    import subprocess
    import sys
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "e2e", "cpu_baseline"):
        assert key in line, key
    assert line["steps"] == 1
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_alias_package_shares_module_objects(gf):
    """``gansformer_b200.x`` must BE ``gansformer-reproducibility-challenge_b200.x`` (one copy of every module-level switch)."""
    import importlib
    real = importlib.import_module("gansformer-reproducibility-challenge_b200")
    assert gf is real
    for sub in ("training", "networks", "attention", "_lib", "ops", "dist", "_state"):
        a = importlib.import_module("gansformer_b200." + sub)
        b = importlib.import_module("gansformer-reproducibility-challenge_b200." + sub)
        assert a is b, sub
    from gansformer_b200.training import Trainer
    assert Trainer is gf.Trainer
    import gansformer_b200.networks as nets
    nets.CACHE_BYPASS = True
    try:
        assert importlib.import_module("gansformer-reproducibility-challenge_b200.networks").CACHE_BYPASS is True
    finally:
        nets.CACHE_BYPASS = False


def test_weight_caches_follow_the_weights_epoch(gf):
    """A parameter changed behind autograd's back (CUDA-graph replay of an optimizer step: no version bump) must not be
    served from the weight-derived caches once the weights epoch moves; deep copies carry no caches or plans."""
    import copy
    import importlib
    nets = importlib.import_module("gansformer_b200.networks")
    state = importlib.import_module("gansformer_b200._state")
    fc = nets.FullyConnected(8, 4)
    x = torch.randn(3, 8)
    with torch.no_grad():
        y0 = fc(x).clone()
        fc.weight.data.mul_(2.0)                      # .data: no version bump, like a graph replay
        assert torch.equal(fc(x), y0)                 # stale by construction ...
        state.bump_weights_epoch()
        y1 = fc(x)
        assert not torch.equal(y1, y0)                # ... until the epoch moves
    G = gf.Generator(resolution=16, components_num=2, latent_dim=8, fmap_base=64, fmap_max=16, mapping_layers=1)
    with torch.no_grad():
        G.mapping(torch.randn(2, 3, 8))
    G.__dict__["_graphs"] = {"k": object()}
    assert any("_icache" in m.__dict__ for m in G.modules())
    plan0 = G.synthesis.layers[1].attention._plan
    G2 = copy.deepcopy(G)
    assert "_graphs" not in G2.__dict__ and not any("_icache" in m.__dict__ for m in G2.modules())
    assert G2.synthesis.layers[1].attention._plan is not plan0 and G.synthesis.layers[1].attention._plan is plan0
    for (n1, p1), (n2, p2) in zip(G.named_parameters(), G2.named_parameters()):
        assert n1 == n2 and torch.equal(p1, p2) and p1.data_ptr() != p2.data_ptr()
    e0 = state.weights_epoch()
    G2.load_state_dict(G.state_dict())
    assert state.weights_epoch() == e0 + 1
    Gi = gf.Generator(resolution=16, components_num=2, latent_dim=8, fmap_base=64, fmap_max=16, kmeans=True, iterative=True, kmeans_iters=2,
                      g_img2ltnt=True)
    a = Gi.synthesis.layers[1].attention
    assert Gi.synthesis.iterative and a.iterative and a.kmeans_iters == 2 and a.img2ltnt and {"wcq", "wi2l", "bi2l"} <= set(a.param_dict())
