"""GPU tests of duplex layers trained with attention dropout (run on a B200: ``pytest -m gpu``).

Forward with the Philox mask against the fp64 oracle given the same mask (oracle/bipartite.py ``att_mult``), the D step's fused
no-grad route against per-layer calls, gradients through the pass-A backward kernels (gf_attn_centroid_recompute /
gf_attn_centroid_bwd) against the oracle's autograd, the two entry points called directly, and the training step."""
import ctypes
import math
from importlib import import_module

import pytest
import torch

from oracle import bipartite as ob
from oracle import philox as ph
from tests.test_gpu_parity import _small_generator, check_close

pytestmark = pytest.mark.gpu

am = import_module("gansformer-reproducibility-challenge_b200.attention")
ag = import_module("gansformer-reproducibility-challenge_b200.autograd")

PASS_A_PARAMS = ("wq2", "wk2", "wv2", "wkc")


def _setup(gf, dev, C, H, W, k, integration, norm, iters, i2l, exact, B=2, pd=0.2, seed_w=4):
    D = p = 16
    g = torch.Generator().manual_seed(C + k + 7 * iters + int(i2l))
    x64 = (torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 1.2 + 0.1).requires_grad_(True)
    y64 = torch.randn(B, k, D, generator=g, dtype=torch.float64).requires_grad_(True)
    w = {n: t.requires_grad_(True) for n, t in ob.init_params(C, D, k, p, integration, True, seed=seed_w, bias_std=0.3, extras=True).items()}
    attn = gf.BipartiteAttention(C, D, k, pos_dim=p, integration=integration, norm=norm, kmeans=True, kmeans_iters=iters, img2ltnt=i2l,
                                 att_dp=pd, exact_fp32=exact).to(dev)
    w = {n: w[n] for n, _ in attn.named_parameters()}
    with torch.no_grad():
        for n, prm in attn.named_parameters():
            prm.copy_(w[n].detach().float())
    seed, step = 24681357, 5
    am.set_dropout_seed(seed, dev, step)
    KP = 16 if k <= 16 else 32
    mult = torch.from_numpy(ph.dropout_mult(pd, seed, step, attn.dp_salt, B * H * W, KP).reshape(B, H * W, KP)[:, :, :k].copy())
    return x64, y64, w, attn, mult, g


FWD_CASES = [  # exact, C, H, W, k, integration, norm, kmeans_iters, img2ltnt
    (True, 64, 8, 16, 4, "both", "layer", 1, False),
    (True, 96, 10, 13, 20, "mul", "layer", 2, True),      # CUDA-core path, ragged n = 130, k > 16
    (True, 128, 16, 16, 16, "add", None, 1, True),
    (False, 128, 16, 16, 16, "mul", "layer", 1, False),   # tcgen05 stage T
    (False, 256, 16, 16, 20, "mul", "layer", 2, False),   # tcgen05, k > 16, two k-means iterations
    (False, 64, 8, 8, 8, "both", None, 1, True),
]


@pytest.mark.parametrize("exact,C,H,W,k,integration,norm,iters,i2l", FWD_CASES)
def test_duplex_dropout_forward_vs_oracle(gf, cuda_dev, exact, C, H, W, k, integration, norm, iters, i2l):
    """gf_attn_duplex_fwd_ex with att_dp > 0 == the oracle given the same Philox mask on pass B's probabilities (pass A never dropped);
    the attention map is the probabilities before dropout; a bumped step draws another mask; eval mode == the no-dropout oracle."""
    x64, y64, w, attn, mult, _ = _setup(gf, cuda_dev, C, H, W, k, integration, norm, iters, i2l, exact)
    wd = {n: t.detach() for n, t in w.items()}
    ref, ratt, _ = ob.transformer_layer(x64.detach(), y64.detach(), wd, integration=integration, norm=norm, duplex=True, return_att=True,
                                        kmeans_iters=iters, img2ltnt=i2l, att_mult=mult)
    xg = x64.detach().permute(0, 2, 3, 1).contiguous().float().to(cuda_dev)
    yg = y64.detach().float().to(cuda_dev)
    attn.train()
    with torch.no_grad():
        out, att, _ = attn(xg, yg, return_att=True)
    path = gf._lib.last_path()
    assert path == ("simt_fp32" if exact else "tcgen05_tf32")
    scale = 2.0 * (1.5 if iters > 1 else 1.0)
    check_close(out, ref.permute(0, 2, 3, 1), path, "duplex-dropout/forward", tol_scale=scale)
    assert (att.cpu().double() - ratt).abs().max() <= (1e-4 if exact else 5e-3)         # pre-dropout probabilities
    with torch.no_grad():
        am.advance_dropout(cuda_dev)
        out3, _, _ = attn(xg, yg)
        attn.eval()
        out4, _, _ = attn(xg, yg)
    assert (out3 - out).abs().max() > 1e-3
    ref0, _, _ = ob.transformer_layer(x64.detach(), y64.detach(), wd, integration=integration, norm=norm, duplex=True,
                                      kmeans_iters=iters, img2ltnt=i2l)
    check_close(out4, ref0.permute(0, 2, 3, 1), path, "duplex-dropout/eval", tol_scale=scale)


@pytest.mark.parametrize("i2l", [False, True], ids=["plain", "img2ltnt"])
def test_d_step_route_with_dropout_matches_per_layer(gf, cuda_dev, i2l, monkeypatch):
    """The D step's fakes: a duplex SynthesisNetwork in training mode under no_grad (batched prologue, fused post-op, fused tRGB where
    eligible) gives the same bits as per-layer calls with the same mask, and differs from eval mode (the mask is applied)."""
    G = _small_generator(gf, cuda_dev, False, kmeans=True, att_dp=0.12, g_img2ltnt=i2l).train()
    z = torch.randn(3, 9, 32, generator=torch.Generator().manual_seed(7)).to(cuda_dev)
    with torch.no_grad():
        am.set_dropout_seed(99, cuda_dev, 3)
        a = G(z).clone()
        monkeypatch.setenv("GF_NO_BATCH_PROLOGUE", "1")
        am.set_dropout_seed(99, cuda_dev, 3)
        b = G(z).clone()
        G.eval()
        c = G(z).clone()
    assert torch.isfinite(a).all()
    assert torch.equal(a, b)
    assert (a - c).abs().max() > 1e-3


GRAD_CASES = [  # exact, C, H, W, k, integration, norm, kmeans_iters, img2ltnt, bound (x / y, parameters)
    (True, 64, 8, 16, 4, "both", "layer", 1, False, (1e-4, 2e-4)),
    (True, 96, 10, 13, 20, "mul", "layer", 1, True, (1e-4, 2e-4)),     # KP = 32, ragged n
    (True, 128, 16, 16, 16, "add", None, 1, False, (1e-4, 2e-4)),
    (True, 64, 16, 12, 7, "mul", "layer", 2, True, (1e-4, 2e-4)),      # two k-means iterations
    (False, 128, 16, 16, 16, "mul", "layer", 1, False, (2e-3, 2e-3)),  # fp32 backward of a TF32 forward
    (False, 64, 8, 8, 8, "both", "layer", 1, True, (2e-3, 2e-3)),
]


@pytest.mark.parametrize("exact,C,H,W,k,integration,norm,iters,i2l,bound", GRAD_CASES)
def test_duplex_dropout_gradients_vs_oracle(gf, cuda_dev, monkeypatch, exact, C, H, W, k, integration, norm, iters, i2l, bound):
    """Gradients of x, y and every parameter through stage T (gf_attn_simplex_bwd_ex, same mask) and pass A (recompute + backward
    kernels) against the oracle's autograd with the same mask; the composite is never used; 3 launches per k-means iteration + 1."""
    x64, y64, w, attn, mult, g = _setup(gf, cuda_dev, C, H, W, k, integration, norm, iters, i2l, exact)
    ref, _, _ = ob.transformer_layer(x64, y64, w, integration=integration, norm=norm, duplex=True, kmeans_iters=iters, img2ltnt=i2l,
                                     att_mult=mult)
    gout = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    ref.backward(gout)
    xr = x64.detach().permute(0, 2, 3, 1).contiguous().float().to(cuda_dev).requires_grad_(True)
    yr = y64.detach().float().to(cuda_dev).requires_grad_(True)
    attn.train()
    out, _, _ = attn(xr, yr)
    check_close(out, ref.detach().permute(0, 2, 3, 1), gf._lib.last_path(), "duplex-dropout/train-forward",
                tol_scale=2.0 * (1.5 if iters > 1 else 1.0))

    def no_composite(*a, **kw):
        raise AssertionError("the composite backward ran")
    monkeypatch.setattr(ag, "composite_forward", no_composite)
    l0 = gf._lib.launch_count()
    out.backward(gout.permute(0, 2, 3, 1).contiguous().float().to(cuda_dev))
    torch.cuda.synchronize()
    assert gf._lib.launch_count() - l0 == 3 * iters + 1       # per iteration: pass-A partials + merge + backward; stage-T backward
    rel = lambda a, b: ((a.double().cpu() - b).norm() / b.norm().clamp_min(1e-30)).item()
    bx, bp = bound
    assert rel(xr.grad, x64.grad.permute(0, 2, 3, 1)) < bx
    assert rel(yr.grad, y64.grad) < bx
    for n, prm in attn.named_parameters():
        if w[n].grad is None:                 # wk: duplex keys come from the centroids through wkc
            assert prm.grad is None, n
            continue
        if w[n].grad.norm() < 1e-9:           # bk (constant over the latents), bk2 (constant over the tokens): round-off only
            assert prm.grad.norm().item() < 1e-3, n
            continue
        assert rel(prm.grad, w[n].grad) < bp, (n, rel(prm.grad, w[n].grad))


@pytest.mark.parametrize("B,H,W,C,k", [(1, 256, 256, 128, 16), (2, 10, 13, 96, 20), (3, 8, 8, 512, 5), (2, 16, 16, 256, 32)])
def test_pass_a_entry_points_vs_autograd(gf, cuda_dev, B, H, W, C, k):
    """gf_attn_centroid_recompute / gf_attn_centroid_bwd called directly against fp64 autograd of Xbar = softmax_t(X M^T + Rt2 + Ct2) X:
    one 256 x 256 image (many splits), padded latents, ragged n; dX is accumulated in place; two calls give the same bits."""
    L = gf._lib
    lib = L.load()
    dev = cuda_dev
    n = H * W
    KP = 16 if k <= 16 else 32
    g = torch.Generator(device=dev).manual_seed(B * 1000 + C + k)
    X = torch.randn(B, n, C, generator=g, device=dev)
    M = torch.randn(B, KP, C, generator=g, device=dev) * (2.0 / math.sqrt(C))
    M[:, k:] = 0.0                                # padded latents as in the workspace layout
    Rt2 = torch.randn(B, H, KP, generator=g, device=dev)
    Rt2[:, :, k:] = -math.inf
    Ct2 = torch.randn(B, W, KP, generator=g, device=dev)
    dXbar = torch.randn(B, k, C, generator=g, device=dev)
    desc = L.make_desc(B, H, W, C, k, 16, pos_dim=16, duplex=1)
    ws = torch.empty(L.workspace_bytes(desc), dtype=torch.uint8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def run(dX0):
        Xbar = torch.empty(B, k, C, device=dev)
        lse = torch.empty(B, k, device=dev)
        L.check(lib.gf_attn_centroid_recompute(ctypes.byref(desc), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(), Xbar.data_ptr(),
                                               lse.data_ptr(), ws.data_ptr(), st), "gf_attn_centroid_recompute")
        dX = dX0.clone()
        dSa = torch.empty(B, n, KP, device=dev)
        L.check(lib.gf_attn_centroid_bwd(ctypes.byref(desc), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(), lse.data_ptr(),
                                         Xbar.data_ptr(), dXbar.data_ptr(), dX.data_ptr(), dSa.data_ptr(), st), "gf_attn_centroid_bwd")
        torch.cuda.synchronize()
        return Xbar, lse, dX, dSa

    Xbar, lse, dX, dSa = run(torch.zeros(B, n, C, device=dev))
    Xbar2, lse2, dX2, dSa2 = run(torch.zeros(B, n, C, device=dev))
    assert torch.equal(Xbar, Xbar2) and torch.equal(lse, lse2) and torch.equal(dX, dX2) and torch.equal(dSa, dSa2)

    Xd, Md, Rd, Cd = (t.double().requires_grad_(True) for t in (X, M[:, :k], Rt2[:, :, :k], Ct2[:, :, :k]))
    Sa = Xd @ Md.transpose(1, 2) + (Rd[:, :, None, :] + Cd[:, None, :, :]).reshape(B, n, k)
    Xbar_ref = torch.softmax(Sa, dim=1).transpose(1, 2) @ Xd
    Xbar_ref.backward(dXbar.double())
    rel = lambda a, b: ((a.double() - b).norm() / b.norm().clamp_min(1e-30)).item()
    assert rel(Xbar, Xbar_ref.detach()) < 1e-4
    assert rel(lse, torch.logsumexp(Sa.detach(), dim=1)) < 1e-5
    assert rel(dX, Xd.grad) < 1e-4
    assert torch.all(dSa[:, :, k:] == 0)
    dM = torch.bmm(dSa.transpose(1, 2), X)
    dS4 = dSa.view(B, H, W, KP)
    assert rel(dM[:, :k], Md.grad) < 1e-4
    assert rel(dS4.sum(dim=2)[:, :, :k], Rd.grad) < 1e-4 and rel(dS4.sum(dim=1)[:, :, :k], Cd.grad) < 1e-4
    dX0 = torch.randn(B, n, C, generator=g, device=dev)
    _, _, dX3, _ = run(dX0)
    assert (dX3 - (dX0 + dX)).abs().max() <= 1e-5 * max(1.0, dX0.abs().max().item())


@pytest.mark.parametrize("i2l", [False, True], ids=["plain", "img2ltnt"])
def test_trainer_duplex_with_dropout(gf, cuda_dev, i2l):
    """Trainer.step and Trainer.step_graphed on a 64x64 duplex generator with att_dp = 0.12: finite losses, the pass-A parameters
    move on every replay, the fakes' loss varies across replays."""
    tr = import_module("gansformer-reproducibility-challenge_b200.training")
    torch.manual_seed(0)
    G = gf.Generator(resolution=64, components_num=8, latent_dim=32, fmap_base=2048, fmap_max=128, mapping_layers=4, kmeans=True,
                     g_img2ltnt=i2l, att_dp=0.12).to(cuda_dev)
    D = tr.Discriminator(64, fmap_base=2048, fmap_max=128).to(cuda_dev)
    trainer = tr.Trainer(G, D, tr.TrainConfig(d_reg_interval=2))
    g = torch.Generator().manual_seed(5)
    z = torch.randn(4, 9, 32, generator=g).to(cuda_dev)
    reals = (torch.rand(4, 3, 64, 64, generator=g) * 2 - 1).to(cuda_dev)
    st = trainer.step(z, reals)
    assert math.isfinite(st.loss_g) and math.isfinite(st.loss_d)
    layer = G.synthesis.layers[2].attention
    snap = lambda: torch.cat([getattr(layer, n).detach().reshape(-1) for n in PASS_A_PARAMS]).clone()
    snaps, stats = [snap()], []
    for _ in range(4):
        stats.append(trainer.step_graphed(z, reals))
        snaps.append(snap())
    assert all(math.isfinite(s.loss_g) and math.isfinite(s.loss_d) for s in stats)
    for a, b in zip(snaps, snaps[1:]):
        assert (a - b).abs().max() > 0
    for n in PASS_A_PARAMS:
        assert torch.isfinite(getattr(layer, n)).all(), n
    assert len({round(s.loss_d, 6) for s in stats}) > 1
