"""CPU tests of the duplex training route: the folded algebra of the pass-A backward (what gf_attn_centroid_bwd computes) against
torch autograd in float64, the torch builder of the pass-A tables against the direct form's scores, argument validation of the two
pass-A entry points, and the refusals that remain for attention dropout.  No kernel is launched here."""
import ctypes
import math
from importlib import import_module

import pytest
import torch

from oracle import bipartite as ob

ag = import_module("gansformer-reproducibility-challenge_b200.autograd")


def centroid_backward_folded(X, M, Rt2, Ct2, dXbar, k, H, W):
    """Pass-A backward in the kernel's form.  X [B,n,C], M [B,KP,C], Rt2 [B,H,KP], Ct2 [B,W,KP], dXbar [B,k,C].
    Returns Xbar, lse, dX (pass A's part), dSa [B,n,KP], dM, dRt2, dCt2; the padded latents j >= k contribute exactly 0."""
    B, n, C = X.shape
    KP = M.shape[1]
    Sa = (X @ M[:, :k].transpose(1, 2) + (Rt2[:, :, None, :k] + Ct2[:, None, :, :k]).reshape(B, n, k))     # [B,n,k]
    lse = torch.logsumexp(Sa, dim=1)                                                 # [B,k]
    A = torch.exp(Sa - lse[:, None, :])
    Xbar = A.transpose(1, 2) @ X                                                     # [B,k,C]
    dA = X @ dXbar.transpose(1, 2)                                                   # x_t . dXbar_j
    r = (Xbar * dXbar).sum(dim=2)                                                    # per image, not per token
    dSa = torch.zeros(B, n, KP, dtype=X.dtype)
    dSa[:, :, :k] = A * (dA - r[:, None, :])
    dX = dSa[:, :, :k] @ M[:, :k] + A @ dXbar
    dM = dSa.transpose(1, 2) @ X
    dS4 = dSa.reshape(B, H, W, KP)
    return Xbar, lse, dX, dSa, dM, dS4.sum(dim=2), dS4.sum(dim=1)


@pytest.mark.parametrize("B,H,W,C,k", [(2, 5, 7, 32, 5), (1, 9, 4, 64, 20), (3, 3, 3, 96, 16)])
def test_pass_a_backward_algebra_matches_autograd(B, H, W, C, k):
    """dX, dM, dRt2, dCt2 of the folded formulas == torch.autograd of Xbar = softmax_t(X M^T + Rt2 + Ct2) X (float64), with padded
    latents (k < KP) and ragged grids."""
    g = torch.Generator().manual_seed(B * 100 + C + k)
    KP = 16 if k <= 16 else 32
    n = H * W
    X = torch.randn(B, n, C, generator=g, dtype=torch.float64)
    M = torch.randn(B, KP, C, generator=g, dtype=torch.float64) * 0.3
    M[:, k:] = 0.0
    Rt2 = torch.randn(B, H, KP, generator=g, dtype=torch.float64)
    Rt2[:, :, k:] = -math.inf
    Ct2 = torch.randn(B, W, KP, generator=g, dtype=torch.float64)
    Ct2[:, :, k:] = 0.0
    dXbar = torch.randn(B, k, C, generator=g, dtype=torch.float64)

    Xa, Ma, Ra, Ca = (t.clone().requires_grad_(True) for t in (X, M, Rt2, Ct2))
    Sa = Xa @ Ma[:, :k].transpose(1, 2) + (Ra[:, :, None, :k] + Ca[:, None, :, :k]).reshape(B, n, k)
    Xbar_ref = torch.softmax(Sa, dim=1).transpose(1, 2) @ Xa
    Xbar_ref.backward(dXbar)

    Xbar, lse, dX, dSa, dM, dRt2, dCt2 = centroid_backward_folded(X, M, Rt2, Ct2, dXbar, k, H, W)
    torch.testing.assert_close(Xbar, Xbar_ref.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(lse, torch.logsumexp(Sa.detach(), dim=1), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(dX, Xa.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(dM, Ma.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(dRt2[:, :, :k], Ra.grad[:, :, :k], rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(dCt2, Ca.grad, rtol=1e-10, atol=1e-12)
    assert torch.all(dSa[:, :, k:] == 0) and torch.all(dM[:, k:] == 0)
    # the softmax over the tokens is shift-invariant per latent: its logit gradient sums to zero over the tokens
    assert dSa.sum(dim=1).abs().max() < 1e-10


@pytest.mark.parametrize("use_pos", [True, False])
def test_pass_a_table_builder_reproduces_the_direct_scores(use_pos):
    """duplex_queries + duplex_query_tables (the differentiable builder of the backward) give x_t.M_j + Rt2 + Ct2 == Qy Kx^T / sqrt(C)
    of oracle/bipartite.py in float64, for the first k-means iteration (queries from the latents) and the second (from the centroids)."""
    B, C, H, W, k, D, p = 2, 64, 6, 5, 7, 16, 16
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    y = torch.randn(B, k, D, generator=g, dtype=torch.float64)
    w = ob.init_params(C, D, k, p, "mul", True, seed=3, bias_std=0.3, extras=True)
    X = x.reshape(B, C, H * W).permute(0, 2, 1)
    Kx = ob._dense(X, w["wk2"], w["bk2"])
    Pl = w["pos_latent"]
    if use_pos:
        Kx = Kx + ob._dense(ob.grid_pos_table(H, W, p, torch.float64), w["wpk2"])[None]
    _, _, cen1 = ob.transformer_layer(x, y, w, duplex=True, use_pos=use_pos)           # centroids of iteration 1
    for it, src in ((0, y), (1, cen1)):
        Qy = ob._dense(src, w["wq2"] if it == 0 else w["wcq"], w["bq2"])
        if use_pos:
            Qy = Qy + ob._dense(Pl, w["wpq2"])[None]
        want = Qy @ Kx.transpose(1, 2) / math.sqrt(C)                                 # [B,k,n]
        qy = ag.duplex_queries(src, w, first=it == 0, use_pos=use_pos)
        M, Rt2, Ct2 = ag.duplex_query_tables(qy, w, H=H, W=W, C=C, use_pos=use_pos)
        assert M.shape == (B, 16, C) and Rt2.shape == (B, H, 16) and Ct2.shape == (B, W, 16)
        got = X @ M[:, :k].transpose(1, 2) + (Rt2[:, :, None, :k] + Ct2[:, None, :, :k]).reshape(B, H * W, k)
        torch.testing.assert_close(got.transpose(1, 2), want, rtol=1e-12, atol=1e-12)
        assert torch.all(M[:, k:] == 0) and torch.all(Rt2[:, :, k:] == -math.inf) and torch.all(Ct2[:, :, k:] == 0)
    # the kmeans_iters = 2 oracle layer takes exactly these second-iteration scores
    _, _, cen2 = ob.transformer_layer(x, y, w, duplex=True, use_pos=use_pos, kmeans_iters=2)
    A2 = torch.softmax(got.transpose(1, 2), dim=2)
    torch.testing.assert_close(A2 @ ob._dense(X, w["wv2"], w["bv2"]), cen2, rtol=1e-10, atol=1e-12)


def test_pass_a_entry_points_validate_before_touching_the_device(gf):
    """gf_attn_centroid_recompute / gf_attn_centroid_bwd: argument errors come back as gf_status + message (no GPU needed)."""
    L = gf._lib
    lib = L.load()
    err = lambda: lib.gf_last_error().decode()
    dup = L.make_desc(2, 8, 8, 64, 5, 16, pos_dim=16, duplex=1)
    simplex = L.make_desc(2, 8, 8, 64, 5, 16, pos_dim=16, duplex=0)
    bad_c = L.make_desc(2, 8, 8, 48, 5, 16, pos_dim=16, duplex=1)
    rec, bwd = lib.gf_attn_centroid_recompute, lib.gf_attn_centroid_bwd
    assert rec(None, 1, 1, 1, 1, 1, 1, 1, None) == -1 and "null descriptor" in err()
    assert rec(ctypes.byref(simplex), 1, 1, 1, 1, 1, 1, 1, None) == -1 and "desc.duplex is 0" in err()
    assert rec(ctypes.byref(bad_c), 1, 1, 1, 1, 1, 1, 1, None) == -2 and "C % 32 == 0" in err()
    assert rec(ctypes.byref(dup), 1, 1, 1, 1, None, 1, 1, None) == -1 and "gf_attn_centroid_recompute: null pointer" in err()
    assert bwd(None, 1, 1, 1, 1, 1, 1, 1, 1, 1, None) == -1 and "null descriptor" in err()
    assert bwd(ctypes.byref(simplex), 1, 1, 1, 1, 1, 1, 1, 1, 1, None) == -1 and "desc.duplex is 0" in err()
    assert bwd(ctypes.byref(dup), 1, 1, 1, 1, 1, 1, 1, None, 1, None) == -1 and "gf_attn_centroid_bwd: null pointer" in err()
    huge_b = L.make_desc(70000, 1, 1, 64, 5, 16, duplex=1)
    assert bwd(ctypes.byref(huge_b), 1, 1, 1, 1, 1, 1, 1, 1, 1, None) == -2 and "B > 65535" in err()


def _layer(gf, **kw):
    return gf.BipartiteAttention(64, 16, 5, pos_dim=16, att_dp=0.12, **kw).train()


def test_remaining_dropout_refusals(gf):
    """What attention dropout still refuses, with a message naming what is missing: multi-head layers (training and the no-grad
    training forward), duplex layers with instance / batch norm under autograd, and the `iterative` centroid carry under autograd."""
    x = torch.randn(2, 8, 8, 64, requires_grad=True)
    y = torch.randn(2, 5, 16)
    with pytest.raises(NotImplementedError, match="single-head"):
        _layer(gf, num_heads=2)(x, y)
    with torch.no_grad(), pytest.raises(NotImplementedError, match="single-head"):
        _layer(gf, num_heads=2)(x, y)
    for norm in ("instance", "batch"):
        with pytest.raises(NotImplementedError, match="instance / batch norm"):
            _layer(gf, kmeans=True, norm=norm)(x, y)
    with pytest.raises(RuntimeError, match="inference feature"):
        _layer(gf, kmeans=True, iterative=True)(x, y, centroids_init=torch.zeros(2, 5, 64))
