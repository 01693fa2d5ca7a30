"""Differentiable wrapper of the fused attention op (needed by the G/D training step, SURVEY row f2).

Forward = the C-ABI CUDA kernels.  Backward of a simplex layer with layer norm (or none): the hand-written stage-T
backward kernel ``gf_attn_simplex_bwd`` (activation gradient + the per-token gradients of logits / control signal), two
batched GEMMs for the reductions over tokens, and torch autograd through the tiny per-image tables of stages W and I
(``folded_tables``).  A duplex layer trained with attention dropout takes the same route for stage T; its pass A (the
centroid softmax over the grid cells) is recomputed and differentiated by ``gf_attn_centroid_recompute`` /
``gf_attn_centroid_bwd`` (``_PassA``), with torch autograd through the [B, k, *] tables around it (``duplex_queries`` /
``duplex_query_tables``).  Everything else (plain duplex layers, instance / batch norm, multi-head layers, CPU tensors):
PyTorch autograd through a recomputation of the direct-form algebra with torch ops (``composite_forward``).
"""
from __future__ import annotations

import math

import torch


def _e(w):
    return w * (1.0 / math.sqrt(w.shape[0]))


def _axis(length, dim, device):
    pos = (torch.arange(length, dtype=torch.float64, device=device) + 0.5) / length * 2.0 - 1.0
    freq = (math.pi / 2.0) * torch.pow(2.0, torch.arange(dim // 2, dtype=torch.float64, device=device))
    ang = pos[:, None] * freq[None, :]
    return torch.cat([torch.sin(ang), torch.cos(ang)], dim=1)            # float64: callers cast to their dtype


def composite_forward(x, y, p, *, integration, norm, duplex, use_pos, centroids=None, kmeans_iters=1, img2ltnt=False, num_heads=1):
    """Same math as the kernels, in torch ops (direct op order), on whatever device x lives on.  x [B,H,W,C]."""
    B, H, W, C = x.shape
    n = H * W
    X = x.reshape(B, n, C)
    s = 1.0 / math.sqrt(C)
    if use_pos:
        pd = p["pos_latent"].shape[1]
        half = pd // 2
        row, col = _axis(H, half, x.device).to(x.dtype), _axis(W, half, x.device).to(x.dtype)
        Pg = torch.cat([row[:, None, :].expand(H, W, half), col[None, :, :].expand(H, W, half)], dim=2).reshape(n, pd)
        Pl = p["pos_latent"]
    cen = None
    if duplex:
        if centroids is not None:
            cen = centroids
        else:
            Qy = y @ _e(p["wq2"]) + p["bq2"]
            Kx = X @ _e(p["wk2"]) + p["bk2"]
            if use_pos:
                Qy = Qy + (Pl @ _e(p["wpq2"]))[None]
                Kx = Kx + (Pg @ _e(p["wpk2"]))[None]
            Vx = X @ _e(p["wv2"]) + p["bv2"]
            for it in range(max(1, kmeans_iters)):
                if it > 0:
                    Qy = cen @ _e(p["wcq"]) + p["bq2"]
                    if use_pos:
                        Qy = Qy + (Pl @ _e(p["wpq2"]))[None]
                A = torch.softmax((Qy @ Kx.transpose(1, 2)) * s, dim=2)
                cen = A @ Vx
        K = cen @ _e(p["wkc"]) + p["bk"]
    else:
        K = y @ _e(p["wk"]) + p["bk"]
    Q = X @ _e(p["wq"]) + p["bq"]
    if use_pos:
        K = K + (Pl @ _e(p["wpk"]))[None]
        Q = Q + (Pg @ _e(p["wpq"]))[None]
    yv = y
    if duplex and img2ltnt:
        ym = y.mean(dim=2, keepdim=True)
        yv = (y - ym) * torch.rsqrt(((y - ym) ** 2).mean(dim=2, keepdim=True) + 1e-8) * (1.0 + cen @ _e(p["wi2l"]) + p["bi2l"])
    V = yv @ _e(p["wv"]) + p["bv"]
    if num_heads == 1:
        P = torch.softmax((Q @ K.transpose(1, 2)) * s, dim=2)
        ctl = (P @ V) @ _e(p["wo"]) + p["bo"]
    else:                                   # heads split the channels; softmax over the latents per head; scale 1/sqrt(C/heads)
        h, kk = num_heads, K.shape[1]
        sp = lambda t, L: t.reshape(B, L, h, C // h).permute(0, 2, 1, 3)
        Ph = torch.softmax((sp(Q, n) @ sp(K, kk).transpose(2, 3)) * (1.0 / math.sqrt(C / h)), dim=3)
        ctl = (Ph @ sp(V, kk)).permute(0, 2, 1, 3).reshape(B, n, C) @ _e(p["wo"]) + p["bo"]
    if norm == "layer":
        mu = X.mean(dim=2, keepdim=True)
        Xn = (X - mu) * torch.rsqrt(((X - mu) ** 2).mean(dim=2, keepdim=True) + 1e-8)
    elif norm in (None, "none"):
        Xn = X
    else:
        dims = (1,) if norm == "instance" else (0, 1)
        mu = X.mean(dim=dims, keepdim=True)
        Xn = (X - mu) * torch.rsqrt(((X - mu) ** 2).mean(dim=dims, keepdim=True) + 1e-8)
    if integration == "mul":
        out = Xn * (1.0 + ctl)
    elif integration == "add":
        out = Xn + ctl
    else:
        out = Xn * (1.0 + ctl[..., :C]) + ctl[..., C:]
    return out.reshape(B, H, W, C), cen


def folded_tables(y, p, *, H, W, C, integration, use_pos, cen=None, img2ltnt=False):
    """Stages W + I in differentiable torch ops: (latents y [B,k,D], raw parameters) -> the per-image tables stage T and its
    backward consume, in the workspace layout: Kp [B,KP,C], Vt [B,Cout,KP], Rt [B,H,KP] (-inf in the padded latents),
    Ct [B,W,KP].  Same algebra as csrc/gf_fold.cu.  Duplex layers: cen [B,k,C] = the centroids, keys from them through wkc;
    img2ltnt: values from the latents modulated by the centroids."""
    B, k, _ = y.shape
    KP = 16 if k <= 16 else 32
    s = 1.0 / math.sqrt(C)
    cols = [_e(p["wq"]).t() * s]
    pd = p["pos_latent"].shape[1] if use_pos else 0
    if use_pos:
        cols.append(_e(p["wpq"]).t() * s)
    cols.append((p["bq"] * s)[:, None])
    qfold = torch.cat(cols, dim=1)                                       # [C, C + pd + 1]
    kconst = p["bk"][None, :].expand(k, C)
    if use_pos:
        kconst = kconst + p["pos_latent"] @ _e(p["wpk"])
    if cen is None:
        kp_all = y @ (_e(p["wk"]) @ qfold) + (kconst @ qfold)[None]      # [B, k, C + pd + 1]
    else:
        kp_all = cen @ (_e(p["wkc"]) @ qfold) + (kconst @ qfold)[None]
    if img2ltnt:
        ym = y.mean(dim=2, keepdim=True)
        y = (y - ym) * torch.rsqrt(((y - ym) ** 2).mean(dim=2, keepdim=True) + 1e-8) * (1.0 + cen @ _e(p["wi2l"]) + p["bi2l"])
    Kp = torch.nn.functional.pad(kp_all[:, :, :C], (0, 0, 0, KP - k))
    kap0 = kp_all[:, :, C + pd]
    if use_pos:
        half = pd // 2
        row, col = _axis(H, half, y.device).to(y.dtype), _axis(W, half, y.device).to(y.dtype)
        rt = torch.einsum("hp,bjp->bhj", row, kp_all[:, :, C:C + half]) + kap0[:, None, :]
        ct = torch.einsum("wp,bjp->bwj", col, kp_all[:, :, C + half:C + pd])
    else:
        rt = kap0[:, None, :].expand(B, H, k)
        ct = torch.zeros(B, W, k, device=y.device, dtype=y.dtype)
    Rt = torch.cat([rt, torch.full((B, H, KP - k), -math.inf, device=y.device, dtype=y.dtype)], dim=2) if KP > k else rt
    Ct = torch.nn.functional.pad(ct, (0, KP - k))
    wo = _e(p["wo"])
    cv = p["bv"] @ wo + p["bo"]
    if integration in ("mul", "both"):
        cv = cv + torch.cat([torch.ones(C, device=y.device, dtype=y.dtype), torch.zeros(cv.numel() - C, device=y.device, dtype=y.dtype)])
    v = y @ (_e(p["wv"]) @ wo) + cv                                      # [B, k, Cout]
    Vt = torch.nn.functional.pad(v.transpose(1, 2), (0, KP - k))
    cb = cv - p["bv"] @ wo                       # bo (+1 on the gain half): the constants attention dropout leaves unscaled
    return Kp.contiguous(), Vt.contiguous(), Rt.contiguous(), Ct.contiguous(), cb.contiguous()


def duplex_queries(src, p, *, first, use_pos):
    """Pass-A queries Qy [B,k,C] of one k-means iteration: from the latents (first iteration) or the previous centroids (wcq)."""
    qy = src @ _e(p["wq2"] if first else p["wcq"]) + p["bq2"]
    if use_pos:
        qy = qy + (p["pos_latent"] @ _e(p["wpq2"]))[None]
    return qy


def duplex_query_tables(qy, p, *, H, W, C, use_pos):
    """Pass-A tables in the workspace layout from the queries: Sa[j,t] = x_t.M[j] + Rt2[h,j] + Ct2[w,j] = Qy_j.Kx_t / sqrt(C),
    Kx = X wk2 + bk2 (+ the grid positional term through wpk2).  M [B,KP,C] (zero rows in the padded latents), Rt2 [B,H,KP]
    (-inf there), Ct2 [B,W,KP].  The bk2 term is constant over the tokens (the forward's fold drops it); it rides in Rt2 so the
    tables reproduce the direct form's scores."""
    B, k, _ = qy.shape
    KP = 16 if k <= 16 else 32
    s = 1.0 / math.sqrt(C)
    M = torch.nn.functional.pad((qy @ _e(p["wk2"]).t()) * s, (0, 0, 0, KP - k))
    kap0 = (qy @ p["bk2"]) * s                                           # [B, k]
    if use_pos:
        half = p["pos_latent"].shape[1] // 2
        qp = (qy @ _e(p["wpk2"]).t()) * s                                # [B, k, pd]
        row, col = _axis(H, half, qy.device).to(qy.dtype), _axis(W, half, qy.device).to(qy.dtype)
        rt = torch.einsum("hp,bjp->bhj", row, qp[:, :, :half]) + kap0[:, None, :]
        ct = torch.einsum("wp,bjp->bwj", col, qp[:, :, half:])
    else:
        rt = kap0[:, None, :].expand(B, H, k)
        ct = torch.zeros(B, W, k, device=qy.device, dtype=qy.dtype)
    Rt2 = torch.cat([rt, torch.full((B, H, KP - k), -math.inf, device=qy.device, dtype=qy.dtype)], dim=2) if KP > k else rt
    Ct2 = torch.nn.functional.pad(ct, (0, KP - k))
    return M.contiguous(), Rt2.contiguous(), Ct2.contiguous()


class _PassA(torch.autograd.Function):
    """Xbar [B,k,C] = softmax over the tokens of (X M^T + Rt2 + Ct2), times X: duplex pass A recomputed in fp32 by
    gf_attn_centroid_recompute.  Backward: gf_attn_centroid_bwd, which adds the activation gradient of pass A into `dx_acc` in
    place (the stage-T gradient, written before autograd reaches this node) instead of returning it; the reductions over the
    tokens are batched GEMMs / sums."""

    @staticmethod
    def forward(ctx, desc, X, dx_acc, M, Rt2, Ct2):
        import ctypes
        from . import _lib
        B, n, C = X.shape
        k = desc.k
        Xbar = torch.empty((B, k, C), dtype=torch.float32, device=X.device)
        lse = torch.empty((B, k), dtype=torch.float32, device=X.device)
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=X.device)
        with torch.cuda.device(X.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
            _lib.check(_lib.load().gf_attn_centroid_recompute(ctypes.byref(desc), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(),
                                                              Xbar.data_ptr(), lse.data_ptr(), ws.data_ptr(), stream), "gf_attn_centroid_recompute")
        ctx.desc, ctx.dx_acc = desc, dx_acc
        ctx.save_for_backward(X, M, Rt2, Ct2, lse, Xbar)
        return Xbar

    @staticmethod
    def backward(ctx, dXbar):
        import ctypes
        from . import _lib
        X, M, Rt2, Ct2, lse, Xbar = ctx.saved_tensors
        d = ctx.desc
        B, n, C = X.shape
        KP = M.shape[1]
        dXbar = dXbar.contiguous()
        dSa = torch.empty((B, n, KP), dtype=torch.float32, device=X.device)
        with torch.cuda.device(X.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
            _lib.check(_lib.load().gf_attn_centroid_bwd(ctypes.byref(d), X.data_ptr(), M.data_ptr(), Rt2.data_ptr(), Ct2.data_ptr(), lse.data_ptr(),
                                                        Xbar.data_ptr(), dXbar.data_ptr(), ctx.dx_acc.data_ptr(), dSa.data_ptr(), stream),
                       "gf_attn_centroid_bwd")
        dM = torch.bmm(dSa.transpose(1, 2), X)                           # [B, KP, C]
        dS4 = dSa.view(B, d.H, d.W, KP)
        return None, None, None, dM, dS4.sum(dim=2), dS4.sum(dim=1)


def _kernel_backward_ok(m, x, dropout=None) -> bool:
    """Simplex layers, and duplex layers trained with attention dropout (plain duplex layers keep the composite)."""
    return ((not m.duplex) or bool(dropout)) and m.norm in ("layer", None, "none") and m.num_heads == 1 and x.is_cuda \
        and x.dtype == torch.float32


class _FusedAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, centroids, return_att, names, x, y, *params):
        from .attention import bipartite_attention_forward
        pd = dict(zip(names, params))
        out, att, cen = bipartite_attention_forward(
            x.detach(), y.detach(), {k: v.detach() for k, v in pd.items()}, module._plan,
            integration=module.integration, norm=module.norm, duplex=module.kmeans_iters if module.duplex else 0, num_heads=module.num_heads,
            use_pos=module.use_pos, return_att=return_att, centroids=centroids, exact_fp32=module.exact_fp32,
            weights_version=tuple((v.data_ptr(), v._version) for v in params), img2ltnt=module.img2ltnt,
            postop=({"act": "linear", "gain": 1.0, **module.dropout_postop(x.device)} if module.dropout_postop(x.device) else None))
        ctx.module, ctx.names, ctx.centroids = module, names, centroids
        ctx.dropout = module.dropout_postop(x.device)                  # the backward regenerates the same mask (same device state)
        ctx.save_for_backward(x, y, *params)
        ctx.mark_non_differentiable(*[t for t in (att, cen) if t is not None])
        return out, att, cen

    @staticmethod
    def backward(ctx, g_out, g_att, g_cen):
        m = ctx.module
        x, y, *params = ctx.saved_tensors
        if _kernel_backward_ok(m, x, ctx.dropout):
            return (None, None, None, None, *_kernel_backward(m, ctx.names, x, y, params, g_out, ctx.dropout, ctx.centroids))
        if ctx.dropout:
            raise NotImplementedError("attention dropout needs the stage-T backward kernel (single-head simplex, layer norm / none)")
        with torch.enable_grad():
            xs = x.detach().requires_grad_(True)
            ys = y.detach().requires_grad_(True)
            ps = [p.detach().requires_grad_(True) for p in params]
            out, _ = composite_forward(xs, ys, dict(zip(ctx.names, ps)), integration=m.integration, norm=m.norm,
                                       duplex=m.duplex, use_pos=m.use_pos, centroids=ctx.centroids, kmeans_iters=m.kmeans_iters,
                                       img2ltnt=m.img2ltnt, num_heads=m.num_heads)
            grads = torch.autograd.grad(out, [xs, ys, *ps], g_out, allow_unused=True)
        return (None, None, None, None, *grads)


def _kernel_backward(m, names, x, y, params, g_out, dropout=None, centroids=None):
    """d(loss)/d(x, y, params) through gf_attn_simplex_bwd (stage T) and, for a duplex layer, _PassA (see the module docstring)."""
    import ctypes
    from . import _lib
    B, H, W, C = x.shape
    n, k = H * W, y.shape[1]
    xc, gc = x.detach().contiguous(), g_out.detach().contiguous()
    dX = torch.empty_like(xc)                    # stage T writes it; pass A's backward adds its part in place
    with torch.enable_grad():
        ys = y.detach().requires_grad_(True)
        ps = [p.detach().requires_grad_(True) for p in params]
        pd = dict(zip(names, ps))
        cen = None
        if m.duplex:
            if centroids is not None:            # given centroids: no pass A to differentiate
                cen = centroids.detach()
            else:
                desc_a = _lib.make_desc(B, H, W, C, k, y.shape[2], heads=1, norm=m.norm, integration=m.integration,
                                        pos_dim=m.pos_dim if m.use_pos else 0, duplex=1, flags=0)
                X = xc.reshape(B, n, C)
                for it in range(m.kmeans_iters):
                    qy = duplex_queries(ys if it == 0 else cen, pd, first=it == 0, use_pos=m.use_pos)
                    M, Rt2, Ct2 = duplex_query_tables(qy, pd, H=H, W=W, C=C, use_pos=m.use_pos)
                    cen = _PassA.apply(desc_a, X, dX, M, Rt2, Ct2) @ _e(pd["wv2"]) + pd["bv2"]
        Kp, Vt, Rt, Ct, cb = folded_tables(ys, pd, H=H, W=W, C=C, integration=m.integration, use_pos=m.use_pos, cen=cen,
                                           img2ltnt=bool(m.duplex and m.img2ltnt))
    KP, Cout = Kp.shape[1], Vt.shape[1]
    dS = torch.empty((B, n, KP), dtype=torch.float32, device=x.device)
    P = torch.empty_like(dS)
    dCtl = torch.empty((B, n, Cout), dtype=torch.float32, device=x.device)
    desc = _lib.make_desc(B, H, W, C, k, y.shape[2], heads=1, norm=m.norm, integration=m.integration,
                          pos_dim=m.pos_dim if m.use_pos else 0, duplex=False, flags=0)
    with torch.cuda.device(x.device):
        dpo = dropout or {}
        _lib.check(_lib.load().gf_attn_simplex_bwd_ex(ctypes.byref(desc), xc.data_ptr(), gc.data_ptr(), Kp.data_ptr(), Vt.data_ptr(),
                                                      Rt.data_ptr(), Ct.data_ptr(), dX.data_ptr(), dS.data_ptr(), P.data_ptr(),
                                                      dCtl.data_ptr(), ctypes.c_float(dpo.get("att_dp", 0.0)), int(dpo.get("dp_salt", 0)),
                                                      dpo["dp_state"].data_ptr() if dpo else None, cb.detach().data_ptr() if dpo else None,
                                                      ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)),
                   "gf_attn_simplex_bwd_ex")
    # reductions over the tokens: plain batched GEMMs / sums
    dKp = torch.bmm(dS.transpose(1, 2), xc.reshape(B, n, C))             # [B, KP, C]
    dVt = torch.bmm(dCtl.transpose(1, 2), P)                             # [B, Cout, KP]
    dS4 = dS.reshape(B, H, W, KP)
    dRt, dCt = dS4.sum(dim=2), dS4.sum(dim=1)
    outs, grads = [Kp, Vt, Rt, Ct], [dKp, dVt, dRt, dCt]
    if dpo:                                      # ctl = sum_j q_j (Vt_j - cb) + cb: the constants' own gradient
        outs.append(cb)
        grads.append((dCtl * (1.0 - P.sum(dim=2, keepdim=True))).sum(dim=(0, 1)))
    gy, *gp = torch.autograd.grad(outs, [ys, *ps], grads, allow_unused=True)
    return (dX, gy, *gp)


def bipartite_attention_autograd(module, x, y, centroids, return_att):
    names = tuple(n for n, _ in module.named_parameters(recurse=False))
    params = tuple(p for _, p in module.named_parameters(recurse=False))
    return _FusedAttention.apply(module, centroids, return_att, names, x, y, *params)
