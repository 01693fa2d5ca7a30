"""Host-side mirror of the reference's attention operator, backed by libgf_attn.so (sm_100a kernels).

Reference interface mirrored (expected ``src/training/network.py`` upstream; the file is NOT in the reference
checkout -- ``/root/reference/.SUBMODULES.json:2`` reports zero payload bytes -- so names/kwargs follow
SURVEY.md section 8a/8b):

    transformer_layer(dim, pos_dim, from_tensor, to_tensor, from_len, to_len, from_pos, to_pos, num_heads,
                      att_dp, integration, norm, kmeans, kmeans_iters, att_vars, iterative, ...)
        -> (from_tensor', att_probs, att_vars)

Here: ``BipartiteAttention(nn.Module)`` owns one layer's parameters and ``transformer_layer(...)`` is the
functional form with the reference's argument names.  Activations are channels-last ``[B, H, W, C]`` fp32 so
the two NCHW<->[B,n,C] transposes of the reference disappear.  PyTorch is used for device memory and streams
only; all arithmetic of the block happens inside the C-ABI calls.  No CPU path exists: a CPU tensor raises.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import torch
from torch import nn

from . import _lib
from ._state import weights_epoch

SIMPLEX_PARAMS = ("wq", "bq", "wpq", "wk", "bk", "wpk", "wv", "bv", "wo", "bo", "pos_latent")
DUPLEX_PARAMS = ("wq2", "bq2", "wpq2", "wk2", "bk2", "wpk2", "wv2", "bv2", "wkc")
KMEANS_PARAMS = ("wcq",)                 # kmeans_iters > 1: centroid -> query projection of the later iterations
IMG2LTNT_PARAMS = ("wi2l", "bi2l")       # g_img2ltnt: centroid -> latent gain


def param_shapes(dim: int, latent_dim: int, components_num: int, pos_dim: int, integration: str, duplex: bool,
                 kmeans_iters: int = 1, img2ltnt: bool = False, iterative: bool = False):
    """Raw parameter shapes, [fan_in, fan_out]; equalised-LR scaling happens inside the library."""
    C, D, k, p = dim, latent_dim, components_num, pos_dim
    cout = 2 * C if integration == "both" else C
    shapes = {"wq": (C, C), "bq": (C,), "wpq": (p, C), "wk": (D, C), "bk": (C,), "wpk": (p, C),
              "wv": (D, C), "bv": (C,), "wo": (C, cout), "bo": (cout,), "pos_latent": (k, p)}
    if duplex:
        shapes.update({"wq2": (D, C), "bq2": (C,), "wpq2": (p, C), "wk2": (C, C), "bk2": (C,), "wpk2": (p, C),
                       "wv2": (C, C), "bv2": (C,), "wkc": (C, C)})
        if kmeans_iters > 1 or iterative:
            shapes["wcq"] = (C, C)
        if img2ltnt:
            shapes.update({"wi2l": (C, D), "bi2l": (D,)})
    return shapes


class StageTimer:
    """Optional CUDA-event timer around the attention launches; bench.py installs one.

    Events are recorded on the stream the kernels are launched on.  Whole call = stages I + T (start-of-call event ->
    end); stage T alone = the dominant kernel."""

    def __init__(self):
        self.records = []            # (stage-T start, end, algorithmic bytes, start of the whole call)
        self.batch_records = []      # (start, end) of batched stage-I launches (prologue_batch)

    def reset(self):
        self.records = []
        self.batch_records = []


STAGE_TIMER: Optional[StageTimer] = None


# ---- attention dropout (att_dp): one device-resident {seed, step} pair per device; the kernels read it when they run, so a
#      replayed CUDA graph draws fresh masks once `advance_dropout` has bumped the step on the device ------------------------------
_DP_STATE: Dict[str, torch.Tensor] = {}
_DP_SALT = [0]


def dropout_state(device) -> torch.Tensor:
    """int64 [2] = {seed, step} on `device` (created with seed 0x5eed1234 on first use; see set_dropout_seed)."""
    key = str(device)
    t = _DP_STATE.get(key)
    if t is None:
        t = _DP_STATE[key] = torch.tensor([0x5EED1234, 0], dtype=torch.int64, device=device)
    return t


def set_dropout_seed(seed: int, device, step: int = 0) -> None:
    dropout_state(device).copy_(torch.tensor([int(seed), int(step)], dtype=torch.int64))


def advance_dropout(device) -> None:
    """step += 1 on the device (stream-ordered, capturable): call between training steps / between the D and G phases."""
    dropout_state(device)[1:].add_(1)


FORCE_REFOLD = False      # set by training.Trainer while it captures a CUDA graph (see networks.CACHE_BYPASS)


class _Plan:
    """Folded weights + workspace for one (shape, config); owns the device buffers the library writes into."""

    def __init__(self):
        self.folded: Optional[torch.Tensor] = None
        self.folded_key = None
        self.ws: Dict[tuple, torch.Tensor] = {}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _check_tensor(t: torch.Tensor, name: str, device) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name}: bipartite attention has no CPU path (tensor is on {t.device})")
    if t.device != device:
        raise RuntimeError(f"{name} is on {t.device}, expected {device}")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


def _make_postop(postop: Optional[dict], B: int, H: int, W: int, C: int, dev):
    """dict -> (GfAttnPostop | None, tensors to keep alive until the launch is enqueued)."""
    if postop is None:
        return None, []
    pst = _lib.GfAttnPostop()
    keep = []
    for fld in ("bias", "noise", "strength"):
        t = postop.get(fld)
        if t is not None:
            t = t.detach()
            _check_tensor(t, "postop." + fld, dev)
            keep.append(t)
            setattr(pst, fld, t.data_ptr())
    nz = postop.get("noise")
    if nz is not None and nz.numel() not in (H * W, B * H * W):
        raise ValueError("postop.noise must have H*W or B*H*W elements")
    if postop.get("bias") is not None and postop["bias"].numel() != C:
        raise ValueError("postop.bias must have C elements")
    pst.noise_bstride = H * W if (nz is not None and nz.numel() == B * H * W and B > 1) else 0
    pst.act = {"linear": 0, "lrelu": 1}[postop.get("act", "lrelu")]
    pst.gain = float(postop.get("gain", 1.0))
    for fld in ("in_scale", "post_scale"):
        t = postop.get(fld)
        if t is None:
            continue
        t = t.detach()
        if t.shape != (B, C) or t.dtype != torch.float32 or t.device != dev:
            raise ValueError(f"postop.{fld} must be a float32 [B, C] tensor on {dev}")
        if not (t.stride(1) == 1 and t.stride(0) % 4 == 0 and t.stride(0) >= C and t.data_ptr() % 16 == 0):
            t = t.contiguous()
        keep.append(t)
        setattr(pst, fld, t.data_ptr())
        setattr(pst, fld + "_ld", t.stride(0))
    if postop.get("rgb_out") is not None:      # fused tRGB: per-sample weights [B,3,C] in, planar image [B,3,H,W] out
        rw, ro, rb = postop.get("rgb_w"), postop["rgb_out"], postop.get("rgb_bias")
        if rw is None or tuple(rw.shape) != (B, 3, C) or tuple(ro.shape) != (B, 3, H, W):
            raise ValueError("postop.rgb_w must be [B, 3, C] and postop.rgb_out [B, 3, H, W]")
        for name, t in (("rgb_w", rw), ("rgb_out", ro)) + ((("rgb_bias", rb),) if rb is not None else ()):
            _check_tensor(t.detach(), "postop." + name, dev)
            keep.append(t)
        pst.rgb_w, pst.rgb_out = rw.data_ptr(), ro.data_ptr()
        pst.rgb_bias = rb.detach().data_ptr() if rb is not None else None
    if postop.get("att_dp", 0.0):                 # attention dropout (training): state = int64 [2] {seed, step} on the device
        st = postop["dp_state"]
        if st.dtype != torch.int64 or st.numel() != 2 or st.device != dev:
            raise ValueError("postop.dp_state must be an int64 [2] tensor on the activation's device")
        keep.append(st)
        pst.att_dp, pst.dp_salt, pst.dp_state = float(postop["att_dp"]), int(postop.get("dp_salt", 0)) & 0xFFFFFFFF, st.data_ptr()
    return pst, keep


def _plan_call(lib, shape, y: torch.Tensor, params: Dict[str, torch.Tensor], plan: _Plan, *, integration, norm, duplex, num_heads,
               use_pos, flags, weights_version=None):
    """Descriptor + folded weights (stage W runs here when a parameter changed) + workspace of one layer call."""
    B, H, W, C = shape
    dev = y.device
    k, D = y.shape[1], y.shape[2]
    pos_dim = params["pos_latent"].shape[1] if use_pos else 0
    desc = _lib.make_desc(B, H, W, C, k, D, heads=num_heads, norm=norm, integration=integration, pos_dim=pos_dim,
                          duplex=duplex, flags=flags)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    names = SIMPLEX_PARAMS + (DUPLEX_PARAMS if duplex else ()) + (KMEANS_PARAMS if (int(duplex) > 1 or flags & _lib.FLAG_CENTROIDS_INIT) else ()) \
        + (IMG2LTNT_PARAMS if (duplex and flags & _lib.FLAG_IMG2LTNT) else ())
    if weights_version is None:
        weights_version = tuple((params[n].data_ptr(), params[n]._version) for n in names)
    fkey = (H, W, k, D, C, pos_dim, integration, int(duplex), num_heads, flags & (_lib.FLAG_IMG2LTNT | _lib.FLAG_CENTROIDS_INIT), str(dev),
            weights_version, weights_epoch())
    if plan.folded is None or plan.folded_key != fkey or FORCE_REFOLD:
        nfl = _lib.folded_floats(desc)
        if plan.folded is None or plan.folded.numel() != nfl or plan.folded.device != dev:
            plan.folded = torch.empty(nfl, dtype=torch.float32, device=dev)
        wstruct = _lib.GfAttnWeights()
        for n in names:
            t = params[n].detach()
            _check_tensor(t, n, dev)
            setattr(wstruct, n, t.data_ptr())
        _lib.check(lib.gf_attn_fold_weights(ctypes.byref(desc), ctypes.byref(wstruct), plan.folded.data_ptr(), stream),
                   "gf_attn_fold_weights")
        plan.folded_key = fkey
    wkey = (B, H, W, C, k, D, pos_dim, integration, norm, int(duplex), num_heads, flags & (_lib.FLAG_IMG2LTNT | _lib.FLAG_CENTROIDS_INIT), str(dev))
    ws = plan.ws.get(wkey)
    if ws is None:
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=dev)
        plan.ws[wkey] = ws
    return desc, ws, stream


def bipartite_attention_forward(x: torch.Tensor, y: torch.Tensor, params: Dict[str, torch.Tensor], plan: _Plan, *,
                                integration: str = "mul", norm: Optional[str] = "layer", duplex: bool = False,
                                num_heads: int = 1, use_pos: bool = True, return_att: bool = False,
                                centroids: Optional[torch.Tensor] = None, exact_fp32: bool = False,
                                out: Optional[torch.Tensor] = None, weights_version=None, postop: Optional[dict] = None,
                                stage: str = "all", x_shape: Optional[Tuple[int, int, int, int]] = None,
                                need_centroids: bool = True, img2ltnt: bool = False, centroids_init: Optional[torch.Tensor] = None):
    """x [B,H,W,C] channels-last fp32 (CUDA), y [B,k,D].  Returns (x', att [B,k,H,W] | None, centroids | None).

    duplex: False / 0 = simplex; True / n >= 1 = duplex with n k-means iterations (kmeans_iters).  img2ltnt: g_img2ltnt.
    centroids: skip pass A and take these as the centroids (GF_FLAG_CENTROIDS_IN).  centroids_init (`iterative`): the previous
    attention layer's centroids [B,k,C]; the first k-means iteration takes its queries from them (GF_FLAG_CENTROIDS_INIT).

    postop (optional): dict(bias [C] | None, noise [H*W] or [B,H*W] | None, strength 0-d tensor | None, act 'lrelu' |
    'linear', gain float, in_scale [B,C] | None, post_scale [B,C] | None, rgb_w [B,3,C] + rgb_out [B,3,H,W] (+ rgb_bias [3]))
    -- the demodulation scale of the preceding convolution (load side) and the noise + fused_bias_act step + next-layer style
    scale (store side), fused into the kernel; with rgb_* also the tRGB 1x1 modulated convolution of the layer output.

    stage: "all" | "prologue" | "token".  "prologue" runs stages W + I for a layer whose activations do not exist yet (x may
    be None, give x_shape; postop needs only in_scale) -- they depend on the latents alone (see ``prologue_batch`` for all
    layers of a network in one launch); "token" then runs the rest on the prepared workspace: stage T for a simplex layer;
    pass A + centroid keys + stage T for a duplex layer (its query tables and V^T are the prepared part)."""
    lib = _lib.load()
    if stage not in ("all", "prologue", "token") or (stage == "prologue" and duplex):
        raise ValueError("stage must be 'all' | 'token', or 'prologue' for a simplex layer (duplex layers: prologue_batch)")
    if x is None:
        if stage != "prologue" or x_shape is None:
            raise ValueError("x may only be omitted (with x_shape) for stage='prologue'")
        B, H, W, C = x_shape
        dev = y.device
    else:
        if x.dim() != 4:
            raise ValueError("x must be [B, H, W, C] (channels-last)")
        dev = x.device
        _check_tensor(x, "x", dev)
        B, H, W, C = x.shape
    _check_tensor(y, "y", dev)
    if y.dim() != 3 or y.shape[0] != B:
        raise ValueError(f"y must be [B, k, D] with B={B}, got {tuple(y.shape)}")
    k = y.shape[1]
    flags = ((_lib.FLAG_FP32_EXACT if exact_fp32 else 0) | (_lib.FLAG_CENTROIDS_IN if (duplex and centroids is not None) else 0)
             | (_lib.FLAG_TABLES_READY if (duplex and stage == "token") else 0)
             | (_lib.FLAG_IMG2LTNT if (duplex and img2ltnt) else 0)
             | (_lib.FLAG_CENTROIDS_INIT if (duplex and centroids_init is not None and centroids is None) else 0))

    with torch.cuda.device(dev):
        desc, ws, stream = _plan_call(lib, (B, H, W, C), y, params, plan, integration=integration, norm=norm, duplex=duplex,
                                      num_heads=num_heads, use_pos=use_pos, flags=flags, weights_version=weights_version)
        if stage != "prologue":
            if out is None:
                out = torch.empty_like(x)
            else:
                _check_tensor(out, "out", dev)
        att = torch.empty((B, H * W, k), dtype=torch.float32, device=dev) if (return_att and stage != "prologue") else None
        pst, keep = _make_postop(postop, B, H, W, C, dev)
        post_ref = ctypes.byref(pst) if pst is not None else None
        timer = STAGE_TIMER
        if timer is not None:
            ev0, ev1, evc = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            evc.record()                                # start of the whole call (stage I + stage T)
        if duplex:
            if timer is not None:
                ev0.record()
            if centroids is None and centroids_init is not None:
                if tuple(centroids_init.shape) != (B, k, C):
                    raise ValueError(f"centroids_init must be [B, k, C] = {(B, k, C)}, got {tuple(centroids_init.shape)}")
                cen = centroids_init.detach().to(torch.float32).clone()        # in/out buffer: carried-in centroids -> this layer's
                _check_tensor(cen, "centroids_init", dev)
            elif centroids is None:
                # need_centroids=False: the keys are built straight from the attention-weighted means (Wv2 / bv2 folded into
                # the key projection), one [B*k, C] x [C, C] product less on the critical path
                cen = torch.empty((B, k, C), dtype=torch.float32, device=dev) if need_centroids else None
            else:
                _check_tensor(centroids, "centroids", dev)
                cen = centroids
            _lib.check(lib.gf_attn_duplex_fwd_ex(ctypes.byref(desc), x.data_ptr(), y.data_ptr(), plan.folded.data_ptr(),
                                                 out.data_ptr(), _ptr(att), _ptr(cen), ws.data_ptr(), post_ref, stream),
                       "gf_attn_duplex_fwd_ex")
        else:
            cen = None
            if stage != "token":
                _lib.check(lib.gf_attn_prologue_ex(ctypes.byref(desc), y.data_ptr(), plan.folded.data_ptr(), ws.data_ptr(), post_ref, stream),
                           "gf_attn_prologue_ex")
            if stage == "prologue":
                return None, None, None
            if timer is not None:
                ev0.record()
            _lib.check(lib.gf_attn_simplex_fwd_ex(ctypes.byref(desc), x.data_ptr(), out.data_ptr(), _ptr(att), ws.data_ptr(),
                                                  post_ref, stream),
                       "gf_attn_simplex_fwd_ex")
        if timer is not None:
            ev1.record()
            timer.records.append((ev0, ev1, 2 * 4 * B * H * W * C, evc))
        del keep
    att_map = att.view(B, H, W, k).permute(0, 3, 1, 2) if att is not None else None   # [B,k,H,W] view
    return out, att_map, cen


def tc_eligible(module: "BipartiteAttention", shape, k: int) -> bool:
    """Will stage T of this layer call run on the tcgen05 kernel (gf_attn_tc_eligible)?  Decides fusions only that kernel serves."""
    B, H, W, C = shape
    desc = _lib.make_desc(B, H, W, C, k, module.latent_dim, heads=module.num_heads, norm=module.norm, integration=module.integration,
                          pos_dim=module.pos_dim if module.use_pos else 0, duplex=module.kmeans_iters if module.duplex else 0,
                          flags=_lib.FLAG_FP32_EXACT if module.exact_fp32 else 0)
    rc = _lib.load().gf_attn_tc_eligible(ctypes.byref(desc))
    if rc < 0:
        _lib.check(rc, "gf_attn_tc_eligible")
    return rc == 1


@torch.no_grad()
def prologue_batch(items) -> None:
    """Stage I of several layers in ONE launch (``gf_attn_prologue_batch``).  items: iterable of
    (module: BipartiteAttention, y [B,k,D], x_shape (B,H,W,C), in_scale [B,C] | None).  Afterwards call each module with
    ``stage="token"`` (same y, same in_scale).  Stage W (weight folding) of a layer runs first if its parameters changed."""
    lib = _lib.load()
    items = list(items)
    if not items:
        return
    dev = items[0][1].device
    n = len(items)
    descs, keep = [], []
    arr_d = (ctypes.c_void_p * n)()
    arr_y = (ctypes.c_void_p * n)()
    arr_f = (ctypes.c_void_p * n)()
    arr_w = (ctypes.c_void_p * n)()
    arr_p = (ctypes.c_void_p * n)()
    timer = STAGE_TIMER
    with torch.cuda.device(dev):
        if timer is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream = None
        for i, (m, y, shape, in_scale) in enumerate(items):
            _check_tensor(y, "y", dev)
            flags = (_lib.FLAG_FP32_EXACT if m.exact_fp32 else 0) | (_lib.FLAG_IMG2LTNT if (m.duplex and m.img2ltnt) else 0)
            desc, ws, stream = _plan_call(lib, tuple(shape), y, m.param_dict(), m._plan, integration=m.integration, norm=m.norm,
                                          duplex=m.kmeans_iters if m.duplex else 0, num_heads=m.num_heads, use_pos=m.use_pos, flags=flags)
            pst, kp = _make_postop(dict(in_scale=in_scale) if in_scale is not None else None, shape[0], shape[1], shape[2], shape[3], dev)
            descs.append(desc)
            keep.extend(kp)
            keep.append(pst)
            arr_d[i] = ctypes.addressof(desc)
            arr_y[i] = y.data_ptr()
            arr_f[i] = m._plan.folded.data_ptr()
            arr_w[i] = ws.data_ptr()
            arr_p[i] = ctypes.addressof(pst) if pst is not None else None
        if timer is not None:
            e0.record()
        _lib.check(lib.gf_attn_prologue_batch(n, arr_d, arr_y, arr_f, arr_w, arr_p, stream), "gf_attn_prologue_batch")
        if timer is not None:
            e1.record()
            timer.batch_records.append((e0, e1))
    del keep, descs


class BipartiteAttention(nn.Module):
    """One bipartite attention layer (simplex, or duplex when ``kmeans=True``) + region-wise modulation.

    kwargs follow the reference's names: ``dim`` (C), ``pos_dim``, ``num_heads``, ``integration`` ('mul' |
    'add' | 'both'), ``norm`` ('layer' | 'instance' | 'batch' | None), ``kmeans`` (duplex), ``kmeans_iters`` (1).
    """

    def __init__(self, dim: int, latent_dim: int, components_num: int, pos_dim: Optional[int] = None,
                 num_heads: int = 1, integration: str = "mul", norm: Optional[str] = "layer", kmeans: bool = False,
                 kmeans_iters: int = 1, use_pos: bool = True, att_dp: float = 0.0, exact_fp32: bool = False, img2ltnt: bool = False,
                 iterative: bool = False):
        super().__init__()
        if kmeans_iters < 1 or kmeans_iters > 16:
            raise ValueError("kmeans_iters must be in 1..16")
        if (kmeans_iters != 1 or img2ltnt) and not kmeans:
            raise ValueError("kmeans_iters > 1 / img2ltnt need kmeans=True (duplex attention)")
        if not 0.0 <= att_dp < 1.0:
            raise ValueError("att_dp must be in [0, 1)")
        self.dim, self.latent_dim, self.components_num = dim, latent_dim, components_num
        self.pos_dim = latent_dim if pos_dim is None else pos_dim
        self.num_heads, self.integration, self.norm = num_heads, integration, norm
        self.duplex, self.use_pos, self.exact_fp32 = bool(kmeans), use_pos, exact_fp32
        self.kmeans_iters, self.img2ltnt, self.iterative = int(kmeans_iters), bool(img2ltnt), bool(iterative and kmeans)
        self.att_dp = float(att_dp)                       # attention dropout, active in training mode only (reference: p ~ 0.12);
        # duplex layers drop pass B's probabilities (over the latents) only, never pass A's softmax over the grid cells
        _DP_SALT[0] += 1
        self.dp_salt = _DP_SALT[0] * 0x9E3779B1 & 0xFFFFFFFF   # distinct masks per layer
        for name, shape in param_shapes(dim, latent_dim, components_num, self.pos_dim, integration, self.duplex, self.kmeans_iters, self.img2ltnt,
                                        self.iterative).items():
            init = torch.zeros(shape) if name.startswith("b") else torch.randn(shape)
            self.register_parameter(name, nn.Parameter(init))
        self._plan = _Plan()

    def param_dict(self) -> Dict[str, torch.Tensor]:
        return {n: p for n, p in self.named_parameters(recurse=False)}

    def dropout_postop(self, device) -> dict:
        """Post-op members that switch attention dropout on for this call ({} in eval mode / att_dp = 0)."""
        if not (self.training and self.att_dp > 0.0):
            return {}
        return dict(att_dp=self.att_dp, dp_salt=self.dp_salt, dp_state=dropout_state(device))

    def forward(self, x: torch.Tensor, y: torch.Tensor, centroids: Optional[torch.Tensor] = None,
                return_att: bool = False, out: Optional[torch.Tensor] = None, postop: Optional[dict] = None,
                stage: str = "all", need_centroids: bool = True, centroids_init: Optional[torch.Tensor] = None):
        """x [B,H,W,C] channels-last, y [B,k,D] -> (x', att [B,k,H,W] | None, centroids [B,k,C] | None).
        stage="token": the latent-only tables were already built by ``prepare`` / ``prologue_batch`` (same y, same in_scale)."""
        if torch.is_grad_enabled() and (x.requires_grad or y.requires_grad or any(p.requires_grad for p in self.parameters())):
            if postop is not None:
                raise RuntimeError("the fused post-op is inference-only; apply noise/bias/activation outside when training")
            if self.att_dp > 0.0 and self.training:
                if self.num_heads != 1:
                    raise NotImplementedError("attention dropout needs a single-head layer: the multi-head backward (torch composite) "
                                              "cannot apply the dropout mask")
                if self.duplex and self.norm not in ("layer", None, "none"):
                    raise NotImplementedError("attention dropout on a duplex layer needs norm 'layer' or None: there is no backward "
                                              "kernel for instance / batch norm")
            if centroids_init is not None:
                raise RuntimeError("iterative centroid carry (centroids_init) is an inference feature in this build")
            from .autograd import bipartite_attention_autograd
            return bipartite_attention_autograd(self, x, y, centroids, return_att)
        dp = self.dropout_postop(x.device)
        if dp:
            if self.num_heads != 1:
                raise NotImplementedError("attention dropout needs a single-head layer (one mask column per latent)")
            postop = {**(postop or {"act": "linear", "gain": 1.0}), **dp}
        return bipartite_attention_forward(x, y, self.param_dict(), self._plan, integration=self.integration,
                                           norm=self.norm, duplex=self.kmeans_iters if self.duplex else 0, num_heads=self.num_heads,
                                           use_pos=self.use_pos, return_att=return_att, centroids=centroids,
                                           exact_fp32=self.exact_fp32, out=out, postop=postop, stage=stage,
                                           need_centroids=need_centroids, img2ltnt=self.img2ltnt,
                                           centroids_init=centroids_init if self.iterative else None)

    @torch.no_grad()
    def prepare(self, y: torch.Tensor, x_shape: Tuple[int, int, int, int], in_scale: Optional[torch.Tensor] = None):
        """Stages W + I of a simplex layer (weights fold + per-image K', V^T, positional tables): they depend on the latents
        (and the demodulation scale folded into K') only, so the generator runs them for every layer up front on a side stream."""
        post = dict(in_scale=in_scale) if in_scale is not None else None
        bipartite_attention_forward(None, y, self.param_dict(), self._plan, integration=self.integration, norm=self.norm,
                                    duplex=self.kmeans_iters if self.duplex else 0, num_heads=self.num_heads, use_pos=self.use_pos,
                                    exact_fp32=self.exact_fp32, postop=post, stage="prologue", x_shape=x_shape)


_FUNCTIONAL_PLANS: Dict[int, _Plan] = {}


def transformer_layer(dim: int, pos_dim: int, from_tensor: torch.Tensor, to_tensor: torch.Tensor, from_len: int,
                      to_len: int, params: Dict[str, torch.Tensor], *, grid_shape: Tuple[int, int],
                      num_heads: int = 1, att_dp: float = 0.0, integration: str = "mul", norm: Optional[str] = "layer",
                      kmeans: bool = False, kmeans_iters: int = 1, att_vars: Optional[dict] = None,
                      iterative: bool = False, use_pos: bool = True, exact_fp32: bool = False):
    """Functional form with the reference's argument names (see module docstring).

    from_tensor [B, from_len, dim] (grid tokens, row-major over grid_shape=(H, W)); to_tensor [B, to_len, D].
    Returns (from_tensor' [B, from_len, dim], att_probs [B, from_len, to_len], att_vars).
    """
    H, W = grid_shape
    B = from_tensor.shape[0]
    if from_len != H * W or from_tensor.shape[1] != from_len or from_tensor.shape[2] != dim or to_tensor.shape[1] != to_len:
        raise ValueError("from_len/to_len/dim do not match the tensors")
    if use_pos and params["pos_latent"].shape[1] != pos_dim:
        raise ValueError("pos_dim does not match params['pos_latent']")
    plan = _FUNCTIONAL_PLANS.setdefault(id(params), _Plan())
    att_vars = dict(att_vars or {})
    cen_in = att_vars.get("centroids") if (kmeans and iterative) else None
    x = from_tensor.reshape(B, H, W, dim)
    post = None
    if att_dp:          # training-time dropout of the probabilities: att_vars may carry "dp_salt"; the {seed, step} state is the device's
        post = dict(act="linear", gain=1.0, att_dp=float(att_dp), dp_salt=int(att_vars.get("dp_salt", 0)), dp_state=dropout_state(x.device))
    out, att, cen = bipartite_attention_forward(x, to_tensor, params, plan, integration=integration, norm=norm,
                                                duplex=(kmeans_iters if kmeans else 0), num_heads=num_heads, use_pos=use_pos,
                                                return_att=True, centroids=cen_in, exact_fp32=exact_fp32,
                                                img2ltnt=bool(kmeans and "wi2l" in params), postop=post)
    if cen is not None:
        att_vars["centroids"] = cen
    att_probs = att.permute(0, 2, 3, 1).reshape(B, from_len, to_len)
    return out.reshape(B, from_len, dim), att_probs, att_vars
