"""Host wrappers of the memory-bound companion ops (include/gf_ops.h): the B200-native equivalents of the
reference's native ops ``dnnlib/tflib/ops/upfirdn_2d.cu`` and ``fused_bias_act.cu`` (expected upstream; not in the
checkout) in the forms the generator uses, plus channel scaling (style modulation / demodulation).

Inference on CUDA fp32 tensors goes through libgf_attn.so.  The plain-torch forms below are the *definition* of each
op (and serve autograd / float64 / CPU plumbing tests of the surrounding host code -- none of this is the attention
hot path, which has no CPU form at all).
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional

import torch
import torch.nn.functional as F

from . import _lib

SQRT2 = math.sqrt(2.0)


def _use_cuda(*tensors) -> bool:
    ts = [t for t in tensors if t is not None]
    if not all(t.is_cuda and t.dtype == torch.float32 for t in ts):
        return False
    return not (torch.is_grad_enabled() and any(t.requires_grad for t in ts))


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def fir_filter(device=None, dtype=torch.float32) -> torch.Tensor:
    f = torch.tensor([1.0, 3.0, 3.0, 1.0], dtype=torch.float64)
    f = torch.outer(f, f)
    return (f / f.sum()).to(device=device, dtype=dtype)


def upfirdn2d_ref(x: torch.Tensor, f: torch.Tensor, up: int = 1, pad=(0, 0, 0, 0), gain: float = 1.0) -> torch.Tensor:
    """Definition: zero-insert upsample by `up`, pad (x0, x1, y0, y1), correlate with the symmetric FIR filter `f`."""
    B, C, H, W = x.shape
    if up > 1:
        x = x.reshape(B, C, H, 1, W, 1)
        x = F.pad(x, [0, up - 1, 0, 0, 0, up - 1])
        x = x.reshape(B, C, H * up, W * up)
    x = F.pad(x, [pad[0], pad[1], pad[2], pad[3]])
    w = (f * gain).to(x.dtype)[None, None].expand(C, 1, *f.shape)
    return F.conv2d(x, w, groups=C)


def _nhwc_view(x: torch.Tensor) -> torch.Tensor:
    """NCHW-shaped tensor -> contiguous [B,H,W,C] view (free when x is channels_last)."""
    v = x.permute(0, 2, 3, 1)
    return v if v.is_contiguous() else v.contiguous()


def _rows(s: torch.Tensor):
    """(tensor, row stride in floats) of a [B, C] matrix that may be a column slice of a wider contiguous matrix."""
    if s.dim() == 2 and s.stride(1) == 1 and s.stride(0) % 4 == 0 and s.data_ptr() % 16 == 0 and s.stride(0) >= s.shape[1]:
        return s, s.stride(0)
    s = s.contiguous()
    return s, s.shape[1]


def chan_scale(x: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
    """x [B,C,H,W] * s [B,C] (style modulation / demodulation as activation scaling)."""
    if _use_cuda(x, s) and x.shape[1] % 4 == 0:
        xv = _nhwc_view(x)
        B, H, W, C = xv.shape
        y = torch.empty_like(xv)
        sr, ld = _rows(s)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_chan_scale_nhwc(xv.data_ptr(), sr.data_ptr(), ld, y.data_ptr(), B, H * W, C,
                                                      _stream(x.device)), "gf_chan_scale_nhwc")
        return y.permute(0, 3, 1, 2)
    return x * s[:, :, None, None].to(x.dtype)


class _Fir4(torch.autograd.Function):
    """Native [1,3,3,1]^2/64 FIR with symmetric padding (gf_fir4_nhwc), differentiable to any order: the filter is symmetric,
    so the gradient of a pad-p blur is the pad-(3-p) blur of the incoming gradient -- the same op again."""

    @staticmethod
    def forward(ctx, x, pad, gain):
        ctx.pad, ctx.gain = pad, gain
        xv = _nhwc_view(x.detach())
        B, H, W, C = xv.shape
        y = torch.empty((B, H + 2 * pad - 3, W + 2 * pad - 3, C), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_fir4_nhwc(xv.data_ptr(), y.data_ptr(), B, H, W, C, pad, ctypes.c_float(gain), _stream(x.device)),
                       "gf_fir4_nhwc")
        return y.permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, gy):
        return _Fir4.apply(gy, 3 - ctx.pad, ctx.gain), None, None


def fir4(x: torch.Tensor, f: torch.Tensor, pad: int, gain: float = 1.0) -> torch.Tensor:
    """Stride-1 FIR blur with the [1,3,3,1] filter and symmetric padding `pad`: x [B,C,H,W] -> [B,C,H+2p-3,W+2p-3].
    CUDA fp32 tensors use the native kernel in both directions (autograd included); anything else the torch definition."""
    if x.is_cuda and x.dtype == torch.float32 and x.shape[1] % 4 == 0 and 0 <= pad <= 3 and min(x.shape[2:]) + 2 * pad > 3:
        return _Fir4.apply(x, int(pad), float(gain))
    return upfirdn2d_ref(x, f.to(x.dtype), pad=(pad, pad, pad, pad), gain=gain)


def blur_up(x: torch.Tensor, f: torch.Tensor, scale: Optional[torch.Tensor] = None, gain: float = 4.0) -> torch.Tensor:
    """FIR blur after a stride-2 transposed conv: x [B,C,2H+1,2W+1] -> [B,C,2H,2W] (pad 1), optional * scale [B,C]."""
    if _use_cuda(x, scale) and x.shape[1] % 4 == 0:
        xv = _nhwc_view(x)
        B, Hin, Win, C = xv.shape
        y = torch.empty((B, Hin - 1, Win - 1, C), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_blur_up_nhwc(xv.data_ptr(), y.data_ptr(), None if scale is None else scale.contiguous().data_ptr(),
                                                   B, Hin - 1, Win - 1, C, float(gain), _stream(x.device)), "gf_blur_up_nhwc")
        return y.permute(0, 3, 1, 2)
    y = fir4(x, f, 1, gain=gain)                                        # training: native FIR both ways, scale in torch
    return y if scale is None else y * scale[:, :, None, None].to(y.dtype)


def upconv_phase_weights(w: torch.Tensor):
    """w [O,I,3,3] (already equalised-LR scaled) -> the four (kernel, padding) pairs whose stride-1 convolutions of the
    low-resolution input give the polyphase components T[2i+a, 2j+b] of conv_transpose2d(x, w^T, stride=2)."""
    out = []
    for a in (0, 1):
        for b in (0, 1):
            wy = w[:, :, 0::2].flip(2) if a == 0 else w[:, :, 1:2]        # taps (2, 0) / (1,) -- slices, no host index tensors
            wk = wy[:, :, :, 0::2].flip(3) if b == 0 else wy[:, :, :, 1:2]   # (capturable in a CUDA graph)
            out.append((wk.contiguous(memory_format=torch.channels_last), (1 - a, 1 - b)))
    return out


def upconv_blur_phases(x: torch.Tensor, phases, scale: Optional[torch.Tensor] = None, gain: float = 4.0) -> torch.Tensor:
    """Stride-2 transposed 3x3 convolution + FIR blur (+ demodulation scale) of the upsampling layers, inference on CUDA:
    four stride-1 convolutions (cuDNN fprop) feeding the polyphase blur kernel.  x [B,I,H,W] -> [B,O,2H,2W]."""
    ps = [_nhwc_view(F.conv2d(x, wk, padding=pad)) for wk, pad in phases]
    B, H, W, C = ps[3].shape
    y = torch.empty((B, 2 * H, 2 * W, C), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().gf_blur_up_phases_nhwc(ps[0].data_ptr(), ps[1].data_ptr(), ps[2].data_ptr(), ps[3].data_ptr(), y.data_ptr(),
                                                      None if scale is None else scale.contiguous().data_ptr(), B, 2 * H, 2 * W, C,
                                                      float(gain), _stream(x.device)), "gf_blur_up_phases_nhwc")
    return y.permute(0, 3, 1, 2)


def upsample2x(x: torch.Tensor, f: torch.Tensor, add: Optional[torch.Tensor] = None) -> torch.Tensor:
    """2x FIR upsampling of an NCHW image (tRGB skip connection), optionally + add."""
    if _use_cuda(x, add):
        xc = x.contiguous()
        B, C, H, W = xc.shape
        y = torch.empty((B, C, 2 * H, 2 * W), dtype=torch.float32, device=x.device)
        ac = None if add is None else add.contiguous()
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_upsample2x_nchw(xc.data_ptr(), None if ac is None else ac.data_ptr(), y.data_ptr(), B, C, H, W,
                                                      _stream(x.device)), "gf_upsample2x_nchw")
        return y
    y = upfirdn2d_ref(x, f, up=2, pad=(2, 1, 2, 1), gain=4.0)
    return y if add is None else y + add


def _bias_act_native(x, bias, act, noise, strength, gain):
    xv = _nhwc_view(x)
    B, H, W, C = xv.shape
    y = torch.empty_like(xv)
    nz = None if noise is None else noise.contiguous()
    bstride = H * W if (nz is not None and nz.numel() == B * H * W and B > 1) else 0
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().gf_bias_act_nhwc(xv.data_ptr(), y.data_ptr(), None if bias is None else bias.contiguous().data_ptr(),
                                                None if nz is None else nz.data_ptr(),
                                                None if strength is None else strength.data_ptr(), bstride, B, H * W, C,
                                                1 if act == "lrelu" else 0, float(gain), _stream(x.device)), "gf_bias_act_nhwc")
    return y.permute(0, 3, 1, 2)


class _BiasAct(torch.autograd.Function):
    """Training form of bias_act on CUDA: native forward; backward = one masked scaling of the incoming gradient (the sign of
    the pre-activation is the sign of the output) plus the bias / noise-strength reductions -- instead of autograd through
    five separate elementwise ops with their saved tensors."""

    @staticmethod
    def forward(ctx, x, bias, noise, strength, act, gain):
        y = _bias_act_native(x.detach(), None if bias is None else bias.detach(), act, noise,
                             None if strength is None else strength.detach(), gain)
        ctx.act, ctx.gain = act, gain
        ctx.has_bias, ctx.has_strength = bias is not None, strength is not None and noise is not None
        ctx.save_for_backward(y, noise if noise is not None else y.new_empty(0))
        return y

    @staticmethod
    def backward(ctx, gy):
        y, noise = ctx.saved_tensors
        g = gy * ctx.gain if ctx.act != "lrelu" else gy * torch.where(y > 0, ctx.gain, 0.2 * ctx.gain)
        gb = g.sum(dim=(0, 2, 3)) if ctx.has_bias else None
        gs = None
        if ctx.has_strength:
            gs = (g.sum(dim=1, keepdim=True) * noise.reshape((-1, 1) + tuple(g.shape[2:]))).sum()
        return g, gb, None, gs, None, None


def bias_act(x: torch.Tensor, bias: Optional[torch.Tensor], act: str = "lrelu", noise: Optional[torch.Tensor] = None,
             strength: Optional[torch.Tensor] = None) -> torch.Tensor:
    """act(x + noise * strength + bias[c]) * gain; x [B,C,H,W]; noise [H,W] (shared) or [B,1,H,W]; lrelu gain sqrt(2)."""
    gain = SQRT2 if act == "lrelu" else 1.0
    cuda32 = all(t is None or (t.is_cuda and t.dtype == torch.float32) for t in (x, bias, noise, strength))
    if cuda32 and x.shape[1] % 4 == 0 and torch.is_grad_enabled() and (noise is None or not noise.requires_grad) \
            and any(t is not None and t.requires_grad for t in (x, bias, strength)):
        return _BiasAct.apply(x, bias, noise, strength, act, gain)
    if _use_cuda(x, bias, noise, strength) and x.shape[1] % 4 == 0:
        xv = _nhwc_view(x)
        B, H, W, C = xv.shape
        y = torch.empty_like(xv)
        nz = None if noise is None else noise.contiguous()
        bstride = H * W if (nz is not None and nz.numel() == B * H * W and B > 1) else 0
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_bias_act_nhwc(xv.data_ptr(), y.data_ptr(), None if bias is None else bias.contiguous().data_ptr(),
                                                    None if nz is None else nz.data_ptr(),
                                                    None if strength is None else strength.data_ptr(), bstride, B, H * W, C,
                                                    1 if act == "lrelu" else 0, float(gain), _stream(x.device)), "gf_bias_act_nhwc")
        return y.permute(0, 3, 1, 2)
    if noise is not None:
        x = x + noise.to(x.dtype) * (1.0 if strength is None else strength.to(x.dtype))
    if bias is not None:
        x = x + bias.to(x.dtype).reshape(1, -1, 1, 1)
    if act == "lrelu":
        x = F.leaky_relu(x, 0.2) * SQRT2
    return x


def demod_coef(styles: torch.Tensor, wsq: torch.Tensor, eps: float = 1e-8) -> torch.Tensor:
    """d[b,o] = rsqrt(sum_i styles[b,i]^2 wsq[o,i] + eps) (StyleGAN2 demodulation, activation-scaling form)."""
    if _use_cuda(styles, wsq):
        B, I = styles.shape
        O = wsq.shape[0]
        d = torch.empty((B, O), dtype=torch.float32, device=styles.device)
        sr, ld = _rows(styles)
        with torch.cuda.device(styles.device):
            _lib.check(_lib.load().gf_demod_coef(sr.data_ptr(), ld, wsq.contiguous().data_ptr(), d.data_ptr(), B, O, I,
                                                 float(eps), _stream(styles.device)), "gf_demod_coef")
        return d
    return torch.rsqrt(styles.square() @ wsq.t() + eps)


def demod_coef_batch(pairs, eps: float = 1e-8):
    """[(styles [B,I_l], wsq [O_l,I_l]), ...] -> [d_l [B,O_l], ...]: every layer's demodulation coefficients in one launch
    (gf_demod_coef_batch).  CUDA fp32 only; the per-layer call serves everything else."""
    if not pairs:
        return []
    if len(pairs) > _lib.DEMOD_MAX_JOBS or not all(_use_cuda(s_, w_) for s_, w_ in pairs):
        return [demod_coef(s_, w_, eps) for s_, w_ in pairs]
    dev = pairs[0][0].device
    B = pairs[0][0].shape[0]
    total = sum(w_.shape[0] for _, w_ in pairs)
    d_all = torch.empty((B * total,), dtype=torch.float32, device=dev)       # one allocation, one [B, O_l] block per layer
    jobs = (_lib.GfDemodJob * len(pairs))()
    outs, keep, off = [], [], 0
    for i, (s_, w_) in enumerate(pairs):
        if s_.shape[0] != B or s_.shape[1] != w_.shape[1]:
            raise ValueError("demod_coef_batch: styles [B, I] / wsq [O, I] mismatch")
        sr, ld = _rows(s_)
        wc = w_.contiguous()
        O, I = wc.shape
        d = d_all[off:off + B * O].view(B, O)
        off += B * O
        jobs[i].styles, jobs[i].wsq, jobs[i].d = sr.data_ptr(), wc.data_ptr(), d.data_ptr()
        jobs[i].s_ld, jobs[i].O, jobs[i].I = ld, O, I
        outs.append(d)
        keep += [sr, wc]
    with torch.cuda.device(dev):
        _lib.check(_lib.load().gf_demod_coef_batch(ctypes.cast(jobs, ctypes.c_void_p), len(pairs), B, float(eps), _stream(dev)),
                   "gf_demod_coef_batch")
    return outs


def torgb(x: torch.Tensor, weight: torch.Tensor, styles: torch.Tensor, bias: Optional[torch.Tensor],
          next_styles: Optional[torch.Tensor] = None):
    """tRGB: 1x1 modulated convolution without demodulation.  x [B,C,H,W], weight [3,C,1,1] (raw; equalised-LR scale
    1/sqrt(C) applied here), styles [B,C], bias [3] -> [B,3,H,W] (planar).  With next_styles [B,C] (inference on CUDA) the same
    read of x also produces x * next_styles (the next block's modulated input) and the call returns (rgb, x_scaled)."""
    O, I = weight.shape[:2]
    wscale = 1.0 / math.sqrt(I)
    if _use_cuda(x, weight, styles, bias, next_styles) and O == 3 and I % 4 == 0 and I <= 512:
        xv = _nhwc_view(x)
        B, H, W, C = xv.shape
        y = torch.empty((B, O, H, W), device=x.device, dtype=torch.float32)
        sr, ld = _rows(styles)
        wv = weight.reshape(O, I).contiguous()
        xs = s2 = None
        ld2 = 0
        if next_styles is not None:
            s2, ld2 = _rows(next_styles)
            xs = torch.empty_like(xv)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().gf_torgb_scale_nhwc(xv.data_ptr(), wv.data_ptr(), sr.data_ptr(), ld,
                                                       bias.data_ptr() if bias is not None else None, ctypes.c_float(wscale),
                                                       y.data_ptr(), None if s2 is None else s2.data_ptr(), ld2,
                                                       None if xs is None else xs.data_ptr(), B, H * W, C, _stream(x.device)),
                       "gf_torgb_scale_nhwc")
        return y if next_styles is None else (y, xs.permute(0, 3, 1, 2))
    wm = weight.reshape(1, O, I).to(x.dtype) * styles[:, None, :].to(x.dtype) * wscale           # [B, 3, C]
    B, C, H, W = x.shape
    xl = x.permute(0, 2, 3, 1).reshape(B, H * W, C)
    rgb = torch.matmul(xl, wm.transpose(1, 2))
    if bias is not None:
        rgb = rgb + bias.to(x.dtype)
    rgb = rgb.transpose(1, 2).reshape(B, O, H, W)
    return rgb if next_styles is None else (rgb, x * next_styles[:, :, None, None].to(x.dtype))


def mapping_fwd(z: torch.Tensor, w_eff: torch.Tensor, b_eff: torch.Tensor, w_avg: Optional[torch.Tensor], psi: float, k: int) -> torch.Tensor:
    """G_mapping in one launch (gf_mapping_fwd): z [B, k+1, D]; w_eff [2, L, D, D] ([in, out], gains folded), b_eff [2, L, D];
    w_avg [2, D] (applied with psi when psi != 1).  CUDA fp32 inference only -- the module keeps the torch form for autograd."""
    B, kp1, D = z.shape
    L = w_eff.shape[1]
    out = torch.empty_like(z)
    wa = w_avg.contiguous() if (w_avg is not None and psi != 1.0) else None
    with torch.cuda.device(z.device):
        _lib.check(_lib.load().gf_mapping_fwd(z.contiguous().data_ptr(), w_eff.data_ptr(), b_eff.data_ptr(), wa.data_ptr() if wa is not None else None,
                                              float(psi), out.data_ptr(), B, k, D, L, _stream(z.device)), "gf_mapping_fwd")
    return out


def conv3x3_pack(weight: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """weight [O, I, 3, 3] -> the tap-major, TF32-rounded [9, O, I] layout gf_conv3x3_nhwc_tf32 consumes (gf_conv3x3_pack_weights)."""
    O, I = weight.shape[:2]
    wt = torch.empty((9, O, I), dtype=torch.float32, device=weight.device)
    with torch.cuda.device(weight.device):
        _lib.check(_lib.load().gf_conv3x3_pack_weights(weight.detach().contiguous().data_ptr(), wt.data_ptr(), O, I, ctypes.c_float(scale),
                                                       _stream(weight.device)), "gf_conv3x3_pack_weights")
    return wt


def conv3x3_native(x: torch.Tensor, wt: torch.Tensor, variant: Optional[tuple] = None) -> torch.Tensor:
    """3x3 stride-1 zero-padded convolution on the tcgen05 implicit-GEMM kernel (row f1, TF32): x [B, I, H, W] (channels-last
    storage), wt from conv3x3_pack -> [B, O, H, W] (channels-last storage).  CUDA fp32 inference only.
    variant: (version, bn, mt) forces one kernel instantiation (gf_conv3x3_nhwc_tf32_ex); None = the shape dispatch."""
    xv = _nhwc_view(x)
    B, H, W, I = xv.shape
    O = wt.shape[1]
    y = torch.empty((B, H, W, O), dtype=torch.float32, device=x.device)
    version, bn, mt = variant if variant is not None else (0, 0, 0)
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().gf_conv3x3_nhwc_tf32_ex(xv.data_ptr(), wt.data_ptr(), y.data_ptr(), B, H, W, I, O, version, bn, mt,
                                                       _stream(x.device)), "gf_conv3x3_nhwc_tf32")
    return y.permute(0, 3, 1, 2)
