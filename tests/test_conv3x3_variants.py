"""The 3x3 convolution kernel (csrc/gf_conv.cu), instantiation by instantiation, against an exact-operand fp64 reference.

The kernel streams x in fp32 and the tensor core reads it as TF32 by dropping the low 13 mantissa bits; the packed weights are
TF32 already (gf_conv3x3_pack_weights rounds them to nearest).  Every product the kernel forms is therefore
trunc_tf32(x) * wt, exact in fp64, and

    ref_exact = ALPHA * conv2d_fp64(trunc_tf32(x), unpack(wt))        (zero padding 1)

differs from the kernel's output only by the fp32 accumulation over 9 * Cin terms and the final multiply by ALPHA.  That is checked
element by element against TAU * ALPHA * (|trunc_tf32(x)| conv |wt|), which a wrong tap, channel slab, tile or padding cell exceeds
by orders of magnitude.  The looser check against the unrounded fp64 convolution stays as the op's semantic contract.  On a B200
the kernel meets ref_exact to 1.6e-6 of (|x| conv |w|), and against the unrounded convolution its output carries no +3.5e-4 bias
(measured -1e-5 .. 0): the tensor core does truncate x, so ALPHA compensates a real bias instead of adding one.

gf_conv3x3_nhwc_tf32_ex forces one of the twelve (version, bn, mt) instantiations; shapes are chosen from the device's SM count so
that each one runs a single wave (one tile per CTA) and a persistent ragged grid (3 or 4 tiles per CTA: accumulator sets reused,
barrier phases flipped).
"""
import ctypes
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

# P.alpha of both launchers in gf_conv.cu: the mean relative TF32 truncation bias of the streamed x (0.7213 * 2^-11), compensated.
ALPHA = 1.000352220
# What is left is the tensor core's fp32 accumulation, and it is not round-to-nearest: on a B200 (148 SMs, 1000 W) y - ref_exact is a
# systematic shrink of about -2.3e-9 per summed term (relative rms 6.4e-7 at 9 * 32 terms, 1.07e-5 at 9 * 512, the same for all
# twelve instantiations), not noise.  Measured worst over every case in this file: 1.55e-6 for the element ratio below (config 2,
# res 64), 1.07e-5 for the relative rms.  A 1e-4 relative error anywhere gives >= 1.1e-5 and ~9e-5.
# Element bound |y - ref_exact| <= TAU * ALPHA * (|trunc(x)| conv |wt|)
TAU = 4e-6
# Relative RMS of y - ref_exact
REL_RMS_EXACT = 3e-5
# Semantic contract against the unrounded fp64 convolution (TF32 operands): rel-RMS, as test_conv3x3_implicit_gemm.
REL_RMS_FP64 = 5e-4

# every instantiation gf_conv.cu compiles: (version, bn, mt); NBUF = 1 for (256, 2), else 2
VARIANTS = [(v, bn, mt) for v in (1, 2) for bn in (256, 128, 64) for mt in (2, 1)]
VID = [f"v{v}-bn{bn}-mt{mt}" for v, bn, mt in VARIANTS]


def _ops():
    from importlib import import_module
    return import_module("gansformer-reproducibility-challenge_b200.ops")


def trunc_tf32(t: torch.Tensor) -> torch.Tensor:
    """fp32 -> TF32 by clearing the low 13 mantissa bits (what the tensor core does to the streamed operand)."""
    return (t.contiguous().view(torch.int32) & -8192).view(torch.float32)


def rne_tf32(t: torch.Tensor) -> torch.Tensor:
    """fp32 -> TF32, round to nearest, ties to even (finite inputs)."""
    b = t.contiguous().view(torch.int32)
    return ((b + 0xFFF + ((b >> 13) & 1)) & -8192).view(torch.float32)


def unpack(wt: torch.Tensor) -> torch.Tensor:
    """[9, O, I] packed weights -> [O, I, 3, 3]."""
    _, O, I = wt.shape
    return wt.reshape(3, 3, O, I).permute(2, 3, 0, 1)


def conv(xv: torch.Tensor, wt: torch.Tensor, variant=None) -> torch.Tensor:
    """xv [B, H, W, Cin] contiguous -> y [B, H, W, Cout] contiguous, on the kernel (variant None = the shape dispatch)."""
    y = _ops().conv3x3_native(xv.permute(0, 3, 1, 2), wt, variant=variant)
    return y.permute(0, 2, 3, 1)


def check_exact(y, xv, wt, idx=None, w_fp64=None, what=""):
    """y vs ref_exact on images idx (all if None): the element bound and the rel-RMS bound; with w_fp64 (the unrounded
    [O, I, 3, 3] weights) also the rel-RMS contract against the unrounded convolution.  Images are independent, so a subset
    of them is checked exactly."""
    if idx is None:
        idx = list(range(xv.shape[0]))
    x = xv[idx].double().permute(0, 3, 1, 2)
    tx = trunc_tf32(xv[idx]).double().permute(0, 3, 1, 2)
    w64 = unpack(wt).double()
    ref = ALPHA * F.conv2d(tx, w64, padding=1)
    mag = ALPHA * F.conv2d(tx.abs(), w64.abs(), padding=1)
    got = y[idx].double().permute(0, 3, 1, 2)
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    err = (got - ref).abs()
    ratio = (err / mag.clamp_min(1e-300)).max().item()
    rel_rms = (err.norm() / ref.norm()).item()
    msg = f"[conv-exact] {what}: max |err| / (|x| conv |w|) = {ratio:.3e}, rel_rms = {rel_rms:.3e}"
    if w_fp64 is not None:
        full = F.conv2d(x, w_fp64.double(), padding=1)
        rel_full = ((got - full).norm() / full.norm()).item()
        r = F.conv2d(x, w64, padding=1)                                   # exact x, the packed weights: the bias ALPHA corrects
        bias = ((got - r) * r).sum().item() / (r * r).sum().item()
        msg += f", vs unrounded fp64: rel_rms = {rel_full:.3e}, bias = {bias:+.3e}"
    print(msg)
    bad = (err > TAU * mag).sum().item()
    assert bad == 0, f"{what}: {bad} elements exceed TAU * (|x| conv |w|) (max ratio {ratio:.3e})"
    assert rel_rms <= REL_RMS_EXACT, f"{what}: rel_rms {rel_rms:.3e} vs ref_exact"
    if w_fp64 is not None:
        assert rel_full <= REL_RMS_FP64, f"{what}: rel_rms {rel_full:.3e} vs the unrounded fp64 convolution"


def sampled(B):
    return sorted({0, B // 2, B - 1})


def tiles(B, H, W, Cout, bn, mt):
    return B * (H // (8 * mt)) * (W // 16) * (Cout // bn)


def problem(B, H, W, Cin, Cout, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    xv = torch.randn(B, H, W, Cin, device=dev, generator=g)
    w = torch.randn(Cout, Cin, 3, 3, device=dev, generator=g)
    scale = 1.0 / math.sqrt(9 * Cin)
    return xv, _ops().conv3x3_pack(w, scale=scale), w.double() * scale


@pytest.fixture(scope="module")
def nsm(cuda_dev):
    return torch.cuda.get_device_properties(cuda_dev).multi_processor_count


# ---------------------------------------------------------------------------------------------------------
# CPU: the selector validates before touching the device
# ---------------------------------------------------------------------------------------------------------
def test_ex_rejects_what_it_cannot_run(gf):
    lib = gf._lib.load()
    err = lambda: lib.gf_last_error().decode()
    P = 256                                                               # fake, 16-byte aligned device pointers: never dereferenced
    ex = lambda H, Cout, v, bn, mt, x=P: lib.gf_conv3x3_nhwc_tf32_ex(x, P, P, 2, H, 32, 64, Cout, v, bn, mt, None)
    for v, bn, mt in [(3, 256, 1), (1, 96, 1), (2, 128, 3), (0, 256, 1), (1, 0, 0), (-1, 64, 1)]:
        assert ex(32, 256, v, bn, mt) == -2 and "no instantiation" in err() and f"version={v}, bn={bn}, mt={mt}" in err()
    assert ex(32, 192, 1, 128, 1) == -2 and "Cout % 128 == 0" in err() and "Cout=192" in err()
    assert ex(24, 256, 2, 64, 2) == -2 and "H % 16 == 0" in err() and "H=24" in err()
    # zeros = the dispatch, with gf_conv3x3_nhwc_tf32's own validation and messages
    assert ex(7, 256, 0, 0, 0) == -2 and "H % 8 == 0" in err()
    assert lib.gf_conv3x3_nhwc_tf32_ex(P, P, P, 2, 8, 16, 48, 64, 0, 0, 0, None) == -2 and "Cin % 32" in err()
    assert lib.gf_conv3x3_nhwc_tf32_ex(None, P, P, 2, 8, 16, 32, 64, 0, 0, 0, None) == -1 and "null pointer" in err()
    assert ex(32, 256, 0, 0, 0, x=P + 4) == -1 and "16-byte aligned" in err()
    assert ex(32, 256, 1, 256, 2, x=P + 4) == -1 and "16-byte aligned" in err()
    # a call that launched nothing reports zeros
    assert gf._lib.conv3x3_last_variant() == (0, 0, 0)
    assert lib.gf_conv3x3_last_variant(None, None, None) == -1 and "null pointer" in err()


def test_alpha_is_the_constant_of_both_launchers():
    src = open(os.path.join(ROOT, "gansformer-reproducibility-challenge_b200", "csrc", "gf_conv.cu")).read()
    found = re.findall(r"P\.alpha\s*=\s*([0-9.eE+-]+)f\s*;", src)
    assert len(found) == 2 and all(float(a) == ALPHA for a in found), found


# ---------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------
def variant_shape(kind, variant, nsm):
    """single: one wave (every CTA runs one tile), Cin = 512 (a long K ring), three tile rows, W = 48 (border and interior
    w tiles).  persistent: >= 3 x SMs tiles and not a multiple of the SM count (CTAs run 3 or 4 tiles, the last wave is
    ragged), Cin = 32 (nine K steps per tile: the ring wraps across tiles), one tile row, W = 64."""
    _, bn, mt = variant
    if kind == "single":
        return 2, 24 * mt, 48, 512, 256
    H, W, Cout = 8 * mt, 64, 2 * bn
    per_image = tiles(1, H, W, Cout, bn, mt)
    B = 3 * nsm // per_image + 1
    while (B * per_image) % nsm == 0:
        B += 1
    return B, H, W, 32, Cout


@gpu
@pytest.mark.parametrize("kind", ["single", "persistent"])
@pytest.mark.parametrize("variant", VARIANTS, ids=VID)
def test_instantiation_matches_exact_operand_reference(gf, cuda_dev, nsm, variant, kind):
    B, H, W, Cin, Cout = variant_shape(kind, variant, nsm)
    n = tiles(B, H, W, Cout, *variant[1:])
    if kind == "single":
        assert n < nsm
    else:
        assert 3 * nsm <= n < 4 * nsm and n % nsm != 0
    xv, wt, w64 = problem(B, H, W, Cin, Cout, cuda_dev, seed=2 * VARIANTS.index(variant) + (kind == "persistent"))
    with torch.no_grad():
        y = conv(xv, wt, variant)
    assert gf._lib.conv3x3_last_variant() == variant
    check_exact(y, xv, wt, w_fp64=w64, what=f"{variant} {kind} B={B} {H}x{W} {Cin}->{Cout} tiles={n}")


@gpu
@pytest.mark.parametrize("version", [1, 2])
def test_instantiations_of_one_version_give_the_same_bits(gf, cuda_dev, nsm, version):
    """Within a version every instantiation sums in the same K order (tap -> channel slab in version 1, channel slab -> dx -> dy in
    version 2), whatever BN, MT and the accumulator count: the outputs are bit-identical, and so are two calls."""
    B, H, W, Cin, Cout = 6, 32, 48, 64, 256                          # every (bn, mt) fits; 36 .. 576 tiles
    xv, wt, _ = problem(B, H, W, Cin, Cout, cuda_dev, seed=version)
    mine = [v for v in VARIANTS if v[0] == version]
    with torch.no_grad():
        ys = [conv(xv, wt, v).view(torch.int32).clone() for v in mine]
        again = conv(xv, wt, mine[0]).view(torch.int32)
    check_exact(ys[0].view(torch.float32), xv, wt, what=f"v{version} bitwise base")
    assert torch.equal(again, ys[0]), "two calls of one instantiation differ"
    for v, y in zip(mine[1:], ys[1:]):
        diff = (y != ys[0]).sum().item()
        assert diff == 0, f"{v} differs from {mine[0]} in {diff} elements"


@gpu
@pytest.mark.parametrize("variant", VARIANTS, ids=VID)
def test_padding_and_addressing_canaries(gf, cuda_dev, nsm, variant):
    """Image b scaled by 8^b (a read across images shows), border rows and columns scaled by 1024 (a wrong padding cell shows),
    x inside a NaN-filled allocation (a read past the tensor map's extent reaches the output), y inside a sentinel-filled one
    (every element around y stays bitwise unchanged).  Power-of-two scales keep the TF32 operands exact."""
    B, H, W, Cin, Cout = 3, 32, 48, 64, 256
    PAD = 4 * 1025                                                        # floats: 16-byte, not 128-byte, aligned
    g = torch.Generator(device=cuda_dev).manual_seed(7)
    x = torch.randn(B, H, W, Cin, device=cuda_dev, generator=g)
    x *= (8.0 ** torch.arange(B, device=cuda_dev, dtype=torch.float32))[:, None, None, None]
    x[:, [0, H - 1]] *= 1024.0
    x[:, :, [0, W - 1]] *= 1024.0
    xbuf = torch.full((PAD + x.numel() + PAD,), float("nan"), device=cuda_dev)
    xv = xbuf[PAD:PAD + x.numel()].view(B, H, W, Cin)
    xv.copy_(x)
    wt = _ops().conv3x3_pack(torch.randn(Cout, Cin, 3, 3, device=cuda_dev, generator=g), scale=1.0 / math.sqrt(9 * Cin))
    SENTINEL = 0x5A5A5A5A
    ny = B * H * W * Cout
    ybuf = torch.full((PAD + ny + PAD,), SENTINEL, dtype=torch.int32, device=cuda_dev)
    yv = ybuf[PAD:PAD + ny].view(torch.float32).view(B, H, W, Cout)
    lib = gf._lib.load()
    with torch.cuda.device(cuda_dev):
        gf._lib.check(lib.gf_conv3x3_nhwc_tf32_ex(xv.data_ptr(), wt.data_ptr(), yv.data_ptr(), B, H, W, Cin, Cout, *variant,
                                                  ctypes.c_void_p(torch.cuda.current_stream(cuda_dev).cuda_stream)),
                      "gf_conv3x3_nhwc_tf32_ex")
    torch.cuda.synchronize()
    assert bool((ybuf[:PAD] == SENTINEL).all()) and bool((ybuf[PAD + ny:] == SENTINEL).all()), "a store landed outside y"
    check_exact(yv, xv, wt, what=f"{variant} canaries")


@gpu
@pytest.mark.parametrize("Cout,Cin", [(64, 32), (7, 5), (1, 1), (33, 129)])
def test_pack_weights_rounds_to_nearest_even(gf, cuda_dev, Cout, Cin):
    """gf_conv3x3_pack_weights = round_to_nearest_even_tf32(w * scale) in the [9][Cout][Cin] layout, bit for bit -- including
    exact ties (low 13 bits 0x1000, both parities of the kept LSB) and their neighbours, and sizes that are not multiples of 4."""
    g = torch.Generator(device=cuda_dev).manual_seed(Cout * 131 + Cin)
    w = torch.randn(Cout, Cin, 3, 3, device=cuda_dev, generator=g)
    bits = w.view(torch.int32)
    sel = torch.randint(0, 4, w.shape, device=cuda_dev, generator=g)
    low = torch.tensor([0x1000, 0x0FFF, 0x1001, 0x1FFF], device=cuda_dev, dtype=torch.int32)[sel]
    ties = ((bits & -8192) | low).view(torch.float32)
    for src, scale in ((w, 1.0 / math.sqrt(9 * Cin)), (ties, 1.0)):
        got = _ops().conv3x3_pack(src, scale=scale)
        want = rne_tf32(src.permute(2, 3, 0, 1).reshape(9, Cout, Cin) * torch.tensor(scale, dtype=torch.float32, device=cuda_dev))
        torch.cuda.synchronize()
        assert got.shape == (9, Cout, Cin)
        diff = (got.view(torch.int32) != want.view(torch.int32)).sum().item()
        assert diff == 0, f"scale={scale}: {diff} packed weights differ from the RNE emulation"


def _bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


# config 2 (256^2, batch 32) on a 148-SM B200: resolution -> (version, bn, mt) the dispatch launches
CONFIG2_ON_148_SMS = {16: (1, 256, 1), 32: (2, 256, 2), 64: (1, 256, 2), 128: (2, 256, 2), 256: (2, 128, 2)}


@gpu
@pytest.mark.parametrize("cfg", [1, 2, 3, 5])
def test_benchmarked_shapes(gf, cuda_dev, nsm, cfg):
    """The stride-1 convolutions that run on the kernel in bench.py's configurations (res >= 16, Cin = Cout = nf(res), the per-GPU
    batch): the shape dispatch against ref_exact on images {0, B/2, B-1}, and bit-identical to forcing the instantiation
    gf_conv3x3_last_variant reports -- which ties the per-instantiation tests above to what the benchmark launches."""
    from importlib import import_module
    nets = import_module("gansformer-reproducibility-challenge_b200.networks")
    c = _bench().CONFIGS[cfg]
    B = c["batch"]
    launched = {}
    res = 16
    while res <= c["res"]:
        C = nets.nf(res)
        xv, wt, w64 = problem(B, res, res, C, C, cuda_dev, seed=res + cfg)
        with torch.no_grad():
            y = conv(xv, wt)
            v = gf._lib.conv3x3_last_variant()
            yf = conv(xv, wt, v)
        launched[res] = v
        what = f"config {cfg} res {res} B={B} {C}->{C} {v}"
        assert v in VARIANTS, what
        assert torch.equal(y.view(torch.int32), yf.view(torch.int32)), f"{what}: dispatch and forced instantiation differ"
        check_exact(y, xv, wt, idx=sampled(B), w_fp64=w64, what=what)
        del xv, y, yf
        res *= 2
    print(f"[conv-dispatch] config {cfg} on {nsm} SMs: {launched}")
    if cfg == 2 and nsm == 148:
        assert launched == CONFIG2_ON_148_SMS
