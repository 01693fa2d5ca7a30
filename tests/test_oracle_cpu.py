"""CPU tests of the oracle itself: golden vectors, folded-vs-direct algebra, algebraic properties (SURVEY section 4).

PARITY UNPINNED: the reference ships no tests/fixtures (and no source) for this path; these pins are ours.
"""
import itertools
import os

import numpy as np
import pytest
import torch

from oracle import bipartite as ob
from oracle import folded as of
from tests.golden import make_golden as mg

GOLD = os.path.join(os.path.dirname(__file__), "golden", "attn_cases.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _run_case(c, seed, dtype=torch.float64):
    x, y, w = mg.make_inputs(c, seed)
    norm = None if c["norm"] == "none" else c["norm"]
    x, y = x.to(dtype), y.to(dtype)
    w = {k: v.to(dtype) for k, v in w.items()}
    return ob.transformer_layer(x, y, w, integration=c["integration"], norm=norm, duplex=c["duplex"],
                                use_pos=c["use_pos"], return_att=True, kmeans_iters=c.get("kmeans_iters", 1), img2ltnt=bool(c.get("img2ltnt")),
                                num_heads=c.get("num_heads", 1))


@pytest.mark.parametrize("idx", range(len(mg.cases())))
def test_oracle_matches_golden(gold, idx):
    c = mg.cases()[idx]
    out, att, cen = _run_case(c, 100 + idx)
    name = mg.case_name(c)
    np.testing.assert_allclose(mg.out_sample(out.permute(0, 2, 3, 1).numpy()), gold[name + "/out_sample"], rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(att.numpy(), gold[name + "/att"], rtol=2e-6, atol=1e-7)
    if cen is not None:
        np.testing.assert_allclose(cen.numpy(), gold[name + "/cen"], rtol=2e-6, atol=2e-6)


@pytest.mark.parametrize("idx", [0, 5, 12, 15, 19])
def test_oracle_fp32_close_to_fp64(idx):
    """e_ref of SURVEY 8c: the fp32 oracle (reference-Python-path stand-in) against fp64 truth."""
    c = mg.cases()[idx]
    out32, _, _ = _run_case(c, 100 + idx, torch.float32)
    ref, _, _ = _run_case(c, 100 + idx)                  # fp64, pinned by test_oracle_matches_golden
    err = (out32 - ref).abs()
    assert (err <= 2e-5 + 2e-4 * ref.abs()).all(), err.max()


@pytest.mark.parametrize("integration,norm,duplex,k,use_pos",
                         list(itertools.product(["mul", "add", "both"], ["layer", "instance", "batch", None],
                                                [False, True], [3, 16], [True, False])))
def test_folded_equals_direct(integration, norm, duplex, k, use_pos):
    """The three-stage folded form (what the CUDA kernels implement) is exact algebra of the direct form."""
    torch.manual_seed(1)
    B, C, H, W, D, p = 2, 32, 4, 8, 8, 8
    w = ob.init_params(C, D, k, p, integration, duplex, seed=1, bias_std=0.5)
    x = torch.randn(B, C, H, W, dtype=torch.float64)
    y = torch.randn(B, k, D, dtype=torch.float64)
    o, att, cen = ob.transformer_layer(x, y, w, integration=integration, norm=norm, duplex=duplex, use_pos=use_pos, return_att=True)
    o2, att2, cen2 = of.transformer_layer_folded(x.permute(0, 2, 3, 1).contiguous(), y, w, integration=integration, norm=norm,
                                                 duplex=duplex, use_pos=use_pos, return_att=True)
    assert (o.permute(0, 2, 3, 1) - o2).abs().max() < 1e-9
    assert (att - att2).abs().max() < 1e-10
    if duplex:
        assert (cen - cen2).abs().max() < 1e-10


def _simple(k=4, duplex=False, integration="mul", seed=3, B=3):
    C, H, W, D, p = 32, 4, 4, 8, 8
    g = torch.Generator().manual_seed(seed)
    w = ob.init_params(C, D, k, p, integration, duplex, seed=seed, bias_std=0.3)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    y = torch.randn(B, k, D, generator=g, dtype=torch.float64)
    return x, y, w


def test_attention_rows_sum_to_one():
    x, y, w = _simple()
    _, att, _ = ob.transformer_layer(x, y, w, return_att=True)
    assert torch.allclose(att.sum(dim=1), torch.ones_like(att.sum(dim=1)), atol=1e-12)
    assert (att >= 0).all()


def test_single_latent_gives_uniform_modulation():
    """k = 1: softmax over one latent is 1, so the gain is the same vector for every grid cell."""
    x, y, w = _simple(k=1)
    out, att, _ = ob.transformer_layer(x, y, w, return_att=True)
    assert torch.allclose(att, torch.ones_like(att))
    B, C, H, W = x.shape
    X = x.reshape(B, C, -1).permute(0, 2, 1)
    gain = out.reshape(B, C, -1).permute(0, 2, 1) / ob.att_norm(X, "layer")
    assert (gain - gain[:, :1]).abs().max() < 1e-8


def test_latent_permutation_equivariance():
    """Permuting the latents together with their positional embeddings leaves x' unchanged and permutes att."""
    x, y, w = _simple(k=5)
    perm = torch.tensor([3, 0, 4, 1, 2])
    out, att, _ = ob.transformer_layer(x, y, w, return_att=True)
    w2 = dict(w)
    w2["pos_latent"] = w["pos_latent"][perm]
    out2, att2, _ = ob.transformer_layer(x, y[:, perm], w2, return_att=True)
    assert (out - out2).abs().max() < 1e-10
    assert (att[:, perm] - att2).abs().max() < 1e-12


@pytest.mark.parametrize("duplex", [False, True])
def test_batch_independence(duplex):
    """Every image is independent through the block (the basis of the data-parallel sharding, SURVEY 8e)."""
    x, y, w = _simple(k=4, duplex=duplex)
    out, _, _ = ob.transformer_layer(x, y, w, duplex=duplex)
    out1, _, _ = ob.transformer_layer(x[1:2], y[1:2], w, duplex=duplex)
    assert (out[1:2] - out1).abs().max() < 1e-10


def test_positional_table_is_separable():
    t = ob.grid_pos_table(4, 8, 8)
    assert t.shape == (32, 8)
    row, col = ob.sinusoidal_axis(4, 4), ob.sinusoidal_axis(8, 4)
    assert torch.equal(t.reshape(4, 8, 8)[2, 5], torch.cat([row[2], col[5]]))


def test_philox_oracle_matches_random123_known_answers():
    """oracle/philox.py against the published Philox4x32-10 known-answer vectors (Random123 kat_vectors) -- the one part of the
    oracle a third party pins; the GPU suite then checks the kernels' mask against this oracle bit for bit."""
    from oracle import philox as ph
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        assert tuple(int(x) for x in ph.philox4x32_10(*ctr, *key)) == want
    m = ph.dropout_mult(0.25, seed=1234567890123, step=7, salt=5, tokens=4096, KP=16)
    assert m.shape == (4096, 16) and set(np.unique(m).tolist()) == {0.0, float(np.float32(1.0) / np.float32(0.75))}
    keep = (m > 0).mean()
    assert abs(keep - 0.75) < 4 * (0.25 * 0.75 / m.size) ** 0.5 + 1e-3
    assert not np.array_equal(m, ph.dropout_mult(0.25, seed=1234567890123, step=8, salt=5, tokens=4096, KP=16))     # next step: new mask
    assert not np.array_equal(m, ph.dropout_mult(0.25, seed=1234567890123, step=7, salt=6, tokens=4096, KP=16))     # another layer


def test_attention_dropout_algebra_of_the_oracle():
    """att_mult: an all-ones mask is the plain layer; an all-zero mask leaves only the un-droppable constants -- the output then does
    not depend on the latents' values (what the kernels re-add as (1 - sum q) * cb)."""
    C, D, k, p = 32, 16, 4, 16
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, C, 8, 8, generator=g, dtype=torch.float64)
    y = torch.randn(2, k, D, generator=g, dtype=torch.float64)
    w = ob.init_params(C, D, k, p, "mul", False, seed=2, bias_std=0.3)
    ref, _, _ = ob.transformer_layer(x, y, w, integration="mul")
    ones = torch.ones(2, 64, k, dtype=torch.float64)
    out1, _, _ = ob.transformer_layer(x, y, w, integration="mul", att_mult=ones)
    assert torch.allclose(out1, ref, atol=1e-12)
    zeros = torch.zeros(2, 64, k, dtype=torch.float64)
    out0a, _, _ = ob.transformer_layer(x, y, w, integration="mul", att_mult=zeros)
    out0b, _, _ = ob.transformer_layer(x, y + 3.0, w, integration="mul", att_mult=zeros)
    assert torch.allclose(out0a, out0b, atol=1e-12) and not torch.allclose(out0a, ref, atol=1e-3)
