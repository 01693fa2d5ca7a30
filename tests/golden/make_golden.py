"""Generates tests/golden/attn_cases.npz from the fp64 oracle (oracle/bipartite.py), fixed seeds.

PARITY UNPINNED: the reference ships no fixtures for this path (no source at all, SURVEY.md section 0), so these
vectors pin the *oracle*, and through it the CUDA kernels, against silent drift -- not against the reference.
Attention probabilities and centroids are stored whole; of each layer output only the fixed sample ``out_sample``
is stored, which keeps the file small (the tests compare the full output with the live fp64 oracle).
Run from the repo root:  python tests/golden/make_golden.py
"""
import itertools
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import bipartite as ob  # noqa: E402

B, C, H, W, D, P = 2, 64, 8, 16, 16, 16
OUT_STRIDE = 5          # coprime with C and W: the sample covers every channel and every pixel column


def out_sample(out_nhwc):
    """The stored sample of a channels-last layer output (numpy array or tensor): every OUT_STRIDE-th element."""
    return out_nhwc.reshape(-1)[::OUT_STRIDE]


def cases():
    out = []
    for integ, norm in itertools.product(["mul", "add", "both"], ["layer", "instance", "batch", "none"]):
        out.append(dict(integration=integ, norm=norm, duplex=False, k=4, use_pos=True))
    for integ in ["mul", "add", "both"]:
        out.append(dict(integration=integ, norm="layer", duplex=True, k=4, use_pos=True))
    for k in (16, 20, 32):
        out.append(dict(integration="mul", norm="layer", duplex=False, k=k, use_pos=True))
    out.append(dict(integration="both", norm="layer", duplex=True, k=16, use_pos=True))
    out.append(dict(integration="mul", norm="layer", duplex=False, k=8, use_pos=False))
    out.append(dict(integration="mul", norm="layer", duplex=True, k=8, use_pos=False))
    # round 2 (appended: earlier cases keep their seeds): k-means iterations > 1 and g_img2ltnt (SURVEY A.3)
    out.append(dict(integration="mul", norm="layer", duplex=True, k=16, use_pos=True, kmeans_iters=2))
    out.append(dict(integration="both", norm="layer", duplex=True, k=8, use_pos=True, img2ltnt=True))
    out.append(dict(integration="mul", norm="layer", duplex=True, k=4, use_pos=True, kmeans_iters=3, img2ltnt=True))
    out.append(dict(integration="mul", norm="layer", duplex=False, k=8, use_pos=True, num_heads=2))
    out.append(dict(integration="both", norm="layer", duplex=False, k=5, use_pos=True, num_heads=4))
    return out


def case_name(c):
    ext = (f"-it{c['kmeans_iters']}" if c.get("kmeans_iters", 1) > 1 else "") + ("-i2l" if c.get("img2ltnt") else "") \
        + (f"-h{c['num_heads']}" if c.get("num_heads", 1) > 1 else "")
    return f"{c['integration']}-{c['norm']}-{'duplex' if c['duplex'] else 'simplex'}-k{c['k']}-{'pos' if c['use_pos'] else 'nopos'}{ext}"


def make_inputs(c, seed):
    """Inputs are regenerated from the seed by the tests (only outputs are stored)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 1.5 + 0.3
    y = torch.randn(B, c["k"], D, generator=g, dtype=torch.float64)
    w = ob.init_params(C, D, c["k"], P, c["integration"], c["duplex"], seed=seed + 1000, bias_std=0.5,
                       extras=c.get("kmeans_iters", 1) > 1 or bool(c.get("img2ltnt")))
    return x, y, w


def main():
    store = {}
    for i, c in enumerate(cases()):
        x, y, w = make_inputs(c, seed=100 + i)
        norm = None if c["norm"] == "none" else c["norm"]
        out, att, cen = ob.transformer_layer(x, y, w, integration=c["integration"], norm=norm, duplex=c["duplex"],
                                             use_pos=c["use_pos"], return_att=True, kmeans_iters=c.get("kmeans_iters", 1),
                                             img2ltnt=bool(c.get("img2ltnt")), num_heads=c.get("num_heads", 1))
        name = case_name(c)
        store[name + "/out_sample"] = out_sample(out.permute(0, 2, 3, 1).contiguous().numpy()).astype(np.float32)   # channels-last
        store[name + "/att"] = att.numpy().astype(np.float32)
        if cen is not None:
            store[name + "/cen"] = cen.numpy().astype(np.float32)
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "attn_cases.npz")
    np.savez_compressed(path, **store)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB,", len(cases()), "cases")


if __name__ == "__main__":
    main()
