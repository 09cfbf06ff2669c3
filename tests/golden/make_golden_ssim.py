"""Generates tests/golden/ssim_small.npz by running the UNMODIFIED reference fused_ssim CUDA kernels (built by
oracle/build_ref.py:build_ssim from litegs/submodules/fused_ssim/{ssim.cu,ext.cpp} with the reference's flags) on a B200:

    python tests/golden/make_golden_ssim.py gpurun_out/golden      # on the GPU box; then copy the .npz into tests/golden/

Inputs are seeded (numpy default_rng(7)): a random image pair and a smooth pair (blurred noise, the regime of real
renders where sigma is small), [2,3,37,53]: ragged against every tile size in play (16x16 in the reference, 64x32 ours).
Stored per mode (0 = SSIM map, 1 = L1 + SSIM loss map with weight 0.2): map, the three partials, and dL/dimg1 for a seeded
upstream gradient.

Also writes tests/golden/ssim_1080p_sample.npz: the L1 + SSIM loss (weight 0.2) of a seeded 1920x1080 pair, its three partials
and dL/dimg1 for a seeded upstream gradient (inputs from ``inputs_1080p``), stored at a fixed seeded sample of SAMPLE_1080P
elements, with each tensor's largest magnitude and the sums of the three inputs (to check that they regenerate).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def inputs():
    rng = np.random.default_rng(7)
    B, CH, H, W = 2, 3, 37, 53
    out = {}
    a = rng.random((B, CH, H, W), dtype=np.float32)
    b = rng.random((B, CH, H, W), dtype=np.float32)
    out["rand"] = (a, b)
    k = np.ones(9, np.float32) / 9
    sm = lambda z: np.apply_along_axis(lambda r: np.convolve(r, k, mode="same"), 3, np.apply_along_axis(lambda r: np.convolve(r, k, mode="same"), 2, z))
    c = sm(a).astype(np.float32)
    d = (c + 0.05 * (sm(b) - 0.5)).astype(np.float32)
    d[0, 0, 3:6, 4:9] = c[0, 0, 3:6, 4:9]              # exact ties: sign(0) = 0 in the L1 gradient
    out["smooth"] = (c, d)
    up = rng.standard_normal((B, CH, H, W)).astype(np.float32)
    return out, up


SAMPLE_1080P = 4096


def inputs_1080p(dev):
    """A 1080p image pair 0.1 apart and an upstream gradient, from torch's CPU generator (seed 2)."""
    g = torch.Generator(device="cpu").manual_seed(2)
    x = torch.rand((1, 3, 1080, 1920), generator=g).to(dev)
    y = (x + 0.1 * (torch.rand((1, 3, 1080, 1920), generator=g).to(dev) - 0.5)).clamp(0, 1)
    up = torch.randn((1, 3, 1080, 1920), generator=g).to(dev)
    return x, y, up


def sample_1080p(ref, dev):
    x, y, up = inputs_1080p(dev)
    idx = np.sort(np.random.default_rng(13).choice(x.numel(), SAMPLE_1080P, replace=False)).astype(np.int64)
    ti = torch.from_numpy(idx).to(dev)
    m, d0, d1, d2 = ref.fusedl1ssim_loss(0.2, 0.01 ** 2, 0.03 ** 2, x, y, True)
    g = ref.fusedl1ssim_loss_backward(0.2, 0.01 ** 2, 0.03 ** 2, x, y, up, d0, d1, d2)
    store = {"index": idx, "input_sums": np.array([float(t.double().sum()) for t in (x, y, up)])}
    for k, v in zip(("map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12", "grad"), (m, d0, d1, d2, g)):
        store[k] = v.reshape(-1)[ti].cpu().numpy()
        store[f"{k}_absmax"] = np.float64(v.abs().max().item())
    return store


def main():
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    from oracle import build_ref
    ref = build_ref.load_ssim()
    if ref is None:
        sys.exit("oracle/_ref/fused_ssim_cuda_ref.so is not built: run `python oracle/build_ref.py` where /root/reference is mounted")
    dev = torch.device("cuda:0")
    C1, C2, w = 0.01 ** 2, 0.03 ** 2, 0.2
    pairs, up = inputs()
    store = {"upstream": up, "C1": np.float64(C1), "C2": np.float64(C2), "ssim_weight": np.float64(w)}
    for name, (a, b) in pairs.items():
        ta, tb, tu = torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), torch.from_numpy(up).to(dev)
        store[f"{name}_img1"], store[f"{name}_img2"] = a, b
        m, d0, d1, d2 = ref.fusedssim(C1, C2, ta, tb, True)
        g = ref.fusedssim_backward(C1, C2, ta, tb, tu, d0, d1, d2)
        for k, v in zip(("map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12", "grad"), (m, d0, d1, d2, g)):
            store[f"{name}_ssim_{k}"] = v.cpu().numpy()
        m, d0, d1, d2 = ref.fusedl1ssim_loss(w, C1, C2, ta, tb, True)
        g = ref.fusedl1ssim_loss_backward(w, C1, C2, ta, tb, tu, d0, d1, d2)
        for k, v in zip(("map", "dm_dmu1", "dm_dsigma1_sq", "dm_dsigma12", "grad"), (m, d0, d1, d2, g)):
            store[f"{name}_l1_{k}"] = v.cpu().numpy()
    path = os.path.join(outdir, "ssim_small.npz")
    np.savez_compressed(path, **store)
    print("wrote", path, os.path.getsize(path), "bytes")
    path = os.path.join(outdir, "ssim_1080p_sample.npz")
    np.savez_compressed(path, **sample_1080p(ref, dev))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
