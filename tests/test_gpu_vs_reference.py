"""Tier-2 (SURVEY 8c): our kernels against the REFERENCE's own kernels (unmodified sources compiled for sm_100a) on a B200,
same seeded inputs, same op chain (tests/golden/make_golden.py:run_backend).  The reference side is what that op chain
returned on the reference's kernels, stored as tests/golden/<case>.npz by tests/golden/make_golden.py.

fp32 per-Gaussian ops must agree to fast-math rounding; integer binning outputs must agree except on pairs that
graze a tile (the reference's count uses --use_fast_math log/sqrt/div); the raster is compared at the tolerance its
packed-half blend allows (SURVEY fact 2 / Appendix B: ~1e-3 on the image, ~1e-2 relative on gradients)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _close(a, b, rtol, atol):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.abs(a - b) <= atol + rtol * np.abs(b)


@pytest.mark.parametrize("name", ["c_small_16x16", "c_small_8x16"])
def test_ours_vs_reference_kernels(cuda, name):
    import torch
    from litegs_b200 import fused
    from tests.golden.make_golden import run_backend
    old = dict(fused.CONFIG)
    fused.CONFIG["fix_last_tile"] = False            # bit-compatible tile ranges for this comparison (SURVEY Q3)
    ref = dict(np.load(os.path.join(GOLD, f"{name}.npz")))
    try:
        ours = run_backend(fused, name, torch, cuda)
    finally:
        fused.CONFIG.update(old)
    # chunk culling + activation + projection: fp32 on both sides
    assert np.array_equal(ref["cull_vis"], ours["cull_vis"]) and np.array_equal(ref["cull_ids"], ours["cull_ids"])
    for k in ("act_pos", "act_scale", "act_rot", "act_color", "act_opacity", "view_pos", "ndc", "T", "J", "cov2d", "inv_cov2d",
              "eig_val", "bw_inv", "bw_cov", "bw_T_q", "bw_T_s", "bw_mvp", "ab_pos", "ab_scale", "ab_rot", "ab_sh0", "ab_shr", "ab_opacity"):
        scale = max(1.0, float(np.abs(ref[k]).max()))
        ok = _close(ours[k], ref[k], 2e-4, 2e-5 * scale)
        assert ok.mean() > 0.9999, (k, 1 - ok.mean())
    # binning: per-splat tile counts equal for (almost) every splat; identical tables when the counts agree
    same = ref["alloc"] == ours["alloc"]
    assert same.mean() > 0.995, 1 - same.mean()
    if same.all():
        assert np.array_equal(ref["table_keys"], ours["table_keys"])
        assert np.array_equal(ref["table_vals"], ours["table_vals"])
        assert np.array_equal(ref["tile_range"], ours["tile_range"])
    # raster: the reference blends in fp16
    d = np.abs(ref["img"] - ours["img"])
    assert np.quantile(d, 0.999) < 6e-3 and d.mean() < 6e-4, (np.quantile(d, 0.999), d.mean())
    dl = np.abs(ref["last"].astype(np.int32) - ours["last"].astype(np.int32))
    assert (dl <= 1).mean() > 0.98
    for k in ("d_ndc", "d_cov2d_inv", "d_color", "d_opacity"):
        r, o = ref[k], ours[k]
        num = np.abs(r - o).sum(); den = np.abs(r).sum() + 1e-30
        assert num / den < 5e-2, (k, num / den)        # L1-relative, fp16 reference
