"""SURVEY 8f rank 4 -- densification statistics and chunk maintenance -- against their definitions:
 * gpu_driven_pipeline_sparse_op: add / min / max over every dtype the reference dispatches (GR/compact.cu:1221-1336);
 * Morton codes, spatial_refine and chunk AABBs on the device vs the numpy restatement and vs what the reference's own
   functions (litegs/scene/point.py:22-154, litegs/scene/cluster.py:29-46) computed on the same inputs
   (tests/golden/scene_reference.npz, written by tests/golden/make_golden_scene.py);
 * litegs_b200.statistics.StatisticsHelper fed by Level A and by the fused Level B: same numbers, equal to the ones derived from
   the oracle's raster statistics (statistic_helper.py:82-156,215-243; wrapper.py:501-506)."""
import os

import numpy as np
import pytest
import torch

import oracle
from litegs_b200 import fused, render, scene, statistics
from litegs_b200.arguments import PipelineParams
from tests.util import PARAM_KEYS, scaled_err, small_scene

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.float32, torch.int32, torch.float64, torch.int64, torch.int16, torch.int8, torch.uint8])
@pytest.mark.parametrize("op", ["add", "min", "max"])
def test_sparse_chunk_op_all_dtypes(cuda, dtype, op):
    rng = np.random.default_rng(0)
    E, C, A, S = 3, 40, 17, 128
    lo, hi = (0, 100) if dtype == torch.uint8 else (-50, 50)
    a = rng.integers(lo, hi, size=(E, C, S)); b = rng.integers(lo, hi, size=(E, A, S))
    ids = rng.permutation(C)[:A].astype(np.int64)
    nvalid = 11                                                   # rows at or past the device-side count are ignored
    At = torch.from_numpy(a).to(dtype).to(cuda); Bt = torch.from_numpy(b).to(dtype).to(cuda)
    fused.gpu_driven_pipeline_sparse_op(At, Bt, torch.from_numpy(ids).to(cuda), torch.tensor([nvalid], dtype=torch.int32, device=cuda), op)
    exp = a.copy()
    f = {"add": np.add, "min": np.minimum, "max": np.maximum}[op]
    exp[:, ids[:nvalid], :] = f(a[:, ids[:nvalid], :], b[:, :nvalid, :])
    assert np.array_equal(At.cpu().numpy().astype(np.int64), exp)
    with pytest.raises(RuntimeError):
        fused.gpu_driven_pipeline_sparse_op(At, Bt, torch.from_numpy(ids).to(cuda), torch.tensor([nvalid], dtype=torch.int32, device=cuda), "mul")


def _morton_numpy(xyz, bits=21):
    """_gen_morton_code restated (point.py:38-81), fp32 arithmetic."""
    lo = xyz.min(axis=1, keepdims=True); hi = xyz.max(axis=1, keepdims=True)
    scale = np.float32((1 << bits) - 1)
    nrm = ((xyz - lo) / np.maximum(hi - lo, np.float32(1e-12))).astype(np.float32) * scale
    q = np.clip(nrm.astype(np.int64), 0, int(scale))
    code = np.zeros(xyz.shape[1], np.int64)
    for b in range(bits):
        code |= ((q[0] >> b) & 1) << (3 * b) | ((q[1] >> b) & 1) << (3 * b + 1) | ((q[2] >> b) & 1) << (3 * b + 2)
    return code


def _reference_golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scene_reference.npz"))


def test_morton_codes_and_spatial_refine(cuda):
    p = scene.make_scene(50_000, sh_degree=1, seed=2, morton=False)
    xyz_c = torch.from_numpy(p["xyz"]).to(cuda)
    C, S = xyz_c.shape[-2:]
    flat = p["xyz"].reshape(3, -1)
    codes = scene.morton_codes_device(xyz_c.reshape(3, -1)).cpu().numpy()
    assert np.array_equal(codes, _morton_numpy(flat))
    T = {k: torch.from_numpy(p[k]).to(cuda) for k in PARAM_KEYS}
    T["exp_avg_xyz"] = torch.randn_like(T["xyz"])                   # an optimizer moment rides along
    out, order = scene.spatial_refine_device(T)
    order_np = np.argsort(_morton_numpy(flat), kind="stable")
    assert np.array_equal(order.cpu().numpy(), order_np)
    for k in T:
        src = T[k].cpu().numpy().reshape(-1, C * S)
        assert np.array_equal(out[k].cpu().numpy().reshape(-1, C * S), src[:, order_np]), k
    # the reference's own spatial_refine in its optimizer form (point.py:104-154: parameters and Adam moments reordered in place;
    # its tensor form, :94-103, passes a tuple to uncluster and cannot run) and its Morton codes, bit for bit
    from tests.golden.make_golden_scene import digest
    ref = _reference_golden()
    mom, _ = scene.spatial_refine_device({"xyz": T["xyz"], **{f"m_{k}": T[k] * 0.5 for k in PARAM_KEYS}, **{f"v_{k}": T[k] * T[k] for k in PARAM_KEYS}})
    for k in PARAM_KEYS:
        assert digest(out[k]) == str(ref[f"refine_{k}_sha256"]), k
        assert digest(mom[f"m_{k}"]) == str(ref[f"refine_exp_avg_{k}_sha256"]), k
        assert digest(mom[f"v_{k}"]) == str(ref[f"refine_exp_avg_sq_{k}_sha256"]), k
    assert digest(torch.from_numpy(codes)) == str(ref["morton_sha256"])


def test_cluster_aabb_device(cuda):
    p = scene.make_scene(30_000, sh_degree=0, seed=4, log_scale_range=(0.01, 0.2))
    x, s, q = (torch.from_numpy(p[k]).to(cuda) for k in ("xyz", "scale", "rot"))
    o, e = scene.cluster_aabb_device(x, s, q)
    o64, e64 = scene.cluster_aabb(p["xyz"], p["scale"], p["rot"])   # fp64 numpy form of cluster.py:29-46
    assert np.abs(o.cpu().numpy() - o64).max() < 1e-5 and np.abs(e.cpu().numpy() - e64).max() < 1e-5
    ref = _reference_golden()                                       # the reference's get_cluster_AABB on the same inputs
    assert np.abs(ref["aabb_origin"] - o.cpu().numpy()).max() < 1e-5 and np.abs(ref["aabb_extend"] - e.cpu().numpy()).max() < 1e-5
    # a box must contain its Gaussians' centres
    assert bool(((x - o[:, :, None]).abs() <= e[:, :, None] + 1e-6).all())


def _expected_statistics(ref, params, w, hw, tile):
    th, tw = tile
    inter = ref["inter"]
    C, S = params["xyz"].shape[-2:]
    ids = ref["visible_chunk_id"]; nvis = ids.shape[0]
    _, _, _, fc, fw, _ = oracle.rasterize_forward(ref["sorted_pid"], ref["ranges"], inter["ndc"], inter["inv_cov2d"], ref["color"], ref["opacity"],
                                                  None, hw[0], hw[1], th, tw, enable_statistic=True)
    g_full = np.zeros_like(ref["img_padded"])
    mask = (ref["img_padded"][..., : hw[0], : hw[1]] >= 0) & (ref["img_padded"][..., : hw[0], : hw[1]] <= 1)
    g_full[..., : hw[0], : hw[1]] = w * mask
    gmax = float(np.abs(g_full).max())
    bw = oracle.rasterize_backward(ref["sorted_pid"], ref["ranges"], inter["ndc"], inter["inv_cov2d"], ref["color"], ref["opacity"], None,
                                   ref["T"], ref["last"], (g_full / gmax).astype(np.float32), None, gmax, hw[0], hw[1], th, tw,
                                   enable_statistic=True, err_mode="reference")

    def dense(a):
        out = np.zeros((*a.shape[:-1], C, S), np.float64)
        out[..., ids, :] = a.reshape(*a.shape[:-1], -1, S)[..., :nvis, :]
        return out.reshape(*a.shape[:-1], -1)
    cnt = dense(fc[0, 0].astype(np.float64))
    s1 = dense(bw[3].astype(np.float64)); s2 = dense((bw[5][0] * gmax * gmax).astype(np.float64))
    _, _, alloc = oracle.get_allocate_size(inter["ndc"], inter["view_pos"][:, 2], inter["inv_cov2d"], ref["opacity"], hw[0], hw[1], th, tw)
    return dict(cnt=cnt, w_mean=dense(fw[0].astype(np.float64)) / (cnt + 1e-9),
                e_var=np.maximum(s2 / (cnt + 1) - (s1 / (cnt + 1)) ** 2, 0), vis=dense((alloc > 0).astype(np.float64)))


@pytest.mark.parametrize("level", ["A", "B", "views"])
def test_statistics_helper_levels_match_oracle(cuda, level):
    SH = statistics.StatisticsHelperInst
    hw, tile, deg = (96, 128), (8, 16), 2
    params, aabb, cam = small_scene(n=4000, hw=hw, tile=tile, seed=5)
    rng = np.random.default_rng(105)
    w = rng.normal(size=(1, 3, *hw)).astype(np.float32)
    o0 = oracle.render_forward_backward(params, aabb, cam, hw, tile, deg, lambda img: w)
    frag = o0["fragile"][:, : hw[0], : hw[1]]
    w = w * (~frag)[:, None]
    ref = oracle.render_forward_backward(params, aabb, cam, hw, tile, deg, lambda img: w)
    exp = _expected_statistics(ref, params, w, hw, tile)
    C, S = params["xyz"].shape[-2:]
    P = {k: torch.from_numpy(params[k]).to(cuda).requires_grad_(True) for k in PARAM_KEYS}
    A = [torch.from_numpy(a).to(cuda) for a in aabb]
    Cm = {k: torch.from_numpy(v).to(cuda) for k, v in cam.items()}
    wt = torch.from_numpy(w).to(cuda)
    pp = PipelineParams(tile_size=tile)
    SH.reset(C, S, lambda epoch: True)
    SH.cur_sample = "view0"
    try:
        with SH.try_start(0):
            if level == "A":
                ids, num, cx, cs, cr, col, cop = render.render_preprocess(A[0], A[1], Cm["frustumplane"], Cm["view"], P["xyz"], P["scale"], P["rot"],
                                                                          P["sh_0"], P["sh_rest"], P["opacity"], None, None, pp, deg)
                img = render.render(Cm["view"], Cm["proj"], cx, cs, cr, col, cop, num * pp.cluster_size, None, None, deg, hw, pp)[0]
                (img * wt).sum().backward()
            elif level == "B":
                img = render.render_view(A[0], A[1], Cm["frustumplane"], Cm["view"], Cm["proj"], P["xyz"], P["scale"], P["rot"], P["sh_0"],
                                         P["sh_rest"], P["opacity"], deg, hw, pp)[0]
                (img * wt).sum().backward()
            else:
                from litegs_b200.dist import GradAccumulator
                acc = GradAccumulator(P)
                render.render_views(1, lambda i: Cm, lambda i, im: (im * wt).sum(), A[0], A[1], P["xyz"], P["scale"], P["rot"], P["sh_0"],
                                    P["sh_rest"], P["opacity"], deg, hw, pp, acc.grads())
        torch.cuda.synchronize()
        got_w, got_cnt = SH.get_mean("fragment_weight")
        assert np.array_equal(got_cnt.cpu().numpy().astype(np.int64), exp["cnt"].astype(np.int64))
        assert scaled_err(got_w.cpu().numpy(), exp["w_mean"]) < 2e-4
        got_var, _ = SH.get_var("fragment_err")
        assert scaled_err(got_var.cpu().numpy(), exp["e_var"]) < 5e-4
        assert np.array_equal(SH.visible_count.cpu().numpy().reshape(-1).astype(np.int64), exp["vis"].reshape(-1).astype(np.int64))
        assert np.array_equal(SH.get_global_culling().cpu().numpy().reshape(-1), exp["vis"].reshape(-1) == 0)
        # tile blend counts -> heaviest-first order for the next time this sample is rendered
        gx, gy = (hw[1] + tile[1] - 1) // tile[1], (hw[0] + tile[0] - 1) // tile[0]
        last = ref["last"][0, 0].astype(np.uint16).astype(np.int64)
        per_tile = last.reshape(gy, tile[0], gx, tile[1]).transpose(0, 2, 1, 3).reshape(gy * gx, -1).max(1)
        okt = ~frag[0].reshape(gy, tile[0], gx, tile[1]).transpose(0, 2, 1, 3).reshape(gy * gx, -1).any(1)
        got_tiles = SH.cached_tiles_blend_count["view0"].cpu().numpy()
        assert np.array_equal(got_tiles[okt], per_tile[okt])
        order = SH.cached_sorted_tile_list["view0"].cpu().numpy()
        assert np.array_equal(np.sort(order), np.arange(1, gx * gy + 1)) and (np.diff(got_tiles[order - 1]) <= 0).all()
    finally:
        SH.reset(0, 0, lambda epoch: False)
        SH.cur_sample = None
        SH.cached_sorted_tile_list.clear(); SH.cached_tiles_blend_count.clear()
