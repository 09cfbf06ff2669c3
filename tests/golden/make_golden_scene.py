"""Generates tests/golden/scene_reference.npz: what the reference's own chunk-maintenance code (litegs/scene/point.py,
litegs/scene/cluster.py, the unmodified Python package staged by ``oracle/build_ref.py:stage_python``, on this repository's
native modules) computes on the seeded inputs of tests/test_gpu_f4.py, on a B200:

    python tests/golden/make_golden_scene.py [outdir]          (default: tests/golden)

* ``spatial_refine`` in its optimizer form (point.py:104-154: parameters and Adam moments reordered in place) and
  ``_gen_morton_code``: bit-exact outputs, stored as the SHA-256 of each array's bytes;
* ``get_cluster_AABB`` (cluster.py:29-46): the chunk origins and extents themselves (float32, [3, chunks]).
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

PARAM_KEYS = ("xyz", "scale", "rot", "sh_0", "sh_rest", "opacity")


def digest(t) -> str:
    """SHA-256 of a tensor's elements in row-major order (dtype included)."""
    a = np.ascontiguousarray(t.detach().cpu().numpy())
    return hashlib.sha256(str(a.dtype).encode() + a.tobytes()).hexdigest()


def reference_scene_module():
    from oracle import build_ref
    from litegs_b200 import shims
    path = build_ref.reference_python_path()
    if path is None:
        sys.exit("the reference Python package is not staged: run __graft_entry__.build() where the reference tree is present")
    shims.install()
    if path not in sys.path:
        sys.path.insert(1, path)
    import litegs
    return litegs.scene


def main():
    import torch
    from litegs_b200 import scene
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    ref = reference_scene_module()
    import litegs.scene.point as refpoint
    dev = torch.device("cuda:0")
    store = {}
    # tests/test_gpu_f4.py::test_morton_codes_and_spatial_refine
    p = scene.make_scene(50_000, sh_degree=1, seed=2, morton=False)
    T = {k: torch.from_numpy(p[k]).to(dev) for k in PARAM_KEYS}
    prm = {k: torch.nn.Parameter(T[k].clone()) for k in PARAM_KEYS}
    opt = torch.optim.Adam([{"params": [prm[k]], "lr": 0.0, "name": k} for k in PARAM_KEYS], lr=0.0, eps=1e-15)
    for k in PARAM_KEYS:
        opt.state[prm[k]] = {"step": torch.tensor(0.0), "exp_avg": (T[k] * 0.5).clone(), "exp_avg_sq": (T[k] * T[k]).clone()}
    store["morton_sha256"] = digest(refpoint._gen_morton_code(T["xyz"].reshape(3, -1)))
    r = ref.spatial_refine(True, opt, prm["xyz"])
    for k, t in zip(PARAM_KEYS, r):
        store[f"refine_{k}_sha256"] = digest(t.reshape(T[k].shape))
        store[f"refine_exp_avg_{k}_sha256"] = digest(opt.state[prm[k]]["exp_avg"].reshape(T[k].shape))
        store[f"refine_exp_avg_sq_{k}_sha256"] = digest(opt.state[prm[k]]["exp_avg_sq"].reshape(T[k].shape))
    # tests/test_gpu_f4.py::test_cluster_aabb_device
    p = scene.make_scene(30_000, sh_degree=0, seed=4, log_scale_range=(0.01, 0.2))
    x, s, q = (torch.from_numpy(p[k]).to(dev) for k in ("xyz", "scale", "rot"))
    ro, re_ = ref.cluster.get_cluster_AABB(x, s.exp(), torch.nn.functional.normalize(q, dim=0))
    store["aabb_origin"] = ro.cpu().numpy()
    store["aabb_extend"] = re_.cpu().numpy()
    path = os.path.join(outdir, "scene_reference.npz")
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in store.items()})
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
