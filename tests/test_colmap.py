"""CPU tests of litegs_b200/colmap.py (SURVEY 8f rank 3: the data format on the input side of the path).

* binary round trip of cameras / images / points3D;
* the files our writer produces are read by the REFERENCE's own reader (litegs/io_manager/colmap.py) to exactly what was
  written, through what that reader decoded from them (tests/golden/colmap_reference_reader.npz);
* camera conversion against the reference's formulas (litegs/data.py:33-51,72-77) and its round trip;
* initial Gaussians from SfM points against litegs/scene/point.py:7-19 with a brute-force k-NN."""
import hashlib
import os

import numpy as np
import pytest

from litegs_b200 import colmap, scene

def _model(n_pts=300, n_views=4, W=160, H=96, seed=0):
    rng = np.random.default_rng(seed)
    cams = {1: colmap.Camera(1, "PINHOLE", W, H, np.array([140.0, 138.0, W / 2, H / 2])),
            7: colmap.Camera(7, "SIMPLE_RADIAL", W, H, np.array([120.0, W / 2, H / 2, 0.01]))}
    images = {}
    for i in range(n_views):
        cam = scene.make_camera(i, n_views, W, H)
        q, t, _ = colmap.camera_to_colmap(cam, W, H)
        m = int(rng.integers(0, 6))
        images[i + 1] = colmap.Image(i + 1, q, t, 1, f"img_{i:03d}.png", rng.random((m, 2)) * 100, rng.integers(-1, 50, m))
    pts = {j + 1: colmap.Point3D(j + 1, rng.uniform(-1, 1, 3), rng.integers(0, 256, 3).astype(np.uint8), float(rng.random()),
                                 rng.integers(0, 100, (int(rng.integers(0, 4)), 2)).astype(np.int32)) for j in range(n_pts)}
    return cams, images, pts


def test_binary_round_trip(tmp_path):
    cams, images, pts = _model()
    colmap.write_model(str(tmp_path), cams, images, pts)
    c2, i2, p2 = colmap.read_model(str(tmp_path))
    assert set(c2) == set(cams) and set(i2) == set(images) and set(p2) == set(pts)
    for k, c in cams.items():
        assert c2[k].model == c.model and (c2[k].width, c2[k].height) == (c.width, c.height) and np.array_equal(c2[k].params, c.params)
    for k, im in images.items():
        assert np.array_equal(i2[k].qvec, im.qvec) and np.array_equal(i2[k].tvec, im.tvec) and i2[k].name == im.name
        assert i2[k].camera_id == im.camera_id and np.array_equal(i2[k].xys, im.xys) and np.array_equal(i2[k].point3D_ids, im.point3D_ids)
    for k, p in pts.items():
        assert np.array_equal(p2[k].xyz, p.xyz) and np.array_equal(p2[k].rgb, p.rgb) and p2[k].error == p.error
        assert np.array_equal(p2[k].track, p.track)


READER_MODEL = dict(n_pts=120, n_views=5)
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "colmap_reference_reader.npz")


def test_reference_reader_reads_what_we_write(tmp_path):
    """tests/golden/colmap_reference_reader.npz holds what the reference's reader decoded from the files our writer produced
    for this model, and their SHA-256 (tests/golden/make_golden_tree.py): the files written now are those bytes, and what the
    reference read from them is exactly what was written."""
    z = np.load(GOLD)
    cams, images, pts = _model(**READER_MODEL)
    d = colmap.write_model(str(tmp_path), cams, images, pts)
    for f, digest in zip(z["file_names"], z["file_sha256"]):
        assert hashlib.sha256(open(os.path.join(d, str(f)), "rb").read()).hexdigest() == str(digest), f
    assert list(z["camera_ids"]) == [1]                            # only PINHOLE cameras are kept (colmap.py:222-224)
    assert tuple(z["camera_wh"][0]) == (160, 96) and np.array_equal(z["camera_params"][0], cams[1].params)
    assert list(z["frame_names"]) == sorted(im.name for im in images.values())
    by_name = {im.name: im for im in images.values()}
    xys = np.split(z["frame_xys"], np.cumsum(z["frame_xys_len"])[:-1])
    for i, name in enumerate(z["frame_names"]):
        im = by_name[str(name)]
        assert z["frame_ids"][i] == im.id and np.array_equal(z["frame_qvec"][i], im.qvec) and np.array_equal(z["frame_tvec"][i], im.tvec)
        assert z["frame_camera_ids"][i] == 1
        assert np.array_equal(xys[i], np.asarray(im.xys).reshape(-1, 2))
    want = [pts[k] for k in pts]
    assert np.array_equal(z["points_xyz"], np.stack([p.xyz for p in want]))
    assert np.array_equal(z["points_rgb"], np.stack([p.rgb for p in want]).astype(np.float64))
    assert np.array_equal(z["points_err"][:, 0], np.array([p.error for p in want]))


def test_camera_conversion_matches_reference_formulas():
    W, H = 200, 120
    q = np.array([0.8, 0.1, -0.5, 0.3]); q /= np.linalg.norm(q)
    t = np.array([0.3, -1.2, 2.5])
    intr = np.array([170.0, 165.0, W / 2, H / 2])
    cam = colmap.camera_from_colmap(q, t, intr, W, H)
    # litegs/utils/__init__.py:7-17,33-38 and litegs/data.py:33-51,77 restated
    w, x, y, z = q
    R = np.array([[1 - 2 * y * y - 2 * z * z, 2 * x * y - 2 * w * z, 2 * z * x + 2 * w * y],
                  [2 * x * y + 2 * w * z, 1 - 2 * x * x - 2 * z * z, 2 * y * z - 2 * w * x],
                  [2 * z * x - 2 * w * y, 2 * y * z + 2 * w * x, 1 - 2 * x * x - 2 * y * y]])
    Rt = np.zeros((4, 4)); Rt[:3, :3] = R; Rt[:3, 3] = t; Rt[3, 3] = 1
    assert np.array_equal(cam["view"][0], np.float32(Rt).T)
    zn, zf = 0.01, 5000.0
    P = np.array([[intr[0] / (W * 0.5), 0, 0, 0], [0, intr[1] / (H * 0.5), 0, 0], [0, 0, zf / (zf - zn), -zf * zn / (zf - zn)], [0, 0, 1, 0]],
                 dtype=np.float32).T
    assert np.array_equal(cam["proj"][0], P)
    # a world point in front of the camera lands where the pinhole model says
    pw = np.array([0.2, -0.1, 0.4, 1.0], np.float32)
    pv = pw @ cam["view"][0]
    ph = pv @ cam["proj"][0]
    ndc = ph[:2] / ph[3]
    pc = R @ pw[:3] + t
    assert np.allclose(pv[:3], pc, atol=1e-6)
    assert np.allclose((ndc + 1) * 0.5 * np.array([W, H]), np.array([intr[0] * pc[0] / pc[2] + W / 2, intr[1] * pc[1] / pc[2] + H / 2]), atol=1e-3)
    q2, t2, i2 = colmap.camera_to_colmap(cam, W, H)
    assert np.allclose(q2, q, atol=1e-6) and np.allclose(t2, t, atol=1e-6) and np.allclose(i2, intr, atol=1e-4)
    for i in range(6):                                             # lattice cameras of the bench round-trip too
        c = scene.make_camera(i, 6, W, H)
        c2 = colmap.camera_from_colmap(*colmap.camera_to_colmap(c, W, H), W, H)
        assert all(np.abs(c[k] - c2[k]).max() < 2e-6 for k in c)


def test_initial_gaussians_follow_the_reference_recipe():
    rng = np.random.default_rng(3)
    n = 700
    xyz = rng.normal(size=(n, 3)); rgb = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    g = colmap.gaussians_from_points(xyz, rgb, sh_degree=3, chunk=128, morton=False)
    C, S = g["xyz"].shape[-2:]
    assert C * S >= n and g["sh_rest"].shape == (15, 3, C, S) and not g["sh_rest"].any()
    flat = lambda a: a.reshape(*a.shape[:-2], -1)[..., :n]
    assert np.allclose(flat(g["xyz"]).T, xyz, atol=1e-6)
    d2 = ((xyz[:, None] - xyz[None]) ** 2).sum(-1); np.fill_diagonal(d2, np.inf)
    want = np.log(np.sqrt(np.maximum(np.sort(d2, 1)[:, :3].mean(1), 1e-7)))          # point.py:8,14
    assert np.allclose(flat(g["scale"]), np.repeat(want[None], 3, 0), atol=1e-5)
    assert np.array_equal(flat(g["rot"])[0], np.ones(n, np.float32)) and not flat(g["rot"])[1:].any()
    assert np.allclose(flat(g["opacity"]), np.log(0.1 / 0.9), atol=1e-6)
    assert np.allclose(flat(g["sh_0"])[0] * colmap.SH_C0 + 0.5, rgb.T / 255.0, atol=1e-6)           # sh0_to_rgb(rgb_to_sh0(c)) = c
    # chunk AABBs contain their points
    lo, hi = g["cluster_origin"] - g["cluster_extend"], g["cluster_origin"] + g["cluster_extend"]
    assert (g["xyz"] >= lo[..., None] - 1e-5).all() and (g["xyz"] <= hi[..., None] + 1e-5).all()
