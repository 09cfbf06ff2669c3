"""Generates the fixtures that pin this repository to the reference's source tree (LiteGS), so that the tests using them
run without that tree:

    python tests/golden/make_golden_tree.py <path of a LiteGS checkout> [outdir]

* ``reference_tree.json``: the line count of every source file under ``litegs/`` (tests/test_citations.py resolves the
  ``file:line`` citations of this repository against it) and the 26 ``litegs_fused`` pybind names with the arity of the C++
  declaration each one binds (tests/test_abi.py).
* ``colmap_reference_reader.npz``: what the reference's own COLMAP reader (``litegs/io_manager/colmap.py``, imported on its
  own with its two heavy imports stubbed) decodes from the files ``litegs_b200.colmap.write_model`` writes for the seeded
  model of tests/test_colmap.py, plus the SHA-256 of those files (tests/test_colmap.py).
CPU only."""
import hashlib
import importlib.util
import json
import os
import re
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

COLMAP_FILES = ("cameras.bin", "images.bin", "points3D.bin")


def line_counts(ref):
    out = {}
    for d, dirs, files in os.walk(os.path.join(ref, "litegs")):
        dirs[:] = sorted(x for x in dirs if x != "__pycache__")
        for f in sorted(files):
            if f.endswith((".cu", ".cuh", ".h", ".py", ".cpp")):
                p = os.path.join(d, f)
                out[os.path.relpath(p, ref)] = sum(1 for _ in open(p, errors="replace"))
    return out


def pybind_arity(ref):
    gr = os.path.join(ref, "litegs", "submodules", "gaussian_raster")
    names = re.findall(r'm\.def\("(\w+)"', open(os.path.join(gr, "ext_cuda.cpp")).read())
    decl = ""
    for h in ("raster.h", "binning.h", "compact.h", "transform.h"):
        decl += open(os.path.join(gr, h)).read()
    decl = re.sub(r"//.*", "", decl)
    out = {}
    for name in names:
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", decl, flags=re.S)
        out[name] = None if m is None else len([a for a in m.group(1).split(",") if a.strip()])
    return out


def reference_colmap_reader(ref):
    """litegs/io_manager/colmap.py imported on its own: `plyfile` and `litegs.data` (pulls in cv2/torch datasets) are replaced
    by stubs that record the constructor arguments."""
    pkg_dir = os.path.join(ref, "litegs")
    path = os.path.join(pkg_dir, "io_manager", "colmap.py")
    saved = {k: sys.modules.get(k) for k in ("plyfile", "litegs", "litegs.data", "litegs.io_manager", "litegs.io_manager.colmap")}
    try:
        ply = types.ModuleType("plyfile"); ply.PlyData = object; ply.PlyElement = object
        pkg = types.ModuleType("litegs"); pkg.__path__ = [pkg_dir]
        iom = types.ModuleType("litegs.io_manager"); iom.__path__ = [os.path.join(pkg_dir, "io_manager")]
        data = types.ModuleType("litegs.data")

        class PinHoleCameraInfo:
            def __init__(self, id, width, height, parameters):
                self.id, self.width, self.height, self.parameters = id, width, height, np.array(parameters)

        class ImageFrame:
            def __init__(self, id, qvec, tvec, camera_id, name, img_source, xys):
                self.id, self.qvec, self.tvec, self.camera_id, self.name, self.img_source, self.xys = id, qvec, tvec, camera_id, name, img_source, xys

        data.PinHoleCameraInfo, data.ImageFrame, data.CameraInfo = PinHoleCameraInfo, ImageFrame, object
        sys.modules.update({"plyfile": ply, "litegs": pkg, "litegs.io_manager": iom, "litegs.data": data})
        spec = importlib.util.spec_from_file_location("litegs.io_manager.colmap", path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules["litegs.io_manager.colmap"] = mod
        spec.loader.exec_module(mod)
        return mod
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def colmap_decoded(ref):
    from litegs_b200 import colmap
    from tests.test_colmap import READER_MODEL, _model
    reader = reference_colmap_reader(ref)
    cams, images, pts = _model(**READER_MODEL)
    with tempfile.TemporaryDirectory() as tmp:
        d = colmap.write_model(tmp, cams, images, pts)
        digests = [hashlib.sha256(open(os.path.join(d, f), "rb").read()).hexdigest() for f in COLMAP_FILES]
        cam_dict, frames = reader.load_frames(tmp, "images")
        xyz, rgb, err = reader.__dict__["__read_points3D_binary"](os.path.join(d, "points3D.bin"))
    ids = sorted(cam_dict)
    return dict(
        file_names=np.array(COLMAP_FILES), file_sha256=np.array(digests),
        camera_ids=np.array(ids, np.int64), camera_wh=np.array([(cam_dict[i].width, cam_dict[i].height) for i in ids], np.int64),
        camera_params=np.stack([np.asarray(cam_dict[i].parameters, np.float64) for i in ids]),
        frame_names=np.array([f.name for f in frames]), frame_ids=np.array([f.id for f in frames], np.int64),
        frame_camera_ids=np.array([f.camera_id for f in frames], np.int64),
        frame_qvec=np.stack([np.asarray(f.qvec, np.float64) for f in frames]), frame_tvec=np.stack([np.asarray(f.tvec, np.float64) for f in frames]),
        frame_xys_len=np.array([np.asarray(f.xys).reshape(-1, 2).shape[0] for f in frames], np.int64),
        frame_xys=np.concatenate([np.asarray(f.xys, np.float64).reshape(-1, 2) for f in frames]),
        points_xyz=np.asarray(xyz, np.float64), points_rgb=np.asarray(rgb, np.float64), points_err=np.asarray(err, np.float64))


def main():
    if len(sys.argv) < 2:
        sys.exit(__doc__)
    ref = sys.argv[1]
    outdir = sys.argv[2] if len(sys.argv) > 2 else os.path.dirname(os.path.abspath(__file__))
    tree = {"line_counts": line_counts(ref), "pybind_arity": pybind_arity(ref)}
    with open(os.path.join(outdir, "reference_tree.json"), "w") as f:
        json.dump(tree, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(outdir, "colmap_reference_reader.npz"), **colmap_decoded(ref))
    print("wrote", len(tree["line_counts"]), "line counts,", len(tree["pybind_arity"]), "pybind names, the COLMAP reader's decode")


if __name__ == "__main__":
    main()
