"""Every reference citation of the form `<file>:<line>[-<line>]` in the C ABI header, the kernels, the host mirror, the
oracle and the design documents must resolve against the reference tree: the file exists and has at least that many lines.  The
tree is represented by the line count of each of its source files (tests/golden/reference_tree.json, written by
tests/golden/make_golden_tree.py)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREE = os.path.join(ROOT, "tests", "golden", "reference_tree.json")
PREFIXES = {"GR/": "litegs/submodules/gaussian_raster/", "fused_ssim/": "litegs/submodules/fused_ssim/", "litegs/": "litegs/"}
BARE = {"wrapper.py": "litegs/utils/wrapper.py", "optimizer.py": "litegs/training/optimizer.py", "trainer.py": "litegs/training/trainer.py",
        "data.py": "litegs/data.py", "densify.py": "litegs/training/densify.py", "statistic_helper.py": "litegs/utils/statistic_helper.py",
        "colmap.py": "litegs/io_manager/colmap.py", "ply.py": "litegs/io_manager/ply.py", "ssim.cu": "litegs/submodules/fused_ssim/ssim.cu",
        "ext.cpp": "litegs/submodules/fused_ssim/ext.cpp", "point.py": "litegs/scene/point.py", "cluster.py": "litegs/scene/cluster.py",
        "arguments.py": "litegs/arguments.py", "render/__init__.py": "litegs/render/__init__.py"}
CITE = re.compile(r"((?:GR/|fused_ssim/|litegs/)[\w./\-]+?\.(?:cu|cuh|h|py|cpp)|(?<![\w/])(?:%s)):(\d+)(?:-(\d+))?" %
                  "|".join(re.escape(k) for k in BARE))


def _sources():
    out = [os.path.join(ROOT, "include", "litegs_b200.h")] + [os.path.join(ROOT, f) for f in ("DESIGN.md", "INTEGRATION.md", "README.md")]
    for d in ("litegs_b200", os.path.join("litegs_b200", "csrc"), "oracle"):
        p = os.path.join(ROOT, d)
        out += [os.path.join(p, f) for f in sorted(os.listdir(p)) if f.endswith((".py", ".cu", ".cuh", ".h", ".c"))]
    return out


def _resolve(name):
    for pre, to in PREFIXES.items():
        if name.startswith(pre):
            cands = [to + name[len(pre):]]
            if pre == "fused_ssim/":
                cands.append(to + "fused_ssim/" + name[len(pre):])          # the package's __init__ lives one level down
            return cands
    return [BARE[name]]


def test_reference_citations_resolve():
    lines_of = json.load(open(TREE))["line_counts"]
    bad, n = [], 0
    for src in _sources():
        text = open(src, errors="replace").read()
        for m in CITE.finditer(text):
            name, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            path = next((p for p in _resolve(name) if p in lines_of), None)
            n += 1
            if path is None:
                bad.append((os.path.relpath(src, ROOT), m.group(0), "no such file"))
                continue
            if not (1 <= a <= b <= lines_of[path]):
                bad.append((os.path.relpath(src, ROOT), m.group(0), f"file has {lines_of[path]} lines"))
    assert n > 150, n
    assert not bad, bad[:20]
