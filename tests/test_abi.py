"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/litegs_b200.h declares (with the argument counts the ctypes layer assumes), and the host mirror
offers the reference's 26 pybind names with the reference's positional arity.  No compute calls."""
import ctypes
import inspect
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_decls():
    h = open(os.path.join(ROOT, "include", "litegs_b200.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    out = {}
    for m in re.finditer(r"\n(?:int|const char\*)\s+(lgs_\w+)\s*\(([^;]*?)\)\s*;", h):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args == "void" else len(args.split(","))
    return out


def test_library_exports_every_declared_symbol():
    from litegs_b200 import _lib, build
    build.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    decls = _header_decls()
    assert len(decls) >= 30
    for name in decls:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert set(decls) == set(_lib.exported_symbols())
    for name, n in decls.items():
        if name in _lib.SIGNATURES:
            assert len(_lib.SIGNATURES[name]) == n, name
    assert lib.lgs_abi_version() == 2


def test_library_contains_sm100a_code_and_bulk_copy():
    """cuobjdump: the cubin is sm_100a and the raster kernels use the TMA engine's bulk copy (UBLKCP)."""
    import shutil
    import subprocess
    from litegs_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass and "LDGSTS" in sass and "MUFU.EX2" in sass and "REDG.E.ADD.F32" in sass


def test_host_mirror_has_the_26_reference_names():
    import litegs_fused
    from litegs_b200 import fused
    assert len(fused.EXPORTS) == 26
    for name in fused.EXPORTS:
        assert callable(getattr(litegs_fused, name))


def test_names_and_arity_match_the_reference_headers():
    """The reference's pybind names (GR/ext_cuda.cpp) and the arity of the declaration each binds (GR/{raster,binning,compact,
    transform}.h), as tests/golden/make_golden_tree.py read them into tests/golden/reference_tree.json."""
    import json
    from litegs_b200 import fused
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_tree.json")))["pybind_arity"]
    assert sorted(ref) == sorted(fused.EXPORTS)
    for name, n_ref in ref.items():
        assert n_ref is not None, name
        fn = getattr(fused, name)
        params = inspect.signature(fn).parameters
        if any(p.kind == p.VAR_POSITIONAL for p in params.values()):      # out-of-scope stubs take *args
            continue
        assert len(params) == n_ref, (name, len(params), n_ref)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from litegs_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.LiteGSB200Error):
        _lib.load()


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under litegs_b200/ (nor the drop-in shims, nor the example) may import it."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = [os.path.join(root, "litegs_fused.py"), os.path.join(root, "fused_ssim.py"), os.path.join(root, "examples", "train_synthetic.py")]
    for d, _, fs in os.walk(os.path.join(root, "litegs_b200")):
        files += [os.path.join(d, f) for f in fs if f.endswith(".py")]
    pat = re.compile(r"^\s*(import\s+oracle\b|from\s+oracle\b)", re.M)
    bad = [f for f in files if os.path.exists(f) and pat.search(open(f).read())]
    assert not bad, bad


def test_fused_ssim_shim_has_the_reference_names():
    """fused_ssim/fused_ssim/__init__.py:5-6,16,44,53,82 and ext.cpp:4-9."""
    import fused_ssim as m
    for n in ("fusedssim", "fusedssim_backward", "fusedl1ssim_loss", "fusedl1ssim_loss_backward", "FusedSSIMMap", "FusedL1SSIMLossMap",
              "fused_ssim", "fused_l1_ssim_loss", "allowed_padding"):
        assert hasattr(m, n), n


def test_no_kernel_of_ours_spills_to_local_memory():
    """cuobjdump -res-usage: every hand-written kernel compiles without local-memory spills (LOCAL:0) and within the
    255-register limit with room to spare (a regression here is a silent 2x slowdown of an issue-bound kernel)."""
    import shutil
    import subprocess
    from litegs_b200 import _lib
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([exe, "-res-usage", _lib.LIB_PATH], capture_output=True, text=True).stdout
    names = re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out)
    ours = [(n, int(r), int(l)) for n, r, s, sh, l in names if "cub" not in n and "thrust" not in n]
    assert len(ours) > 60, len(ours)
    assert all(l == 0 for _, _, l in ours), [n for n, _, l in ours if l]
    assert max(r for _, r, _ in ours) <= 168, max(ours, key=lambda t: t[1])
