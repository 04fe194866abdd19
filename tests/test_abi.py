"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every symbol the header
declares; the Python surface mirrors the reference's operator (names, fields, error behaviour); no CPU path exists."""
import os
import re

import pytest
import torch

import helpers  # noqa: F401  (sets sys.path)
from dreamgaussian_b200 import _lib, build

ROOT = helpers.ROOT


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "dgr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dgr_[a-z_0-9]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
    path = build.build()
    assert os.path.exists(path)
    lib = _lib.load()
    declared = _declared_functions()
    assert len(declared) >= 12
    for name in declared:
        assert hasattr(lib, name), "libdgr_b200.so does not export %s" % name
    assert set(_lib.EXPORTS) <= set(declared)
    assert lib.dgr_abi_version() == _lib.ABI_VERSION == 4


def test_scratch_size_queries_need_no_gpu():
    lib = _lib.load()
    g1, g2 = lib.dgr_geom_bytes(1000, 800, 800), lib.dgr_geom_bytes(100000, 800, 800)
    assert 0 < g1 < g2 and g2 >= 100000 * (48 + 48 + 4)
    assert lib.dgr_image_bytes(800, 800) >= 800 * 800 * 8
    assert lib.dgr_binning_bytes(1000000, 800, 800) >= 1000000 * 60
    assert lib.dgr_geom_bytes(0, 16, 16) > 0 and lib.dgr_binning_bytes(0, 16, 16) > 0


def test_tuning_word_is_validated_and_its_switch_bits_are_accepted():
    """dgr_set_tuning: sub-tile shapes are checked, the bit field (A/B switches up to bit 28, include/dgr_b200.h) is accepted and
    needs no GPU; the defaults are restored."""
    lib = _lib.load()
    assert lib.dgr_set_tuning(3, 1, 1) != 0 and b"ppl" in lib.dgr_last_error()
    for bits in (1 << 3, 1 << 20, 1 << 21, 2 << 22, 1 << 24, 1 << 25, 1 << 26, 1 << 28, (7 << 24) | (1 << 28), 0x7fffffff):
        assert lib.dgr_set_tuning(1, 2, 1 | bits) == 0
    assert lib.dgr_set_tuning(1, 1, 1) == 0


def test_misaligned_input_views_get_their_own_aligned_allocation():
    """The kernels read rotations / SH rows with 128-bit loads (include/dgr_b200.h, DgrGaussians): the host layer re-allocates a
    contiguous view that starts off a 16-byte boundary and leaves aligned tensors alone (no copy)."""
    import torch
    from dreamgaussian_b200 import rasterizer as R
    flat = torch.arange(41, dtype=torch.float32)
    view = flat[1:].view(10, 4)
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    fixed = R._aligned16(view)
    assert fixed.data_ptr() % 16 == 0 and torch.equal(fixed, view)
    assert R._aligned16(flat) is flat and R._aligned16(flat[:0]).numel() == 0


def test_python_surface_matches_reference_operator():
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    # the 12 fields the reference passes by keyword at gs_renderer.py:745-758, in the op's order
    assert GaussianRasterizationSettings._fields == (
        "image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix", "projmatrix",
        "sh_degree", "campos", "prefiltered", "debug")
    rs = GaussianRasterizationSettings(image_height=8, image_width=8, tanfovx=0.5, tanfovy=0.5, bg=torch.zeros(3),
                                       scale_modifier=1.0, viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=0,
                                       campos=torch.zeros(3), prefiltered=False, debug=False)
    r = GaussianRasterizer(raster_settings=rs)
    assert isinstance(r, torch.nn.Module) and hasattr(r, "markVisible")
    P = 4
    m, o = torch.zeros(P, 3), torch.zeros(P, 1)
    with pytest.raises(Exception, match="SHs or precomputed colors"):
        r(means3D=m, means2D=m, opacities=o, scales=torch.ones(P, 3), rotations=torch.ones(P, 4))
    with pytest.raises(Exception, match="SHs or precomputed colors"):
        r(means3D=m, means2D=m, opacities=o, shs=torch.zeros(P, 1, 3), colors_precomp=torch.zeros(P, 3),
          scales=torch.ones(P, 3), rotations=torch.ones(P, 4))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m, means2D=m, opacities=o, shs=torch.zeros(P, 1, 3))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m, means2D=m, opacities=o, shs=torch.zeros(P, 1, 3), scales=torch.ones(P, 3), rotations=torch.ones(P, 4),
          cov3D_precomp=torch.zeros(P, 6))


def test_no_cpu_path():
    """CPU tensors must fail loudly instead of silently running somewhere else."""
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    rs = GaussianRasterizationSettings(image_height=8, image_width=8, tanfovx=0.5, tanfovy=0.5, bg=torch.zeros(3),
                                       scale_modifier=1.0, viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=0,
                                       campos=torch.zeros(3), prefiltered=False, debug=False)
    P = 4
    with pytest.raises(RuntimeError, match="no CPU path"):
        GaussianRasterizer(rs)(means3D=torch.zeros(P, 3), means2D=torch.zeros(P, 3), opacities=torch.zeros(P, 1),
                               shs=torch.zeros(P, 1, 3), scales=torch.ones(P, 3), rotations=torch.ones(P, 4))


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under dreamgaussian_b200/ or diff_gaussian_rasterization/ may use it."""
    for pkg in ("dreamgaussian_b200", "diff_gaussian_rasterization", "simple_knn"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    txt = open(os.path.join(dirpath, f)).read()
                    assert "oracle" not in txt.replace("no oracle", ""), "%s mentions the oracle" % os.path.join(dirpath, f)


def test_compiled_host_layer_builds_loads_and_has_no_cpu_path():
    """csrc/dgr_torch.cpp -> lib/dgr_torch_host.so: the PyTorch binding of the same C-ABI calls (no arithmetic of its own)."""
    from dreamgaussian_b200 import rasterizer as R
    path = build.build_host()
    assert os.path.exists(path)
    assert R.set_fast_host(True), "the compiled host layer did not load"
    mod = R._FAST
    assert mod.abi_version() == _lib.ABI_VERSION and all(hasattr(mod, n) for n in ("forward", "backward", "State", "get_hint", "set_hint"))
    z = torch.zeros(3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        mod.forward(8, 8, 0.5, 0.5, 1.0, 0, False, False, z, torch.zeros(16), torch.zeros(16), z, torch.zeros(4, 3), None,
                    torch.zeros(4, 3), torch.zeros(4, 1), torch.zeros(4, 3), torch.zeros(4, 4), None, None, False)
    mod.set_hint(0, 123, 8, 8, 4096, True)
    assert mod.get_hint(0, 123, 8, 8) == (4096, True) and mod.get_hint(0, 124, 8, 8) is None


def test_reference_caller_imports_against_the_drop_in_packages():
    """Every name the original project's gs_renderer.py imports from diff_gaussian_rasterization and simple_knn._C (as bound
    when it ran on this repo's packages: tests/golden/make_golden_caller.py) resolves in the drop-in packages, to the same
    objects the rest of the repo uses; the GPU run is tests/test_reference_caller_gpu.py."""
    import importlib

    import numpy as np
    import diff_gaussian_rasterization as ours
    import simple_knn._C as knn
    imports = list(np.load(os.path.join(ROOT, "tests", "golden", "reference_caller_vectors.npz"))["imports"])
    assert {"diff_gaussian_rasterization:GaussianRasterizer", "diff_gaussian_rasterization:GaussianRasterizationSettings",
            "simple_knn._C:distCUDA2"} <= set(imports)
    for entry in imports:
        module, name = str(entry).split(":")
        assert hasattr(importlib.import_module(module), name), entry
    from dreamgaussian_b200 import knn as own_knn, rasterizer as R
    assert ours.GaussianRasterizer is R.GaussianRasterizer and knn.distCUDA2 is own_knn.distCUDA2
