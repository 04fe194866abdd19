"""Batched multi-view rendering without a GPU: the new C-ABI symbols and scratch-size queries, the SASS / resource contract of the
two multi-view kernels (cuobjdump reads the sm_100a library), and the argument validation of the Python layer."""
import re
import shutil
import subprocess

import pytest
import torch

import helpers  # noqa: F401  (sets sys.path)
from dreamgaussian_b200 import _lib, build
from dreamgaussian_b200 import rasterizer as R
from dreamgaussian_b200.fused import BatchedFusedGaussianRasterizer

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
BATCH_SYMBOLS = ("dgr_batch_geom_bytes", "dgr_batch_image_bytes", "dgr_forward_preprocess_batch", "dgr_backward_batch")


def test_batch_symbols_are_exported_and_the_scratch_queries_need_no_gpu():
    lib = _lib.load()
    for name in BATCH_SYMBOLS:
        assert name in _lib.EXPORTS and hasattr(lib, name)
    for V, P, H, W in ((1, 1000, 64, 64), (8, 500000, 512, 512), (16, 100001, 70, 100)):
        g, i = lib.dgr_geom_bytes(P, H, W), lib.dgr_image_bytes(H, W)
        assert g % 256 == 0 and i % 256 == 0                                      # documented per-view strides
        assert lib.dgr_batch_geom_bytes(V, P, H, W) == V * g and lib.dgr_batch_image_bytes(V, H, W) == V * i
    assert lib.dgr_batch_geom_bytes(0, 10, 16, 16) == 0


@pytest.fixture(scope="module")
def resources():
    import os
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not found")
    path = build.build()
    out = subprocess.run([CUOBJDUMP, "--dump-resource-usage", path], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    res, name = {}, None
    for line in out.stdout.splitlines():
        m = re.match(r"\s*Function\s+(\S+?):?\s*$", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+)\s+STACK:(\d+)\s+SHARED:(\d+)", line)
        if m and name:
            res[name] = dict(reg=int(m.group(1)), stack=int(m.group(2)), shared=int(m.group(3)))
            name = None
    return path, res


def _ops(path, fn):
    out = subprocess.run([CUOBJDUMP, "-sass", "-fun", fn, path], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    return [m.group(1) for m in (re.match(r"\s*/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", l) for l in out.stdout.splitlines()) if m]


def test_multiview_kernels_resource_contract(resources):
    """Both kernels are designed for two 256-thread CTAs per SM (<= 128 registers, no spills: DESIGN.md §4), stage each warp's inputs
    with bulk TMA on an mbarrier, and use no tensor-core instructions."""
    path, res = resources
    count = lambda ops, prefix: sum(1 for o in ops if o.startswith(prefix))
    for kind in ("preprocess_fwd_multiview_kernel", "preprocess_bwd_multiview_kernel"):
        names = [k for k in res if kind in k]
        assert len(names) == 8, (kind, names)                                 # SH degree 0..3 x plain / raw parameters
        for k in names:
            assert res[k]["reg"] <= 128 and res[k]["stack"] == 0, (k, res[k])
        for k in names:
            ops = _ops(path, k)
            assert len(ops) > 100, k
            assert count(ops, "UBLKCP") >= 5 and count(ops, "SYNCS.ARRIVE.TRANS64") >= 1 and count(ops, "SYNCS.PHASECHK") >= 1, k
            assert not any(o.startswith(("HMMA", "UTCHMMA", "UTCQMMA", "UTCMMA", "LDTM", "STTM")) for o in ops), k
    # the step kernels' own lookups keep matching exactly one kernel each (tests/test_sass_contract.py)
    for parts in ("preprocess_fwd_kernelILi3ELb1ELb0ELb0ELb1E", "preprocess_bwd_kernelILi3ELb1ELb0ELb0ELb1E"):
        assert sum(1 for k in res if parts in k) == 1


def _settings(H=32, W=32, deg=0, dev="cpu", **kw):
    base = dict(image_height=H, image_width=W, tanfovx=0.5, tanfovy=0.5, bg=torch.zeros(3, device=dev), scale_modifier=1.0,
                viewmatrix=torch.eye(4, device=dev), projmatrix=torch.eye(4, device=dev), sh_degree=deg,
                campos=torch.zeros(3, device=dev), prefiltered=False, debug=False)
    base.update(kw)
    return R.GaussianRasterizationSettings(**base)


@pytest.mark.parametrize("cls", [R.BatchedGaussianRasterizer, BatchedFusedGaussianRasterizer])
def test_batch_settings_validation(cls):
    with pytest.raises(ValueError, match="1 to 16 views"):
        cls([])
    with pytest.raises(ValueError, match="1 to 16 views"):
        cls([_settings()] * 17)
    for bad in (dict(H=48), dict(W=48), dict(deg=1), dict(scale_modifier=2.0), dict(debug=True)):
        with pytest.raises(ValueError, match="must share"):
            cls([_settings(), _settings(**bad)])
    # fov, bg and the camera may differ
    ok = cls([_settings(), _settings(tanfovx=0.7, bg=torch.ones(3), viewmatrix=2 * torch.eye(4), campos=torch.ones(3))] * 8)
    assert isinstance(ok, torch.nn.Module) and len(ok.settings_list) == 16


def test_batch_rejects_precomputed_colours_and_covariances_and_cpu_tensors():
    P = 4
    r = R.BatchedGaussianRasterizer([_settings(), _settings()])
    args = (torch.zeros(P, 3), torch.zeros(P, 1), torch.zeros(P, 1, 3), torch.ones(P, 3), torch.ones(P, 4))
    with pytest.raises(ValueError, match="colors_precomp and cov3D_precomp are not supported"):
        r(*args, colors_precomp=torch.zeros(P, 3))
    with pytest.raises(ValueError, match="colors_precomp and cov3D_precomp are not supported"):
        r(*args, cov3D_precomp=torch.zeros(P, 6))
    with pytest.raises(ValueError, match="num_views, num_points, 3"):
        r(*args, means2D=torch.zeros(P, 3))
    with pytest.raises(RuntimeError, match="no CPU path"):
        r(*args)
    f = BatchedFusedGaussianRasterizer([_settings()])
    with pytest.raises(RuntimeError, match="no CPU path"):
        f(torch.zeros(P, 3), torch.zeros(P, 1, 3), torch.zeros(P, 0, 3), torch.zeros(P, 1), torch.zeros(P, 3), torch.ones(P, 4))


def test_c_abi_rejects_bad_batches_without_touching_a_device():
    """The batched entry points check their arguments before anything is enqueued."""
    import ctypes
    lib = _lib.load()
    z3 = (ctypes.c_float * 3)()
    s = _lib.DgrSettings(32, 32, 0.5, 0.5, 1.0, 0, 0, 0, ctypes.addressof(z3), ctypes.addressof(z3), ctypes.addressof(z3), ctypes.addressof(z3))
    g = _lib.DgrGaussians(64, 1, 16, 16, None, 16, 16, 16, None, None, 0)
    arr = (_lib.DgrSettings * 2)(s, s)
    assert lib.dgr_forward_preprocess_batch(arr, 0, ctypes.byref(g), 256, 256, 256, None) != 0 and b"1 to 16" in lib.dgr_last_error()
    assert lib.dgr_forward_preprocess_batch(arr, 17, ctypes.byref(g), 256, 256, 256, None) != 0
    arr[1].image_width = 48
    assert lib.dgr_forward_preprocess_batch(arr, 2, ctypes.byref(g), 256, 256, 256, None) != 0 and b"same for every view" in lib.dgr_last_error()
    arr[1].image_width = 32
    g2 = _lib.DgrGaussians(64, 1, 16, 16, None, 16, None, None, 16, None, 0)          # cov3D_precomp
    assert lib.dgr_forward_preprocess_batch(arr, 2, ctypes.byref(g2), 256, 256, 256, None) != 0 and b"cov3D_precomp" in lib.dgr_last_error()
    g3 = _lib.DgrGaussians(64, 1, 20, 16, None, 16, 16, 16, None, None, 0)            # means3D off a 16-byte boundary
    assert lib.dgr_forward_preprocess_batch(arr, 2, ctypes.byref(g3), 256, 256, 256, None) != 0 and b"16-byte aligned" in lib.dgr_last_error()
