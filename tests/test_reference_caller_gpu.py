"""The original project's own caller of the rasterizer on the drop-in packages of this repo (SURVEY.md §8 row A0).

The original's `Renderer.initialize` -> `GaussianModel.create_from_pcd` -> `simple_knn._C.distCUDA2` and `Renderer.render`
(transposed-view `viewmatrix` of MiniCam, the retain_grad dummy `means2D`, `clamp(0, 1)`) followed by
`add_densification_stats` were run once on this repo's `diff_gaussian_rasterization` / `simple_knn._C`, and what that caller
passed and got back was stored: tests/golden/reference_caller_vectors.npz (tests/golden/make_golden_caller.py).  Here
`_initialize` and `_render` restate that caller; the stored camera and settings are the call's arguments, and the stored
samples pin the restated Gaussians.  Everything the caller gets back (image, alpha, depth, radii, leaf gradients,
viewspace-point gradients, densification statistics) is compared with the CPU oracle fed the same tensors, and at the stored
samples with what the original caller got.
"""
import os
import types

import numpy as np
import pytest
import torch

import helpers as h

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_caller_vectors.npz")
SH_C0 = 0.28209479177387814


def _training_args():
    # configs/image.yaml:67-75 of the original
    return types.SimpleNamespace(position_lr_init=0.001, position_lr_final=0.00002, position_lr_delay_mult=0.02,
                                 position_lr_max_steps=500, feature_lr=0.01, opacity_lr=0.05, scaling_lr=0.005,
                                 rotation_lr=0.005, percent_dense=0.01)


CASES = {
    # BASELINE.json configs[0]: what `python main.py --config configs/image.yaml` renders first (image.yaml:65-66, 12, 41-44)
    "image_yaml_init": dict(sh_degree=0, num_pts=5000, W=256, H=256, elev=0.0, azim=0.0, scaling_modifier=1.0, bg=None, ups=0),
    # SH degree 3 active, non-square image, scaling modifier, explicit background, perturbed parameters
    "deg3_perturbed": dict(sh_degree=3, num_pts=20000, W=320, H=200, elev=-20.0, azim=130.0, scaling_modifier=1.15,
                           bg=(0.1, 0.4, 0.7), ups=3),
}


def _initialize(num_pts, max_sh_degree):
    """Renderer.initialize(num_pts) of the original: points uniform in a ball of radius 0.5 and colours SH2RGB(U(0, 1) / 255),
    drawn from numpy's global generator in this order; then create_from_pcd: SH DC = RGB2SH(colour) in float32, higher
    bands zero, scale = log sqrt(max(distCUDA2, 1e-7)) on all three axes, identity rotation, opacity logit(0.1)."""
    from simple_knn._C import distCUDA2
    phi = np.random.random((num_pts,)) * 2 * np.pi
    theta = np.arccos(np.random.random((num_pts,)) * 2 - 1)
    r = 0.5 * np.cbrt(np.random.random((num_pts,)))
    xyz = np.stack((r * np.sin(theta) * np.cos(phi), r * np.sin(theta) * np.sin(phi), r * np.cos(theta)), axis=1)
    rgb = np.random.random((num_pts, 3)) / 255.0 * SH_C0 + 0.5
    xyz = torch.tensor(xyz).float().cuda()
    M = (max_sh_degree + 1) ** 2
    dist2 = torch.clamp_min(distCUDA2(xyz), 0.0000001)
    op = 0.1 * torch.ones((num_pts, 1), dtype=torch.float, device="cuda")
    p = dict(xyz=xyz, features_dc=((torch.tensor(rgb).float().cuda() - 0.5) / SH_C0).reshape(num_pts, 1, 3),
             features_rest=torch.zeros((num_pts, M - 1, 3), device="cuda"),
             opacity=torch.log(op / (1 - op)), scaling=torch.log(torch.sqrt(dist2))[..., None].repeat(1, 3),
             rotation=torch.tensor([[1.0, 0.0, 0.0, 0.0]], device="cuda").repeat(num_pts, 1))
    return {k: v.contiguous().requires_grad_(True) for k, v in p.items()}


def _render(p, g, H, W, bg):
    """Renderer.render of the original with the stored camera: activations, the rasterizer call by keyword, clamp(0, 1)."""
    import diff_gaussian_rasterization as ours
    screenspace = torch.zeros_like(p["xyz"], requires_grad=True) + 0
    screenspace.retain_grad()
    t = lambda a: torch.tensor(a, device="cuda")
    rs = ours.GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=float(g["tanfov"][0]), tanfovy=float(g["tanfov"][1]), bg=bg,
        scale_modifier=float(g["scaling_modifier"]), viewmatrix=t(g["viewmatrix"]), projmatrix=t(g["projmatrix"]),
        sh_degree=int(g["sh_degree"]), campos=t(g["campos"]), prefiltered=False, debug=False)
    image, radii, depth, alpha = ours.GaussianRasterizer(raster_settings=rs)(
        means3D=p["xyz"], means2D=screenspace, shs=torch.cat((p["features_dc"], p["features_rest"]), dim=1), colors_precomp=None,
        opacities=torch.sigmoid(p["opacity"]), scales=torch.exp(p["scaling"]),
        rotations=torch.nn.functional.normalize(p["rotation"]), cov3D_precomp=None)
    return dict(image=image.clamp(0, 1), depth=depth, alpha=alpha, viewspace_points=screenspace, visibility_filter=radii > 0,
                radii=radii), rs


@pytest.mark.parametrize("name", list(CASES))
def test_reference_renderer_runs_unmodified_on_the_drop_in(name):
    c = CASES[name]
    gz = np.load(GOLDEN)
    g = {k.split("/", 1)[1]: gz[k] for k in gz.files if k.startswith(name + "/")}
    H, W = c["H"], c["W"]

    np.random.seed(7)
    torch.manual_seed(7)
    p = _initialize(c["num_pts"], c["sh_degree"])
    accum, denom = torch.zeros((c["num_pts"], 1), device="cuda"), torch.zeros((c["num_pts"], 1), device="cuda")
    if c["ups"]:
        with torch.no_grad():                                # leave the symmetric initial state: anisotropy, rotations, colour detail
            p["features_rest"].normal_(0.0, 0.1)
            p["scaling"].add_(0.3 * torch.randn_like(p["scaling"]))
            p["rotation"].copy_(torch.randn_like(p["rotation"]))
            p["opacity"].copy_(torch.logit(torch.rand_like(p["opacity"]) * 0.9 + 0.05))
    rows = g["rows"]
    for k, v in p.items():                                   # the Gaussians the original caller rendered (features_rest: first band)
        got = v.detach().cpu().numpy()[rows]
        np.testing.assert_allclose(got[:, :3] if k == "features_rest" else got, g[k], rtol=1e-6, atol=1e-7, err_msg=k)
    assert int(g["sh_degree"]) == min(c["ups"], c["sh_degree"])

    bg = torch.tensor(g["bg"], device="cuda")
    out, rs = _render(p, g, H, W, bg)
    assert out["image"].shape == (3, H, W) and out["alpha"].shape == (1, H, W) and out["depth"].shape == (1, H, W)
    assert out["radii"].dtype == torch.int32 and out["visibility_filter"].dtype == torch.bool

    gC, gD, gA = h.upstream_grads(H, W, seed=5, depth=False)
    t = lambda a: torch.tensor(a, device="cuda")
    loss = (out["image"] * t(gC)).sum() + (out["alpha"] * t(gA)).sum()
    loss.backward()
    vis = out["visibility_filter"]                           # add_densification_stats of the original
    accum[vis] += torch.norm(out["viewspace_points"].grad[vis, :2], dim=-1, keepdim=True)
    denom[vis] += 1

    # ---- the oracle on the very tensors the caller handed to the op
    f64 = lambda x: x.detach().double().cpu().numpy()
    settings = dict(image_height=H, image_width=W, tanfovx=float(g["tanfov"][0]), tanfovy=float(g["tanfov"][1]),
                    bg=np.asarray(g["bg"], np.float64), scale_modifier=float(g["scaling_modifier"]),
                    viewmatrix=np.asarray(g["viewmatrix"], np.float64), projmatrix=np.asarray(g["projmatrix"], np.float64),
                    sh_degree=int(g["sh_degree"]), campos=np.asarray(g["campos"], np.float64))
    raw = {k: f64(v) for k, v in p.items()}
    # clamp(0, 1) of the caller: gradient passes where the un-clamped colour lies in [0, 1] (torch's rule); the un-clamped
    # colour is what one more (deterministic) call of the op with the same tensors returns
    import diff_gaussian_rasterization as ours
    with torch.no_grad():
        pre, radii2, _, _ = ours.GaussianRasterizer(rs)(
            means3D=p["xyz"], means2D=torch.zeros_like(p["xyz"]), shs=torch.cat((p["features_dc"], p["features_rest"]), dim=1),
            opacities=torch.sigmoid(p["opacity"]), scales=torch.exp(p["scaling"]), rotations=torch.nn.functional.normalize(p["rotation"]))
    assert torch.equal(radii2, out["radii"]) and torch.equal(pre.clamp(0, 1), out["image"])
    passes = ((pre >= 0) & (pre <= 1)).cpu().numpy()
    ref = h.run_oracle_raw(settings, raw, (gC * passes, None, gA))
    cu = dict(color=pre.cpu().numpy(), depth=out["depth"].detach().cpu().numpy(), alpha=out["alpha"].detach().cpu().numpy(),
              radii=out["radii"].cpu().numpy(),
              grads=dict(xyz=p["xyz"].grad, features_dc=p["features_dc"].grad, features_rest=p["features_rest"].grad,
                         opacity=p["opacity"].grad, scaling=p["scaling"].grad, rotation=p["rotation"].grad,
                         means2D=out["viewspace_points"].grad))
    cu["grads"] = {k: (v.detach().cpu().numpy() if v is not None else np.zeros(ref["grads"][k].shape, np.float32))
                   for k, v in cu["grads"].items()}
    ok, rep = h.compare(cu, ref, max_ambig_frac=0.10)
    assert ok, rep
    assert int((out["radii"] > 0).sum()) > c["num_pts"] // 2

    # densification statistics as the original's method computes them from OUR viewspace gradient
    vis = ref["radii"] > 0
    want = np.linalg.norm(ref["grads"]["means2D"][:, :2], axis=-1)
    got = accum[:, 0].cpu().numpy()
    clean = (ref["ambig_g"] == 0) & vis
    assert np.abs(got[clean] - want[clean]).max() <= 1e-3 * max(want.max(), 1e-12)
    assert np.array_equal(denom[:, 0].cpu().numpy()[ref["ambig_g"] == 0], vis[ref["ambig_g"] == 0].astype(np.float32))

    # ---- what the original caller got back, at the stored samples (same tolerances as against the oracle)
    px, clean_px = g["px"], ~ref["ambig_px"].astype(bool).reshape(-1)[g["px"]]
    for k in ("image", "alpha", "depth"):
        v = out[k].detach().cpu().numpy()
        d = np.abs(v.reshape(v.shape[0], -1)[:, px] - g[k])[:, clean_px]
        scale = max(1.0, float(np.abs(g[k]).max())) if k == "depth" else 1.0
        assert d.max() / scale <= 2 * h.IMG_ATOL, (k, float(d.max()))
    clean_g = ref["ambig_g"][rows] == 0
    assert np.array_equal(out["radii"].cpu().numpy()[rows][clean_g], g["radii"][clean_g])
    assert np.array_equal(denom[:, 0].cpu().numpy()[rows][clean_g], g["denom"][clean_g])
    acc_scale = max(float(g["xyz_gradient_accum"].max()), 1e-12)
    assert np.abs(got[rows][clean_g] - g["xyz_gradient_accum"][clean_g]).max() <= 2e-3 * acc_scale
