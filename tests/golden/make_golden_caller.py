"""Generate tests/golden/reference_caller_vectors.npz: what the original project's own caller (gs_renderer.Renderer,
GaussianModel, MiniCam; cam_utils.OrbitCamera / orbit_camera) hands to the rasterizer and what it derives from the result,
on the cases of tests/test_reference_caller_gpu.py.  Needs a GPU and the original caller (oracle/ref_caller.py).

Per case `<case>/...`:
  * the call: viewmatrix, projmatrix, campos, tanfov (x, y), bg, sh_degree, scaling_modifier;
  * the Gaussians the caller rendered (initialisation + the test's perturbation), at a fixed, seeded sample of `rows`:
    xyz, features_dc, features_rest (first band), opacity, scaling, rotation (raw parameters);
  * what the caller returned, at the same rows: radii, xyz_gradient_accum, denom; and at a fixed sample of pixels `px`
    (flat index into H x W): image (clamped), alpha, depth.
`imports`: the names the original caller binds from the drop-in packages, as "<module>:<name>".

  python tests/golden/make_golden_caller.py [OUT.npz]
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

ROWS = 512
PIXELS = 4096


def run_case(name, c, cam_utils, gs):
    import torch
    import helpers as h
    from test_reference_caller_gpu import _training_args
    np.random.seed(7)
    torch.manual_seed(7)
    r = gs.Renderer(sh_degree=c["sh_degree"])
    r.initialize(num_pts=c["num_pts"])
    gm = r.gaussians
    gm.training_setup(_training_args())
    for _ in range(c["ups"]):
        gm.oneupSHdegree()
    if c["ups"]:
        with torch.no_grad():
            gm._features_rest.normal_(0.0, 0.1)
            gm._scaling.add_(0.3 * torch.randn_like(gm._scaling))
            gm._rotation.copy_(torch.randn_like(gm._rotation))
            gm._opacity.copy_(torch.logit(torch.rand_like(gm._opacity) * 0.9 + 0.05))
    oc = cam_utils.OrbitCamera(c["W"], c["H"], r=2, fovy=49.1)
    cam = gs.MiniCam(cam_utils.orbit_camera(c["elev"], c["azim"], 2), c["W"], c["H"], oc.fovy, oc.fovx, oc.near, oc.far)
    bg = None if c["bg"] is None else torch.tensor(c["bg"], dtype=torch.float32, device="cuda")
    out = r.render(cam, scaling_modifier=c["scaling_modifier"], bg_color=bg)
    H, W = c["H"], c["W"]
    gC, gD, gA = h.upstream_grads(H, W, seed=5, depth=False)
    t = lambda a: torch.tensor(a, device="cuda")
    ((out["image"] * t(gC)).sum() + (out["alpha"] * t(gA)).sum()).backward()
    gm.add_densification_stats(out["viewspace_points"], out["visibility_filter"])

    f32 = lambda x: x.detach().float().cpu().numpy()
    P = gm.get_xyz.shape[0]
    rows = np.sort(np.random.default_rng(11).choice(P, min(ROWS, P), replace=False))
    px = np.sort(np.random.default_rng(12).choice(H * W, min(PIXELS, H * W), replace=False))
    bg_used = r.bg_color if bg is None else bg
    d = dict(viewmatrix=f32(cam.world_view_transform), projmatrix=f32(cam.full_proj_transform), campos=f32(cam.camera_center),
             tanfov=np.array([np.tan(cam.FoVx * 0.5), np.tan(cam.FoVy * 0.5)], np.float64), bg=f32(bg_used),
             sh_degree=np.int32(gm.active_sh_degree), scaling_modifier=np.float64(c["scaling_modifier"]),
             rows=rows.astype(np.int32), px=px.astype(np.int32))
    for k in ("xyz", "features_dc", "features_rest", "opacity", "scaling", "rotation"):
        d[k] = f32(getattr(gm, "_" + k))[rows]
    d["features_rest"] = d["features_rest"][:, :3]          # first band only: pins the perturbation at a fraction of the size
    d["radii"] = out["radii"].cpu().numpy()[rows].astype(np.int32)
    d["xyz_gradient_accum"] = f32(gm.xyz_gradient_accum)[rows, 0]
    d["denom"] = f32(gm.denom)[rows, 0]
    for k in ("image", "alpha", "depth"):
        v = f32(out[k])
        d[k] = v.reshape(v.shape[0], -1)[:, px]
    return {"%s/%s" % (name, k): v for k, v in d.items()}


def main(out):
    import diff_gaussian_rasterization
    import simple_knn._C
    from oracle import ref_caller
    from test_reference_caller_gpu import CASES
    assert ref_caller.available(), "the original caller is not available (oracle/ref_caller.py)"
    cam_utils, gs, _ = ref_caller.load()
    imports = sorted("%s:%s" % (m.__name__, n) for m in (diff_gaussian_rasterization, simple_knn._C)
                     for n, v in vars(gs).items() if not n.startswith("_") and hasattr(m, n) and getattr(m, n) is v)
    data = {"imports": np.array(imports)}
    for name, c in CASES.items():
        data.update(run_case(name, c, cam_utils, gs))
    np.savez_compressed(out, **data)
    print("wrote", out, imports)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_caller_vectors.npz"))
