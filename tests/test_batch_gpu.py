"""Batched multi-view rendering on the GPU: a batch of V views must give what V single-view calls give (images and radii per
view, gradients summed over the views, means2D gradients and densification statistics per view), every view must pass both
oracles, and the capacity re-run, accumulate and retain_graph paths must work as they do for one view."""
import numpy as np
import pytest
import torch

import helpers as h
from dreamgaussian_b200 import rasterizer as R
from dreamgaussian_b200 import scene
from dreamgaussian_b200.fused import BatchedFusedGaussianRasterizer, DensifyStats, FusedGaussianRasterizer

pytestmark = pytest.mark.gpu

DEV = "cuda"
PLAIN_KEYS = ("means3D", "shs", "opacities", "scales", "rotations")


def _t(a):
    return torch.tensor(np.asarray(a, np.float32), device=DEV)


def _rs(cam, deg, bg, scale_modifier=1.0):
    return R.GaussianRasterizationSettings(
        image_height=cam.image_height, image_width=cam.image_width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=_t(bg),
        scale_modifier=scale_modifier, viewmatrix=_t(cam.world_view_transform), projmatrix=_t(cam.full_proj_transform), sh_degree=deg,
        campos=_t(cam.camera_center), prefiltered=False, debug=False)


def _away_camera(W, H):
    """A camera at distance 2 looking AWAY from the cloud (radius 0.5 around the origin): it culls everything."""
    pose = scene.orbit_pose(0.0, 0.0, 2.0)
    pose[:3, 0] *= -1.0
    pose[:3, 2] *= -1.0
    return scene.make_camera(pose, W, H)


def _views(V, W, H, deg, away=None, scale_modifier=1.0):
    cams = scene.bench_views(V, W, H)
    if away is not None:
        cams[away] = _away_camera(W, H)
    rng = np.random.default_rng(V)
    return [_rs(c, deg, rng.random(3), scale_modifier) for c in cams]


def _upstream(V, H, W, seed=11):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn((V, 3, H, W), device=DEV, generator=g), torch.randn((V, 1, H, W), device=DEV, generator=g),
            torch.randn((V, 1, H, W), device=DEV, generator=g))


def _loss(color, depth, alpha, up):
    return (color * up[0]).sum() + (depth * up[1]).sum() + (alpha * up[2]).sum()


def run_loop(sets, params, up, raw=False, stats=None):
    """V single-view calls, each backward adding into the same leaves (what a Python loop over views does)."""
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    imgs, m2d = [], []
    for v, rs in enumerate(sets):
        m = torch.zeros((params["xyz" if raw else "means3D"].shape[0], 3), device=DEV, requires_grad=True)
        if raw:
            out = FusedGaussianRasterizer(rs)(leaves["xyz"], leaves["features_dc"], leaves["features_rest"], leaves["opacity"],
                                              leaves["scaling"], leaves["rotation"], means2D=m, stats=stats)
        else:
            out = R.GaussianRasterizer(rs)(means3D=leaves["means3D"], means2D=m, shs=leaves["shs"], opacities=leaves["opacities"],
                                           scales=leaves["scales"], rotations=leaves["rotations"])
        color, radii, depth, alpha = out
        _loss(color, depth, alpha, (up[0][v], up[1][v], up[2][v])).backward()
        imgs.append((color.detach(), radii, depth.detach(), alpha.detach()))
        m2d.append(m.grad)
    grads = {k: (l.grad if l.grad is not None else torch.zeros_like(l)) for k, l in leaves.items()}
    return dict(color=torch.stack([i[0] for i in imgs]), radii=torch.stack([i[1] for i in imgs]), depth=torch.stack([i[2] for i in imgs]),
                alpha=torch.stack([i[3] for i in imgs]), grads=grads, means2D=torch.stack(m2d))


def run_batch(sets, params, up, raw=False, stats=None, retain=False):
    leaves = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    P = params["xyz" if raw else "means3D"].shape[0]
    m = torch.zeros((len(sets), P, 3), device=DEV, requires_grad=True)
    if raw:
        out = BatchedFusedGaussianRasterizer(sets)(leaves["xyz"], leaves["features_dc"], leaves["features_rest"], leaves["opacity"],
                                                   leaves["scaling"], leaves["rotation"], means2D=m, stats=stats)
    else:
        out = R.BatchedGaussianRasterizer(sets)(leaves["means3D"], leaves["opacities"], leaves["shs"], leaves["scales"], leaves["rotations"],
                                                means2D=m)
    color, radii, depth, alpha = out
    for o, shape in ((color, (3,)), (depth, (1,)), (alpha, (1,))):
        assert o.is_contiguous() and tuple(o.shape) == (len(sets),) + shape + tuple(color.shape[-2:])
    assert radii.dtype == torch.int32 and tuple(radii.shape) == (len(sets), P) and radii.is_contiguous()
    loss = _loss(color, depth, alpha, up)
    names = list(leaves)
    first = torch.autograd.grad(loss, [leaves[k] for k in names] + [m], retain_graph=retain, allow_unused=True)
    res = dict(color=color.detach(), radii=radii, depth=depth.detach(), alpha=alpha.detach(),
               grads={k: (g if g is not None else torch.zeros_like(leaves[k])) for k, g in zip(names, first[:-1])}, means2D=first[-1])
    if retain:
        second = torch.autograd.grad(loss, [leaves[k] for k in names] + [m], allow_unused=True)
        res["second"] = ({k: (g if g is not None else torch.zeros_like(leaves[k])) for k, g in zip(names, second[:-1])}, second[-1])
    return res


def _grad_check(got, want, tol, outliers):
    """Per-Gaussian max |got - want| against tol x the tensor's scale: at most `outliers` x P Gaussians above it, all below 2e-2."""
    scale = float(want.abs().max())
    err = (got - want).abs().reshape(want.shape[0], -1).max(dim=1).values if want.numel() else want.reshape(-1)
    n_bad = int((err > tol * scale + 1e-12).sum())
    worst = float(err.max()) / (scale + 1e-30) if err.numel() else 0.0
    ok = n_bad <= int(outliers * want.shape[0]) and worst <= (2e-2 if outliers else tol)
    return ok, dict(outliers=n_bad, of=int(want.shape[0]), worst_rel=worst)


def assert_equivalent(loop, batch, V, grad_outliers=0.0):
    """grad_outliers: fraction of Gaussians whose gradient may exceed the bound (up to 2e-2 of the scale).  Needed only where float32
    view depths of consecutive contributors tie (configs[2]: ~2000-entry pixel lists): a last-bit difference of a record's depth
    from per-instantiation FMA fusion may flip such a pair, which changes the gradients of the Gaussians involved."""
    for k in ("color", "depth", "alpha"):
        for v in range(V):
            a, b = loop[k][v].cpu().numpy(), batch[k][v].cpu().numpy()
            d = np.abs(a - b) / max(1.0, float(np.abs(a).max()))
            assert float((d > 2e-6).mean()) <= 1e-4 and float(d.max()) <= 1e-2, (k, v, float(d.max()), float((d > 2e-6).mean()))
    for v in range(V):
        assert int((loop["radii"][v] != batch["radii"][v]).sum()) <= 2, v
    for k, want in loop["grads"].items():                      # float atomics: summation order differs
        ok, rep = _grad_check(batch["grads"][k], want, 2e-4, grad_outliers)
        assert ok, (k, rep)
    for v in range(V):
        ok, rep = _grad_check(batch["means2D"][v], loop["means2D"][v], 2e-5, grad_outliers)
        assert ok, ("means2D", v, rep)


def _plain(P, deg, seed=0, sigma=0.04):
    return {k: _t(v) for k, v in scene.make_cloud(P, deg, seed=seed, sigma=sigma).items()}


def _raw(P, deg, seed=0, sigma=0.04):
    return {k: _t(v) for k, v in scene.to_raw_parameters(scene.make_cloud(P, deg, seed=seed, sigma=sigma)).items()}


CASES = {
    "plain_deg0": dict(P=3001, W=96, H=96, deg=0, V=4),
    "plain_deg3": dict(P=5000, W=128, H=128, deg=3, V=3),
    "odd_size_deg1": dict(P=2500, W=100, H=70, deg=1, V=5),                     # P and H, W off the warp / tile grid
    "one_view": dict(P=2000, W=64, H=64, deg=3, V=1),
    "sixteen_views": dict(P=3000, W=64, H=64, deg=1, V=16),
    "one_view_culls_all": dict(P=4000, W=80, H=80, deg=2, V=4, away=2),
    "scale_modifier": dict(P=1500, W=72, H=72, deg=2, V=3, scale_modifier=1.3),
}


@pytest.mark.parametrize("name", list(CASES))
def test_batch_equals_loop_of_single_views(name):
    c = CASES[name]
    params = _plain(c["P"], c["deg"], seed=3)
    sets = _views(c["V"], c["W"], c["H"], c["deg"], away=c.get("away"), scale_modifier=c.get("scale_modifier", 1.0))
    up = _upstream(c["V"], c["H"], c["W"])
    loop, batch = run_loop(sets, params, up), run_batch(sets, params, up)
    if "away" in c:
        assert int(batch["radii"][c["away"]].max()) == 0 and int(batch["radii"].max()) > 0
    assert_equivalent(loop, batch, c["V"])


def test_batch_raw_path_with_densify_stats_equals_loop():
    P, W, H, deg, V = 4001, 100, 70, 3, 4
    params = _raw(P, deg, seed=5)
    sets = _views(V, W, H, deg)
    up = _upstream(V, H, W)
    s_loop, s_batch = DensifyStats(P, DEV), DensifyStats(P, DEV)
    s_loop.max_radii2D.fill_(2.0); s_batch.max_radii2D.fill_(2.0)
    loop = run_loop(sets, params, up, raw=True, stats=s_loop)
    batch = run_batch(sets, params, up, raw=True, stats=s_batch)
    assert_equivalent(loop, batch, V)
    same = (loop["radii"] == batch["radii"]).all(dim=0)                 # Gaussians whose radii agree in every view
    assert int((~same).sum()) <= 2 * V
    assert torch.equal(s_batch.denom[same], s_loop.denom[same])
    assert torch.equal(s_batch.max_radii2D[same], s_loop.max_radii2D[same])
    tol = 1e-4 * float(s_loop.xyz_gradient_accum.max())
    assert float((s_batch.xyz_gradient_accum[same] - s_loop.xyz_gradient_accum[same]).abs().max()) <= tol
    vis = (batch["radii"] > 0).sum(dim=0).float()
    assert torch.equal(s_batch.denom, vis)


def test_batch_padded_sh_storage_with_lower_active_degree():
    P, W, H, V = 1800, 72, 72, 3
    params = _plain(P, 1, seed=2)
    rng = np.random.default_rng(4)
    params["shs"] = torch.cat([params["shs"], _t(rng.normal(size=(P, 12, 3)))], dim=1)        # M = 16, 4 in use
    sets = _views(V, W, H, 1)
    up = _upstream(V, H, W)
    loop, batch = run_loop(sets, params, up), run_batch(sets, params, up)
    assert_equivalent(loop, batch, V)
    assert tuple(batch["grads"]["shs"].shape) == (P, 16, 3) and not batch["grads"]["shs"][:, 4:].any()


def test_batch_of_an_empty_cloud():
    sets = _views(3, 40, 40, 0)
    z = lambda *shape: torch.zeros(*shape, device=DEV, requires_grad=True)
    leaves = [z(0, 3), z(0, 1), z(0, 1, 3), z(0, 3), z(0, 4)]
    color, radii, depth, alpha = R.BatchedGaussianRasterizer(sets)(*leaves)
    assert tuple(radii.shape) == (3, 0) and float(alpha.abs().max()) == 0.0 and float(depth.abs().max()) == 0.0
    for v, rs in enumerate(sets):
        assert torch.allclose(color[v], rs.bg[:, None, None].expand_as(color[v]))
    (color.sum() + alpha.sum()).backward()
    assert all(l.grad is not None and l.grad.numel() == 0 for l in leaves)


def test_every_view_of_a_batch_passes_both_oracles():
    """Each view's images / radii and, with the upstream gradient of that view alone, its gradients, against the float64 and the
    float32 CPU oracle (the rule of tests/test_parity_gpu.py)."""
    P, res, deg, V = 1500, 64, 3, 3
    cloud = scene.make_cloud(P, deg, seed=9, sigma=0.04)
    cams = scene.bench_views(V, res, res)
    params = {k: _t(v) for k, v in cloud.items()}
    sets = [_rs(c, deg, np.full(3, 0.25 * (i + 1))) for i, c in enumerate(cams)]
    for v, cam in enumerate(cams):
        s = dict(image_height=res, image_width=res, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=np.full(3, 0.25 * (v + 1), np.float32),
                 scale_modifier=1.0, viewmatrix=cam.world_view_transform, projmatrix=cam.full_proj_transform, sh_degree=deg,
                 campos=cam.camera_center)
        g = h.upstream_grads(res, res, seed=40 + v)
        up = [torch.zeros((V, 3, res, res), device=DEV), torch.zeros((V, 1, res, res), device=DEV), torch.zeros((V, 1, res, res), device=DEV)]
        for j in range(3):
            up[j][v] = _t(g[j])
        b = run_batch(sets, params, up)
        cu = dict(color=b["color"][v].cpu().numpy(), depth=b["depth"][v].cpu().numpy(), alpha=b["alpha"][v].cpu().numpy(),
                  radii=b["radii"][v].cpu().numpy(), grads={k: b["grads"][k].cpu().numpy() for k in PLAIN_KEYS})
        cu["grads"]["means2D"] = b["means2D"][v].cpu().numpy()
        ok32, rep32 = h.compare_f32(cu, h.run_oracle(s, cloud, g, dtype=np.float32))
        ok64, rep64 = h.compare(cu, h.run_oracle(s, cloud, g))
        h.report("batch_view%d" % v, vs_f64=rep64, vs_f32=rep32)
        assert ok64, (v, "float64 oracle", rep64)
        assert ok32, (v, "float32 oracle", rep32)


def test_cfg3_full_size_batch_equals_loop():
    """BASELINE.json configs[2]: 500k Gaussians, 512x512, SH degree 3, the 8 benchmark views.  Float32 depth ties between consecutive
    contributors occur here (DESIGN.md §2), so gradients follow the outlier rule of helpers.compare_f32 (<= 2e-4 of the Gaussians)."""
    P, res, deg, V = 500000, 512, 3, 8
    params = {k: _t(v) for k, v in scene.make_cloud(P, deg, seed=0, sigma=0.0075).items()}
    sets = [_rs(c, deg, np.ones(3)) for c in scene.bench_views(V, res, res)]
    up = _upstream(V, res, res, seed=3)
    up = (up[0], torch.zeros_like(up[1]), up[2])
    assert_equivalent(run_loop(sets, params, up), run_batch(sets, params, up), V, grad_outliers=2e-4)


def test_batch_capacity_guess_too_small_is_repaired():
    P, res, deg, V = 3000, 128, 1, 4
    params = _plain(P, deg, seed=1, sigma=0.05)
    sets = _views(V, res, res, deg)
    args = (params["means3D"], params["shs"], params["opacities"], params["scales"], params["rotations"])
    color, radii, depth, alpha, state = R.forward_batch_impl(sets, *args)
    ref = [o.clone() for o in (color, radii, depth, alpha)]
    key = (torch.cuda.current_device(), P, res, res)
    counts = sorted(state.num_rendered)
    assert counts[0] < counts[-1]
    for cap, big in ((counts[-1] - 1, True), (64, False)):       # only the largest view re-runs / every view re-runs
        R.set_capacity_hint(*key, cap, big)
        out = R.forward_batch_impl(sets, *args)
        for a, b in zip(ref, out[:4]):
            assert torch.equal(a, b)
        assert R.get_capacity_hint(*key)[0] > cap
        assert out[4].capacities.count(cap) == sum(1 for n in out[4].num_rendered if n <= cap)


def test_batch_backward_accumulate_adds_into_the_buffers():
    P, res, deg, V = 2500, 80, 2, 3
    params = _plain(P, deg, seed=6)
    sets = _views(V, res, res, deg)
    args = (params["means3D"], params["shs"], params["opacities"], params["scales"], params["rotations"])
    *_, state = R.forward_batch_impl(sets, *args)
    f = lambda *shape: torch.empty(shape, device=DEV)
    shapes = [(P, 3), (V, P, 3), (P, 9, 3), (P, 1), (P, 3), (P, 4)]
    ups = [_upstream(V, res, res, seed=s) for s in (1, 2)]
    single = []
    for up in ups:
        bufs = [f(*s) for s in shapes]
        R.backward_batch_impl(state, *up, *bufs)
        single.append(bufs)
    bufs = [f(*s) for s in shapes]
    R.backward_batch_impl(state, *ups[0], *bufs)
    R.backward_batch_impl(state, *ups[1], *bufs, accumulate=True)
    for a, b, c in zip(single[0], single[1], bufs):
        scale = float((a + b).abs().max())
        assert float((a + b - c).abs().max()) <= 2e-5 * scale + 1e-12


def test_batch_backward_twice_of_one_forward_gives_the_same_gradients():
    P, res, deg, V = 4000, 96, 2, 3
    params = _raw(P, deg, seed=8)
    sets = _views(V, res, res, deg)
    stats = DensifyStats(P, DEV)
    b = run_batch(sets, params, _upstream(V, res, res), raw=True, stats=stats, retain=True)
    grads2, m2d2 = b["second"]
    for k, a in b["grads"].items():
        scale = float(a.abs().max()) + 1e-20
        assert float((a - grads2[k]).abs().max()) <= 2e-5 * scale, k
    assert float((b["means2D"] - m2d2).abs().max()) <= 2e-5 * (float(b["means2D"].abs().max()) + 1e-20)
    assert torch.equal(stats.denom, (b["radii"] > 0).sum(dim=0).float())       # the second backward does not count the views again
