"""SURVEY.md §8 row f1: the rasterizer taking GaussianModel's RAW parameters, activations fused into the kernels.

The reference renders with (gs_renderer.py:196-216, :762-806)

    means3D = _xyz;  opacity = sigmoid(_opacity);  scales = exp(_scaling);  rotations = F.normalize(_rotation)
    shs = torch.cat((_features_dc, _features_rest), dim=1)

i.e. four element-wise passes over the parameters, a 12·M-byte-per-Gaussian concatenation copy, and the mirror-image
passes in the backward — then, after the optimiser step (main.py:279-281, gs_renderer.py:625-627),

    max_radii2D[vis] = max(max_radii2D[vis], radii[vis]);  xyz_gradient_accum[vis] += |means2D.grad[vis, :2]|;  denom[vis] += 1

Here the per-Gaussian kernels read the raw tensors directly (`DgrGaussians.activations`), apply the activations in
registers, return gradients with respect to the raw tensors, and update the three densification statistics in the same
backward kernel.  Same C ABI entry points as the plain path (include/dgr_b200.h)."""
from typing import Optional

import torch
import torch.nn as nn

from . import rasterizer as _r


class DensifyStats:
    """The three per-Gaussian statistics of the reference's densification (float32 [P]; the reference keeps [P,1] / [P])."""

    def __init__(self, P: int, device):
        self.xyz_gradient_accum = torch.zeros((P,), dtype=torch.float32, device=device)
        self.denom = torch.zeros((P,), dtype=torch.float32, device=device)
        self.max_radii2D = torch.zeros((P,), dtype=torch.float32, device=device)

    def as_tuple(self):
        return (self.xyz_gradient_accum, self.denom, self.max_radii2D)


class _RasterizeRaw(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, means2D, features_dc, features_rest, opacity_raw, scaling_raw, rotation_raw, raster_settings, stats):
        if _r._FAST is not None:
            color, radii, depth, alpha, state = _r.forward_impl(raster_settings, xyz, features_dc, None, opacity_raw, scaling_raw, rotation_raw,
                                                                None, sh_rest=features_rest, activations=True)
            ctx.state, ctx.stats = state, stats
            ctx.mark_non_differentiable(radii)
            return color, radii, depth, alpha
        xyz = _r._dev_f32(xyz, "xyz")
        dc = _r._dev_f32(features_dc, "features_dc")
        rest = _r._opt(features_rest, "features_rest")
        if rest is not None and rest.numel() == 0:
            rest = None
        op, sc, rot = _r._dev_f32(opacity_raw, "opacity"), _r._dev_f32(scaling_raw, "scaling"), _r._dev_f32(rotation_raw, "rotation")
        color, radii, depth, alpha, state = _r.forward_impl(raster_settings, xyz, dc, None, op, sc, rot, None, sh_rest=rest,
                                                            activations=True)
        ctx.state, ctx.stats = state, stats
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha):
        state = ctx.state
        # the statistics describe the RENDER, not the backward call: a retain_graph / second backward of the same forward
        # must not count the view twice (gs_renderer.py:625-627 runs once per render)
        if getattr(state, "stats_applied", False):
            ctx.stats = None
        state.stats_applied = True
        if state.fast is not None:
            stats = ctx.stats.as_tuple() if ctx.stats is not None else (None, None, None)
            g = _r._FAST.backward(state.fast, grad_color, grad_depth, grad_alpha, False, [], *stats)
            return g[0], g[1], g[2], g[8], g[4], g[5], g[6], None, None
        xyz, dc, _, op, sc, rot, _, rest = state.tensors
        P = state.frame.P
        f32 = dict(dtype=torch.float32, device=xyz.device)
        gC = _r._dev_f32(grad_color, "grad_color") if grad_color is not None else None
        gD = _r._dev_f32(grad_depth, "grad_depth") if grad_depth is not None else None
        gA = _r._dev_f32(grad_alpha, "grad_alpha") if grad_alpha is not None else None
        d_xyz, d_m2d = torch.empty((P, 3), **f32), torch.empty((P, 3), **f32)
        d_dc = torch.empty((P, 1, 3), **f32)
        d_rest = torch.empty(rest.shape, **f32) if rest is not None else None
        d_op, d_sc, d_rot = torch.empty((P, 1), **f32), torch.empty((P, 3), **f32), torch.empty((P, 4), **f32)
        stats = ctx.stats.as_tuple() if ctx.stats is not None else None
        _r.backward_impl(state, gC, gD, gA, d_xyz, d_m2d, d_dc, None, d_op, d_sc, d_rot, None, d_sh_rest=d_rest, densify=stats)
        return d_xyz, d_m2d, d_dc, d_rest, d_op, d_sc, d_rot, None, None


class FusedGaussianRasterizer(nn.Module):
    """`GaussianRasterizer` for raw parameters.  forward(xyz, features_dc, features_rest, opacity, scaling, rotation,
    means2D=None, stats=None) -> (color [3,H,W], radii int32 [P], depth [1,H,W], alpha [1,H,W]); `stats` (DensifyStats) is
    updated during the backward."""

    def __init__(self, raster_settings: _r.GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def forward(self, xyz, features_dc, features_rest, opacity, scaling, rotation, means2D: Optional[torch.Tensor] = None,
                stats: Optional[DensifyStats] = None):
        if means2D is None:
            means2D = torch.zeros_like(xyz, requires_grad=xyz.requires_grad)
        return _RasterizeRaw.apply(xyz, means2D, features_dc, features_rest, opacity, scaling, rotation, self.raster_settings, stats)


def render_gaussian_model(gaussians, raster_settings, stats: Optional[DensifyStats] = None):
    """Renders an object with the reference GaussianModel's attribute names (_xyz, _features_dc, _features_rest, _opacity,
    _scaling, _rotation: gs_renderer.py:140-160).  Returns the reference Renderer.render's dict (gs_renderer.py:812-822)."""
    xyz = gaussians._xyz
    means2D = torch.zeros_like(xyz, requires_grad=True)
    color, radii, depth, alpha = FusedGaussianRasterizer(raster_settings)(
        xyz, gaussians._features_dc, gaussians._features_rest, gaussians._opacity, gaussians._scaling, gaussians._rotation,
        means2D=means2D, stats=stats)
    return {"image": color.clamp(0, 1), "depth": depth, "alpha": alpha, "viewspace_points": means2D,
            "visibility_filter": radii > 0, "radii": radii}


class _RasterizeRawBatch(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, means2D, features_dc, features_rest, opacity_raw, scaling_raw, rotation_raw, settings_list, stats):
        xyz = _r._dev_f32(xyz, "xyz")
        dc = _r._dev_f32(features_dc, "features_dc")
        rest = _r._opt(features_rest, "features_rest")
        if rest is not None and rest.numel() == 0:
            rest = None
        op, sc, rot = _r._dev_f32(opacity_raw, "opacity"), _r._dev_f32(scaling_raw, "scaling"), _r._dev_f32(rotation_raw, "rotation")
        color, radii, depth, alpha, state = _r.forward_batch_impl(settings_list, xyz, dc, op, sc, rot, sh_rest=rest, activations=True)
        ctx.state, ctx.stats = state, stats
        ctx.rest_shape = None if features_rest is None else tuple(features_rest.shape)
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha):
        state = ctx.state
        # the statistics describe the RENDERS: a retain_graph / second backward must not count the views twice
        stats = ctx.stats if not getattr(state, "stats_applied", False) else None
        state.stats_applied = True
        xyz, dc, op, sc, rot, rest = state.tensors
        V, P = state.frame.V, state.frame.P
        f32 = dict(dtype=torch.float32, device=xyz.device)
        d_xyz, d_m2d = torch.empty((P, 3), **f32), torch.empty((V, P, 3), **f32)
        d_dc = torch.empty((P, 1, 3), **f32)
        d_rest = torch.empty(rest.shape, **f32) if rest is not None else None
        d_op, d_sc, d_rot = torch.empty((P, 1), **f32), torch.empty((P, 3), **f32), torch.empty((P, 4), **f32)
        _r.backward_batch_impl(state, *_r._batch_grads(state, grad_color, grad_depth, grad_alpha), d_xyz, d_m2d, d_dc, d_op, d_sc, d_rot,
                               d_sh_rest=d_rest, densify=stats.as_tuple() if stats is not None else None)
        if d_rest is None and ctx.rest_shape is not None:
            d_rest = torch.zeros(ctx.rest_shape, **f32)
        return d_xyz, d_m2d, d_dc, d_rest, d_op, d_sc, d_rot, None, None


class BatchedFusedGaussianRasterizer(nn.Module):
    """`BatchedGaussianRasterizer` for raw parameters: V views (1 to 16) of one GaussianModel in one call.
    forward(xyz, features_dc, features_rest, opacity, scaling, rotation, means2D=None, stats=None) -> (color [V,3,H,W],
    radii int32 [V,P], depth [V,1,H,W], alpha [V,1,H,W]).  Gradients of the raw tensors are summed over the views; means2D, when
    given, is [V,P,3] and receives each view's screen-space gradient; `stats` (DensifyStats) is updated once per view, as V
    single-view renders would update it."""

    def __init__(self, settings_list):
        super().__init__()
        self.settings_list = _r.check_batch_settings(settings_list)

    def forward(self, xyz, features_dc, features_rest, opacity, scaling, rotation, means2D: Optional[torch.Tensor] = None,
                stats: Optional[DensifyStats] = None):
        V = len(self.settings_list)
        if means2D is None:
            means2D = torch.zeros((V,) + tuple(xyz.shape), dtype=torch.float32, device=xyz.device, requires_grad=xyz.requires_grad)
        elif tuple(means2D.shape) != (V,) + tuple(xyz.shape):
            raise ValueError("means2D must have dimensions (num_views, num_points, 3)")
        return _RasterizeRawBatch.apply(xyz, means2D, features_dc, features_rest, opacity, scaling, rotation, self.settings_list, stats)
