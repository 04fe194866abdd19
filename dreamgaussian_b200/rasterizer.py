"""Host-side mirror of the reference's rasterizer operator: ``GaussianRasterizationSettings`` / ``GaussianRasterizer``.

Drop-in for the import at /root/reference/gs_renderer.py:10-13 and the call at gs_renderer.py:745-809:

    rasterizer = GaussianRasterizer(raster_settings=GaussianRasterizationSettings(...12 fields...))
    color, radii, depth, alpha = rasterizer(means3D=, means2D=, shs=, colors_precomp=, opacities=,
                                            scales=, rotations=, cov3D_precomp=)

Same names, argument meaning, return shapes/dtypes (color [3,H,W], radii int32 [P], depth [1,H,W], alpha [1,H,W]) and
error behaviour (the two "Please provide ..." exceptions) as the un-vendored package the reference imports [EXT].
All arithmetic runs in libdgr_b200.so (hand-written sm_100a CUDA) through the C ABI of include/dgr_b200.h; torch is
used for device memory, the current stream and autograd plumbing only.  There is no CPU path: non-CUDA tensors raise.
"""
import ctypes
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

from . import _lib


def _load_fast():
    """The compiled host layer (csrc/dgr_torch.cpp -> lib/dgr_torch_host.so): same C-ABI calls, ~10x less host time per
    call than ctypes.  Optional: without it (or with DGR_NO_FASTHOST=1) the ctypes path below does the same work."""
    import importlib.util
    import os
    if os.environ.get("DGR_NO_FASTHOST") == "1":
        return None
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "dgr_torch_host.so")
    if not os.path.exists(path):
        return None
    try:
        from . import build as _build
        if not os.path.exists(_build.HOST_HASH) or open(_build.HOST_HASH).read().strip() != _build._host_hash():
            import warnings
            warnings.warn("dgr_torch_host.so is stale (csrc/dgr_torch.cpp or include/dgr_b200.h changed since it was built): "
                          "using the ctypes host layer; run dreamgaussian_b200/build.py", RuntimeWarning)
            return None
        _lib.load()
        spec = importlib.util.spec_from_file_location("dgr_torch_host", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod if mod.abi_version() == _lib.ABI_VERSION else None
    except Exception as e:  # noqa: BLE001  (a torch / compiler mismatch: fall back to ctypes, never to a CPU path)
        import warnings
        warnings.warn("dgr_torch_host.so could not be loaded (%r): using the ctypes host layer" % (e,), RuntimeWarning)
        return None


_FAST = _load_fast()


def set_fast_host(enabled: bool):
    """Switch between the compiled host layer and the ctypes one (tests exercise both)."""
    global _FAST
    _FAST = _load_fast() if enabled else None
    return _FAST is not None


def get_capacity_hint(device_index, P, H, W):
    if _FAST is not None:
        return _FAST.get_hint(device_index, P, H, W)
    return _CAPACITY_HINT.get((device_index, P, H, W))


def set_capacity_hint(device_index, P, H, W, cap, big):
    if _FAST is not None:
        _FAST.set_hint(device_index, P, H, W, cap, big)
    else:
        _CAPACITY_HINT[(device_index, P, H, W)] = (cap, big)


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _dev_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError(
            "%s is on %s: this rasterizer has no CPU path (it runs as sm_100a CUDA kernels in libdgr_b200.so)" % (name, t.device))
    if t.dtype != torch.float32:
        t = t.float()
    return _aligned16(t.contiguous())


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """The kernels read rotations / SH rows with 128-bit loads and stage their inputs with bulk TMA: a contiguous view that starts
    off a 16-byte boundary (e.g. ``flat[1:].view(P, 4)``) gets its own allocation, which is aligned."""
    if t.numel() > 0 and t.data_ptr() % 16 != 0:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


def _opt(t, name):
    if t is None or (isinstance(t, torch.Tensor) and t.numel() == 0 and t.dim() <= 1):
        return None
    return _dev_f32(t, name)


class _Frame:
    """ctypes views of one forward call's settings + inputs (keeps the tensors alive)."""

    def __init__(self, rs: GaussianRasterizationSettings, means3D, sh, colors_precomp, opacities, scales, rotations, cov3D,
                 sh_rest=None, activations=False):
        self.keep = []
        k = self.keep.append
        self.bg = _dev_f32(rs.bg, "bg"); k(self.bg)
        self.view = _dev_f32(rs.viewmatrix, "viewmatrix"); k(self.view)
        self.proj = _dev_f32(rs.projmatrix, "projmatrix"); k(self.proj)
        self.campos = _dev_f32(rs.campos, "campos"); k(self.campos)
        if self.bg.numel() != 3 or self.view.numel() != 16 or self.proj.numel() != 16 or self.campos.numel() != 3:
            raise ValueError("bg/campos must have 3 elements, viewmatrix/projmatrix 16")
        self.settings = _lib.DgrSettings(
            int(rs.image_height), int(rs.image_width), float(rs.tanfovx), float(rs.tanfovy), float(rs.scale_modifier),
            int(rs.sh_degree), int(bool(rs.prefiltered)), int(bool(rs.debug)),
            _ptr(self.bg), _ptr(self.view), _ptr(self.proj), _ptr(self.campos))
        if means3D.dim() != 2 or means3D.shape[1] != 3:
            raise ValueError("means3D must have dimensions (num_points, 3)")
        P = means3D.shape[0]
        M = 0
        if sh is not None:
            if sh.dim() != 3 or sh.shape[0] != P or sh.shape[2] != 3:
                raise ValueError("shs must have dimensions (num_points, num_coeffs, 3)")
            M = sh.shape[1]
        if activations:
            # raw GaussianModel parameters: sh = _features_dc [P,1,3], sh_rest = _features_rest [P,M-1,3]
            if sh is None or sh.shape[1] != 1:
                raise ValueError("features_dc must have dimensions (num_points, 1, 3)")
            if sh_rest is not None and sh_rest.numel() > 0:
                if sh_rest.dim() != 3 or sh_rest.shape[0] != P or sh_rest.shape[2] != 3:
                    raise ValueError("features_rest must have dimensions (num_points, num_coeffs - 1, 3)")
                M = 1 + sh_rest.shape[1]
            else:
                sh_rest = None
        for t, n, w in ((colors_precomp, "colors_precomp", 3), (scales, "scales", 3), (rotations, "rotations", 4), (cov3D, "cov3D_precomp", 6)):
            if t is not None and (t.numel() != P * w):
                raise ValueError("%s must have dimensions (num_points, %d)" % (n, w))
        if opacities.numel() != P:
            raise ValueError("opacities must have dimensions (num_points, 1)")
        self.P, self.M = P, M
        self.gaussians = _lib.DgrGaussians(P, M, _ptr(means3D), _ptr(sh), _ptr(colors_precomp), _ptr(opacities),
                                           _ptr(scales), _ptr(rotations), _ptr(cov3D), _ptr(sh_rest if activations else None),
                                           1 if activations else 0)


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class ForwardState:
    """Everything one forward leaves behind for its backward (upstream: ctx + geom/binning/img buffers)."""
    __slots__ = ("rs", "frame", "num_rendered", "capacity", "geom", "binning", "image", "radii", "alpha", "tensors", "fast",
                 "stats_applied")


def forward_impl(rs, means3D, sh, colors_precomp, opacities, scales, rotations, cov3D, sh_rest=None, activations=False):
    """Runs both forward stages through the C ABI. Inputs are validated CUDA float32 tensors (or None).
    Returns (color, radii, depth, alpha, ForwardState).

    No host round trip sits between the kernels: the instance buffer is sized from a per-shape capacity hint, every
    kernel of the forward is enqueued, and only then does the host wait for the (early) instance-count event.  If the
    guess was too small, stage 2 is re-run with a large enough buffer (the kernels clip safely to the capacity)."""
    if _FAST is not None:
        color, radii, depth, alpha, cst = _FAST.forward(
            int(rs.image_height), int(rs.image_width), float(rs.tanfovx), float(rs.tanfovy), float(rs.scale_modifier), int(rs.sh_degree),
            bool(rs.prefiltered), bool(rs.debug), rs.bg, rs.viewmatrix, rs.projmatrix, rs.campos, means3D, sh, colors_precomp, opacities,
            scales, rotations, cov3D, sh_rest, bool(activations))
        state = ForwardState()
        state.fast, state.rs, state.num_rendered, state.capacity = cst, rs, cst.num_rendered, cst.capacity
        state.radii, state.alpha = radii, None
        state.tensors = (means3D, sh, colors_precomp, opacities, scales, rotations, cov3D, sh_rest)
        return color, radii, depth, alpha, state
    lib = _lib.load()
    dev = means3D.device
    with torch.cuda.device(dev):
        fr = _Frame(rs, means3D, sh, colors_precomp, opacities, scales, rotations, cov3D, sh_rest, activations)
        H, W, P = int(rs.image_height), int(rs.image_width), fr.P
        u8 = dict(dtype=torch.uint8, device=dev)
        color = torch.empty((3, H, W), dtype=torch.float32, device=dev)
        depth = torch.empty((1, H, W), dtype=torch.float32, device=dev)
        alpha = torch.empty((1, H, W), dtype=torch.float32, device=dev)
        radii = torch.empty((P,), dtype=torch.int32, device=dev)
        geom = torch.empty((lib.dgr_geom_bytes(P, H, W),), **u8)
        image = torch.empty((lib.dgr_image_bytes(H, W),), **u8)
        n_host, event = _host_sync_objects(dev)
        st = _stream_ptr(dev)
        _lib.check(lib.dgr_forward_preprocess(ctypes.byref(fr.settings), ctypes.byref(fr.gaussians), _ptr(geom), _ptr(image),
                                              _ptr(radii), st))
        out = _lib.DgrImages(_ptr(color), _ptr(depth), _ptr(alpha), _ptr(radii))
        key = (dev.index, P, H, W)
        cap, big = _CAPACITY_HINT.get(key, (max(65536, 16 * P), True))
        rerun = 0
        while True:
            binning = torch.empty((lib.dgr_binning_bytes(cap, H, W),), **u8)
            _lib.check(lib.dgr_forward_render(ctypes.byref(fr.settings), ctypes.byref(fr.gaussians), _ptr(geom), _ptr(binning),
                                              ctypes.c_uint64(cap), _ptr(image), ctypes.byref(out), (1 if big else 0) | rerun,
                                              ctypes.c_void_p(n_host.data_ptr()), ctypes.c_uint64(0), event, st))
            _lib.check(lib.dgr_event_synchronize(event))
            n_inst, n_big = int(n_host[0]), int(n_host[1])
            if n_inst <= cap and (big or n_big == 0):
                break
            cap = max(cap, int(n_inst * 1.25) + 4096)  # a guess was wrong: redo stage 2 (rare)
            big = big or n_big > 0
            rerun = 2                                   # DGR_FLAG_RERUN
        _CAPACITY_HINT[key] = (max(int(n_inst * 1.25) + 4096, 65536), n_big > 0)
    state = ForwardState()
    state.fast = None
    state.rs, state.frame, state.num_rendered, state.capacity = rs, fr, n_inst, cap
    # alpha is a differentiable OUTPUT: storing it here would close the cycle state -> alpha -> grad_fn -> ctx -> state and leave
    # ~100 MB of scratch per call to the cyclic garbage collector (the C ABI's out_alpha argument is unused)
    state.geom, state.binning, state.image, state.radii, state.alpha = geom, binning, image, radii, None
    state.tensors = (means3D, sh, colors_precomp, opacities, scales, rotations, cov3D, sh_rest)
    return color, radii, depth, alpha, state


_SYNC = {}
_CAPACITY_HINT = {}


def _host_sync_objects(dev):
    """(pinned uint64 for the instance count, cudaEvent handle) per (host thread, device)."""
    import threading
    key = (threading.get_ident(), dev.index)
    t = _SYNC.get(key)
    if t is None:
        ev = _lib.load().dgr_event_create()
        if not ev:
            raise RuntimeError("libdgr_b200: could not create a CUDA event")
        t = (torch.zeros((4,), dtype=torch.int64).pin_memory(), ctypes.c_void_p(ev))
        _SYNC[key] = t
    return t


def backward_impl(state, grad_color, grad_depth, grad_alpha, d_means3D, d_means2D, d_sh, d_col, d_opac, d_scales, d_rot,
                  d_cov, accumulate=False, d_sh_rest=None, densify=None, push=None):
    """Runs the backward through the C ABI, writing (or accumulating) into the given gradient tensors.
    densify = (xyz_gradient_accum, denom, max_radii2D) float32 [P] tensors (any may be None) updated in the same kernel.
    push = a _lib.DgrPeerPush (multi-GPU: rows of Gaussians another rank owns go straight to that rank, include/dgr_b200.h)."""
    push_addr = ctypes.addressof(push) if push is not None else 0
    if state.fast is not None:
        _FAST.backward(state.fast, grad_color, grad_depth, grad_alpha, bool(accumulate),
                       [d_means3D, d_means2D, d_sh, d_col, d_opac, d_scales, d_rot, d_cov, d_sh_rest], *(densify or (None, None, None)),
                       push_addr)
        return
    lib = _lib.load()
    fr = state.frame
    dev = state.radii.device
    with torch.cuda.device(dev):
        gin = _lib.DgrImageGrads(_ptr(grad_color), _ptr(grad_depth), _ptr(grad_alpha))
        gout = _lib.DgrGaussianGrads(_ptr(d_means3D), _ptr(d_means2D), _ptr(d_sh), _ptr(d_col), _ptr(d_opac), _ptr(d_scales),
                                     _ptr(d_rot), _ptr(d_cov), 1 if accumulate else 0, _ptr(d_sh_rest),
                                     *((_ptr(t) for t in densify) if densify is not None else (None, None, None)), push_addr or None)
        _lib.check(lib.dgr_backward(ctypes.byref(fr.settings), ctypes.byref(fr.gaussians), _ptr(state.geom), _ptr(state.binning),
                                    ctypes.c_uint64(state.capacity), _ptr(state.image), _ptr(state.radii), _ptr(state.alpha),
                                    ctypes.byref(gin), ctypes.byref(gout), _stream_ptr(dev)))


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings):
        means3D = _dev_f32(means3D, "means3D")
        opacities = _dev_f32(opacities, "opacities")
        sh, colors_precomp = _opt(sh, "shs"), _opt(colors_precomp, "colors_precomp")
        scales, rotations, cov3D = _opt(scales, "scales"), _opt(rotations, "rotations"), _opt(cov3Ds_precomp, "cov3D_precomp")
        color, radii, depth, alpha, state = forward_impl(raster_settings, means3D, sh, colors_precomp, opacities, scales,
                                                         rotations, cov3D)
        ctx.state = state
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha):
        state = ctx.state
        if state.fast is not None:
            g = _FAST.backward(state.fast, grad_color, grad_depth, grad_alpha, False, [], None, None, None)      # undefined -> None
            return g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7], None
        means3D, sh, colors_precomp, opacities, scales, rotations, cov3D, _ = state.tensors
        dev = means3D.device
        P, M = state.frame.P, state.frame.M
        f32 = dict(dtype=torch.float32, device=dev)
        gC = _dev_f32(grad_color, "grad_color") if grad_color is not None else None
        gD = _dev_f32(grad_depth, "grad_depth") if grad_depth is not None else None
        gA = _dev_f32(grad_alpha, "grad_alpha") if grad_alpha is not None else None
        d_means3D = torch.empty((P, 3), **f32)
        d_means2D = torch.empty((P, 3), **f32)
        d_opac = torch.empty((P, 1), **f32)
        d_sh = torch.empty((P, M, 3), **f32) if sh is not None else None
        d_col = torch.empty((P, 3), **f32) if colors_precomp is not None else None
        d_scales = torch.empty((P, 3), **f32) if scales is not None else None
        d_rot = torch.empty((P, 4), **f32) if rotations is not None else None
        d_cov = torch.empty((P, 6), **f32) if cov3D is not None else None
        backward_impl(state, gC, gD, gA, d_means3D, d_means2D, d_sh, d_col, d_opac, d_scales, d_rot, d_cov)
        # ctx.state stays: a retain_graph backward runs again from the same buffers (they go away with the graph node)
        return d_means3D, d_means2D, d_sh, d_col, d_opac, d_scales, d_rot, d_cov, None


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, raster_settings):
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                     raster_settings)


class GaussianRasterizer(nn.Module):
    """Constructed per render call by the reference (gs_renderer.py:760): construction is trivial."""

    def __init__(self, raster_settings: GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        with torch.no_grad():
            rs = self.raster_settings
            lib = _lib.load()
            pos = _dev_f32(positions, "positions")
            view, proj = _dev_f32(rs.viewmatrix, "viewmatrix"), _dev_f32(rs.projmatrix, "projmatrix")
            present = torch.empty((pos.shape[0],), dtype=torch.uint8, device=pos.device)
            with torch.cuda.device(pos.device):
                _lib.check(lib.dgr_mark_visible(pos.shape[0], _ptr(pos), _ptr(view), _ptr(proj), _ptr(present), _stream_ptr(pos.device)))
            return present.bool()

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None, cov3D_precomp=None):
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception("Please provide excatly one of either SHs or precomputed colors!")
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")
        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp,
                                   self.raster_settings)


# ---------------------------------------------------------------------------------------------------------------------------------
# Batched views: V cameras of ONE cloud at one resolution in one forward / backward (include/dgr_b200.h, "Batched views").  The
# per-Gaussian stages run once for all views (inputs read once, summed gradient written once); binning, sort and both render
# kernels run per view on that view's slice of the scratch.

MAX_BATCH_VIEWS = 16
_BATCH_SHARED = ("image_height", "image_width", "sh_degree", "scale_modifier", "prefiltered", "debug")


def check_batch_settings(settings_list):
    """The views of a batch share image size, SH degree, scale_modifier, prefiltered and debug; 1 to 16 views."""
    settings_list = list(settings_list)
    if not 1 <= len(settings_list) <= MAX_BATCH_VIEWS:
        raise ValueError("a batch renders 1 to %d views, got %d" % (MAX_BATCH_VIEWS, len(settings_list)))
    first = settings_list[0]
    for i, rs in enumerate(settings_list[1:], 1):
        for name in _BATCH_SHARED:
            a, b = getattr(first, name), getattr(rs, name)
            if (bool(a) != bool(b)) if name in ("prefiltered", "debug") else (a != b):
                raise ValueError("view %d of the batch has %s = %r, view 0 has %r: the views of a batch must share %s"
                                 % (i, name, b, a, ", ".join(_BATCH_SHARED)))
    return settings_list


def _reject_precomputed(colors_precomp, cov3D_precomp):
    if colors_precomp is not None or cov3D_precomp is not None:
        raise ValueError("the batched rasterizer takes SHs and scales / rotations: colors_precomp and cov3D_precomp are not supported")


class _BatchFrame:
    """ctypes views of one batched call's V settings + inputs (keeps the tensors alive)."""

    def __init__(self, settings_list, means3D, sh, opacities, scales, rotations, sh_rest=None, activations=False):
        self.frames = [_Frame(rs, means3D, sh, None, opacities, scales, rotations, None, sh_rest, activations) for rs in settings_list]
        self.V = len(self.frames)
        self.settings = (_lib.DgrSettings * self.V)(*[f.settings for f in self.frames])
        self.gaussians = self.frames[0].gaussians
        self.P, self.M = self.frames[0].P, self.frames[0].M


_TICKET = [0]


def _batch_counts(dev, V):
    """Pinned (device-mapped) [16, 4] uint64 count slots, one row per view, per (host thread, device)."""
    import threading
    key = ("batch", threading.get_ident(), dev.index)
    t = _SYNC.get(key)
    if t is None:
        t = torch.zeros((MAX_BATCH_VIEWS, 4), dtype=torch.int64).pin_memory()
        _SYNC[key] = t
    return t


def _wait_tickets(counts, tickets, stream):
    """Polls the ticket every view's scan kernel stores after its counts (no copy or event between the kernels)."""
    arr = counts.numpy()
    pending = list(range(len(tickets)))
    spins = 0
    while pending:
        pending = [v for v in pending if int(arr[v, 2]) != tickets[v]]
        spins += 1
        if pending and spins % 2048 == 0 and stream.query():
            pending = [v for v in pending if int(arr[v, 2]) != tickets[v]]
            if pending:
                raise RuntimeError("libdgr_b200: the instance counts of views %s never arrived" % pending)


def forward_batch_impl(settings_list, means3D, sh, opacities, scales, rotations, sh_rest=None, activations=False):
    """Both forward stages of V views.  Inputs are validated CUDA float32 tensors.  Returns (color [V,3,H,W], radii [V,P],
    depth [V,1,H,W], alpha [V,1,H,W], BatchState).

    Stage 1 is one batched call; then stage 2 of every view is enqueued with the shape's capacity hint before the host waits for
    any instance count, and only a view whose guess was too small runs stage 2 again."""
    lib = _lib.load()
    dev = means3D.device
    with torch.cuda.device(dev):
        fr = _BatchFrame(settings_list, means3D, sh, opacities, scales, rotations, sh_rest, activations)
        V, P = fr.V, fr.P
        H, W = int(settings_list[0].image_height), int(settings_list[0].image_width)
        u8 = dict(dtype=torch.uint8, device=dev)
        color = torch.empty((V, 3, H, W), dtype=torch.float32, device=dev)
        depth = torch.empty((V, 1, H, W), dtype=torch.float32, device=dev)
        alpha = torch.empty((V, 1, H, W), dtype=torch.float32, device=dev)
        radii = torch.empty((V, P), dtype=torch.int32, device=dev)
        geom_stride, image_stride = lib.dgr_geom_bytes(P, H, W), lib.dgr_image_bytes(H, W)
        geom = torch.empty((lib.dgr_batch_geom_bytes(V, P, H, W),), **u8)
        image = torch.empty((lib.dgr_batch_image_bytes(V, H, W),), **u8)
        st = _stream_ptr(dev)
        _lib.check(lib.dgr_forward_preprocess_batch(fr.settings, V, ctypes.byref(fr.gaussians), _ptr(geom), _ptr(image), _ptr(radii), st))
        hint = get_capacity_hint(dev.index, P, H, W)
        cap0, big0 = hint if hint is not None else (max(65536, 16 * P), True)
        caps, bigs, binnings, outs = [cap0] * V, [bool(big0)] * V, [None] * V, [None] * V
        counts = _batch_counts(dev, V)
        cnt_base = counts.data_ptr()

        def stage2(v, flags, ticket, event=None):
            binnings[v] = torch.empty((lib.dgr_binning_bytes(caps[v], H, W),), **u8)
            outs[v] = _lib.DgrImages(_ptr(color[v]), _ptr(depth[v]), _ptr(alpha[v]), _ptr(radii[v]))
            _lib.check(lib.dgr_forward_render(ctypes.byref(fr.settings[v]), ctypes.byref(fr.gaussians),
                                              ctypes.c_void_p(geom.data_ptr() + v * geom_stride), _ptr(binnings[v]), ctypes.c_uint64(caps[v]),
                                              ctypes.c_void_p(image.data_ptr() + v * image_stride), ctypes.byref(outs[v]),
                                              (1 if bigs[v] else 0) | flags, ctypes.c_void_p(cnt_base + 32 * v), ctypes.c_uint64(ticket),
                                              event, st))

        tickets = []
        for v in range(V):
            _TICKET[0] += 1
            tickets.append(_TICKET[0])
            stage2(v, 0, tickets[v])
        _wait_tickets(counts, tickets, torch.cuda.current_stream(dev))
        n_inst = [int(counts[v, 0]) for v in range(V)]
        n_big = [int(counts[v, 1]) for v in range(V)]
        for v in range(V):
            while n_inst[v] > caps[v] or (n_big[v] > 0 and not bigs[v]):       # this view's guess was wrong: redo its stage 2 (rare)
                caps[v] = max(caps[v], int(n_inst[v] * 1.25) + 4096)
                bigs[v] = bigs[v] or n_big[v] > 0
                event = _host_sync_objects(dev)[1]
                stage2(v, 2, 0, event)                                         # DGR_FLAG_RERUN; counts copied into row v, then the event
                _lib.check(lib.dgr_event_synchronize(event))
                n_inst[v], n_big[v] = int(counts[v, 0]), int(counts[v, 1])
        set_capacity_hint(dev.index, P, H, W, max(max(int(n * 1.25) + 4096 for n in n_inst), 65536), any(b > 0 for b in n_big))
    state = BatchState()
    state.frame, state.geom, state.image, state.binnings, state.capacities = fr, geom, image, binnings, caps
    state.radii, state.num_rendered = radii, n_inst
    state.tensors = (means3D, sh, opacities, scales, rotations, sh_rest)
    return color, radii, depth, alpha, state


class BatchState:
    """What a batched forward leaves behind for its backward: V scratch slices, V binning buffers and their capacities."""
    __slots__ = ("frame", "geom", "image", "binnings", "capacities", "radii", "num_rendered", "tensors", "stats_applied")


def backward_batch_impl(state, grad_color, grad_depth, grad_alpha, d_means3D, d_means2D, d_sh, d_opac, d_scales, d_rot,
                        accumulate=False, d_sh_rest=None, densify=None):
    """The backward of a batched forward: per-view upstream gradients [V, ...] (any may be None = zeros) in; means3D / shs (/ shs_rest)
    / opacities / scales / rotations gradients summed over the views written (or added with accumulate) into the given tensors;
    d_means2D is [V, P, 3].  densify = (xyz_gradient_accum, denom, max_radii2D), updated once per view."""
    lib = _lib.load()
    fr = state.frame
    V = fr.V
    dev = state.radii.device
    with torch.cuda.device(dev):
        view = lambda t, v: None if t is None else ctypes.c_void_p(t[v].data_ptr())
        gin = (_lib.DgrImageGrads * V)(*[_lib.DgrImageGrads(view(grad_color, v), view(grad_depth, v), view(grad_alpha, v)) for v in range(V)])
        binning = (ctypes.c_void_p * V)(*[b.data_ptr() for b in state.binnings])
        caps = (ctypes.c_uint64 * V)(*state.capacities)
        gout = _lib.DgrGaussianGrads(_ptr(d_means3D), _ptr(d_means2D), _ptr(d_sh), None, _ptr(d_opac), _ptr(d_scales), _ptr(d_rot), None,
                                     1 if accumulate else 0, _ptr(d_sh_rest),
                                     *((_ptr(t) for t in densify) if densify is not None else (None, None, None)), None)
        _lib.check(lib.dgr_backward_batch(fr.settings, V, ctypes.byref(fr.gaussians), _ptr(state.geom), binning, caps, _ptr(state.image),
                                          _ptr(state.radii), gin, ctypes.byref(gout), _stream_ptr(dev)))


def _batch_upstream(g, name, shape):
    if g is None:
        return None
    g = _dev_f32(g, name)
    if tuple(g.shape) != tuple(shape):
        raise ValueError("%s must have shape %s" % (name, tuple(shape)))
    return g


class _RasterizeBatch(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, opacities, scales, rotations, settings_list):
        means3D, opacities = _dev_f32(means3D, "means3D"), _dev_f32(opacities, "opacities")
        sh, scales, rotations = _dev_f32(sh, "shs"), _dev_f32(scales, "scales"), _dev_f32(rotations, "rotations")
        color, radii, depth, alpha, state = forward_batch_impl(settings_list, means3D, sh, opacities, scales, rotations)
        ctx.state = state
        ctx.mark_non_differentiable(radii)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_color, grad_radii, grad_depth, grad_alpha):
        state = ctx.state
        means3D, sh, opacities, scales, rotations, _ = state.tensors
        V, P = state.frame.V, state.frame.P
        f32 = dict(dtype=torch.float32, device=means3D.device)
        d_means3D, d_means2D = torch.empty((P, 3), **f32), torch.empty((V, P, 3), **f32)
        d_sh, d_opac = torch.empty(sh.shape, **f32), torch.empty((P, 1), **f32)
        d_scales, d_rot = torch.empty((P, 3), **f32), torch.empty((P, 4), **f32)
        backward_batch_impl(state, *_batch_grads(state, grad_color, grad_depth, grad_alpha), d_means3D, d_means2D, d_sh, d_opac, d_scales, d_rot)
        # ctx.state stays: a retain_graph backward runs again from the same buffers (they go away with the graph node)
        return d_means3D, d_means2D, d_sh, d_opac, d_scales, d_rot, None


def _batch_grads(state, grad_color, grad_depth, grad_alpha):
    s = state.frame.frames[0].settings
    V, H, W = state.frame.V, int(s.image_height), int(s.image_width)
    return (_batch_upstream(grad_color, "grad_color", (V, 3, H, W)), _batch_upstream(grad_depth, "grad_depth", (V, 1, H, W)),
            _batch_upstream(grad_alpha, "grad_alpha", (V, 1, H, W)))


class BatchedGaussianRasterizer(nn.Module):
    """V views (1 to 16) of one cloud in one call.  The views share image size, SH degree, scale_modifier, prefiltered and
    debug; fov, bg, view / projection matrices and camera position may differ.

    forward(means3D, opacities, shs, scales, rotations, means2D=None) -> (color [V,3,H,W], radii int32 [V,P], depth [V,1,H,W],
    alpha [V,1,H,W]).  The gradients of means3D / shs / opacities / scales / rotations are summed over the views; means2D, when
    given, is the [V,P,3] per-view screen-space dummy whose .grad receives each view's own gradient."""

    def __init__(self, settings_list):
        super().__init__()
        self.settings_list = check_batch_settings(settings_list)

    def forward(self, means3D, opacities, shs, scales, rotations, means2D=None, colors_precomp=None, cov3D_precomp=None):
        _reject_precomputed(colors_precomp, cov3D_precomp)
        if shs is None or scales is None or rotations is None:
            raise ValueError("the batched rasterizer needs shs, scales and rotations")
        V = len(self.settings_list)
        if means2D is None:
            means2D = torch.zeros((V,) + tuple(means3D.shape), dtype=torch.float32, device=means3D.device,
                                  requires_grad=means3D.requires_grad)
        elif tuple(means2D.shape) != (V,) + tuple(means3D.shape):
            raise ValueError("means2D must have dimensions (num_views, num_points, 3)")
        return _RasterizeBatch.apply(means3D, means2D, shs, opacities, scales, rotations, self.settings_list)
