#!/usr/bin/env python
"""bench.py — splats/sec of the differentiable Gaussian-splat rasterize (forward + backward), BASELINE.json's metric.

A "step" = one forward + backward pass of the rasterizer over ONE synthetic view per GPU (views are the data-parallel
axis, SURVEY.md §8e); with N GPUs every rank renders its own view of the same replicated cloud, accumulates the
per-Gaussian gradients into one flat buffer and the ranks all-reduce it over NCCL (weak scaling).
Workload at N=1: BASELINE.json configs[1] — 100k Gaussians, 800x800, SH degree 3 (synthetic DreamGaussian-like cloud,
dreamgaussian_b200/scene.py).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # our sm_100a path (the product)
  python bench.py --impl reference ...                           # the CPU oracle port, timed on the host cores
  python bench.py ... --dump-outputs DIR                         # + the last timed step's gradients as DIR/*.npy

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


# BASELINE.json configs that are bench workloads (configs[0] and [3] are parity / loop cases: tests/, next_rows.f2)
WORKLOADS = {
    "cfg2": dict(points=100000, res=800, views_per_gpu=1, views=8, steps=1000,
                 what="BASELINE.json configs[1]: 100k Gaussians, 800x800, SH degree 3, forward+backward, one view per GPU per step"),
    "cfg3": dict(points=500000, res=512, views_per_gpu=8, views=64, steps=60,
                 what="BASELINE.json configs[2]: 500k Gaussians, 512x512, 64 views per iteration sharded 8 per GPU (8 views per GPU "
                      "per step accumulate into the flat gradient, one all-reduce per step)"),
    "cfg5": dict(points=2000000, res=1600, views_per_gpu=1, views=8, steps=100,
                 what="BASELINE.json configs[4]: 2M Gaussians, 1600x1600, SH degree 3, forward+backward, one view per GPU per step"),
}
DUMP_BYTES = 64 << 20          # --dump-outputs: cap on what one run writes


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS), help="cfg2 = the metric's configuration (default)")
    ap.add_argument("--points", type=int, default=None)
    ap.add_argument("--res", type=int, default=None)
    ap.add_argument("--views-per-gpu", type=int, default=None)
    ap.add_argument("--sh-degree", type=int, default=3)
    ap.add_argument("--opacity", default="trained", choices=["trained", "init"])
    ap.add_argument("--views", type=int, default=None, help="size of the fixed camera set that steps cycle through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-rows", action="store_true", help="skip the short measurements of the SURVEY §8f rows (f1-f4)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the per-Gaussian gradients of the last timed step as DIR/<name>.npy "
                         "(float32; above %d MB in all, the same seeded sample of Gaussians from every array)" % (DUMP_BYTES >> 20))
    a = ap.parse_args()
    w = WORKLOADS[a.workload]
    for k in ("points", "res", "views_per_gpu", "views", "steps"):
        if getattr(a, k) is None:
            setattr(a, k, w[k])
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dump_outputs(out_dir, arrays, seed):
    """arrays: name -> CUDA float32 tensor [P, ...], all with the same P.  Written whole when they fit DUMP_BYTES together,
    else each restricted to the same rows: a sorted sample drawn from numpy's default_rng(seed), so that two builds dumped
    with the same arguments hold the same Gaussians."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    P = next(iter(arrays.values())).shape[0]
    row_bytes = sum(v[0].numel() * 4 for v in arrays.values()) if P else 0
    rows = None
    if P * row_bytes > DUMP_BYTES:
        pick = np.sort(np.random.default_rng(seed).choice(P, DUMP_BYTES // row_bytes, replace=False))
        rows = torch.tensor(pick, device=next(iter(arrays.values())).device)
    for name, v in arrays.items():
        x = v if rows is None else v.index_select(0, rows)
        np.save(os.path.join(out_dir, name + ".npy"), x.float().cpu().numpy())


def workload_name(a):
    return "%dk Gaussians, %dx%d, SH degree %d, forward+backward, opacity=%s, anisotropic%s" % (
        a.points // 1000, a.res, a.res, a.sh_degree, a.opacity,
        "" if a.views_per_gpu == 1 else ", %d views per GPU per step" % a.views_per_gpu)


def algorithmic_bytes(P, M, H, W, n_inst):
    """SURVEY.md §8(d): B_alg = P (148 + 36 M) + H W 52 + N_inst 44 bytes per view, forward + backward."""
    return P * (148 + 36 * M) + H * W * 52 + n_inst * 44


def kernel_algorithmic_bytes(name, P, M, H, W, n_inst):
    """Per-kernel algorithmic bytes (what the kernel must read + write once), DESIGN.md §Kernels."""
    px = H * W
    table = {
        "preprocess_fwd": P * (44 + 12 * M) + P * (4 + 48 + 4),              # inputs; radii + record + touched
        "tile_scan": (H // 16 + 1) * (W // 16 + 1) * 24,                    # counts in; ranges + cursor + order out
        "emit_instances": P * 12 + n_inst * 8,                              # aabb + depth + touched; keys
        "tile_sort_gather": n_inst * (8 + 4 + 48 + 48),                     # key in; id out; record gather + sorted record
        "tile_sort_gather_big": n_inst * (8 + 4 + 48 + 48),                 # the big-tile walker does the same per instance (upper bound: all instances)
        "render_fwd": n_inst * 48 + px * 28,                                 # sorted records; rgb+depth+alpha+n_contrib+T
        "render_bwd": n_inst * 52 + px * 28 + P * 48,                        # records+ids; grads+n_contrib+T; moments
        "preprocess_bwd": P * (44 + 12 * M) + P * 52 + P * (56 + 12 * M),   # inputs; moments+radii; grads
    }
    return table.get(name)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def wait_first_sample(self, timeout=3.0):
        """nvidia-smi needs ~100 ms to start: block until it has produced a row so a short run is still covered."""
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        return len(self.rows)

    def stop(self, window=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows, where = self.rows, "whole run (timed region shorter than the 20 ms sampling period)"
        if window and window[1] - window[0] >= 3:
            rows, where = self.rows[window[0]:window[1]], "timed region"
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": where}


def build_scene(a):
    from dreamgaussian_b200 import scene
    # base scale = 3-NN distance of the cloud (kd-tree) as the reference's initialisation derives it; above 500k points its
    # closed form 0.595 P^(-1/3) (fitted at 5k / 100k / 500k to 1 %) replaces the minutes-long kd-tree query
    sigma = None if a.points <= 500000 else 0.595 * a.points ** (-1.0 / 3.0)
    cloud = scene.make_cloud(a.points, a.sh_degree, seed=a.seed, opacity=a.opacity, anisotropic=True, sigma=sigma)
    cams = scene.bench_views(a.views, a.res, a.res)
    rng = np.random.default_rng(a.seed + 17)
    ups = [(rng.normal(size=(3, a.res, a.res)).astype(np.float32), None, rng.normal(size=(1, a.res, a.res)).astype(np.float32))
           for _ in range(min(a.views, 4))]
    return cloud, cams, ups


def cam_settings(cam, a, bg):
    return dict(image_height=a.res, image_width=a.res, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=bg, scale_modifier=1.0,
                viewmatrix=cam.world_view_transform, projmatrix=cam.full_proj_transform, sh_degree=a.sh_degree,
                campos=cam.camera_center)


def host_threads():
    """Threads for the CPU legs: the physical cores this process may run on.  (One OpenMP thread per LOGICAL CPU made the
    oracle 10x slower on the 2 x 32-core / 128-thread boxes; a cgroup CPU quota, if any, caps it further.)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def measure_other_shapes(dev):
    """Short device-timed measurements of the OTHER BASELINE.json shapes and of configs[1] at the reference's initial opacity
    (0.1 everywhere: no early termination — the hard case), so that the default run carries them next to the headline line.
    Same protocol as the headline (CUDA events per step, L2 flushed between steps), fewer steps."""
    import torch
    from dreamgaussian_b200 import _lib, multiview
    from dreamgaussian_b200.rasterizer import GaussianRasterizationSettings
    lib = _lib.load()
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    rows = {}
    shapes = (("cfg2_init_opacity", "cfg2", dict(opacity="init"), 40),
              ("cfg3_8_views_per_gpu", "cfg3", {}, 6),
              ("cfg5", "cfg5", {}, 12))
    for key, wl, over, steps in shapes:
        try:
            a = argparse.Namespace(sh_degree=3, opacity="trained", seed=0, workload=wl, **{k: WORKLOADS[wl][k] for k in ("points", "res", "views_per_gpu", "views")})
            for k, v in over.items():
                setattr(a, k, v)
            cloud, cams, ups = build_scene(a)
            t = lambda x: torch.tensor(np.asarray(x, np.float32), device=dev)
            params = {k: t(v) for k, v in cloud.items()}
            bg = t(np.ones(3, np.float32))
            settings = [GaussianRasterizationSettings(
                image_height=a.res, image_width=a.res, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=bg, scale_modifier=1.0,
                viewmatrix=t(c.world_view_transform), projmatrix=t(c.full_proj_transform), sh_degree=3,
                campos=t(c.camera_center), prefiltered=False, debug=False) for c in cams]
            ups_d = [(t(u[0]), None, t(u[2])) for u in ups]
            vsr = multiview.ViewShardedRasterizer(a.points, 16, dev)
            vpg = a.views_per_gpu

            def step(i):
                vs = [(i * vpg + k) % len(settings) for k in range(vpg)]
                vsr.render_views(params, [settings[v] for v in vs], [ups_d[v % len(ups_d)] for v in vs])
            for i in range(3):
                step(i)
            torch.cuda.synchronize(dev)
            evs = []
            for i in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); step(3 + i); e1.record(); evs.append((e0, e1))
            torch.cuda.synchronize(dev)
            ms = float(np.mean([x.elapsed_time(y) for x, y in evs]))
            lib.dgr_profile_enable(1)
            for i in range(2):
                flush.zero_(); step(i)
            torch.cuda.synchronize(dev)
            kern = {}
            for name, v in _lib.profile_collect():
                kern.setdefault(name, []).append(v)
            lib.dgr_profile_enable(0)
            rows[key] = {"workload": workload_name(a), "ms_per_step": ms, "splats_per_s": a.points * vpg / (ms * 1e-3), "steps": steps,
                         "kernels_us_per_view": {k: round(float(np.sum(v)) / (2 * vpg) * 1e3, 1) for k, v in kern.items()}}
            del vsr, params, settings, ups_d
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            rows[key] = {"error": repr(e)[:300]}
    return rows


def measure_next_rows(dev):
    """Short, guarded measurements of the rows next to the hot path (SURVEY.md §8f; DESIGN.md §7) — reported beside the
    headline metric, never part of it.  Each entry: this library's time and what it is compared with."""
    import numpy as np
    import torch
    from dreamgaussian_b200 import fields, scene, stage1
    from dreamgaussian_b200.fused import DensifyStats, FusedGaussianRasterizer
    from dreamgaussian_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    from simple_knn._C import distCUDA2
    rows = {}

    def ev_median(fn, n):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        evs = []
        for i in range(n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(i); e1.record(); evs.append((e0, e1))
        torch.cuda.synchronize()
        return float(np.median([x.elapsed_time(y) for x, y in evs]))

    try:        # f1: raw-parameter step (fwd + bwd + densification statistics) at the bench shape
        P, res = 100000, 800
        cloud = scene.make_cloud(P, 3, seed=0, opacity="trained", anisotropic=True)
        raw = {k: torch.tensor(v, device=dev).requires_grad_(True) for k, v in scene.to_raw_parameters(cloud).items()}
        t = lambda x: torch.tensor(np.asarray(x, np.float32), device=dev)
        cams = scene.bench_views(4, res, res)
        rs = [GaussianRasterizationSettings(image_height=res, image_width=res, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=t(np.ones(3)),
              scale_modifier=1.0, viewmatrix=t(c.world_view_transform), projmatrix=t(c.full_proj_transform), sh_degree=3,
              campos=t(c.camera_center), prefiltered=False, debug=False) for c in cams]
        rng = np.random.default_rng(17)
        gC, gA = t(rng.normal(size=(3, res, res))), t(rng.normal(size=(1, res, res)))
        stats = DensifyStats(P, dev)
        acc, den, mr = torch.zeros((P, 1), device=dev), torch.zeros((P, 1), device=dev), torch.zeros((P,), device=dev)

        def zero():
            for v in raw.values():
                v.grad = None

        def ref_form(i):
            zero()
            m2d = torch.zeros_like(raw["xyz"], requires_grad=True)
            c, r, d, al = GaussianRasterizer(rs[i % 4])(means3D=raw["xyz"], means2D=m2d, shs=torch.cat((raw["features_dc"], raw["features_rest"]), dim=1),
                                                       opacities=torch.sigmoid(raw["opacity"]), scales=torch.exp(raw["scaling"]),
                                                       rotations=torch.nn.functional.normalize(raw["rotation"]))
            torch.autograd.backward([c, al], [gC, gA])
            with torch.no_grad():
                vis = r > 0
                mr[vis] = torch.max(mr[vis], r[vis].float()); acc[vis] += torch.norm(m2d.grad[vis, :2], dim=-1, keepdim=True); den[vis] += 1

        def fused(i):
            zero()
            c, r, d, al = FusedGaussianRasterizer(rs[i % 4])(raw["xyz"], raw["features_dc"], raw["features_rest"], raw["opacity"], raw["scaling"],
                                                            raw["rotation"], stats=stats)
            torch.autograd.backward([c, al], [gC, gA])
        rows["f1_raw_parameter_step"] = {"ours_ms": ev_median(fused, 40), "torch_activations_plus_plain_op_ms": ev_median(ref_form, 40),
                                         "shape": "100k / 800x800 / deg 3, fwd+bwd+densify stats through autograd"}
        del raw, stats
    except Exception as e:  # noqa: BLE001
        rows["f1_raw_parameter_step"] = {"error": repr(e)[:200]}
    try:        # f2: BASELINE.json configs[3]
        out = {}
        for name, fz in (("ours", True), ("reference_formulation", False)):
            stage1.Stage1Trainer(stage1.Stage1Config(), fused=fz).train(10)
            tr = stage1.Stage1Trainer(stage1.Stage1Config(), fused=fz)
            torch.cuda.synchronize(); t0 = time.perf_counter(); tr.train(500); torch.cuda.synchronize()
            out[name + "_s_per_500_iters"] = time.perf_counter() - t0
            out[name + "_final_points"] = tr.gaussians.num_points
        out["shape"] = "configs/image.yaml stage-1 loop, synthetic RGBA, guidance stubbed, 500 iterations"
        rows["f2_stage1_loop"] = out
    except Exception as e:  # noqa: BLE001
        rows["f2_stage1_loop"] = {"error": repr(e)[:200]}
    try:        # f3: distCUDA2 against the reference's own CUDA code (oracle/_ref), 100k points of the reference's init ball
        from oracle import knn_oracle
        pts = torch.tensor(scene.make_cloud(100000, 0, seed=1, anisotropic=False, sigma=1.0)["means3D"], device=dev)
        r = {"ours_ms": ev_median(lambda i: distCUDA2(pts), 20), "shape": "100k points"}
        if os.path.exists(knn_oracle.REF_LIB):
            knn_oracle.reference_dist_cuda2(pts); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                ref = knn_oracle.reference_dist_cuda2(pts)
            r["reference_simple_knn_ms"] = (time.perf_counter() - t0) / 5 * 1e3
            r["bit_identical_to_reference"] = bool(torch.equal(ref, distCUDA2(pts)))
        rows["f3_distCUDA2"] = r
    except Exception as e:  # noqa: BLE001
        rows["f3_distCUDA2"] = {"error": repr(e)[:200]}
    try:        # f4: extract_fields, reference defaults
        rawf = scene.to_raw_parameters(scene.make_cloud(100000, 0, seed=4, sigma=0.0128))
        tf = [torch.tensor(rawf[k], device=dev) for k in ("xyz", "opacity", "scaling", "rotation")]
        rows["f4_extract_fields"] = {"ours_ms": ev_median(lambda i: fields.extract_fields(*tf, resolution=128), 5), "shape": "100k Gaussians, 128^3, 16^3 blocks"}
    except Exception as e:  # noqa: BLE001
        rows["f4_extract_fields"] = {"error": repr(e)[:200]}
    return rows


def time_cpu_oracle(a, cloud, cams, ups, steps, warmup):
    """The CPU arm: the oracle port (float32, OpenMP over all host threads), one full view fwd+bwd per step."""
    from oracle import c_oracle
    c_oracle.set_threads(host_threads())            # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    bg = np.ones(3, np.float32)
    inputs = dict(means3D=cloud["means3D"], opacities=cloud["opacities"], shs=cloud["shs"], scales=cloud["scales"],
                  rotations=cloud["rotations"])
    times = []
    for i in range(warmup + steps):
        cam = cams[i % len(cams)]
        gC, gD, gA = ups[i % len(ups)]
        t0 = time.perf_counter()
        r = c_oracle.forward(**cam_settings(cam, a, bg), **inputs, dtype=np.float32)
        r.backward(gC, gD, gA)
        r.close()
        t1 = time.perf_counter()
        if i >= warmup:
            times.append(t1 - t0)
    sec = float(np.mean(times))
    return a.points / sec, sec, c_oracle.num_threads()


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(a, rank, world):
    if rank != 0:
        return
    cloud, cams, ups = build_scene(a)
    steps, warmup = max(1, min(a.steps, 5)), max(1, min(a.warmup, 1))
    val, sec, threads = time_cpu_oracle(a, cloud, cams, ups, steps, warmup)
    out = {
        "impl": "reference", "metric": "splats/sec fwd+bwd @ %dx%d" % (a.res, a.res), "value": val, "unit": "splats/s",
        "n_gpus": a.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "note": "CPU oracle port (oracle/dgr_oracle.c), the reference has no CPU path "
                   "and its CUDA op is not vendored (SURVEY.md §8c); steps capped at 5 to bound the run"},
        "cpu_baseline": {"value": val, "unit": "splats/s", "cores": threads, "kind": "port",
                         "sample": "%d full views fwd+bwd of the same workload" % steps, "cpu": cpu_model()},
        "e2e": {"value": val, "unit": "splats/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def collective_check(vsr, dev, rank, world):
    """N > 1, before anything is timed: the library's own all-reduce on a buffer of per-rank noise must agree with NCCL's
    all_reduce of the same data and must leave the same bits on every rank."""
    import torch
    import torch.distributed as dist
    g = torch.Generator(device=dev); g.manual_seed(4321 + rank)
    n = vsr.grads.flat.numel()
    src = torch.randn(n, device=dev, generator=g)
    ref = src.clone()
    dist.all_reduce(ref)                                           # NCCL
    vsr.grads.flat.copy_(src)
    torch.cuda.synchronize(dev); dist.barrier()
    got = vsr.all_reduce().clone()
    torch.cuda.synchronize(dev)
    diff = float((got - ref).abs().max()); scale = float(ref.abs().max())
    hi, lo = got.clone(), got.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX); dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    same = bool(torch.equal(hi, lo))
    ok = torch.tensor([1.0 if (diff <= 1e-5 * scale and same) else 0.0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    vsr.grads.data.zero_()
    torch.cuda.synchronize(dev); dist.barrier()
    return {"ok": bool(ok.item() == 1.0), "max_abs_diff_vs_nccl": diff, "scale": scale, "identical_on_all_ranks": same,
            "floats": n, "kernel": vsr.collective}


def lib_source_stamp():
    from dreamgaussian_b200 import build
    return build.step_kernel_hash()[:16]


def committed_ncu(kind):
    """ncu-derived per-launch numbers (DRAM traffic, warp instructions) are only trusted when the capture was taken from
    the SAME kernel sources: profiles/r2_ncu_kernels.json carries the source hash of the library it profiled."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_kernels.json")))
        if d.get("lib_source_hash") != lib_source_stamp():
            return None, "stale (kernel sources changed since the capture)"
        return d.get(kind), d.get("source")
    except Exception:
        return None, "no capture committed"


def run_ours(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from dreamgaussian_b200 import _lib, hostmem, multiview
    from dreamgaussian_b200.rasterizer import GaussianRasterizationSettings

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    cloud, cams, ups = build_scene(a)
    P, M, H, W = a.points, (a.sh_degree + 1) ** 2, a.res, a.res
    vpg = a.views_per_gpu
    t = lambda x: torch.tensor(np.asarray(x, np.float32), device=dev)
    names = ("means3D", "shs", "opacities", "scales", "rotations")
    # ONE packed device buffer for the Gaussian inputs (segments 256-byte aligned): the e2e leg fills it with one copy
    seg, off = {}, 0
    for k in names:
        n = int(np.prod(cloud[k].shape))
        seg[k] = (off, n, cloud[k].shape); off += (n + 63) // 64 * 64
    packed_floats = off

    def views_of(buf):
        return {k: buf[o:o + n].view(shape) for k, (o, n, shape) in seg.items()}

    dev_packed = torch.empty((packed_floats,), dtype=torch.float32, device=dev)
    params = views_of(dev_packed)
    for k in names:
        params[k].copy_(t(cloud[k]))
    bg = t(np.ones(3, np.float32))
    settings = [GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=bg, scale_modifier=1.0,
        viewmatrix=t(c.world_view_transform), projmatrix=t(c.full_proj_transform), sh_degree=a.sh_degree,
        campos=t(c.camera_center), prefiltered=False, debug=False) for c in cams]
    ups_d = [(t(u[0]), None, t(u[2])) for u in ups]
    vsr = multiview.ViewShardedRasterizer(P, M, dev)
    flush_buf = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)    # > 126 MB L2

    def local_views(i):
        return [((i * world + rank) * vpg + k) % len(settings) for k in range(vpg)]

    def step(i):
        vs = local_views(i)
        vsr.render_views(params, [settings[v] for v in vs], [ups_d[v % len(ups_d)] for v in vs])
        if world > 1:
            vsr.all_reduce()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    check = collective_check(vsr, dev, rank, world) if world > 1 else None
    if check is not None and not check["ok"]:
        # never time a collective that gives wrong sums: fall back to NCCL for the whole run and say so in the line
        vsr.use_nccl("the library's own kernel failed the pre-run check")
        check["fallback"] = vsr.collective

    # nvidia-smi samples every 20 ms; it is started before the warm-up so that even a short timed region is covered
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first_sample()
    for i in range(max(a.warmup, 3)):
        step(i)
    barrier()
    n_inst = 0
    # ---------------- timed region: K steps, device-resident inputs, L2 flushed between steps ----------------
    lib.dgr_reset_launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    barrier()
    mark0 = sampler.mark()
    wall0 = time.perf_counter()
    for i in range(a.steps):
        flush_buf.zero_()
        evs[i][0].record()
        step(a.warmup + i)
        evs[i][1].record()
    barrier()
    wall1 = time.perf_counter()
    launches = int(lib.dgr_launch_count())
    clocks = sampler.stop((mark0, sampler.mark())) if rank == 0 else None
    ms_local = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    ms_t = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_total = float(ms_t.item())
    ms_per_step = ms_total / a.steps
    value = P * vpg * world * a.steps / (ms_total * 1e-3)
    # what the last timed step handed back: the flat gradient (summed over this rank's views, all-reduced when N > 1)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"grad_" + k: v for k, v in vsr.grads.views.items() if v is not None}, a.seed)

    # ---------------- per-kernel CUDA-event timing (separate pass, same workload, this rank's stream) ----------------
    kern = {}
    if rank == 0:
        lib.dgr_profile_enable(1)
        nprof = max(1, min(a.steps, 8))
        for i in range(nprof):
            flush_buf.zero_()
            vs = local_views(i)
            vsr.render_views(params, [settings[v] for v in vs], [ups_d[v % len(ups_d)] for v in vs])
        torch.cuda.synchronize(dev)
        for name, ms in _lib.profile_collect():
            kern.setdefault(name, []).append(ms)
        lib.dgr_profile_enable(0)
        kern = {k: float(np.sum(v)) / (nprof * vpg) for k, v in kern.items()}       # average per VIEW
        # instance count of the bench views (host read-back the forward already does)
        _, _, _, _, st = __import__("dreamgaussian_b200.rasterizer", fromlist=["forward_impl"]).forward_impl(
            settings[0], params["means3D"], params["shs"], None, params["opacities"], params["scales"], params["rotations"], None)
        n_inst = int(st.num_rendered)
    if world > 1:
        barrier()

    # ---------------- end to end through the public API with HOST buffers ----------------
    # Every step: ONE cudaMemcpyAsync of the packed Gaussian inputs (pinned host -> device), forward + backward of this
    # rank's views through ViewShardedRasterizer (the call a multi-view user makes; gradients accumulate into the flat buffer,
    # N > 1: the library's own all-reduce), the loss of the step, then ONE cudaMemcpyAsync of the flat gradient (+ the loss)
    # back to pinned host memory.  Upload / compute / download of consecutive steps overlap on three streams over a ring of
    # three buffer sets (PCIe is full duplex); every byte of every step moves inside the timed region.
    e2e = None
    if not a.no_e2e:
        RING = 3
        host_in = hostmem.pinned_empty((packed_floats,), torch.float32, dev)          # NUMA-local pinned (hostmem.py)
        hv = views_of(host_in)
        for k in names:
            hv[k].copy_(torch.tensor(cloud[k]))
        dev_in = [torch.empty((packed_floats,), dtype=torch.float32, device=dev) for _ in range(RING)]
        dev_views = [views_of(b) for b in dev_in]
        rings = [vsr] + [multiview.ViewShardedRasterizer(P, M, dev) for _ in range(RING - 1)]
        if check is not None and not check["ok"]:
            for r_ in rings[1:]:
                r_.use_nccl("the library's own kernel failed the pre-run check")
        nflat = vsr.grads.flat.numel()
        host_out = [hostmem.pinned_empty((nflat + 64,), torch.float32, dev) for _ in range(RING)]
        h2d = packed_floats * 4
        d2h = nflat * 4 + 4
        s_up, s_comp, s_down = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        ev_up = [torch.cuda.Event() for _ in range(RING)]
        ev_comp = [torch.cuda.Event() for _ in range(RING)]
        ev_down = [torch.cuda.Event() for _ in range(RING)]
        losses = [torch.zeros((1,), device=dev) for _ in range(RING)]

        def upload(i):
            r = i % RING
            with torch.cuda.stream(s_up):
                s_up.wait_event(ev_comp[r])                 # the previous user of this buffer set has finished computing
                dev_in[r].copy_(host_in, non_blocking=True)
                ev_up[r].record(s_up)

        def compute(i):
            r = i % RING
            vs = local_views(i)
            with torch.cuda.stream(s_comp):
                s_comp.wait_event(ev_up[r])
                s_comp.wait_event(ev_down[r])               # its gradients of RING steps ago have been downloaded
                imgs = rings[r].render_views(dev_views[r], [settings[v] for v in vs], [ups_d[v % len(ups_d)] for v in vs], keep_images=True)
                loss = None
                for v, (color, radii, depth, alpha) in zip(vs, imgs):
                    gC, _, gA = ups_d[v % len(ups_d)]
                    l = (color * gC).sum() + (alpha * gA).sum()
                    loss = l if loss is None else loss + l
                losses[r].copy_(loss.reshape(1))
                if world > 1:
                    rings[r].all_reduce()
                ev_comp[r].record(s_comp)

        def download(i):
            r = i % RING
            with torch.cuda.stream(s_down):
                s_down.wait_event(ev_comp[r])
                host_out[r][:nflat].copy_(rings[r].grads.flat, non_blocking=True)
                host_out[r][nflat:nflat + 1].copy_(losses[r], non_blocking=True)
                ev_down[r].record(s_down)

        def run(nsteps, first):
            upload(first)
            for i in range(first, first + nsteps):
                if i + 1 < first + nsteps:
                    upload(i + 1)
                compute(i)
                download(i)

        for r in range(RING):
            ev_comp[r].record(s_comp); ev_down[r].record(s_down)
        run(max(3, min(a.warmup, 6)), 0)
        barrier()
        e2e_steps = max(3, min(a.steps, 300))
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()                                          # default stream: ordered before the side streams by barrier()
        for st_ in (s_up, s_comp, s_down):
            st_.wait_event(e0)
        run(e2e_steps, 100)
        for st_ in (s_up, s_comp, s_down):
            torch.cuda.current_stream(dev).wait_stream(st_)
        e1.record()
        barrier()
        ms_e = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
        # achieved host-link rates: each direction timed alone on this rank, same buffers
        link = {}
        for nm, fn, nbytes in (("h2d_gbs", lambda: dev_in[0].copy_(host_in, non_blocking=True), h2d),
                               ("d2h_gbs", lambda: host_out[0][:nflat].copy_(vsr.grads.flat, non_blocking=True), d2h)):
            torch.cuda.synchronize(dev)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(5):
                fn()
            c1.record(); torch.cuda.synchronize(dev)
            link[nm] = nbytes * 5 / (c0.elapsed_time(c1) * 1e-3) / 1e9
        step_ms = float(ms_e.item()) / e2e_steps
        # the overlap, shown (there is no nsys in this image): a short untimed pass of the same pipeline with a timing event on
        # either side of every upload / compute / download on its own stream -> start and end of each stage on one clock
        timeline = None
        if world == 1:
            TL = 12
            marks = {k: [] for k in ("up", "comp", "down")}

            def staged(kind, stream, fn, i):
                b_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                fn(i, lambda: b_.record(stream), lambda: e_.record(stream))
                marks[kind].append((b_, e_))

            def up_t(i, mark_b, mark_e):
                r = i % RING
                with torch.cuda.stream(s_up):
                    s_up.wait_event(ev_comp[r]); mark_b(); dev_in[r].copy_(host_in, non_blocking=True); mark_e(); ev_up[r].record(s_up)

            def comp_t(i, mark_b, mark_e):
                r = i % RING
                vs = local_views(i)
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(ev_up[r]); s_comp.wait_event(ev_down[r]); mark_b()
                    rings[r].render_views(dev_views[r], [settings[v] for v in vs], [ups_d[v % len(ups_d)] for v in vs])
                    mark_e(); ev_comp[r].record(s_comp)

            def down_t(i, mark_b, mark_e):
                r = i % RING
                with torch.cuda.stream(s_down):
                    s_down.wait_event(ev_comp[r]); mark_b(); host_out[r][:nflat].copy_(rings[r].grads.flat, non_blocking=True); mark_e(); ev_down[r].record(s_down)

            torch.cuda.synchronize(dev)
            origin = torch.cuda.Event(enable_timing=True); origin.record()
            for st_ in (s_up, s_comp, s_down):
                st_.wait_event(origin)
            staged("up", s_up, up_t, 200)
            for i in range(200, 200 + TL):
                if i + 1 < 200 + TL:
                    staged("up", s_up, up_t, i + 1)
                staged("comp", s_comp, comp_t, i)
                staged("down", s_down, down_t, i)
            torch.cuda.synchronize(dev)
            iv = {k: [(origin.elapsed_time(b_), origin.elapsed_time(e_)) for b_, e_ in v] for k, v in marks.items()}

            def covered(a, others):          # fraction of interval a that some interval of `others` covers
                tot = 0.0
                for b_, e_ in others:
                    tot += max(0.0, min(a[1], e_) - max(a[0], b_))
                return min(1.0, tot / max(a[1] - a[0], 1e-9))
            mid = slice(3, TL - 1)            # steady state
            timeline = {
                "steps": TL, "ms_mean": {k: round(float(np.mean([e_ - b_ for b_, e_ in v[mid]])), 4) for k, v in iv.items()},
                "period_ms": round((iv["down"][TL - 2][1] - iv["down"][3][1]) / (TL - 5), 4),
                "compute_under_upload": round(float(np.mean([covered(c_, iv["up"]) for c_ in iv["comp"][mid]])), 3),
                "compute_under_download": round(float(np.mean([covered(c_, iv["down"]) for c_ in iv["comp"][mid]])), 3),
                "upload_under_download": round(float(np.mean([covered(u_, iv["down"]) for u_ in iv["up"][mid]])), 3),
                "intervals_ms_first_6_steps": {k: [[round(b_, 3), round(e_, 3)] for b_, e_ in v[:6]] for k, v in iv.items()},
                "note": "CUDA events around every stage on its own stream, one clock; fractions = share of the stage's duration during which a stage of the other kind was running"}
        e2e = {"value": P * vpg * world * e2e_steps / (float(ms_e.item()) * 1e-3), "unit": "splats/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": step_ms, "steps": e2e_steps,
               "wall_ms_per_step": (time.perf_counter() - t0) * 1e3 / e2e_steps,
               "copies_per_step": {"h2d": 1, "d2h": 2}, "link_gbs_alone": link,
               "link_gbs_in_pipeline": {"h2d": h2d / (step_ms * 1e-3) / 1e9, "d2h": d2h / (step_ms * 1e-3) / 1e9},
               "host_buffers_numa_local": bool(hostmem.gpu_local_cpus(dev)), "loss": float(host_out[(100 + e2e_steps - 1) % RING][nflat]),
               "collective": rings[0].collective if world > 1 else "none", "timeline": timeline,
               "note": "public API (ViewShardedRasterizer.render_views [+ all_reduce]); packed inputs from / flat gradient + loss to "
                       "pinned host memory every step, one copy per direction (+4 bytes of loss); upload, compute and download of "
                       "consecutive steps overlap on 3 streams"}

    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
    known = {k: v for k, v in kern.items() if kernel_algorithmic_bytes(k, P, M, H, W, n_inst)}
    dom = max(known, key=known.get) if known else None
    roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None, "peak_source": peak_src}
    if dom:
        kb = kernel_algorithmic_bytes(dom, P, M, H, W, n_inst)
        ach = kb / (kern[dom] * 1e-3) / 1e9
        step_bytes = algorithmic_bytes(P, M, H, W, n_inst) * vpg
        roof.update({"kernel": dom, "kernel_ms": kern[dom], "kernel_algorithmic_bytes": kb, "achieved": ach, "frac": ach / peak,
                     "kernels_ms_per_view": kern,
                     "kernels_frac": {k: (kernel_algorithmic_bytes(k, P, M, H, W, n_inst) or 0) / (v * 1e-3) / 1e9 / peak
                                      for k, v in kern.items()},
                     "step": {"algorithmic_bytes": step_bytes, "n_inst": n_inst, "achieved": step_bytes / (ms_per_step * 1e-3) / 1e9,
                              "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak},
                     "note": "render kernels are issue-bound, not HBM-bound (DESIGN.md): see `issue` for the bound that applies"})
        tr, src = committed_ncu("dram_bytes_per_launch")
        if tr and a.workload == "cfg2" and a.opacity == "trained" and dom in tr:
            roof["traffic"] = tr[dom]
        roof["traffic_source"] = src
        # the bound that does apply to the render kernels: warp instructions issued vs the SMs' issue rate
        inst, src = committed_ncu("warp_inst_per_launch")
        if inst and a.workload == "cfg2" and a.opacity == "trained" and clocks and clocks.get("sm_mhz"):
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            peak_issue = sms * 4 * clocks["sm_mhz"] * 1e6              # warp instructions per second (1 per SMSP per clock)
            roof["issue"] = {"unit": "warp-inst/s", "peak": peak_issue, "source": src,
                             "kernels": {k: {"warp_inst": inst[k], "achieved": inst[k] / (kern[k] * 1e-3), "frac": inst[k] / (kern[k] * 1e-3) / peak_issue}
                                         for k in kern if k in inst}}
    out = {
        "metric": "splats/sec fwd+bwd @ %dx%d" % (H, W), "value": value, "unit": "splats/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "baseline_config": WORKLOADS[a.workload]["what"], "views_per_gpu_per_step": vpg,
                   "view_set": a.views, "l2_flush_between_steps": True,
                   "n_inst_view0": n_inst, "parallelism": "view-sharded dp%d, replicated Gaussians, 1 all-reduce of %d MB per step (%s)"
                   % (world, vsr.grads.nbytes() >> 20, vsr.collective) if world > 1 else "single GPU",
                   "collective_check": check,
                   "wall_ms_per_step_incl_flush": (wall1 - wall0) * 1e3 / a.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "e2e": e2e,
    }
    if world == 1 and not a.no_cpu_baseline:
        nv = 2 if P <= 200000 else 1
        val, sec, threads = time_cpu_oracle(a, cloud, cams, ups, nv, 1 if P <= 200000 else 0)
        out["cpu_baseline"] = {"value": val, "unit": "splats/s", "cores": threads, "kind": "port",
                               "sample": "%d full view(s) fwd+bwd of the same workload (oracle/dgr_oracle.c, float32, OpenMP)" % nv,
                               "seconds_per_view": sec, "cpu": cpu_model()}
    if world == 1 and not a.no_rows and a.workload == "cfg2":
        out["other_shapes"] = measure_other_shapes(dev)
        out["next_rows"] = measure_next_rows(dev)
    print(json.dumps(out), flush=True)


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        run_ours(a, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
