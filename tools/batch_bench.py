"""Batched multi-view rendering vs the loop of single-view calls: forward + backward of V views of one cloud per step.

For each shape both ways run in the same process, alternated step by step after a warm-up, with the 256 MB L2 flush between
steps that bench.py uses and CUDA events around each step:
  loop:    multiview.ViewShardedRasterizer.render_views (V single-view forwards, V backwards accumulating into one flat buffer);
  batched: rasterizer.forward_batch_impl + backward_batch_impl (one batched per-Gaussian stage each way).
Reports median / spread per step, splats/s = P V / step, per-kernel microseconds (dgr_profile_enable, separate pass), peak scratch
memory of one step, the agreement of the two ways' outputs at the timed size, and the GPU's name, power limit and clocks.

    python tools/batch_bench.py --out profiles/batch_bench.json [--steps 30 --warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dreamgaussian_b200 import _lib, multiview, scene  # noqa: E402
from dreamgaussian_b200 import rasterizer as R  # noqa: E402

SHAPES = (("cfg3_500k_512_deg3_v8", 500000, 512, 3, 8),
          ("100k_800_deg3_v8", 100000, 800, 3, 8),
          ("stage1_20k_256_deg0_v4", 20000, 256, 0, 4))


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + q, "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=60).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(), "nvidia-smi": repr(e)}


def run_shape(name, P, res, deg, V, steps, warmup):
    dev = torch.device("cuda")
    t = lambda a: torch.tensor(np.asarray(a, np.float32), device=dev)
    cloud = scene.make_cloud(P, deg, seed=0, sigma=0.595 * P ** (-1.0 / 3.0), opacity="trained")
    params = {k: t(v) for k, v in cloud.items()}
    M = (deg + 1) ** 2
    cams = scene.bench_views(V, res, res)
    sets = [R.GaussianRasterizationSettings(image_height=res, image_width=res, tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=t(np.ones(3)),
                                            scale_modifier=1.0, viewmatrix=t(c.world_view_transform), projmatrix=t(c.full_proj_transform),
                                            sh_degree=deg, campos=t(c.camera_center), prefiltered=False, debug=False) for c in cams]
    g = torch.Generator(device=dev).manual_seed(1)
    gC = torch.randn((V, 3, res, res), device=dev, generator=g)
    gA = torch.randn((V, 1, res, res), device=dev, generator=g)
    ups = [(gC[v], None, gA[v]) for v in range(V)]
    vsr = multiview.ViewShardedRasterizer(P, M, dev)
    bg = {k: torch.empty_like(v) for k, v in params.items()}
    bm2d = torch.empty((V, P, 3), device=dev)
    args = (params["means3D"], params["shs"], params["opacities"], params["scales"], params["rotations"])
    out = {}

    def loop():
        vsr.render_views(params, sets, ups)

    def batched():
        color, radii, depth, alpha, st = R.forward_batch_impl(sets, args[0], args[1], args[2], args[3], args[4])
        R.backward_batch_impl(st, gC, None, gA, bg["means3D"], bm2d, bg["shs"], bg["opacities"], bg["scales"], bg["rotations"])
        out["last"] = (color, radii)

    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    for _ in range(warmup):
        loop(); batched()
    torch.cuda.synchronize()
    times = {"loop": [], "batched": []}
    for i in range(steps):
        for way, fn in (("loop", loop), ("batched", batched)) if i % 2 == 0 else (("batched", batched), ("loop", loop)):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            times[way].append(e0.elapsed_time(e1))
    res_d = {"P": P, "res": res, "sh_degree": deg, "views": V, "opacity": "trained", "steps": steps, "warmup": warmup,
             "l2_flush_between_steps": True}
    for way, ts in times.items():
        ts = np.asarray(ts)
        res_d[way] = {"ms_per_step_median": float(np.median(ts)), "ms_p10": float(np.percentile(ts, 10)), "ms_p90": float(np.percentile(ts, 90)),
                      "ms_min": float(ts.min()), "ms_max": float(ts.max()), "splats_per_s": P * V / (float(np.median(ts)) * 1e-3)}
    res_d["batched_over_loop"] = res_d["batched"]["ms_per_step_median"] / res_d["loop"]["ms_per_step_median"]
    # per-kernel time (separate pass, events around every launch), microseconds per STEP
    lib = _lib.load()
    for way, fn in (("loop", loop), ("batched", batched)):
        lib.dgr_profile_enable(1)
        n = 4
        for _ in range(n):
            flush.zero_(); fn()
        torch.cuda.synchronize()
        k = {}
        for kn, ms in _lib.profile_collect():
            k[kn] = k.get(kn, 0.0) + ms * 1e3 / n
        lib.dgr_profile_enable(0)
        res_d[way]["kernel_us_per_step"] = {a: round(b, 2) for a, b in sorted(k.items(), key=lambda x: -x[1])}
    # peak memory of one step (scratch + outputs + gradients), over what the inputs / buffers already hold
    for way, fn in (("loop", loop), ("batched", batched)):
        torch.cuda.synchronize(); base = torch.cuda.memory_allocated(); torch.cuda.reset_peak_memory_stats()
        fn(); torch.cuda.synchronize()
        res_d[way]["peak_step_bytes"] = int(torch.cuda.max_memory_allocated() - base)
    # agreement at the timed size: images / radii per view against single-view forwards, summed gradients against the loop
    loop(); batched(); torch.cuda.synchronize()
    color_b, radii_b = out["last"]
    img_max, rad_mis = 0.0, 0
    for v in range(V):
        c, r, _, _, _ = R.forward_impl(sets[v], args[0], args[1], None, args[2], args[3], args[4], None)
        img_max = max(img_max, float((c - color_b[v]).abs().max()))
        rad_mis = max(rad_mis, int((r != radii_b[v]).sum()))
    gerr = {}
    for k in ("means3D", "shs", "opacities", "scales", "rotations"):
        want = vsr.grads.views[k]
        gerr[k] = float((bg[k] - want).abs().max()) / (float(want.abs().max()) + 1e-30)
    res_d["agreement"] = {"color_max_abs_diff": img_max, "radii_mismatch_max_per_view": rad_mis, "grad_max_rel_diff": gerr,
                          "ok": img_max <= 1e-2 and rad_mis <= 2 and max(gerr.values()) <= 2e-4}
    return res_d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batch_bench.json"))
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shapes", default="all", help="comma-separated shape names, or 'all'")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_bench needs a CUDA device")
    info = {"gpu_before": gpu_info(), "host_layer_of_the_loop": "compiled" if R._FAST is not None else "ctypes",
            "host_layer_of_the_batch": "ctypes"}
    shapes = [s for s in SHAPES if a.shapes == "all" or s[0] in a.shapes.split(",")]
    results = {}
    for s in shapes:
        results[s[0]] = run_shape(*s, steps=a.steps, warmup=a.warmup)
        print(json.dumps({s[0]: {w: results[s[0]][w]["ms_per_step_median"] for w in ("loop", "batched")},
                          "agreement_ok": results[s[0]]["agreement"]["ok"]}), flush=True)
    info["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump({"gpu": info, "shapes": results}, f, indent=1)


if __name__ == "__main__":
    main()
