#!/usr/bin/env python
"""Experiment driver (not a bench line): what a gradient of a view costs against the view itself.

C3 (2400 x 1800, reference solids, round_through_float = 0). The script alternates c5_render_raw and
c5_render_grad (both gradients, g ~ N(0, 1) per pixel) --rounds times in one process and prints one JSON
line per call kind with the wall clock per call. Then it profiles one render_grad with torch.profiler and
prints the device time of the depth pass (pixel + grazing-ray kernel), the gradient pixel kernel, the
gradient grazing-ray kernel, the H2D copy of g and the D2H copies of the gradients. The atomics' cost is
measured, not estimated: the same profile with g = 0 runs the same gradient arithmetic but issues no
atomic (a contribution of 0 is not added). The first line names the GPU, its power limit and max SM
clock, read in the same run.

    python scripts/time_grad.py > profiles/r07_grad_c3_one_b200.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from course5_b200 import api, hostlib, synth  # noqa: E402

KERNELS = {"depth_pixel": "tet_walk_depth", "depth_graze": "grazing_rays_depth", "grad_pixel": "tet_walk_grad",
           "grad_graze": "grazing_rays_grad"}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        line = f"unavailable: {e}"
    return dict(gpu=line, query=q)


def device_times(ctx, view, g):
    """Device milliseconds of one render_grad, by kernel and copy kind (torch.profiler / CUPTI)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx.render_grad(view, g)  # warm
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.render_grad(view, g)
        torch.cuda.synchronize()
    out = {k: 0.0 for k in list(KERNELS) + ["h2d", "d2h", "other"]}
    for ev in prof.events():
        dt = getattr(ev, "device_time_total", None)
        if dt is None:
            dt = ev.cuda_time_total
        if not dt:
            continue
        name = ev.name
        key = next((k for k, sub in KERNELS.items() if sub in name), None)
        if key is None:
            key = "h2d" if "HtoD" in name else "d2h" if "DtoH" in name else "other"
        out[key] += dt / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    print(json.dumps(gpu_info()), flush=True)
    mesh, vk = synth.make_config("C3")
    roche, sphere = hostlib.make_solids(vk["D"])
    view = api.make_view(vk["res_x"], vk["res_y"], X=vk["X"], Y=vk["Y"], I=vk["I"], alpha_limit=vk["alpha_limit"],
                         round_through_float=0)
    g = np.random.default_rng(args.seed).normal(size=(vk["res_y"], vk["res_x"], 2))
    with api.Context(devices=(0,)) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        ctx.render_raw(view)
        ctx.render_grad(view, g)
        walls = {"render_raw": [], "render_grad": []}
        stats = {}
        for _ in range(args.rounds):
            t0 = time.perf_counter()
            img = ctx.render_raw(view)
            walls["render_raw"].append((time.perf_counter() - t0) * 1e3)
            stats["render_raw"] = img.stats
            t0 = time.perf_counter()
            ctx.render_grad(view, g)
            walls["render_grad"].append((time.perf_counter() - t0) * 1e3)
            stats["render_grad"] = ctx.last_stats
        common = dict(workload="C3", res=[vk["res_x"], vk["res_y"]], n_tets=int(mesh.n_tets),
                      tet_steps=int(stats["render_raw"]["tet_steps"]), grazing_rays=int(stats["render_raw"]["grazing_rays"]))
        for k, w in walls.items():
            print(json.dumps(dict(common, call=k, ms_wall_median=float(np.median(w)), ms_wall=w,
                                  ms_walk=stats[k]["ms_walk"], ms_d2h=stats[k]["ms_d2h"], ms_total=stats[k]["ms_total"])),
                  flush=True)
        for name, gg in (("g_normal", g), ("g_zero", np.zeros_like(g))):
            t = device_times(ctx, view, gg)
            print(json.dumps(dict(common, profile=name, device_ms=t,
                                  bytes_h2d=int(g.nbytes), bytes_d2h=int(2 * 8 * mesh.n_tets))), flush=True)


if __name__ == "__main__":
    main()
