#!/usr/bin/env python
"""Experiment driver (not a bench line): gradients on host memory against gradients on device memory.

C3 (2400 x 1800, reference solids, round_through_float = 0), one process, one GPU:
- alternates c5_render_grad (host g in, host gradients out) and c5_render_grad_device (g and gradients in
  torch CUDA tensors, no stats), each followed by a device synchronisation, --rounds times, and prints the
  wall clock per call;
- profiles one c5_render_grad_device and one c5_update_fields_device with torch.profiler and prints the
  device time of the gradient scatter and the field gather;
- times one fit step, autograd.render forward (field upload + image) + loss + backward, on CUDA tensors
  against CPU tensors.
Then, on C4's grid at 1200 x 900 with the reference solids, the backward of autograd.light_curve over
--views views (CUDA tensors), per view. The first line names the GPU, its power limit and max SM clock,
read in the same run.

    python scripts/time_grad_device.py > profiles/r08_grad_device_one_b200.jsonl
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from course5_b200 import api, autograd, hostlib, synth  # noqa: E402
from time_grad import gpu_info  # noqa: E402

OPS = {"scatter": "GradScatterOp", "gather": "FieldGatherOp"}


def setup(name, res=None):
    mesh, vk = synth.make_config(name)
    roche, sphere = hostlib.make_solids(vk["D"])
    res_x, res_y = res or (vk["res_x"], vk["res_y"])
    view = api.make_view(res_x, res_y, X=vk["X"], Y=vk["Y"], I=vk["I"], alpha_limit=vk["alpha_limit"],
                         round_through_float=0)
    ctx = api.Context(devices=(0,))
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    ctx.upload_solids(roche, True)
    ctx.upload_solids(sphere, False)
    return ctx, mesh, view, vk


def op_times(ctx, view, d_g, ga, gq, a, q):
    """Device milliseconds of the scatter (in one render_grad_device) and the gather (one update_fields_device)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stats=False)
        ctx.update_fields_device(a.data_ptr(), q.data_ptr())
        torch.cuda.synchronize()
    out = {k: 0.0 for k in OPS}
    for ev in prof.events():
        dt = getattr(ev, "device_time_total", None)
        if dt is None:
            dt = ev.cuda_time_total
        for k, sub in OPS.items():
            if dt and sub in ev.name:
                out[k] += dt / 1e3
    return out


def fit_step(ctx, view, alpha, q):
    """autograd.render forward (update_fields + image), a loss over the pixels outside the solids, backward."""
    import torch
    a = alpha.clone().requires_grad_(True)
    b = q.clone().requires_grad_(True)
    img = autograd.render(ctx, view, a, b)
    loss = torch.nan_to_num(img, nan=0.0).pow(2).sum()
    loss.backward()
    if a.is_cuda:
        torch.cuda.synchronize()
    return a.grad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--views", type=int, default=16)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    print(json.dumps(gpu_info()), flush=True)

    ctx, mesh, view, vk = setup("C3")
    with ctx:
        common = dict(workload="C3", res=[view.res_x, view.res_y], n_tets=int(mesh.n_tets))
        g = np.random.default_rng(args.seed).normal(size=(view.res_y, view.res_x, 2))
        d_g = torch.tensor(g, device="cuda")
        ga = torch.empty(mesh.n_tets, dtype=torch.float64, device="cuda")
        gq = torch.empty_like(ga)
        ctx.render_grad(view, g)
        ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr())  # makes the device permutation
        walls = {"render_grad": [], "render_grad_device": []}
        for _ in range(args.rounds):
            t0 = time.perf_counter()
            ha, hq = ctx.render_grad(view, g)
            torch.cuda.synchronize()
            walls["render_grad"].append((time.perf_counter() - t0) * 1e3)
            host_stats = ctx.last_stats
            t0 = time.perf_counter()
            ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stats=False)
            torch.cuda.synchronize()
            walls["render_grad_device"].append((time.perf_counter() - t0) * 1e3)
        dev_stats = ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr())
        err = max(float(np.abs(ga.cpu().numpy() - ha).max() / np.abs(ha).max()),
                  float(np.abs(gq.cpu().numpy() - hq).max() / np.abs(hq).max()))
        for k, w in walls.items():
            st = host_stats if k == "render_grad" else dev_stats
            print(json.dumps(dict(common, call=k, ms_wall_median=float(np.median(w)), ms_wall=w,
                                  ms_walk=st["ms_walk"], ms_d2h=st["ms_d2h"], ms_total=st["ms_total"],
                                  tet_steps=int(st["tet_steps"]), grazing_rays=int(st["grazing_rays"]))), flush=True)
        print(json.dumps(dict(common, check="device vs host gradients", max_err_rel_to_max=err)), flush=True)

        a = torch.tensor(mesh.alpha, device="cuda")
        q = torch.tensor(mesh.q, device="cuda")
        op_times(ctx, view, d_g, ga, gq, a, q)  # warm
        t = op_times(ctx, view, d_g, ga, gq, a, q)
        print(json.dumps(dict(common, profile="ops", device_ms=t, bytes_scatter=int(2 * (8 + 8) * mesh.n_tets + 4 * mesh.n_tets),
                              bytes_gather=int((8 + 8 + 8 + 8) * mesh.n_tets + 4 * mesh.n_tets))), flush=True)

        steps = {"cuda": [], "cpu": []}
        fields = {"cuda": (a, q), "cpu": (a.cpu(), q.cpu())}
        for dev in steps:  # warm
            fit_step(ctx, view, *fields[dev])
        for _ in range(args.rounds):
            for dev in steps:
                t0 = time.perf_counter()
                fit_step(ctx, view, *fields[dev])
                steps[dev].append((time.perf_counter() - t0) * 1e3)
        for dev, w in steps.items():
            print(json.dumps(dict(common, call=f"autograd.render step ({dev} tensors)", ms_wall_median=float(np.median(w)),
                                  ms_wall=w)), flush=True)

    ctx, mesh, view, vk = setup("C4")
    with ctx:
        views = []
        for k in range(args.views):
            v = api.make_view(view.res_x, view.res_y, X=vk["X"] + 2.0 * k / args.views, Y=vk["Y"], I=vk["I"],
                              alpha_limit=vk["alpha_limit"], round_through_float=0)
            views.append(v)
        w = torch.randn(len(views), 2, dtype=torch.float64, device="cuda")
        walls = []
        for r in range(args.rounds + 1):
            a = torch.tensor(mesh.alpha, device="cuda", requires_grad=True)
            q = torch.tensor(mesh.q, device="cuda", requires_grad=True)
            lc = autograd.light_curve(ctx, views, a, q)
            loss = (lc * w).sum()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loss.backward()
            torch.cuda.synchronize()
            if r:
                walls.append((time.perf_counter() - t0) * 1e3 / len(views))
        print(json.dumps(dict(workload="C4", res=[view.res_x, view.res_y], n_tets=int(mesh.n_tets), views=len(views),
                              call="light_curve backward (cuda tensors), per view",
                              ms_wall_median=float(np.median(walls)), ms_wall=walls)), flush=True)


if __name__ == "__main__":
    main()
