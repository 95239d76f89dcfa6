#!/usr/bin/env python
"""Experiment driver (not a bench line): the gradient of a light curve, view by view against one
c5_render_flux_grad_device call on the lanes.

Cases, each with the reference solids and round_through_float = 0: C4's grid at 1200 x 900 with 16 and with
64 views, and C3 at 2400 x 1800 with 8 views (views spread over X, as in time_grad_device.py). For each case,
in one process and alternated --rounds times after a warm-up round:
- (a) the view-by-view backward that autograd.light_curve ran before, rebuilt here from public calls: per
  view a device fill of a band-sized g with the view's upstream pair, c5_render_grad_device, and a torch
  add into the sums, all on the current stream;
- (b) c5_render_flux_grad_device over all views with 1, 2, 3 and 4 lanes (set_views_in_flight).
Each call is timed by the host clock between two device synchronisations and reported per view; before it,
the arm's lane count is set and one untimed call made, so that making and freeing lanes is not timed. Then a whole
fit step (light curve forward, squared-error loss, backward, an Adam step) on CUDA tensors, alternated the same
way: the light curve as it was before (per-view blocking c5_render_flux forward, arm (a) backward) against
autograd.light_curve at 1 to 4 lanes. The first line names the GPU, its power limit and max SM clock, read in
the same run.

    python scripts/time_flux_grad.py > profiles/r10_flux_grad_one_b200.jsonl
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

LANES = (1, 2, 3, 4)
CASES = (("C4", 16), ("C4", 64), ("C3", 8))


def setup(name):
    mesh, vk = synth.make_config(name)
    roche, sphere = hostlib.make_solids(vk["D"])
    ctx = api.Context(devices=(0,))
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    ctx.upload_solids(roche, True)
    ctx.upload_solids(sphere, False)
    return ctx, mesh, vk


def make_views(vk, n):
    return [api.make_view(vk["res_x"], vk["res_y"], X=vk["X"] + 2.0 * k / n, Y=vk["Y"], I=vk["I"],
                          alpha_limit=vk["alpha_limit"], round_through_float=0) for k in range(n)]


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def loop_backward(ctx, views, go, like):
    """The view-by-view backward: fill, render_grad_device, add."""
    import torch
    sums = [torch.zeros_like(like), torch.zeros_like(like)]
    for k, v in enumerate(views):
        g = go[k].expand(v.res_y, v.res_x, 2).contiguous()  # whole-image views: the band is the image
        ga, gq = torch.empty_like(like), torch.empty_like(like)
        ctx.render_grad_device(v, g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=_stream(), stats=False)
        sums[0] += ga
        sums[1] += gq
    return sums


def lanes_backward(ctx, views, go, like):
    import torch
    ga, gq = torch.empty_like(like), torch.empty_like(like)
    ctx.render_flux_grad_device(views, go.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=_stream(), stats=False)
    return [ga, gq]


def _parent_light_curve():
    """autograd.light_curve on CUDA tensors as it was before c5_render_flux_grad_device."""
    import torch

    class LightCurve(torch.autograd.Function):
        @staticmethod
        def forward(fn_ctx, ctx, views, alpha, q):
            ctx.update_fields_device(alpha.detach().data_ptr(), q.detach().data_ptr(), _stream())
            totals = np.stack([ctx.render_flux(v)[1][0] for v in views])
            fn_ctx.c5, fn_ctx.views = ctx, views
            fn_ctx.save_for_backward(alpha)
            return torch.from_numpy(totals).to(alpha.device)

        @staticmethod
        def backward(fn_ctx, grad_output):
            alpha, = fn_ctx.saved_tensors
            go = grad_output.detach().to(torch.float64)
            ga, gq = loop_backward(fn_ctx.c5, fn_ctx.views, go, alpha)
            return None, None, ga, gq

    return LightCurve.apply


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--cases", default=",".join(f"{c}:{n}" for c, n in CASES), help="config:views,...")
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    print(json.dumps(gpu_info()), flush=True)
    parent_lc = _parent_light_curve()
    contexts = {}
    for case in args.cases.split(","):
        name, n_views = case.split(":")
        n_views = int(n_views)
        if name not in contexts:
            for c in contexts.values():
                c[0].close()
            contexts = {name: setup(name)}
        ctx, mesh, vk = contexts[name]
        views = make_views(vk, n_views)
        common = dict(workload=name, res=[vk["res_x"], vk["res_y"]], n_tets=int(mesh.n_tets), views=n_views)
        a0 = torch.tensor(mesh.alpha, device="cuda")
        q0 = torch.tensor(mesh.q, device="cuda")
        ctx.update_fields_device(a0.data_ptr(), q0.data_ptr(), _stream())
        go = torch.tensor(np.random.default_rng(args.seed).normal(size=(n_views, 2)), device="cuda")

        # each arm's lane count is set, and one call made, outside the timed region: a change of
        # set_views_in_flight makes or frees lanes and their buffers, which a fit loop does once
        arms = {"loop": (1, lambda: loop_backward(ctx, views, go, a0))}
        for n in LANES:
            arms[f"lanes_{n}"] = (n, lambda: lanes_backward(ctx, views, go, a0))
        walls = {k: [] for k in arms}
        ref = None
        err = {}
        for r in range(args.rounds + 1):  # round 0 warms every arm
            for k, (lanes, fn) in arms.items():
                ctx.set_views_in_flight(lanes)
                timed(fn)
                ms, out = timed(fn)
                if r:
                    walls[k].append(ms / n_views)
                if k == "loop":
                    ref = [x.cpu().numpy() for x in out]
                else:
                    e = max(float(np.abs(x.cpu().numpy() - y).max() / np.abs(y).max()) for x, y in zip(out, ref))
                    err[k] = max(err.get(k, 0.0), e)
        ctx.set_views_in_flight(4)
        scratch = torch.empty_like(a0)
        st = ctx.render_flux_grad_device(views, go.data_ptr(), scratch.data_ptr(), 0)
        for k, w in walls.items():
            line = dict(common, call="backward: view-by-view loop (fill, render_grad_device, add)" if k == "loop"
                        else f"backward: render_flux_grad_device, {k.split('_')[1]} lanes",
                        ms_per_view_median=float(np.median(w)), ms_per_view=w)
            if k != "loop":
                line["max_err_rel_to_max_vs_loop"] = err[k]
            print(json.dumps(line), flush=True)
        print(json.dumps(dict(common, stats_4_lanes=dict(ms_total=st["ms_total"], tet_steps=int(st["tet_steps"]),
                                                         grazing_rays=int(st["grazing_rays"]),
                                                         pixels=int(st["pixels"])))), flush=True)

        target = None
        steps = {"before": None}
        steps.update({f"after_{n}": n for n in LANES})
        fits = {}
        for k in steps:
            a = a0.clone().requires_grad_(True)
            b = q0.clone().requires_grad_(True)
            fits[k] = (a, b, torch.optim.Adam([a, b], lr=1e-4))
        with torch.no_grad():
            target = autograd.light_curve(ctx, views, a0, q0) * 1.01
        walls = {k: [] for k in steps}

        def fit_step(k):
            a, b, opt = fits[k]
            opt.zero_grad()
            if steps[k] is None:
                lc = parent_lc(ctx, views, a, b)
            else:
                lc = autograd.light_curve(ctx, views, a, b)
            loss = ((lc - target) / target).pow(2).sum()
            loss.backward()
            opt.step()

        for r in range(args.rounds + 1):
            for k in steps:
                ctx.set_views_in_flight(steps[k] or 1)
                timed(lambda: fit_step(k))
                ms, _ = timed(lambda: fit_step(k))
                if r:
                    walls[k].append(ms)
        for k, w in walls.items():
            call = ("fit step before: per-view render_flux forward, view-by-view backward" if k == "before" else
                    f"fit step after: autograd.light_curve, {steps[k]} lanes")
            print(json.dumps(dict(common, call=call + " (forward, loss, backward, Adam)",
                                  ms_step_median=float(np.median(w)), ms_step=w)), flush=True)
    for c in contexts.values():
        c[0].close()


if __name__ == "__main__":
    main()
