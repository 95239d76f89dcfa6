#!/usr/bin/env python
"""Experiment driver (not a bench line): a light curve and its J v, view by view against one device call on the
lanes (c5_render_flux_device, c5_render_flux_jvp_device).

Cases, each with the reference solids and round_through_float = 0: C4's grid at 1200 x 900 with 16 and with 64
views, and C3 at 2400 x 1800 with 8 views (views spread over X, as in time_flux_grad.py). For each case, in one
process and alternated --rounds times after a warm-up round:
- jvp loop: the J v that autograd.light_curve ran before, rebuilt from public calls: per view c5_render_jvp_device
  into a whole-image tangent tensor, then a torch nansum, all on the current stream;
- jvp lanes n: c5_render_flux_jvp_device over all views with n = 1 .. 4 lanes;
- forward loop: the forward that autograd.light_curve ran before: sweep.render_light_curve (the pipelined
  c5_render_flux_submit loop, 3 lanes) and the copy of the totals to the device;
- forward lanes n: c5_render_flux_device into a CUDA tensor, n = 1 .. 4 lanes;
- J^T J v: c5_render_flux_jvp_device then c5_render_flux_grad_device with the tangent as g, 3 lanes.
Each call is timed by the host clock between two device synchronisations and reported per view (median, min and
max over the rounds); before it, the arm's lane count is set and one untimed call made, so that making and freeing
lanes is not timed. The fields and the direction are a fixed seeded draw; each arm's result is compared with the
loop's. The first line names the GPU, its power limit and max SM clock, read in the same run.

    python scripts/time_flux_jvp.py > profiles/r12_flux_jvp_one_b200.jsonl
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

from course5_b200 import sweep  # noqa: E402
from time_flux_grad import CASES, LANES, _stream, make_views, setup, timed  # noqa: E402
from time_grad import gpu_info  # noqa: E402


def loop_jvp(ctx, views, va, vq):
    """The view-by-view J v: a whole-image tangent per view, then nansum."""
    import torch
    sums = []
    for v in views:
        tangent = torch.zeros((v.res_y, v.res_x, 2), dtype=torch.float64, device="cuda")
        ctx.render_jvp_device(v, va.data_ptr(), vq.data_ptr(), tangent.data_ptr(), stream=_stream(), stats=False)
        sums.append(tangent.nansum(dim=(0, 1)))
    return torch.stack(sums)


def lanes_jvp(ctx, views, va, vq):
    import torch
    t = torch.empty((len(views), 2), dtype=torch.float64, device="cuda")
    ctx.render_flux_jvp_device(views, va.data_ptr(), vq.data_ptr(), t.data_ptr(), stream=_stream(), stats=False)
    return t


def loop_forward(ctx, views):
    import torch
    return torch.from_numpy(sweep.render_light_curve(ctx, views, in_flight=3)[0][:, 0]).to("cuda")


def lanes_forward(ctx, views):
    import torch
    t = torch.empty((len(views), 2), dtype=torch.float64, device="cuda")
    ctx.render_flux_device(views, t.data_ptr(), _stream(), stats=False)
    return t


def jtjv(ctx, views, va, vq, like):
    import torch
    t = torch.empty((len(views), 2), dtype=torch.float64, device="cuda")
    ga, gq = torch.empty_like(like), torch.empty_like(like)
    ctx.render_flux_jvp_device(views, va.data_ptr(), vq.data_ptr(), t.data_ptr(), stream=_stream(), stats=False)
    ctx.render_flux_grad_device(views, t.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=_stream(), stats=False)
    return ga


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--cases", default=",".join(f"{c}:{n}" for c, n in CASES), help="config:views,...")
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    print(json.dumps(gpu_info()), flush=True)
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
        rng = np.random.default_rng(args.seed)
        va = torch.tensor(rng.normal(size=mesh.n_tets) * mesh.alpha, device="cuda")
        vq = torch.tensor(rng.normal(size=mesh.n_tets) * mesh.q, device="cuda")

        arms = {"jvp loop": (1, "jvp", lambda: loop_jvp(ctx, views, va, vq))}
        for n in LANES:
            arms[f"jvp lanes {n}"] = (n, "jvp", lambda: lanes_jvp(ctx, views, va, vq))
        arms["forward loop"] = (3, "forward", lambda: loop_forward(ctx, views))
        for n in LANES:
            arms[f"forward lanes {n}"] = (n, "forward", lambda: lanes_forward(ctx, views))
        arms["JtJv lanes 3"] = (3, "jtjv", lambda: jtjv(ctx, views, va, vq, a0))
        walls = {k: [] for k in arms}
        ref = {}
        err = {}
        for r in range(args.rounds + 1):  # round 0 warms every arm
            for k, (lanes, kind, fn) in arms.items():
                ctx.set_views_in_flight(lanes)
                timed(fn)
                ms, out = timed(fn)
                if r:
                    walls[k].append(ms / n_views)
                out = out.cpu().numpy()
                if k.endswith("loop") or kind == "jtjv":
                    ref[kind] = out
                else:
                    e = float(np.abs(out - ref[kind]).max() / np.abs(ref[kind]).max())
                    err[k] = max(err.get(k, 0.0), e)
        for k, w in walls.items():
            line = dict(common, call=k, ms_per_view_median=float(np.median(w)), ms_per_view_min=float(np.min(w)),
                        ms_per_view_max=float(np.max(w)), ms_per_view=w)
            if k in err:
                line["max_err_rel_to_max_vs_loop"] = err[k]
            print(json.dumps(line), flush=True)
    for c in contexts.values():
        c[0].close()


if __name__ == "__main__":
    main()
