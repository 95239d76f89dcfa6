#!/usr/bin/env python
"""Experiment driver (not a bench line): what a light-curve frame costs through the flux calls against
moving its image to the host.

C3 (2400 x 1800, reference solids). For the cells' own fields ("plain") and for K seeded channel pairs,
K in --channels, the script alternates batches of --views views of the same view in one process:
- image path: plain renders through c5_render_submit with --in-flight views in flight into page-locked
  images; K-channel renders through c5_render_channels into a page-locked image (channels have no
  pipelined image call);
- flux path: c5_render_flux_submit with --in-flight views in flight (sweep.render_light_curve).
Per path it prints one JSON line with the medians over --rounds batches of the wall clock per view, and
the medians over all views of ms_walk (pixel + grazing-ray kernels) and ms_d2h (image path: the image
copy; flux path: the reduction plus the copy of the row sums). The first line names the GPU, its power
limit and max SM clock, read in the same run.

    python scripts/time_flux.py --channels 0,1,2,4,8 > profiles/r05_flux_c3_one_b200.jsonl
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

from course5_b200 import api, hostlib, sweep, synth  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        line = f"unavailable: {e}"
    return dict(gpu=line, query=q)


def median(stats, key):
    return float(np.median([s[key] for s in stats]))


def image_batch(ctx, view, k, n_views, in_flight, pinned):
    """Wall clock per view and per-view stats of the image path."""
    t0 = time.perf_counter()
    if k == 0:
        _, stats = sweep.render_sweep(ctx, [view] * n_views, in_flight=in_flight)
    else:
        stats = [ctx.render_channels(view, out=pinned)[1] for _ in range(n_views)]
    return (time.perf_counter() - t0) * 1e3 / n_views, stats


def flux_batch(ctx, view, k, n_views, in_flight):
    t0 = time.perf_counter()
    totals, stats = sweep.render_light_curve(ctx, [view] * n_views, in_flight=in_flight, channels=k > 0)
    return (time.perf_counter() - t0) * 1e3 / n_views, stats, totals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", default="0,1,2,4,8", help="pair counts; 0 = the cells' own fields")
    ap.add_argument("--views", type=int, default=20, help="views per batch")
    ap.add_argument("--rounds", type=int, default=5, help="alternating batches per path")
    ap.add_argument("--in-flight", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()
    import torch
    ks = [int(x) for x in args.channels.split(",")]
    print(json.dumps(gpu_info()), flush=True)
    mesh, vk = synth.make_config("C3")
    roche, sphere = hostlib.make_solids(vk["D"])
    rng = np.random.default_rng(args.seed)
    k_max = max(max(ks), 1)
    alpha = rng.uniform(0.1, 4.0, (k_max, mesh.n_tets))
    q = rng.uniform(0.1, 4.0, (k_max, mesh.n_tets))
    view = api.make_view(vk["res_x"], vk["res_y"], X=vk["X"], Y=vk["Y"], I=vk["I"], alpha_limit=vk["alpha_limit"])
    with api.Context(devices=(0,)) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        for k in ks:
            if k:
                ctx.upload_channels(alpha[:k], q[:k])
            pinned = torch.zeros((vk["res_y"], vk["res_x"], k, 2), dtype=torch.float64).pin_memory().numpy() if k else None
            image_batch(ctx, view, k, args.in_flight + 1, args.in_flight, pinned)   # warm-up
            flux_batch(ctx, view, k, args.in_flight + 1, args.in_flight)
            img_wall, img_stats, flux_wall, flux_stats = [], [], [], []
            for _ in range(args.rounds):
                w, st = image_batch(ctx, view, k, args.views, args.in_flight, pinned)
                img_wall.append(w)
                img_stats += st
                w, st, totals = flux_batch(ctx, view, k, args.views, args.in_flight)
                flux_wall.append(w)
                flux_stats += st
            assert all(np.array_equal(t, totals[0]) for t in totals)
            assert flux_stats[-1]["tet_steps"] == img_stats[-1]["tet_steps"] and flux_stats[-1]["walk_errors"] == 0
            common = dict(workload="C3", res=[vk["res_x"], vk["res_y"]], channels=k, views=args.views,
                          rounds=args.rounds, tet_steps=int(flux_stats[-1]["tet_steps"]))
            print(json.dumps(dict(common, path="image",
                                  call="c5_render_submit, %d in flight, page-locked" % args.in_flight if k == 0 else
                                  "c5_render_channels, page-locked",
                                  ms_wall_per_view=float(np.median(img_wall)), ms_wall_batches=img_wall,
                                  ms_walk=median(img_stats, "ms_walk"), ms_d2h=median(img_stats, "ms_d2h"))), flush=True)
            print(json.dumps(dict(common, path="flux", call="c5_render_flux_submit, %d in flight" % args.in_flight,
                                  ms_wall_per_view=float(np.median(flux_wall)), ms_wall_batches=flux_wall,
                                  ms_walk=median(flux_stats, "ms_walk"), ms_d2h=median(flux_stats, "ms_d2h"),
                                  total=totals[0].tolist())), flush=True)


if __name__ == "__main__":
    main()
