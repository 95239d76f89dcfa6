#!/usr/bin/env python
"""Experiment driver (not a bench line): the pixel kernel of one view alone, C3 (2400 x 1800, reference solids) or
another workload of synth.CONFIGS, one view at a time on one context. Per view the stats' events give ms_walk (mask
done -> grazing-ray kernel done: counter zeroing, the ray order, the pixel kernel and the grazing-ray kernel) and
ms_graze (the grazing-ray kernel alone); their difference is the pixel kernel with the two small steps before it.
Also reads the card's name, power limit and max SM clock. Prints one JSON line. `--oblique` renders the oblique
view (X = 0.4, Y = 0.3) instead.

    python scripts/time_pixel_kernel.py [--workload C5t] [--oblique] --views 20 --label this
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from course5_b200 import api, hostlib, synth  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": int(q[2])} if len(q) == 3 else {"gpu": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="C3", choices=sorted(synth.CONFIGS))
    ap.add_argument("--oblique", action="store_true")
    ap.add_argument("--label", default="")
    args = ap.parse_args()
    mesh, vk = synth.make_config(args.workload)
    roche, sphere = hostlib.make_solids(vk["D"])
    flags = dict(X=0.4, Y=0.3, I=vk["I"]) if args.oblique else dict(X=vk["X"], Y=vk["Y"], I=vk["I"])
    rows = []
    with api.Context(devices=(0,)) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        view = api.make_view(vk["res_x"], vk["res_y"], alpha_limit=vk["alpha_limit"], **flags)
        for k in range(args.warmup + args.views):
            _, st = ctx.render(view)
            if k >= args.warmup:
                rows.append((st["ms_walk"] - st["ms_graze"], st["ms_graze"], st["ms_walk"], st["ms_total"]))
    a = np.asarray(rows)
    med = np.median(a, axis=0)
    print(json.dumps({"label": args.label, "workload": args.workload, "oblique": args.oblique, **card(), "views": args.views,
                      "ms_pixel_kernel_median": med[0], "ms_pixel_kernel_min": a[:, 0].min(), "ms_graze_median": med[1],
                      "ms_walk_median": med[2], "ms_total_median": med[3], "ms_total_min": a[:, 3].min()}), flush=True)


if __name__ == "__main__":
    main()
