#!/usr/bin/env python
"""Experiment driver (not a bench line): times c5_render on one context over the given devices
(the C3 workload, 2400 x 1800, reference solids), alternating a pageable and a page-locked host image
view by view. Prints one JSON line per image kind: host wall time per view (the call is synchronous),
the stats' ms_total / ms_d2h, and a digest of the last image. C5GPU_LIBRARY picks the build.

    C5GPU_LIBRARY=/path/to/libc5gpu.so python scripts/time_context.py --devices 0,1 --label new
"""
import argparse
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from course5_b200 import api, hostlib, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", default="0", help="CUDA ordinals of the one context, comma separated (may repeat)")
    ap.add_argument("--views", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--label", default="", help="copied into every line (which build ran)")
    args = ap.parse_args()
    devices = tuple(int(x) for x in args.devices.split(","))
    mesh, vk = synth.make_config("C3")
    roche, sphere = hostlib.make_solids(vk["D"])
    outs = {m: np.zeros((vk["res_y"], vk["res_x"], 2)) for m in ("pageable", "pinned")}
    wall = {m: [] for m in outs}
    stats = {m: [] for m in outs}
    with api.Context(devices=devices) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        view = api.make_view(vk["res_x"], vk["res_y"], X=vk["X"], Y=vk["Y"], I=vk["I"], alpha_limit=vk["alpha_limit"])
        ctx.host_register(outs["pinned"])
        for k in range(args.warmup + args.views):
            for m, out in outs.items():
                t0 = time.perf_counter()
                _, st = ctx.render(view, out=out)
                if k >= args.warmup:
                    wall[m].append((time.perf_counter() - t0) * 1e3)
                    stats[m].append(st)
        ctx.host_unregister(outs["pinned"])
    for m, out in outs.items():
        w = np.array(wall[m])
        print(json.dumps(dict(
            label=args.label, devices=list(devices), out=m, views=args.views, warmup=args.warmup,
            ms_median=float(np.median(w)), ms_p10=float(np.percentile(w, 10)), ms_p90=float(np.percentile(w, 90)),
            ms_min=float(w.min()), ms_max=float(w.max()),
            ms_total_median=float(np.median([s["ms_total"] for s in stats[m]])),
            ms_d2h_median=float(np.median([s["ms_d2h"] for s in stats[m]])),
            tet_steps=int(stats[m][-1]["tet_steps"]), n_devices=int(stats[m][-1]["n_devices"]),
            image_sha256=hashlib.sha256(out.tobytes()).hexdigest())), flush=True)


if __name__ == "__main__":
    main()
