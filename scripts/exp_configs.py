#!/usr/bin/env python
"""Experiment driver (not a bench line): renders named configurations on one GPU and prints one
JSON line per (config, precision, row band) with per-phase device times and the walk kernel's
algorithmic GB/s.

    python scripts/exp_configs.py C1 C3 --debug mask_tile=1604
"""
import argparse
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
    ap.add_argument("configs", nargs="+")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-solids", action="store_true")
    ap.add_argument("--view", default=None, help="X,Y override (units of pi)")
    ap.add_argument("--res", default=None, help="res_x,res_y override")
    ap.add_argument("--precision", default="64")
    ap.add_argument("--rows", default=None, help="semicolon-separated row bands a,b;c,d to render separately")
    ap.add_argument("--debug", default="", help="c5_debug_set knobs, key=value[,key=value]")
    args = ap.parse_args()
    import torch
    dev = torch.device("cuda", 0)
    for name in args.configs:
        t0 = time.perf_counter()
        mesh, view = synth.make_config(name)
        t_gen = time.perf_counter() - t0
        if args.view:
            view["X"], view["Y"] = (float(x) for x in args.view.split(","))
        if args.res:
            view["res_x"], view["res_y"] = (int(x) for x in args.res.split(","))
        solids = None if args.no_solids else hostlib.make_solids(view["D"])
        ctx = api.Context(devices=(0,))
        for kv in (kv for kv in args.debug.split(",") if kv):
            ctx.debug_set(kv.split("=")[0], int(kv.split("=")[1]))
        t0 = time.perf_counter()
        info = ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        t_up = time.perf_counter() - t0
        if solids is not None:
            ctx.upload_solids(solids[0], True)
            ctx.upload_solids(solids[1], False)
        out = torch.empty((view["res_y"], view["res_x"], 2), dtype=torch.float64, device=dev)
        bands = [None] if not args.rows else [tuple(int(x) for x in b.split(",")) for b in args.rows.split(";")]
        for prec, band in ((int(p), bb) for p in args.precision.split(",") for bb in bands):
            extra = {} if band is None else dict(row_begin=band[0], row_end=band[1])
            v = api.make_view(view["res_x"], view["res_y"], X=view["X"], Y=view["Y"], I=view["I"],
                              alpha_limit=view["alpha_limit"], precision=prec, **extra)
            for _ in range(2):
                st = ctx.render_device(v, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
            acc = {k: [] for k in ("ms_rotate", "ms_bvh", "ms_mask", "ms_walk", "ms_graze", "ms_total")}
            for _ in range(args.reps):
                st = ctx.render_device(v, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
                for k in acc:
                    acc[k].append(st[k])
            walk = float(np.median(acc["ms_walk"]))
            pixels = view["res_x"] * (view["res_y"] if band is None else band[1] - band[0])
            gbs = (st["tet_steps"] * 72 + pixels * 16) / (walk * 1e-3) / 1e9
            print(json.dumps({
                "config": name, "view": [view["X"], view["Y"]], "precision": prec, "grazing_rays": st["grazing_rays"], "rows": band, "n_tets": mesh.n_tets,
                "res": [view["res_x"], view["res_y"]], "tet_steps": st["tet_steps"],
                "hit_pixels": st["hit_pixels"], "solid_pixels": st["solid_pixels"],
                **{k: round(float(np.median(x)), 4) for k, x in acc.items()},
                "walk_Gsteps_per_s": round(st["tet_steps"] / walk / 1e6, 2), "walk_alg_GBps": round(gbs, 1),
                "frac_of_6455.9": round(gbs / 6455.9, 3), "gen_s": round(t_gen, 2), "upload_s": round(t_up, 3),
                "device_MB": round(info.device_bytes / 1e6, 1), "bfaces": info.n_boundary_faces,
                "debug": args.debug, "library": os.path.basename(os.environ.get("C5GPU_LIBRARY", "libc5gpu.so"))}), flush=True)
        ctx.close()
        del mesh


if __name__ == "__main__":
    main()
