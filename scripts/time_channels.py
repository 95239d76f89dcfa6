#!/usr/bin/env python
"""Experiment driver (not a bench line): what K channels in one walk cost against K walks.

C3 (2400 x 1800, reference solids) with K seeded channel pairs, K in --channels. For each K the
script alternates, view by view, one plain render (c5_render, the cells' own fields) and one
K-channel render (c5_render_channels), and prints one JSON line per K with the device phase times
per view (medians): ms_walk (pixel + grazing-ray kernels), ms_total and ms_d2h. no_zero_copy is set,
so the image always leaves through a device-to-host copy and ms_walk holds no PCIe stores (a K-channel
host image is K x 69 MB). The K = 1 channel render is the cost of one single-pair pass: `vs_k_passes`
is ms_walk(K) / (K * ms_walk(1)), below 1 when one K-channel walk is cheaper than K passes. The first
line names the GPU, its power limit and max SM clock, read in the same run.

    python scripts/time_channels.py --channels 1,2,4,8 --views 20 > profiles/r04_channels_c3_one_b200.jsonl
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", default="1,2,4,8")
    ap.add_argument("--views", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()
    ks = [int(x) for x in args.channels.split(",")]
    print(json.dumps(gpu_info()), flush=True)
    mesh, vk = synth.make_config("C3")
    roche, sphere = hostlib.make_solids(vk["D"])
    rng = np.random.default_rng(args.seed)
    k_max = max(ks)
    alpha = rng.uniform(0.1, 4.0, (k_max, mesh.n_tets))
    q = rng.uniform(0.1, 4.0, (k_max, mesh.n_tets))
    view = api.make_view(vk["res_x"], vk["res_y"], X=vk["X"], Y=vk["Y"], I=vk["I"], alpha_limit=vk["alpha_limit"])
    ms_walk_one = None
    with api.Context(devices=(0,)) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        ctx.debug_set("no_zero_copy", 1)
        plain_out = np.zeros((vk["res_y"], vk["res_x"], 2))
        for k in ks:
            ctx.upload_channels(alpha[:k], q[:k])
            out = np.zeros((vk["res_y"], vk["res_x"], k, 2))
            plain, chan = [], []
            for v in range(args.warmup + args.views):
                _, sp = ctx.render(view, out=plain_out)
                _, sc = ctx.render_channels(view, out=out)
                if v >= args.warmup:
                    plain.append(sp)
                    chan.append(sc)
            assert chan[-1]["tet_steps"] == plain[-1]["tet_steps"] and chan[-1]["walk_errors"] == 0
            walk = median(chan, "ms_walk")
            if k == 1:
                ms_walk_one = walk
            line = dict(
                workload="C3", res=[vk["res_x"], vk["res_y"]], channels=k, views=args.views, warmup=args.warmup,
                no_zero_copy=1, tet_steps=int(chan[-1]["tet_steps"]),
                ch_ms_walk=walk, ch_ms_graze=median(chan, "ms_graze"), ch_ms_total=median(chan, "ms_total"),
                ch_ms_d2h=median(chan, "ms_d2h"),
                plain_ms_walk=median(plain, "ms_walk"), plain_ms_graze=median(plain, "ms_graze"),
                plain_ms_total=median(plain, "ms_total"), plain_ms_d2h=median(plain, "ms_d2h"),
                ch_ms_walk_per_channel=walk / k,
                vs_k_plain_walks=walk / (k * median(plain, "ms_walk")),
                vs_k_plain_totals=median(chan, "ms_total") / (k * median(plain, "ms_total")))
            if ms_walk_one is not None:
                line["vs_k_passes"] = walk / (k * ms_walk_one)
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
