"""In-process view sweep: the mesh stays resident and only the rotations change per frame.

Replaces the reference's process-per-frame tooling (utility/rotate_traces.py:11-21: 1 500 launches
of `course ... -Y theta`, each re-reading the VTK file, regenerating the solids and re-allocating
~0.8 KB per pixel). Frames go through c5_render_submit / c5_render_wait, a few in flight per GPU, so
the device renders frames k+1, k+2 while the host consumes (writes) frame k. Under torchrun the frames
are dealt round-robin to the ranks (one whole view per GPU): frames are independent, so there is NO
collective on the data path.

    python -m course5_b200.sweep --config C4 --frames 360 [--out-dir frames/]
    python -m course5_b200.sweep --config C4 --frames 360 --light-curve curve.csv
    python -m torch.distributed.run --nproc-per-node 8 -m course5_b200.sweep --config C4 --frames 360
"""
from __future__ import annotations

import argparse
import json
import os
import time

import numpy as np

from . import api, hostlib, synth


def sweep_views(res_x, res_y, *, X, I, alpha_limit, y_from=0.0, y_to=2.0, frames=360, **extra):
    """The frame list of a full turn about y (angles in units of pi, like the CLI)."""
    return [api.make_view(res_x, res_y, X=X, Y=y_from + (y_to - y_from) * k / frames, I=I,
                          alpha_limit=alpha_limit, **extra) for k in range(frames)]


def render_sweep(ctx: api.Context, views, *, in_flight: int = 3, consume=None) -> tuple[int, list[dict]]:
    """Renders `views` in order through c5_render_submit / c5_render_wait with `in_flight` views on the
    device at a time, each into a page-locked host image of its own. `consume(k, image, stats)` is
    called with frame k's finished image (valid until it returns: the buffer is then reused) while the
    next frames are already being rendered. Returns (total tet-steps, per-frame stats)."""
    import collections
    import torch
    if not views:
        return 0, []
    ctx.set_views_in_flight(in_flight)
    res_y, res_x = views[0].res_y, views[0].res_x
    pinned = [torch.empty((res_y, res_x, 2), dtype=torch.float64).pin_memory() for _ in range(in_flight)]
    images = [t.numpy() for t in pinned]
    tickets = collections.deque()
    stats, steps = [], 0
    for k in range(len(views) + in_flight):
        if k >= in_flight:
            kk = k - in_flight
            st = ctx.render_wait(tickets.popleft())
            steps += st["tet_steps"]
            stats.append(st)
            if consume is not None:
                consume(kk, images[kk % in_flight], st)
        if k < len(views):
            tickets.append(ctx.render_submit(views[k], images[k % in_flight]))
    return steps, stats


def render_light_curve(ctx: api.Context, views, *, in_flight: int = 3, channels: bool = False):
    """The light curve of `views`: the pipelined loop of render_sweep over c5_render_flux_submit, so no
    image leaves the device. Returns (totals of shape (frames, n, 2), per-frame stats), [k, c, 0] = sum of
    tau and [k, c, 1] = sum of I of frame k and pair c (n = 1, or the uploaded channels with channels=True)."""
    import collections
    n = ctx.n_channels if channels else 1
    totals = np.zeros((len(views), n, 2), dtype=np.float64)
    if not views:
        return totals, []
    ctx.set_views_in_flight(in_flight)
    tickets = collections.deque()
    stats = []
    for k in range(len(views) + in_flight):
        if k >= in_flight:
            ticket, total = tickets.popleft()
            stats.append(ctx.render_wait(ticket))
            totals[k - in_flight] = total
        if k < len(views):
            ticket, _, total = ctx.render_flux_submit(views[k], channels=channels)
            tickets.append((ticket, total))
    return totals, stats


def write_light_curve(path: str, rows) -> None:
    """rows: (frame, Y_pi, hit_pixels, solid_pixels, tau_sum, I_sum) in frame order; %.17g round-trips."""
    with open(path, "w") as f:
        f.write("frame,Y_pi,hit_pixels,solid_pixels,tau_sum,I_sum\n")
        for frame, y, hit, solid, tau, inten in rows:
            f.write(f"{frame},{y:.17g},{hit},{solid},{tau:.17g},{inten:.17g}\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C4")
    ap.add_argument("--frames", type=int, default=360)
    ap.add_argument("--n", type=int, default=None, help="lattice size override")
    ap.add_argument("--out-dir", default=None, help="write frame_%04d.vti here")
    ap.add_argument("--in-flight", type=int, default=3, help="views in flight per GPU")
    ap.add_argument("--light-curve", default=None,
                    help="write the sums of tau and I of every frame to this CSV instead of moving images to the host")
    ap.add_argument("--no-zero-copy", action="store_true",
                    help="render into device memory and let the copy engine bring each image to the host, instead of "
                         "the walk kernels storing into the page-locked host image in place")
    args = ap.parse_args()

    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    from .dist import bind_to_device_numa_node
    numa = bind_to_device_numa_node(local)       # page-locked images on the GPU's own NUMA node
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    mesh, view = synth.make_config(args.config, n=args.n)
    roche, sphere = hostlib.make_solids(view["D"])
    ctx = api.Context(devices=(local,))
    if args.no_zero_copy:
        ctx.debug_set("no_zero_copy", 1)
    t0 = time.perf_counter()
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    ctx.upload_solids(roche, True)
    ctx.upload_solids(sphere, False)
    upload_s = time.perf_counter() - t0
    y_of = [2.0 * k / args.frames for k in range(args.frames)]   # sweep_views' angles
    views = sweep_views(view["res_x"], view["res_y"], X=view["X"], I=view["I"], alpha_limit=view["alpha_limit"],
                        frames=args.frames)
    mine = list(range(rank, args.frames, world))       # frames dealt round-robin: no collective on the data path
    if args.out_dir and rank == 0:
        os.makedirs(args.out_dir, exist_ok=True)
    if world > 1:
        dist.barrier()

    def write(k, image, st):
        hostlib.write_vti(os.path.join(args.out_dir, f"frame_{mine[k]:04d}.vti"), image)

    curve = None
    if args.light_curve:
        render_light_curve(ctx, [views[k] for k in mine[: args.in_flight + 1]], in_flight=args.in_flight)   # warm-up
    else:
        render_sweep(ctx, [views[k] for k in mine[: args.in_flight + 1]], in_flight=args.in_flight)   # warm-up
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    if args.light_curve:
        totals, frame_stats = render_light_curve(ctx, [views[k] for k in mine], in_flight=args.in_flight)
        steps = sum(st["tet_steps"] for st in frame_stats)
        curve = [(k, y_of[k], st["hit_pixels"], st["solid_pixels"], float(t[0, 0]), float(t[0, 1]))
                 for k, t, st in zip(mine, totals, frame_stats)]
    else:
        steps, _ = render_sweep(ctx, [views[k] for k in mine], in_flight=args.in_flight,
                                consume=write if args.out_dir else None)
    dt = time.perf_counter() - t0
    tot = torch.tensor([dt, float(steps)], dtype=torch.float64, device="cuda")
    if world > 1:
        t_max = tot.clone()
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dt, steps = float(t_max[0]), float(tot[1])
    if curve is not None:   # a few KB per rank
        parts = [None] * world if rank == 0 else None
        if world > 1:
            dist.gather_object(curve, parts, dst=0)
        else:
            parts = [curve]
        if rank == 0:
            write_light_curve(args.light_curve, sorted(r for part in parts for r in part))
    if rank == 0:
        print(json.dumps({"config": args.config, "frames": args.frames, "n_gpus": world, "seconds": dt,
                          "views_per_sec": args.frames / dt, "ms_per_view": 1e3 * dt / args.frames,
                          "tet_steps_per_sec": steps / dt, "tet_steps": steps, "views_in_flight": args.in_flight, "image_path": "light curve: row sums only" if args.light_curve else "copy engine" if args.no_zero_copy else "stored in place",
                          "res": [view["res_x"], view["res_y"]], "n_tets": mesh.n_tets,
                          "flags": {k: view[k] for k in ("X", "D", "I", "alpha_limit")},
                          "upload_and_topology_s": upload_s, "numa": numa,
                          "includes": ("per view: rotate + BVH refit + solid mask + walk + grazing rays + light curve: row sums "
                                       "reduced on the device, row sums to the host (c5_render_flux_submit / c5_render_wait), "
                                       "whole sweep wall clock, max over ranks; + CSV write on rank 0"
                                       if args.light_curve else
                                       "per view: rotate + BVH refit + solid mask + walk + grazing rays + image to page-locked "
                                       "host memory (c5_render_submit / c5_render_wait), whole sweep wall clock, max over ranks"
                                       + ("; + .vti write" if args.out_dir else ""))}))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
