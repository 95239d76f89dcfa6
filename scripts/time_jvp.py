#!/usr/bin/env python
"""Experiment driver (not a bench line): the cost of a forward-mode product against an image and a gradient.

C3 (2400 x 1800, reference solids, round_through_float = 0), one process, one GPU, everything on device
memory and on torch's current stream with no stats (enqueue only). After a warm-up of every call, --rounds
rounds alternate, in this order:
- c5_render_device                  the image alone;
- c5_render_jvp_device              J v along a random {v_alpha, v_Q} (the gather of the direction included);
- c5_render_grad_device             J^T g for a random g;
- J v, then J^T (J v)               the Gauss-Newton product J^T J v: the tangent image, read in place as g.
Each call is timed by CUDA events around it on the stream; the round ends with a synchronisation. Each call
prints one JSON line with the median, min, max and every sample. Checks in the same run: two J v calls give
the same bits, and the device form gives the host form's bits. The first line names the GPU, its power limit
and max SM clock, read in the same run.

    python scripts/time_jvp.py > profiles/r11_jvp_c3_one_b200.jsonl
"""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from time_grad import gpu_info  # noqa: E402
from time_grad_device import setup  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--seed", type=int, default=2026)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    print(json.dumps(gpu_info()), flush=True)

    ctx, mesh, view, vk = setup("C3")
    with ctx:
        common = dict(workload="C3", res=[view.res_x, view.res_y], n_tets=int(mesh.n_tets))
        rng = np.random.default_rng(args.seed)
        va = torch.tensor(rng.normal(size=mesh.n_tets) * mesh.alpha, device="cuda")
        vq = torch.tensor(rng.normal(size=mesh.n_tets) * mesh.q, device="cuda")
        g = torch.tensor(rng.normal(size=(view.res_y, view.res_x, 2)), device="cuda")
        img = torch.empty((view.res_y, view.res_x, 2), dtype=torch.float64, device="cuda")
        tangent = torch.empty_like(img)
        ga = torch.empty(mesh.n_tets, dtype=torch.float64, device="cuda")
        gq = torch.empty_like(ga)
        stream = torch.cuda.current_stream().cuda_stream

        def image():
            ctx.render_device(view, img.data_ptr(), stream, stats=False)

        def jvp():
            ctx.render_jvp_device(view, va.data_ptr(), vq.data_ptr(), tangent.data_ptr(), 0, stream, stats=False)

        def grad():
            ctx.render_grad_device(view, g.data_ptr(), ga.data_ptr(), gq.data_ptr(), 0, stream, stats=False)

        def gauss_newton():
            jvp()
            ctx.render_grad_device(view, tangent.data_ptr(), ga.data_ptr(), gq.data_ptr(), 0, stream, stats=False)

        calls = {"render_device": image, "render_jvp_device": jvp, "render_grad_device": grad,
                 "jvp then grad against it (J^T J v)": gauss_newton}
        for f in calls.values():  # warm: modules, the device permutation, the tangent field, scratch buffers
            f()
        torch.cuda.synchronize()
        stats = {"render_device": ctx.render_device(view, img.data_ptr(), stream),
                 "render_jvp_device": ctx.render_jvp_device(view, va.data_ptr(), vq.data_ptr(), tangent.data_ptr(), 0,
                                                            stream)}
        ms = {k: [] for k in calls}
        for _ in range(args.rounds):
            events = []
            for k, f in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                events.append((k, e0, e1))
            torch.cuda.synchronize()
            for k, e0, e1 in events:
                ms[k].append(e0.elapsed_time(e1))
        for k, w in ms.items():
            st = stats.get(k, {})
            print(json.dumps(dict(common, call=k, ms_median=float(np.median(w)), ms_min=float(np.min(w)),
                                  ms_max=float(np.max(w)), ms=w, tet_steps=int(st.get("tet_steps", 0)),
                                  grazing_rays=int(st.get("grazing_rays", 0)))), flush=True)

        jvp()
        first = tangent.cpu().numpy()
        jvp()
        again = tangent.cpu().numpy()
        host = ctx.render_jvp(view, va.cpu().numpy(), vq.cpu().numpy())
        print(json.dumps(dict(common, check="J v bit-reproducible (two device calls; device vs host form)",
                              two_calls=bool(np.array_equal(first, again, equal_nan=True)),
                              device_vs_host=bool(np.array_equal(first, host, equal_nan=True)))), flush=True)


if __name__ == "__main__":
    main()
