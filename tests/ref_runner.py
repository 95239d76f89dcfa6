"""Runs the UNMODIFIED reference (oracle/_ref/libc5ref.so) on a named configuration in a process
of its own and saves what the parity gate needs. Where oracle/_ref was not built it runs the C
restatement (oracle/c5_oracle.c, held bit for bit against the reference's vectors in tests/golden)
with the reference's solids from the host generator (pinned by the reference's digests), the way
smoke() and bench.py fall back. TEST INFRASTRUCTURE ONLY.

    python tests/ref_runner.py C3 out.npz '[{"res_x": 2400, "res_y": 1800}, {"Y": 0.4, ...}]'

A process of its own because the reference reports a degenerate ray (through a vertex or an
edge) by throwing inside an OpenMP region (/root/reference/project/src/plane.cpp:39-41,
line.cpp:45), i.e. std::terminate: the caller then sees a non-zero exit code instead of losing
its own process. Every view in the JSON list overrides the configuration's flags
(course5_b200.synth.CONFIGS); arrays are saved as tau{k}, inten{k}, steps{k}, solid{k} (pre-cast
doubles, per-pixel record counts, solid mask) plus total_steps{k} and seconds{k} (the
reference's own timed region, main.cpp:126-130).
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    name, out_path, views_json = sys.argv[1], sys.argv[2], sys.argv[3]
    from course5_b200 import synth
    from oracle import refbind
    mesh, base = synth.make_config(name)
    tet_pts = mesh.tet_points()
    if os.path.exists(refbind.REF_SO):
        ref = refbind.Ref()

        def render(view):
            return ref.render(tet_pts, mesh.alpha, mesh.q, res_x=view["res_x"], res_y=view["res_y"], X=view["X"],
                              Y=view["Y"], D=view["D"], I=view["I"], alpha_limit=view["alpha_limit"],
                              threads=min(32, os.cpu_count() or 1), solids=1 if view.get("solids", 1) else 0, raw=True)
    else:
        from course5_b200 import hostlib
        port, solids = refbind.Port(), {}

        def render(view):
            roche = sphere = None
            if view.get("solids", 1):
                if view["D"] not in solids:
                    solids[view["D"]] = hostlib.make_solids(view["D"])
                roche, sphere = solids[view["D"]]
            return port.render(tet_pts, mesh.alpha, mesh.q, res_x=view["res_x"], res_y=view["res_y"], X=view["X"],
                               Y=view["Y"], I=view["I"], alpha_limit=view["alpha_limit"], solid_rot=roche,
                               solid_static=sphere)
    results = {}
    for k, override in enumerate(json.loads(views_json)):
        view = dict(base, **override)
        img = render(view)
        results[f"tau{k}"], results[f"inten{k}"] = img.tau, img.inten
        results[f"steps{k}"], results[f"solid{k}"] = img.steps, img.solid
        results[f"total_steps{k}"] = np.uint64(img.total_steps)
        results[f"seconds{k}"] = img.timings["ctor"] + img.timings["find"] + img.timings["trace"]
    np.savez(out_path, **results)


if __name__ == "__main__":
    main()
