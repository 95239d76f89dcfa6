"""Where a pipelined run's time goes between pixel kernels, from a `bench.py --timeline FILE` file.

For each lane: the mean duration of each phase of a view, each from the moment before it (start -> rotated ->
refitted -> mask -> pixel kernel -> grazing-ray kernel), and how long a view's prologue waited after its lane's
previous view (previous grazing-ray kernel done -> start). Over all lanes: the intervals between consecutive
pixel-kernel completions in time order, and the gap per view over a back-to-back interval: `--k4-ms` (the pixel
kernel's time alone, measured elsewhere) or, without it, the 10th percentile of the intervals themselves.

    python scripts/timeline_gaps.py run.json [--k4-ms 3.45] [--json]
"""
from __future__ import annotations

import argparse
import json

import numpy as np

PHASES = ["start", "rotated", "refitted", "mask", "pixel_kernel", "grazing_kernel"]


def analyse(path: str, k4_ms: float | None = None) -> dict:
    with open(path) as f:
        d = json.load(f)
    rank = d["ranks"][0]
    lanes = [np.asarray(tl, dtype=np.float64).reshape(-1, len(PHASES)) for tl in rank["lanes"]]
    per_lane = []
    for k, tl in enumerate(lanes):
        tl = tl[np.argsort(tl[:, 0])]
        phase_ms = {PHASES[p]: float(np.mean(tl[:, p] - tl[:, p - 1])) for p in range(1, len(PHASES))}
        wait = tl[1:, 0] - tl[:-1, 5]
        per_lane.append({"lane": k, "views": int(tl.shape[0]), "phase_ms": phase_ms,
                         "start_after_previous_grazing_ms": float(np.mean(wait)) if wait.size else None})
    done = np.sort(np.concatenate([tl[:, 4] for tl in lanes]))
    iv = np.diff(done)
    back_to_back = float(k4_ms) if k4_ms else float(np.percentile(iv, 10))
    mean = float(np.mean(iv))
    return {"file": path, "lanes": len(lanes), "views": int(done.size),
            "ms_per_view_elapsed": rank["elapsed_ms"] / max(d["steps"], 1),
            "pixel_kernel_interval_ms": {"mean": mean, "min": float(iv.min()), "p10": float(np.percentile(iv, 10)),
                                         "median": float(np.median(iv)), "p90": float(np.percentile(iv, 90)),
                                         "max": float(iv.max())},
            "back_to_back_ms": back_to_back, "back_to_back_from": "--k4-ms" if k4_ms else "p10 of the intervals",
            "gap_ms_per_view": mean - back_to_back,
            "intervals_over_back_to_back_plus_0.1ms": int(np.sum(iv > back_to_back + 0.1)),
            "per_lane": per_lane}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("files", nargs="+")
    ap.add_argument("--k4-ms", type=float, default=None, help="the pixel kernel's time alone (back-to-back interval)")
    ap.add_argument("--json", action="store_true", help="one JSON line per file")
    args = ap.parse_args()
    for path in args.files:
        r = analyse(path, args.k4_ms)
        if args.json:
            print(json.dumps(r))
            continue
        iv = r["pixel_kernel_interval_ms"]
        print(f"{path}: {r['lanes']} lanes, {r['views']} views, {r['ms_per_view_elapsed']:.3f} ms per view (elapsed)")
        print(f"  pixel kernel completions: interval mean {iv['mean']:.3f}  min {iv['min']:.3f}  median {iv['median']:.3f}"
              f"  p90 {iv['p90']:.3f}  max {iv['max']:.3f} ms")
        print(f"  back to back {r['back_to_back_ms']:.3f} ms ({r['back_to_back_from']}): gap {r['gap_ms_per_view']:.3f} ms per view,"
              f" {r['intervals_over_back_to_back_plus_0.1ms']} intervals over it by > 0.1 ms")
        for ln in r["per_lane"]:
            ph = "  ".join(f"{k} {v:.3f}" for k, v in ln["phase_ms"].items())
            w = ln["start_after_previous_grazing_ms"]
            print(f"  lane {ln['lane']}: {ph}  | start after previous grazing {w:.3f}" if w is not None else f"  lane {ln['lane']}: {ph}")


if __name__ == "__main__":
    main()
