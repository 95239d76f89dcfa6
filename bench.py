#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: tet-steps/s (and pixels/s) of the per-pixel
ray pass at 2400 x 1800 (BASELINE.json `metric`, configs[2]: synthetic 8M-tet grid, 2400 x 1800,
--alpha_limit 3.0 -X 0.5, plus the Roche lobe and sphere the reference always renders).

    python bench.py [--gpus N] [--steps K] [--warmup W]                    # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # the reference's OpenMP path
    python bench.py [...] --dump-outputs DIR                               # + the last timed view's image

A "step" is one view: rotate -> BVH refit -> solid mask -> entry + tet walk -> grazing rays (at N > 1
each rank renders a row band and the walk kernels store their pixels into rank 0's image over NVLink).
  value     tet-steps/s with everything resident in HBM, output left on the device (CUDA events on
            the launching stream, max over ranks).
  e2e       the same metric through the C-ABI calls a user makes (c5_render_submit / c5_render_wait)
            with page-locked HOST images: view parameters go host->device, the image device->host,
            inside the timed region; every image is complete in host memory when its wait returns.
  roofline  the walk kernels: algorithmic bytes (72 B per tet-step + 16 B per pixel, SURVEY.md §8d /
            DESIGN.md) / their CUDA-event time, against the measured HBM copy peak.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, built from /root/reference in the build
            container) on this box's host cores on the SAME workload at the SAME resolution
            (N = 1, rank 0 only), and `parity`: this run's image held against the reference's.
The oracle is only ever the thing compared against or the baseline — never the thing measured as ours.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from course5_b200 import api, synth  # noqa: E402

BYTES_PER_STEP = 72      # 16 B connectivity + 16 B neighbours + 24 B one new vertex + 16 B (alpha, Q)
BYTES_PER_PIXEL = 16     # {tau, I} doubles written
REL_TOL, ABS_FLOOR = 1e-9, 1e-13   # the parity gate (tests/parity.py, BASELINE.json north_star)
DUMP_LIMIT_BYTES = 64_000_000      # --dump-outputs: an image larger than this (64 MB) is written as a sample
DUMP_SAMPLE_PIXELS = 1 << 21       # (42 MB: tau and I doubles, solid mask floats)


def E2E_AUTO(world: int) -> str:
    """How the image reaches the page-locked host buffer when --e2e-mode is left alone."""
    return "inplace"


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_capture():
    """What the committed `ncu --set full` capture of the walk says (profiles/walk_traffic.json), if it exists."""
    path = os.path.join(ROOT, "profiles", "walk_traffic.json")
    try:
        with open(path) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Polls SM clock and throttle reasons through NVML; only samples taken while `armed` count.

    NVML is initialised in the constructor and the thread is started well BEFORE the timed region:
    the first NVML queries of a process are slow (tens of milliseconds at 8 processes per node) and,
    measured, stall CUDA submission in the processes of the same node while they run
    (profiles/r02_timeline_c3_n8_*_a.json: 15-20 ms holes at the start of the timed region on some
    ranks). So the poller is already in steady state when arm() is called right before the first
    timed view, and only what it sees between arm() and stop() is reported."""

    def __init__(self, index: int, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.armed = False
        self.polls = 0
        self._last_unarmed = None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        return mhz, mask

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                armed = self.armed
                mhz, mask = self._poll()
                self.polls += 1
                if armed:
                    self.samples.append(mhz)
                    for bit, name in names.items():
                        if mask & bit:
                            self.reasons.add(name)
                else:
                    self._last_unarmed = (mhz, [name for bit, name in names.items() if mask & bit])
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def wait_warm(self, polls=3, timeout_s=2.0):
        """Returns once the poller has completed a few queries (their first-call cost is behind us)."""
        t0 = time.monotonic()
        while self.nv is not None and self.polls < polls and time.monotonic() - t0 < timeout_s:
            time.sleep(0.002)

    def arm(self):
        self.armed = True

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
               "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if not self.samples and self._last_unarmed is not None:
            # a timed region shorter than one polling period: the poll just before it, taken under the same
            # load (the untimed pipelined round), is what there is
            out.update(sm_mhz=float(self._last_unarmed[0]), reasons=sorted(self._last_unarmed[1]),
                       note="timed region shorter than one poll; sample taken during the untimed pipelined round right before it")
        return out


class Watchdog(threading.Thread):
    """Ends the process if the run stops making progress. A multi-GPU run that deadlocks (a collective
    some rank never joins) would otherwise sit on its GPUs until an outer limit kills it; this way it
    fails fast, says in which phase, and frees the devices."""

    def __init__(self, rank: int, limit_s: float):
        super().__init__(daemon=True)
        self.rank, self.limit_s = rank, limit_s
        self.phase, self.t_phase, self.t0 = "start", time.monotonic(), time.monotonic()
        self.verbose = os.environ.get("C5_BENCH_VERBOSE") == "1"

    def tick(self, phase: str, limit_s: float | None = None):
        now = time.monotonic()
        if self.verbose or self.rank == 0:
            print(f"[bench rank {self.rank}] +{now - self.t0:6.1f}s {phase}", file=sys.stderr, flush=True)
        self.phase, self.t_phase = phase, now
        if limit_s is not None:
            self.limit_s = limit_s

    def run(self):
        while True:
            time.sleep(2.0)
            stalled = time.monotonic() - self.t_phase
            if stalled > self.limit_s:
                print(f"[bench rank {self.rank}] WATCHDOG: no progress for {stalled:.0f}s in phase '{self.phase}'; "
                      "exiting (exit code 3)", file=sys.stderr, flush=True)
                os._exit(3)


def reference_solids(D):
    """The reference's Roche lobe + sphere from the host-side generator (bit-identical to the
    reference's own, tests/test_host.py)."""
    from course5_b200 import hostlib
    return hostlib.make_solids(D)


def dump_outputs(directory, image):
    """Writes the (res_y, res_x, 2) image {tau, I} of the last timed view, so that two builds run with the same
    arguments can be compared value for value, as finite arrays: directory/tau.npy and intensity.npy (float64)
    and solid.npy (float32, 1 where a solid covers the pixel, 0 elsewhere). The image marks a solid pixel with
    NaN in both components; those pixels are written as 0 in tau and intensity, so the image is
    np.where(solid, nan, value) of the three. When the three arrays together exceed DUMP_LIMIT_BYTES they hold
    a fixed sample instead: the DUMP_SAMPLE_PIXELS pixels np.random.default_rng(0) draws from the row-major
    image without replacement, as 1-D arrays in ascending pixel order (the same pixels on every run at that
    resolution)."""
    os.makedirs(directory, exist_ok=True)
    image = np.asarray(image, dtype=np.float64)
    tau, inten = image[..., 0], image[..., 1]
    if tau.size * (8 + 8 + 4) > DUMP_LIMIT_BYTES:
        pick = np.sort(np.random.default_rng(0).choice(tau.size, DUMP_SAMPLE_PIXELS, replace=False))
        tau, inten = tau.reshape(-1)[pick], inten.reshape(-1)[pick]
    solid = np.isnan(tau) | np.isnan(inten)
    np.save(os.path.join(directory, "tau.npy"), np.where(solid, 0.0, tau))
    np.save(os.path.join(directory, "intensity.npy"), np.where(solid, 0.0, inten))
    np.save(os.path.join(directory, "solid.npy"), solid.astype(np.float32))


def config_dict(name, mesh, view):
    """The workload, in the same words for both arms (what ran it goes under `execution`)."""
    return {
        "workload": (f"{name}: synthetic Kuhn-split grid, {mesh.n_tets} tets / {mesh.n_points} points, "
                     f"{view['res_x']}x{view['res_y']}, -X {view['X']} -Y {view['Y']} --alpha_limit "
                     f"{view['alpha_limit']}, reference Roche lobe + sphere as solids"),
        "res_x": view["res_x"], "res_y": view["res_y"], "n_tets": mesh.n_tets, "n_points": mesh.n_points,
        "flags": {k: view[k] for k in ("X", "Y", "D", "I", "alpha_limit")},
        "l2": "inputs larger than L2 (cell records alone are 64 B x n_tets >> 126 MB); no explicit flush",
    }


# ------------------------------------------------------------------------------------------------
# the reference's own CPU implementation of the path on this box's host cores
# ------------------------------------------------------------------------------------------------

def time_reference(mesh, view, *, steps, warmup, raw=False, keep_image=False, tick=None):
    """oracle/_ref (the unmodified reference) — or, where it was never built, the C restatement — on
    the workload at its own resolution. raw=False is the reference's timed flow (plane ctor +
    find_intersections + trace_rays, main.cpp:126-130); raw=True drives the same per-pixel loop
    (plane.cpp:161-169) from the harness so the pre-cast doubles survive for the parity gate."""
    from oracle import refbind
    cores = os.cpu_count() or 1
    threads = min(32, cores)           # MAX_NUMBER_OF_THREADS = 32 (config.hpp:39)
    tet_pts = mesh.tet_points()
    kind = "reference" if os.path.exists(refbind.REF_SO) else "port"
    flags = dict(X=view["X"], Y=view["Y"], D=view["D"], I=view["I"], alpha_limit=view["alpha_limit"])
    times, img = [], None
    if kind == "reference":
        ref = refbind.Ref()
        for k in range(warmup + steps):
            if tick:
                tick(f"reference step {k - warmup}" if k >= warmup else f"reference warm-up {k}")
            img = ref.render(tet_pts, mesh.alpha, mesh.q, res_x=view["res_x"], res_y=view["res_y"],
                             threads=threads, solids=1, raw=raw, **flags)
            if k >= warmup:
                times.append(img.timings["ctor"] + img.timings["find"] + img.timings["trace"])
    else:
        port = refbind.Port()
        threads = cores
        roche, sphere = reference_solids(view["D"])
        for k in range(warmup + steps):
            if tick:
                tick(f"port step {k - warmup}" if k >= warmup else f"port warm-up {k}")
            img = port.render(tet_pts, mesh.alpha, mesh.q, res_x=view["res_x"], res_y=view["res_y"], threads=threads,
                              X=flags["X"], Y=flags["Y"], I=flags["I"], alpha_limit=flags["alpha_limit"],
                              solid_rot=roche, solid_static=sphere)
            if k >= warmup:
                times.append(img.timings["trace"])
    t_step = float(np.mean(times))
    return dict(value=img.total_steps / t_step, seconds_per_step=t_step, tet_steps=img.total_steps, kind=kind,
                cores=threads, pixels=view["res_x"] * view["res_y"], image=img if keep_image else None)


def parity_record(ours, want, *, against):
    """This run's image (api.RawImage, pre-cast doubles) against the oracle's (refbind.OracleImage):
    the gate of tests/parity.py, as numbers. `ok` is the conjunction the tests assert."""
    got = ours.image
    solid_equal = bool(np.array_equal(ours.solid.astype(bool), want.solid.astype(bool)))
    hits_equal = bool(np.array_equal(ours.steps > 0, want.steps > 0))
    steps_equal = bool(np.array_equal(ours.steps, want.steps))
    worst_rel, worst_abs, bad = 0.0, 0.0, 0
    for comp, ref in ((got[..., 0], want.tau), (got[..., 1], want.inten)):
        nan = np.isnan(ref)
        err = np.abs(np.where(nan, 0.0, comp - ref))
        mag = np.abs(np.where(nan, 0.0, ref))
        bad += int((err > REL_TOL * mag + ABS_FLOOR).sum()) + int((np.isnan(comp) != nan).sum())
        worst_abs = max(worst_abs, float(err.max()))
        # relative error where the value is not itself at the rounding floor of a silhouette-grazing pixel
        worst_rel = max(worst_rel, float(np.where(mag >= 1e-3, err / np.maximum(mag, 1e-3), 0.0).max()))
    rec = {"against": against, "gate": f"|got - want| <= {REL_TOL:g} |want| + {ABS_FLOOR:g} per pixel on pre-cast doubles; "
                                       "identical hit/miss sets, solid masks and per-pixel tets crossed",
           "pixels": int(want.steps.size), "hit_pixels": int((want.steps > 0).sum()),
           "solid_pixels": int(want.solid.astype(bool).sum()),
           "hit_sets_equal": hits_equal, "solid_masks_equal": solid_equal, "per_pixel_steps_equal": steps_equal,
           "tet_steps": [int(ours.stats["tet_steps"]), int(want.total_steps)],
           "pixels_out_of_tolerance": bad, "max_abs_err": worst_abs, "max_rel_err_where_value_ge_1e-3": worst_rel}
    rec["ok"] = bool(hits_equal and solid_equal and steps_equal and bad == 0 and
                     int(ours.stats["tet_steps"]) == int(want.total_steps))
    return rec


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dog = Watchdog(0, limit_s=1800.0)
    dog.start()
    mesh, view = synth.make_config(args.workload)
    r = time_reference(mesh, view, steps=args.steps, warmup=args.warmup, keep_image=bool(args.dump_outputs), tick=dog.tick)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.stack([r["image"].tau, r["image"].inten], axis=-1))
    sample_txt = (f"{args.workload} mesh ({mesh.n_tets} tets) + reference solids at {view['res_x']}x{view['res_y']}, the whole "
                  f"workload: {r['tet_steps']} tet-steps per step; timed region = plane ctor + find_intersections + "
                  "trace_rays (main.cpp:126-130)")
    line = {
        "impl": "reference", "metric": "tet_steps_per_sec", "value": r["value"], "unit": "tet-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * r["seconds_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "pixels_per_sec": r["pixels"] / r["seconds_per_step"],
        "tet_steps_per_view": r["tet_steps"],
        "config": config_dict(args.workload, mesh, view),
        "execution": {"where": f"host CPU, OpenMP, {r['cores']} threads", "gpus_used": 0},
        "cpu_baseline": {"value": r["value"], "unit": "tet-steps/s", "cores": r["cores"], "kind": r["kind"],
                         "sample": sample_txt},
        "e2e": {"value": r["value"], "unit": "tet-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist
    from course5_b200.dist import BandRenderer, SharedHostImage

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path "
                         "(use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from course5_b200.dist import bind_to_device_numa_node
    all_cpus = os.sched_getaffinity(0)        # the cpu_baseline leg gets every core back
    numa = {"bound": False, "note": "--no-numa-bind"} if args.no_numa_bind else bind_to_device_numa_node(local_rank)
    dog = Watchdog(rank, limit_s=float(os.environ.get("C5_BENCH_STALL_LIMIT", "150" if world == 1 else "90")))
    dog.start()
    dog.tick("init process group" if world > 1 else "single process")
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=device)

    dog.tick("synthetic mesh + solids on the host")
    mesh, view = synth.make_config(args.workload)
    solids = reference_solids(view["D"])

    dog.tick("upload (topology, BVH)")
    ctx = api.Context(devices=(local_rank,))
    for kv in (kv for kv in args.debug.split(",") if kv):
        ctx.debug_set(kv.split("=")[0], int(kv.split("=")[1]))
    t0 = time.perf_counter()
    info = ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    ctx.upload_solids(solids[0], True)
    ctx.upload_solids(solids[1], False)
    upload_s = time.perf_counter() - t0
    v = api.make_view(view["res_x"], view["res_y"], X=view["X"], Y=view["Y"], I=view["I"],
                      alpha_limit=view["alpha_limit"], lib=ctx.lib)
    # views in flight (measured, profiles/README.md round 2): one GPU rendering whole views is saturated by two
    # (4.41 ms per view, steady; four: 4.44-4.66); a band of 1/N of the image is a single wave of blocks and wants
    # four (0.65 vs 0.75 ms); on the 50M-tet mesh four views evict each other from L2 (6.2 vs 5.7 ms)
    big = mesh.n_tets > 16_000_000
    lanes = args.lanes if args.lanes > 0 else (2 if (world == 1 or big) else 4)
    # e2e: the host submits a view only when an earlier one has come back, so short views (bands) need more in
    # flight to keep every lane's queue fed: N = 8, 0.91 ms per view with eight against 1.0 with four (N = 4: no gain)
    e2e_in_flight = args.e2e_in_flight or (args.lanes if args.lanes > 0 else (3 if big else api.MAX_IN_FLIGHT if world >= 8 else 4))
    # view groups (dist.py). Measured at N = 8, 20 timed views (profiles/r02_bench_*_n8_groups*.json): on C3 eight
    # bands per view, two groups of four and four groups of two run within 4 % of each other (0.717 / 0.706 / 0.688
    # ms per view), so the plain row bands of the north_star stay; on the 50M-tet mesh the prologue every rank
    # repeats (rotate + refit, 0.21 ms) and the lower rate of thin bands make the groups much faster (C5t: 1.26-1.35
    # ms as eight bands, 0.90 as 2 x 4, 0.82 as 4 x 2), so big meshes render two bands per view.
    groups = args.view_groups if args.view_groups > 0 else (world // 2 if (big and world >= 8 and world % 2 == 0) else 1)
    br = BandRenderer(ctx, device=device, rank=rank, world=world, gather=args.gather, lanes=lanes, groups=groups)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    # ---- warm-up: also settles the band cuts -----------------------------------------------------
    # tet-steps of the previous view, weighted by the time each band took (a few iterations; a sweep
    # does the same from frame to frame)
    n_warm = max(args.warmup, 3)
    for k in range(n_warm):
        dog.tick(f"warm-up view {k}")
        br.render(v, rebalance="steps")
    if world > 1:
        # bands cut so that every rank sustains the same pipelined time per view (a sweep does the same
        # from frame to frame): rounds of a few views each, no exchange, re-cut after each
        dog.tick("band calibration")
        br.calibrate(v, rounds=args.calibrate, views=32)
        n_warm += 1 + args.calibrate * (32 + br.n_lanes + 2)
    bands = br.bands(view["res_y"])
    dog.tick(f"bands {bands}")
    barrier()

    # ---- N > 1: the assembled image against one rank's own render of the whole view ---------------
    parity, parity_failed = None, False
    if world > 1:
        dog.tick("parity of the assembled image")
        whole = ctx.render(v)[0] if rank == 0 else None
        same, rows = True, np.zeros(0, dtype=np.int64)
        for _ in range(br.groups):          # consecutive views go to consecutive view groups: every group once
            img_dev, _, _ = br.render(v, rebalance=False)
            torch.cuda.synchronize(device)
            barrier()
            if rank == 0:
                got = img_dev.cpu().numpy()
                same = same and bool(np.array_equal(got, whole, equal_nan=True))
                rows = np.union1d(rows, np.where(~np.all((got == whole) | (np.isnan(got) & np.isnan(whole)), axis=(1, 2)))[0])
        if rank == 0:
            parity = {"against": f"rank 0's own render of the whole view (bit for bit); one rank against oracle/_ref: "
                                 "the N = 1 line and tests/test_gpu_parity.py",
                      "assembled_image_equals_single_rank_render": same, "rows_that_differ": int(rows.size),
                      "n_ranks": world, "gather": br.gather_mode, "ok": same}
        barrier()

    # ---- value: everything resident, output stays on the device -----------------------------------
    # The views are only enqueued (no host readback between them; statistics come from a second
    # pass): consecutive views rotate over the lanes — the context and siblings that share its mesh,
    # each on its own stream — so the tail of one view's walk and its grazing-ray kernel overlap the
    # next views. N > 1, gather=p2p: the walk stores straight into rank 0's image over NVLink and the
    # barrier of view k is left in flight (2 lanes + 1 images); gather=sendrecv: the same with one
    # grouped ncclSend/ncclRecv per view.
    # one untimed pipelined round with the final bands: every lane, every image set and every lazily
    # created mapping has been used once before the clock starts
    # ... and the clock poller is started before it, so that NVML's slow first queries (which stall CUDA
    # submission in every process of the node while they run) are over when the clock starts
    br.prepare(v)
    sampler = None if args.no_clock_sampler else ClockSampler(local_rank)
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    ev1.record()        # (both events exist before the clock starts)
    for _ in range(2 * br.n_lanes + 2):
        br.render(v, rebalance=False, stats=False, pipeline=True)
    br.finish()
    if args.timeline:
        br.enable_timeline(args.steps)
    if sampler:
        sampler.wait_warm()
    dog.tick(f"timed region: {args.steps} views, {br.n_lanes} in flight, gather={br.gather_mode}")
    barrier()
    launches0 = br.kernel_launches()
    host_t = []
    if sampler:
        sampler.arm()
    ev0.record()
    t_host0 = time.perf_counter()
    for _ in range(args.steps):
        last_image, _, _ = br.render(v, rebalance=False, stats=False, pipeline=True, gather=not args.experiment_no_exchange)
        host_t.append(time.perf_counter() - t_host0)
    br.finish()
    ev1.record()
    barrier()
    clocks = sampler.stop() if sampler else {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "--no-clock-sampler"}
    launches = br.kernel_launches() - launches0
    elapsed_ms = max(ev0.elapsed_time(ev1), 1e-6)
    host_enqueue_ms = 1e3 * host_t[-1] / args.steps
    if args.dump_outputs and last_image is not None:      # rank 0 holds the assembled image
        dump_outputs(args.dump_outputs, last_image.cpu().numpy())
    timeline = None
    if args.timeline:
        lanes_tl = br.timeline(ev0.cuda_event)
        timeline = {"rank": rank, "view_group": br.group, "band": list(bands[br.band_index]), "host_enqueue_done_ms": [1e3 * t for t in host_t],
                    "phases": ["start", "rotated", "refitted", "mask", "pixel_kernel", "grazing_kernel"],
                    "lanes": [tl.tolist() for tl in lanes_tl], "elapsed_ms": elapsed_ms}
        br.enable_timeline(0)

    dog.tick("statistics pass")
    walk_ms, stats_last = [], None
    for _ in range(3):
        _, st, _ = br.render(v, rebalance=False, gather=False)    # every rank its own band, no exchange
        walk_ms.append(st["ms_walk"])
        stats_last = st
    barrier()
    band_steps = stats_last["tet_steps"]

    # ---- e2e: the public C-ABI calls with page-locked HOST images ----------------------------------
    # c5_render_submit / c5_render_wait with `lanes` views in flight. N = 1: the images are pinned
    # buffers. N > 1: ONE shared-memory segment every rank pins; each rank's walk writes its band in
    # place over its own PCIe link and publishes "band of view k done" in the segment; rank 0 takes the
    # image when all bands are in. Wall clock around the calls a user makes; every step's image is
    # complete in host memory (and its stats read) inside the timed region.
    dog.tick("e2e: host images")
    L = e2e_in_flight
    ctx.set_views_in_flight(L)
    e2e_mode = args.e2e_mode
    if e2e_mode == "auto":
        e2e_mode = E2E_AUTO(world)
    if e2e_mode == "copy":
        ctx.debug_set("no_zero_copy", 1)
    lo, hi = bands[br.band_index]
    G = br.groups
    group_ranks = [list(range(g * br.per_group, (g + 1) * br.per_group)) for g in range(G)]
    n_img = L + 1 if world == 1 else 2 * L * G + 1   # N > 1: a rank may run a round of views ahead of the slowest one
    shared = SharedHostImage(ctx, view["res_x"], view["res_y"], rank=rank, world=world, sets=n_img)

    def e2e_run(n_views, base):
        """Views base .. base + n_views - 1 (the flags in the segment count views since its creation). View k is
        rendered by view group k % G; a rank has up to L of its own views in flight. Rank 0 takes every image, in
        order, as soon as its bands are in — but waits for one only when it needs that image's set back, so that it
        is no more tightly coupled to the slowest rank than the others are."""
        tickets = collections.deque()
        steps_seen, own = 0, 0
        end = base + n_views
        taken = base                      # rank 0: images base .. taken - 1 have been taken and released

        def take(must_reach):
            nonlocal taken
            while taken < end:
                who = group_ranks[taken % G]
                if taken >= must_reach and int(shared._flags[who].min()) < taken + 1:
                    return
                image = shared.wait_image(taken, who)      # complete in host memory here
                assert image.shape[0] == view["res_y"]
                shared.release(taken)
                taken += 1

        for k in range(n_views + L * G):
            if k >= L * G:
                kk = base + k - L * G
                if kk % G == br.group:
                    steps_seen += shared.complete_band(tickets.popleft(), kk)["tet_steps"]
                    own += 1
            if k < n_views and (base + k) % G == br.group:
                if rank == 0:
                    take(base + k - n_img + 1)             # the set view base + k reuses must have been released
                tickets.append(shared.submit_band(v, (lo, hi), base + k))
            elif rank == 0:
                take(base)                                 # whatever is ready
        if rank == 0:
            take(end)
        return steps_seen, own

    e2e_run(2 * L * G, 0)
    barrier()
    t0 = time.perf_counter()
    e2e_steps, e2e_own = e2e_run(args.steps, 2 * L * G)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_image_ok = True
    if rank == 0:   # the last host image is the view (spot check: same NaN mask and finite elsewhere)
        last = shared.arrays[(2 * L * G + args.steps - 1) % n_img]
        e2e_image_ok = bool(np.isnan(last).any() and np.isfinite(last[~np.isnan(last)]).all() and (last != 0).any())
    shared.close()
    assert e2e_steps == band_steps * e2e_own, (e2e_steps, band_steps, e2e_own)

    dog.tick("reduce over ranks")
    t = torch.tensor([elapsed_ms, e2e_s * 1e3, float(np.mean(walk_ms)), host_enqueue_ms], dtype=torch.float64, device=device)
    s = torch.tensor([band_steps, launches], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
    elapsed_ms, e2e_ms, walk_ms_max, host_enqueue_ms = (float(x) for x in t.cpu())
    total_steps, total_launches = (int(x) for x in s.cpu())
    total_steps //= br.groups            # every band is held by one rank of every view group
    # the roofline line describes the walk of the band with the most tet-steps (rank 0's may be empty)
    mine = torch.tensor([float(band_steps), float((hi - lo) * view["res_x"]), float(np.mean(walk_ms)),
                         float(stats_last["ms_graze"]), float(stats_last["ms_mask"]), float(stats_last["ms_total"])],
                        dtype=torch.float64, device=device)
    per_rank = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, mine)
    else:
        per_rank = [mine]
    per_rank = [p.cpu().tolist() for p in per_rank]
    busiest = max(range(world), key=lambda r: per_rank[r][0])
    if timeline is not None:
        gathered = [None] * world
        if world > 1:
            dist.all_gather_object(gathered, timeline)
        else:
            gathered = [timeline]
        if rank == 0:
            with open(args.timeline, "w") as f:
                json.dump({"n_gpus": world, "steps": args.steps, "lanes": br.n_lanes, "gather": br.gather_mode, "ranks": gathered}, f)

    if rank == 0:
        pixels = view["res_x"] * view["res_y"]
        ms_per_step = elapsed_ms / args.steps
        value = total_steps / (ms_per_step * 1e-3)
        e2e_value = total_steps / (e2e_ms * 1e-3 / args.steps)
        peak, peak_src = measured_hbm_peak()
        cap = ncu_capture()
        # dominant kernels (tet_walk_fp64 + grazing_rays_fp64) on the busiest band; at N = 1 the whole image
        k_steps, k_pixels, k_ms = per_rank[busiest][:3]
        k_ms = max(k_ms, 1e-9)
        alg_bytes = k_steps * BYTES_PER_STEP + k_pixels * BYTES_PER_PIXEL
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic = cap.get("dram_bytes_per_launch") if world == 1 else None
        line = {
            "metric": "tet_steps_per_sec", "value": value, "unit": "tet-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "pixels_per_sec": pixels / (ms_per_step * 1e-3),
            "tet_steps_per_view": total_steps,
            "config": config_dict(args.workload, mesh, view),
            "execution": {
                "views_in_flight": br.n_lanes, "view_groups": br.groups, "bands_per_view": br.per_group,
                "walk": "pixel kernel, then the grazing-ray kernel on the same stream (no kernel waits for another)",
                "parallelism": "single GPU" if world == 1 else
                               (f"{world} row bands (time-balanced), mesh replicated, " if br.groups == 1 else
                                f"{br.groups} view groups of {br.per_group} ranks take alternate views, each view in {br.per_group} row bands "
                                "(time-balanced), mesh replicated, every image assembled in rank 0's memory, ") +
                               ("bands stored into rank 0's image over NVLink peer mappings by the walk kernels, one 4-byte all-reduce per view as the barrier"
                                if br.gather_mode == "p2p" else "one grouped ncclSend/ncclRecv gather-v to rank 0 per view"),
                "host_enqueue_ms_per_view": host_enqueue_ms,
                "numa": numa},
            "e2e": {"value": e2e_value, "unit": "tet-steps/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": int(api.C.sizeof(api.View)) * br.per_group,
                    "d2h_bytes_per_step": pixels * 16 + br.per_group * (64 + 8 * view["res_y"]),
                    "views_in_flight": L, "image_spot_check": e2e_image_ok, "mode": e2e_mode,
                    "api": "c5_render_submit / c5_render_wait into page-locked host images " +
                           ("written in place by the walk kernels" if e2e_mode == "inplace" else
                            "(band rendered in device memory, brought over by the copy engine)") +
                           ("" if world == 1 else " (one shared-memory image per view, every rank its band over its own PCIe link; completion flags in the segment)")},
            "gpu_launches": total_launches,
            "roofline": {"kernel": "tet_walk_fp64 + grazing_rays_fp64", "rank": busiest, "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "frac_of_8000_GBps_nominal": achieved / 8000.0, "traffic": traffic,
                         "peak_source": peak_src, "kernel_ms": k_ms,
                         "kernel_ms_note": "CUDA events around the two kernels of ONE view rendered alone (statistics pass); ms_per_step is "
                                           "the pipelined rate with several views in flight, which hides each view's tail, so it can be lower",
                         "algorithmic_bytes_per_launch": int(alg_bytes),
                         "limiter": "L1 data-pipe wavefronts and load latency, not DRAM: `achieved` is a normalised throughput "
                                    "(algorithmic bytes / time); rays share tets in L1/L2, so real DRAM traffic is `traffic`",
                         "dram_frac_of_peak": (traffic / (k_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "ncu": {k: cap.get(k) for k in ("l1_hit_rate_pct", "l2_hit_rate_pct",
                                                         "l1_data_pipe_wavefronts_pct_of_peak", "source")}},
            "bands": [list(b) for b in bands],
            "per_rank": [{"tet_steps": int(p[0]), "walk_ms": p[2], "graze_ms": p[3], "mask_ms": p[4], "view_ms_alone": p[5]} for p in per_rank],
            "phases_ms": {k: stats_last[k] for k in ("ms_rotate", "ms_bvh", "ms_mask", "ms_walk", "ms_graze", "ms_total")},
            "one_off": {"upload_and_topology_s": upload_s, "device_bytes": int(info.device_bytes),
                        "boundary_faces": int(info.n_boundary_faces)},
            "clocks": clocks,
        }
        if parity is not None:
            line["parity"] = parity
        if args.experiment_no_exchange:
            line["INVALID"] = "--experiment-no-exchange: the timed views were not assembled into one image"
        if br.calibration_log:
            # per calibration round: the cut that was timed and the sustained ms per view every rank measured for
            # its band alone (no exchange); the last entry is the round BEFORE the final re-cut
            line["calibration"] = br.calibration_log
        if os.environ.get("C5_BENCH_ATTEMPTS"):
            line["attempts"] = json.loads(os.environ["C5_BENCH_ATTEMPTS"])   # configurations left before this one
        if world == 1 and not args.no_cpu_baseline:
            dog.tick("cpu_baseline + parity: the reference on the host cores, same workload, same resolution", limit_s=1800.0)
            vraw = api.View.from_buffer_copy(v)
            vraw.round_through_float = 0
            ours = ctx.render_raw(vraw)
            os.sched_setaffinity(0, all_cpus)
            r = time_reference(mesh, view, steps=1, warmup=0, raw=True, keep_image=True)
            line["cpu_baseline"] = {
                "value": r["value"], "unit": "tet-steps/s", "cores": r["cores"], "kind": r["kind"],
                "seconds": r["seconds_per_step"],
                "sample": (f"the whole workload once: {args.workload} mesh + reference solids at {view['res_x']}x{view['res_y']}, "
                           f"{r['tet_steps']} tet-steps; plane ctor + find_intersections + the per-pixel loop of "
                           "plane.cpp:161-169 driven by the harness without the float cast (the pre-cast doubles feed `parity`)")}
            line["parity"] = parity_record(ours, r["image"], against=(
                "oracle/_ref (the unmodified reference) on this box, same mesh, flags, solids and resolution"
                if r["kind"] == "reference" else "oracle/c5_oracle.c (C restatement; oracle/_ref was not built)"))
        print(json.dumps(line), flush=True)
        if line.get("parity") and not line["parity"]["ok"]:
            print("[bench] PARITY FAILED: " + json.dumps(line["parity"]), file=sys.stderr, flush=True)
            parity_failed = True
    dog.tick("teardown", limit_s=120.0)
    br.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if parity_failed:
        raise SystemExit(4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default="C3", choices=sorted(synth.CONFIGS),
                    help="named configuration (course5_b200.synth.CONFIGS); C3 is BASELINE.json's metric configuration")
    ap.add_argument("--lanes", type=int, default=0, choices=range(0, api.MAX_IN_FLIGHT + 1),
                    help="views in flight per GPU (the context and lanes-1 siblings sharing its mesh, one stream each), for the "
                         "device-timed value and for e2e alike; 0 = chosen from N and the mesh size (see run_ours)")
    ap.add_argument("--gather", choices=["auto", "p2p", "sendrecv"], default="p2p",
                    help="N > 1: how bands reach rank 0's image. p2p = stored by the walk kernels straight into rank 0's image "
                         "over NVLink peer mappings (CUDA IPC); sendrecv = one grouped ncclSend/ncclRecv per view (the baseline)")
    ap.add_argument("--e2e-in-flight", type=int, default=0, choices=range(0, api.MAX_IN_FLIGHT + 1),
                    help="e2e: views in flight per GPU through c5_render_submit / c5_render_wait (0 = --lanes, or 4; 3 on big meshes)")
    ap.add_argument("--view-groups", type=int, default=0,
                    help="N > 1: split the ranks into this many groups that render alternate views, each by N / groups row "
                         "bands (1 = every rank a band of every view; 0 = 1, except N / 2 groups of two ranks for meshes "
                         "above 16M tets from N = 8 on)")
    ap.add_argument("--calibrate", type=int, default=8, help="N > 1: rounds of band calibration before the timed region")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline + parity leg (profiling runs)")
    ap.add_argument("--e2e-mode", choices=["auto", "inplace", "copy"], default="auto",
                    help="e2e: the walk kernels store into the page-locked host image in place (default), or render into "
                         "device memory and let the copy engine bring the image to the host (c5_debug_set no_zero_copy)")
    ap.add_argument("--debug", default="", help="c5_debug_set knobs for experiments, key=value[,key=value]")
    ap.add_argument("--experiment-no-exchange", action="store_true",
                    help="EXPERIMENT, not a measurement of the product path: the timed views skip the image exchange and its "
                         "per-view barrier, to see what the coupling of the ranks costs (the line is marked invalid)")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="do not restrict each rank to the CPUs (and so the memory) of its GPU's NUMA node")
    ap.add_argument("--no-clock-sampler", action="store_true", help="experiments: no NVML polling at all")
    ap.add_argument("--timeline", default=None, metavar="FILE",
                    help="write per-rank, per-view phase times of the timed region (CUDA events) and host enqueue times as JSON")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed views, write the image the last one computed to DIR as .npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("C5_BENCH_CHILD") is None:
        run_with_fallback(args)
    else:
        run_ours(args)


def _die_with_parent():
    """In the child, before exec: if the launcher kills this rank, its measurement process goes too
    (no orphan left on a GPU)."""
    import ctypes
    import signal
    try:
        ctypes.CDLL("libc.so.6", use_errno=True).prctl(1, int(signal.SIGKILL), 0, 0, 0)   # PR_SET_PDEATHSIG
    except Exception:
        pass


def run_with_fallback(args):
    """N > 1: every rank runs the measurement in a CHILD process and falls back to the baseline
    transport if the first configuration does not finish. A multi-process GPU run that deadlocks cannot
    be rescued from inside (the collective never returns); the child's own watchdog ends it, every rank
    sees a non-zero exit code at about the same time, and all of them start the next attempt — on a
    fresh rendezvous port, since the first attempt's store is dead. The parent touches neither CUDA
    nor NCCL, so a killed child leaves the devices free. What was attempted and why it was left is
    recorded in the line that finally prints ("attempts")."""
    import subprocess
    rank = int(os.environ.get("RANK", "0"))
    base_port = int(os.environ.get("MASTER_PORT", "29500"))
    attempts = [dict(gather=args.gather, lanes=args.lanes)]
    safe = dict(gather="sendrecv", lanes=2)     # round 1's measured configuration
    if attempts[0] != safe:
        attempts.append(safe)
    log = []
    for i, a in enumerate(attempts):
        # a port of its own per attempt, the same on every rank, away from the launcher's (whose next run may
        # well use base_port + 1)
        port = 31000 + (base_port + 17 * (i + 1)) % 2000
        env = dict(os.environ, C5_BENCH_CHILD="1", MASTER_PORT=str(port), TORCHELASTIC_USE_AGENT_STORE="False",
                   C5_BENCH_ATTEMPTS=json.dumps(log))
        cmd = [sys.executable, os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--gather", a["gather"], "--lanes", str(a["lanes"]), "--workload", args.workload,
               "--e2e-mode", args.e2e_mode, "--calibrate", str(args.calibrate), "--debug", args.debug,
               "--view-groups", str(args.view_groups), "--e2e-in-flight", str(args.e2e_in_flight)]
        if args.no_cpu_baseline:
            cmd.append("--no-cpu-baseline")
        if args.timeline:
            cmd += ["--timeline", args.timeline]
        if args.dump_outputs:
            cmd += ["--dump-outputs", args.dump_outputs]
        if args.no_clock_sampler:
            cmd.append("--no-clock-sampler")
        if args.no_numa_bind:
            cmd.append("--no-numa-bind")
        if args.experiment_no_exchange:
            cmd.append("--experiment-no-exchange")
        try:   # stderr passes through; the hard limit is a second line of defence behind the child's watchdog
            p = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, text=True, preexec_fn=_die_with_parent,
                               timeout=float(os.environ.get("C5_BENCH_ATTEMPT_LIMIT", "600")))
        except subprocess.TimeoutExpired:
            p = subprocess.CompletedProcess(cmd, returncode=124, stdout="")
        if p.returncode == 0:
            if rank == 0:   # the JSON line only (NCCL prints its version banner on stdout)
                for out_line in p.stdout.splitlines():
                    if out_line.startswith("{"):
                        print(out_line, flush=True)
            return
        log.append(dict(a, exit_code=p.returncode))
        print(f"[bench rank {rank}] attempt {a} ended with exit code {p.returncode}"
              + ("; falling back" if i + 1 < len(attempts) else ""), file=sys.stderr, flush=True)
    raise SystemExit(3)


if __name__ == "__main__":
    main()
