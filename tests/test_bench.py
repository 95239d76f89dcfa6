"""bench.py on CPU: what can be checked without a GPU — the reference arm (the one place besides
tests/ that may execute oracle/), the parity record it attaches to a line, and that both arms
describe the workload in the same words. The CUDA arm itself refuses to run without a device; on a
B200, its --dump-outputs image is checked against a render of the same view."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _line(out: str) -> dict:
    lines = [l for l in out.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out
    return json.loads(lines[0])


def test_reference_arm_prints_a_line_on_the_named_workload(built):
    """--impl reference on BASELINE.json configs[0] (the reference's own CPU-runnable case; the
    default workload, configs[2], needs ~8 GB and half a minute per step)."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    d = _line(p.stdout)
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["unit"] == "tet-steps/s"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "tet-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    import bench
    from course5_b200 import synth
    mesh, view = synth.make_config("C1")
    assert d["config"] == bench.config_dict("C1", mesh, view)        # the same words as the CUDA arm's line
    assert "600x450" in d["config"]["workload"] and "600x450" in d["cpu_baseline"]["sample"]
    assert d["tet_steps_per_view"] > 6_000_000


def test_reference_arm_other_ranks_stay_silent(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_cuda_arm_refuses_to_run_without_a_device(built):
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("only meaningful without a CUDA device")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "no CPU path" in (p.stderr + p.stdout) and "{" not in p.stdout


def _load_dump(directory):
    """(image with NaN under solids, as bench.py's image is, rebuilt from the dump; the dumped arrays)."""
    arrays = {n: np.load(os.path.join(directory, n + ".npy")) for n in ("tau", "intensity", "solid")}
    for name, a in arrays.items():
        assert np.isfinite(a).all(), f"{name}.npy is not finite"
    assert arrays["tau"].dtype == arrays["intensity"].dtype == np.float64 and arrays["solid"].dtype == np.float32
    assert set(np.unique(arrays["solid"]).tolist()) <= {0.0, 1.0}
    solid = arrays["solid"] == 1.0
    image = np.stack([np.where(solid, np.nan, arrays["tau"]), np.where(solid, np.nan, arrays["intensity"])], axis=-1)
    return image, arrays


def test_reference_arm_dumps_the_last_image(built, port, tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1",
                        "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    got, arrays = _load_dump(tmp_path / "out")
    assert got.shape == (450, 600, 2)
    if _line(p.stdout)["cpu_baseline"]["kind"] == "port":
        import bench
        from course5_b200 import synth
        mesh, view = synth.make_config("C1")
        roche, sphere = bench.reference_solids(view["D"])
        want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=600, res_y=450, X=view["X"], Y=view["Y"],
                           I=view["I"], alpha_limit=view["alpha_limit"], solid_rot=roche, solid_static=sphere)
        assert np.array_equal(got, np.stack([want.tau, want.inten], axis=-1), equal_nan=True)
    assert arrays["solid"].any() and (arrays["intensity"] > 0).any()


@pytest.mark.gpu
def test_cuda_arm_dump_equals_a_render_of_the_benchmark_view(gpu_lib, tmp_path):
    """bench.py's render plus the dump round trip. Every timed step renders the same view, so this cannot
    tell the last step's image from an earlier one's."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", "3", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out")],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    assert _line(p.stdout)["steps"] == 3
    got, arrays = _load_dump(tmp_path / "out")
    import bench
    from course5_b200 import api, synth
    mesh, view = synth.make_config("C1")
    roche, sphere = bench.reference_solids(view["D"])
    with api.Context(devices=(0,), lib=gpu_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(roche, True)
        ctx.upload_solids(sphere, False)
        want, _ = ctx.render(api.make_view(view["res_x"], view["res_y"], X=view["X"], Y=view["Y"], I=view["I"],
                                           alpha_limit=view["alpha_limit"], lib=gpu_lib))
    assert got.shape == (450, 600, 2) and arrays["solid"].any()
    assert np.array_equal(got, want, equal_nan=True)


def test_dump_of_a_large_image_is_a_fixed_sample(tmp_path):
    import bench
    image = np.random.default_rng(7).normal(size=(1800, 2400, 2))
    image[100:300, 200:900] = np.nan                  # a solid
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), image)
        assert sorted(os.listdir(tmp_path / run)) == ["intensity.npy", "solid.npy", "tau.npy"]
        assert sum(os.path.getsize(tmp_path / run / n) for n in os.listdir(tmp_path / run)) <= 64_000_000
    a, arrays = _load_dump(tmp_path / "a")
    b, _ = _load_dump(tmp_path / "b")
    assert a.shape == (bench.DUMP_SAMPLE_PIXELS, 2) and np.array_equal(a, b, equal_nan=True)
    assert arrays["solid"].any()
    pick = np.sort(np.random.default_rng(0).choice(1800 * 2400, bench.DUMP_SAMPLE_PIXELS, replace=False))
    assert np.array_equal(a, image.reshape(-1, 2)[pick], equal_nan=True)


def test_parity_record(hostsim_lib, port):
    """The record bench.py attaches to its line: green on a faithful image, red (with counts) on a
    perturbed one. (Here the device functions' host build stands in for the GPU.)"""
    import bench
    from course5_b200 import api, synth
    mesh = synth.kuhn_cube(8, seed=81)
    with api.Context(lib=hostsim_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ours = ctx.render_raw(api.make_view(120, 90, X=0.4, Y=0.3, lib=hostsim_lib, round_through_float=0))
    want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=120, res_y=90, X=0.4, Y=0.3)
    rec = bench.parity_record(ours, want, against="the C restatement")
    assert rec["ok"] and rec["pixels_out_of_tolerance"] == 0 and rec["max_rel_err_where_value_ge_1e-3"] < 1e-9
    assert rec["hit_sets_equal"] and rec["per_pixel_steps_equal"] and rec["solid_masks_equal"]
    assert rec["tet_steps"][0] == rec["tet_steps"][1] == want.total_steps
    j, i = np.argwhere(want.steps > 0)[5]
    ours.image[j, i, 1] *= 1.0 + 1e-7
    ours.steps[0, 0] += 1
    rec = bench.parity_record(ours, want, against="the C restatement")
    assert not rec["ok"] and rec["pixels_out_of_tolerance"] == 1 and not rec["per_pixel_steps_equal"]
    assert 0.9e-7 < rec["max_rel_err_where_value_ge_1e-3"] < 1.1e-7 or rec["max_abs_err"] > 0
