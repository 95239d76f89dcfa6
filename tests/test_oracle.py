"""The oracle itself: the C restatement (oracle/c5_oracle.c) against the committed golden vectors
generated from the unmodified reference, against the reference run live (where oracle/_ref was
built), and against known answers derived from line.cpp:176-227."""
import numpy as np
import pytest

from cases import GOLDEN_CASES, GOLDEN_INDEX, golden_case, reference_solids, view_kwargs
from course5_b200 import synth


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_port_reproduces_golden_bitwise(port, name):
    mesh, meta, gold = golden_case(name)
    solid_rot = solid_static = None
    if meta["solids"]:
        sol = reference_solids(meta["flags"]["D"])
        if sol is None:
            pytest.skip("solids need oracle/_ref")
        solid_rot, solid_static = sol
    img = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=meta["res_x"], res_y=meta["res_y"],
                      solid_rot=solid_rot, solid_static=solid_static, threads=4, **view_kwargs(meta))
    assert img.anomalies == 0
    assert img.total_steps == meta["total_steps"]
    assert np.array_equal(img.steps, gold["steps"])
    assert np.array_equal(img.solid, gold["solid"])
    assert np.array_equal(img.tau, gold["tau"], equal_nan=True)      # bit for bit
    assert np.array_equal(img.inten, gold["inten"], equal_nan=True)


@pytest.mark.parametrize("flags", [dict(X=0.0, Y=0.0, I=0.0), dict(X=0.4, Y=1.1, I=-0.03), dict(X=0.5, Y=0.25, I=0.2)])
def test_port_matches_live_reference_bitwise(port, ref, flags):
    mesh = synth.kuhn_cube(9, seed=21)
    a = ref.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=160, res_y=120, alpha_limit=1.7, threads=4, **flags)
    b = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=160, res_y=120, alpha_limit=1.7, threads=4, **flags)
    assert np.array_equal(a.steps, b.steps)
    assert np.array_equal(a.tau, b.tau)
    assert np.array_equal(a.inten, b.inten)


def test_thread_count_does_not_change_the_port(port):
    mesh = synth.kuhn_cube(7, seed=3)
    kw = dict(res_x=120, res_y=90, X=0.3, Y=0.6, alpha_limit=2.5)
    a = port.render(mesh.tet_points(), mesh.alpha, mesh.q, threads=1, **kw)
    b = port.render(mesh.tet_points(), mesh.alpha, mesh.q, threads=5, **kw)
    assert np.array_equal(a.tau, b.tau) and np.array_equal(a.inten, b.inten)


def test_float_rounded_reference_flow_matches_raw(ref):
    """mode 0 of the harness is the reference's own trace_rays (float cast, plane.cpp:165-166)."""
    mesh = synth.kuhn_cube(6, seed=5)
    kw = dict(res_x=96, res_y=72, X=0.4, Y=0.2, alpha_limit=2.5, threads=2)
    raw = ref.render(mesh.tet_points(), mesh.alpha, mesh.q, raw=True, **kw)
    cast = ref.render(mesh.tet_points(), mesh.alpha, mesh.q, raw=False, **kw)
    assert np.array_equal(raw.tau.astype(np.float32).astype(np.float64), cast.tau)
    assert np.array_equal(raw.inten.astype(np.float32).astype(np.float64), cast.inten)


# ---- known answers (SURVEY.md §8c) --------------------------------------------------------------

def test_kat_pixel_coordinates_are_accumulated(port):
    xs, ys = port.pixel_coords(600, 450)
    assert xs[0] == -0.2 and ys[0] == -0.9
    assert xs[599] == 2.2000000000000028          # not -0.2 + 599 * step (plane.cpp:304-314)
    assert ys[449] == 0.89999999999999813


def test_kat_uniform_medium_telescopes(port):
    """alpha = a, Q = q everywhere: tau = a L and I = (q / a^)(1 - exp(-a^ L)), a^ = min(a, limit)."""
    mesh = synth.kuhn_cube(6, seed=8, scalars="const")  # a = 1.5, q = 0.75
    for limit in (2.5, 0.9):
        img = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=96, res_y=72, X=0.35, Y=0.8,
                          alpha_limit=limit, threads=2)
        hit = img.hit
        L = img.tau[hit] / 1.5
        a_hat = min(1.5, limit)
        want = 0.75 / a_hat * (1.0 - np.exp(-a_hat * L))
        assert np.allclose(img.inten[hit], want, rtol=1e-12, atol=1e-15)
        assert np.all(img.tau[~hit] == 0) and np.all(img.inten[~hit] == 0)   # a miss is (0, 0)


def test_kat_transparent_cells_leave_I_unchanged(port):
    mesh = synth.kuhn_cube(5, seed=9)
    alpha = mesh.alpha.copy()
    alpha[::2] = 1e-17                      # < DBL_EPSILON: skipped by line.cpp:221
    q = mesh.q.copy()
    q[::2] = 1e6                            # would dominate I if those cells emitted
    kw = dict(res_x=80, res_y=60, X=0.4, Y=0.4, alpha_limit=2.5, threads=2)
    img = port.render(mesh.tet_points(), alpha, q, **kw)
    assert img.inten.max() < 100.0


def test_kat_solid_wins_regardless_of_depth(port):
    mesh = synth.kuhn_cube(4, seed=10)
    kw = dict(res_x=80, res_y=60, X=0.0, Y=0.0, alpha_limit=2.5, threads=2)
    # one solid tet far BEHIND the grid (z = -5) and one far in front (z = +5)
    base = np.array([[0.9, -0.1, 0.0], [1.1, -0.1, 0.0], [1.0, 0.1, 0.0], [1.0, 0.0, 0.05]])
    sol = np.stack([base + [0, 0, -5.0], base + [0, 0.3, 5.0]])
    img = port.render(mesh.tet_points(), mesh.alpha, mesh.q, solid_static=sol, **kw)
    plain = port.render(mesh.tet_points(), mesh.alpha, mesh.q, **kw)
    assert img.solid.sum() > 0
    assert np.all(np.isnan(img.tau[img.solid == 1])) and np.all(np.isnan(img.inten[img.solid == 1]))
    assert np.array_equal(img.tau[img.solid == 0], plain.tau[img.solid == 0])


def test_kat_solid_object_sizes():
    """On the reference run live where oracle/_ref was built, else on the sizes of its output stored
    by tests/golden/make_golden.py (tests/golden/index.json)."""
    import os
    from oracle import refbind
    if os.path.exists(refbind.REF_SO):
        roche, sphere = refbind.Ref().solids(0.0)
        shapes = roche.shape, sphere.shape
    else:
        pin = GOLDEN_INDEX["_solids"]["0"]
        shapes = (pin["n_roche"], 4, 3), (pin["n_sphere"], 4, 3)
    assert shapes[0] == (130560, 4, 3)    # 255 x 256 rings x points x 2
    assert shapes[1] == (522242, 4, 3)    # 511 x 511 x 2


def test_reference_file_to_file_flow_matches_in_memory(ref, tmp_path):
    """main.cpp:96-137 end to end through the stand-in reader/writer == the in-memory harness."""
    from course5_b200 import hostlib
    mesh = synth.kuhn_cube(4, seed=61)
    src, dst = str(tmp_path / "g.vtk"), str(tmp_path / "ref.vti")
    synth.write_legacy_vtk(src, mesh)
    kw = dict(res_x=64, res_y=48, threads=2, X=0.4, Y=0.3, D=0.1, I=-0.03, alpha_limit=2.0)
    assert ref.run_files(src, dst, **kw) == 0
    img = hostlib.read_vti(dst)
    mem = ref.render(mesh.tet_points(), mesh.alpha, mesh.q, solids=1, raw=False, **kw)
    assert np.array_equal(img[..., 0], mem.tau, equal_nan=True)
    assert np.array_equal(img[..., 1], mem.inten, equal_nan=True)
