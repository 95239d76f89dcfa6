"""Flux renders (c5_render_flux / c5_render_flux_submit): per-row sums of a view reduced on the device,
for light curves. Every check runs on the host-loop build of the device code (tests/hostsim) and, with
-m gpu, on the CUDA library.

The contract of include/c5gpu.h is restated below in numpy (256-stride partials per row, halving tree,
sequential total) and applied to the image and mask the image calls give for the same view: the sums
must match it bit for bit, whatever the row band, device count or number of views in flight."""
import math

import numpy as np
import pytest

from cases import reference_solids
from course5_b200 import api, sweep, synth

LIBS = [pytest.param("hostsim_lib", id="hostsim"), pytest.param("gpu_lib", id="gpu", marks=pytest.mark.gpu)]
PORT_VIEWS = [dict(X=0.0, Y=0.0), dict(X=0.4, Y=0.7, I=-0.03, alpha_limit=1.2), dict(X=0.5, Y=1.9, I=0.3)]
THREADS = 256


@pytest.fixture(params=LIBS)
def lib(request):
    return request.getfixturevalue(request.param)


def fields(mesh, n, seed):
    rng = np.random.default_rng(seed)
    alpha = rng.uniform(0.0, 4.0, (n, mesh.n_tets))
    alpha[:, ::17] = 0.0
    q = rng.uniform(0.1, 4.0, (n, mesh.n_tets))
    return alpha, q


def make_context(lib, mesh, *, channels=None, solids=None, debug=None, devices=(0,)):
    ctx = api.Context(devices=devices, lib=lib)
    for key, value in (debug or {}).items():
        ctx.debug_set(key, value)
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    if solids is not None:
        ctx.upload_solids(solids[0], True)
        ctx.upload_solids(solids[1], False)
    if channels is not None:
        ctx.upload_channels(*channels)
    return ctx


def view_of(lib, res, flags, **over):
    return api.make_view(res[0], res[1], lib=lib, **{"round_through_float": 0, **flags, **over})


def contract_rows(image, solid):
    """The documented order. image: (res_y, res_x, n, 2); solid: (res_y, res_x). Thread t of row j adds
    the pixels x = t, t + 256, ... not under the mask, in increasing x; p[t] += p[t + s], s = 128 .. 1."""
    res_y, res_x, n, _ = image.shape
    vals = image.reshape(res_y, res_x, 2 * n)
    mask = solid.astype(bool)
    p = np.zeros((res_y, THREADS, 2 * n))
    for k in range(0, res_x, THREADS):
        xs = np.arange(k, min(k + THREADS, res_x))
        t = xs - k
        keep = ~mask[:, xs, None]
        p[:, t] = np.where(keep, p[:, t] + vals[:, xs], p[:, t])
    s = THREADS // 2
    while s:
        p[:, :s] = p[:, :s] + p[:, s:2 * s]
        s //= 2
    return p[:, 0].reshape(res_y, n, 2)


def sequential_total(rows):
    total = np.zeros(rows.shape[1:])
    for j in range(rows.shape[0]):
        total = total + rows[j]
    return total


def check_contract(rows, total, image, solid):
    want = contract_rows(image, solid)
    assert rows.shape == want.shape
    assert np.array_equal(rows, want), "row sums differ from the documented order"
    assert np.array_equal(total, sequential_total(want))
    keep = ~solid.astype(bool)
    for c in range(image.shape[2]):
        for w in range(2):
            exact = math.fsum(image[:, :, c, w][keep].tolist())
            assert abs(total[c, w] - exact) <= 1e-12 * abs(exact), (c, w)


def flux_and_image(ctx, v, channels):
    rows, total, st = ctx.render_flux(v, channels=channels)
    if channels:
        image, _, solid, ist = ctx.render_channels(v, raw=True)
    else:
        raw = ctx.render_raw(v)
        image, solid, ist = raw.image[:, :, None, :], raw.solid, raw.stats
    return rows, total, st, image, solid, ist


# ---- the contract ------------------------------------------------------------------------------------

@pytest.mark.parametrize("rtf", [0, 1])
def test_flux_contract_plain_with_solids(lib, rtf):
    mesh = synth.kuhn_cube(10, seed=41)
    with make_context(lib, mesh, solids=reference_solids(0.0)) as ctx:
        for flags in PORT_VIEWS + [dict(X=0.45, Y=0.3)]:
            v = view_of(lib, (300, 150), flags, round_through_float=rtf)
            rows, total, st, image, solid, ist = flux_and_image(ctx, v, False)
            check_contract(rows, total, image, solid)
            for key in ("tet_steps", "hit_pixels", "solid_pixels", "grazing_rays", "pixels", "walk_errors"):
                assert st[key] == ist[key], key
        assert solid.sum() > 0


@pytest.mark.parametrize("n", [1, 3, 8])
@pytest.mark.parametrize("rtf", [0, 1])
def test_flux_contract_channels(lib, n, rtf):
    mesh = synth.kuhn_cube(9, seed=42)
    alpha, q = fields(mesh, n, seed=100 + n)
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.0)) as ctx:
        for flags in PORT_VIEWS:
            v = view_of(lib, (270, 120), flags, round_through_float=rtf)
            rows, total, st, image, solid, ist = flux_and_image(ctx, v, True)
            assert rows.shape == (120, n, 2) and total.shape == (n, 2)
            check_contract(rows, total, image, solid)
            assert st["tet_steps"] == ist["tet_steps"]


def test_flux_fp32_view(lib):
    mesh = synth.kuhn_cube(8, seed=43)
    with make_context(lib, mesh) as ctx:
        v = view_of(lib, (200, 100), dict(X=0.4, Y=0.3), precision=32)
        rows, total, _, image, solid, _ = flux_and_image(ctx, v, False)
        check_contract(rows, total, image, solid)


def test_flux_includes_grazing_rays(lib):
    """Deferred rays are finished by the grazing-ray kernel; the reduction runs after it."""
    mesh = synth.kuhn_cube(12, seed=48)
    with make_context(lib, mesh) as ctx:
        for flags in (dict(X=0.5, Y=0.0), dict(X=0.0, Y=0.5)):
            rows, total, st, image, solid, _ = flux_and_image(ctx, view_of(lib, (240, 180), flags), False)
            assert st["grazing_rays"] > 0
            check_contract(rows, total, image, solid)
    mesh = synth.kuhn_cube(10, seed=55, scalars="sphere", carve_sphere=True)
    alpha, q = fields(mesh, 2, seed=12)
    with make_context(lib, mesh, channels=(alpha, q), debug={"query_budget": 3}) as ctx:
        v = view_of(lib, (200, 150), dict(X=0.3, Y=0.4))
        for channels in (False, True):
            rows, total, st, image, solid, _ = flux_and_image(ctx, v, channels)
            assert st["grazing_rays"] > 0
            check_contract(rows, total, image, solid)


# ---- invariance --------------------------------------------------------------------------------------

def test_flux_row_bands(lib):
    mesh = synth.kuhn_cube(8, seed=31)
    alpha, q = fields(mesh, 3, seed=14)
    flags = dict(X=0.4, Y=0.9)
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.2)) as ctx:
        for channels in (False, True):
            full, _, _ = ctx.render_flux(view_of(lib, (150, 111), flags), channels=channels)
            for lo, hi in ((0, 37), (37, 80), (80, 111), (50, 51), (3, 106)):
                rows, total, st = ctx.render_flux(view_of(lib, (150, 111), flags, row_begin=lo, row_end=hi),
                                                  channels=channels)
                assert np.array_equal(rows[lo:hi], full[lo:hi])
                assert np.all(rows[:lo] == 0.0) and np.all(rows[hi:] == 0.0)
                assert np.array_equal(total, sequential_total(rows))
                assert st["pixels"] == (hi - lo) * 150


@pytest.mark.parametrize("in_flight", [1, 2, 4])
def test_flux_pipelined_sweep(lib, in_flight):
    mesh = synth.kuhn_cube(8, seed=33)
    alpha, q = fields(mesh, 2, seed=15)
    views = sweep.sweep_views(160, 90, X=0.4, I=-0.03, alpha_limit=2.0, frames=7, round_through_float=0)
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.1)) as ctx:
        for channels in (False, True):
            want = [ctx.render_flux(v, channels=channels) for v in views]
            totals, stats = sweep.render_light_curve(ctx, views, in_flight=in_flight, channels=channels)
            assert totals.shape == (7, 2 if channels else 1, 2)
            for k, (rows, total, st) in enumerate(want):
                assert np.array_equal(totals[k], total), k
                assert stats[k]["tet_steps"] == st["tet_steps"]
            # the row sums of submitted views, too
            ctx.set_views_in_flight(in_flight)
            sub = [ctx.render_flux_submit(v, channels=channels) for v in views[:in_flight]]
            for (ticket, rows, total), (w_rows, w_total, _) in zip(sub, want):
                ctx.render_wait(ticket)
                assert np.array_equal(rows, w_rows) and np.array_equal(total, w_total)


def test_flux_multi_device_context(lib):
    """A context over devices (0, 0): two parts on one device, each reducing its band."""
    mesh = synth.kuhn_cube(8, seed=36)
    alpha, q = fields(mesh, 3, seed=19)
    views = [view_of(lib, (160, 121), dict(X=0.4, Y=y)) for y in (0.1, 0.8, 1.3)]
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.0)) as one:
        want = [[one.render_flux(v, channels=c) for v in views] for c in (False, True)]
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.0), devices=(0, 0)) as many:
        for c, channels in enumerate((False, True)):
            for v, (w_rows, w_total, w_st) in zip(views, want[c]):
                rows, total, st = many.render_flux(v, channels=channels)
                assert np.array_equal(rows, w_rows) and np.array_equal(total, w_total)
                assert st["n_devices"] == 2 and st["tet_steps"] == w_st["tet_steps"]


@pytest.mark.gpu
def test_flux_distinct_devices(gpu_lib):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mesh = synth.kuhn_cube(8, seed=37)
    alpha, q = fields(mesh, 2, seed=24)
    v = view_of(gpu_lib, (160, 120), dict(X=0.4, Y=0.5))
    with make_context(gpu_lib, mesh, channels=(alpha, q)) as one:
        want = [one.render_flux(v, channels=c)[:2] for c in (False, True)]
    with make_context(gpu_lib, mesh, channels=(alpha, q), devices=(0, 1)) as many:
        for c, channels in enumerate((False, True)):
            rows, total, _ = many.render_flux(v, channels=channels)
            assert np.array_equal(rows, want[c][0]) and np.array_equal(total, want[c][1])


# ---- plumbing ----------------------------------------------------------------------------------------

def test_flux_errors(lib):
    mesh = synth.kuhn_cube(5, seed=35)
    alpha, q = fields(mesh, 2, seed=16)
    v = view_of(lib, (64, 48), dict(X=0.3, Y=0.2))
    rows, total = np.zeros(48 * 2 * 2), np.zeros(2 * 2)
    r, t = rows.ctypes.data_as(api._dp), total.ctypes.data_as(api._dp)
    ticket = api.C.c_uint64(0)

    def flux(ctx, channels=0, rows=r, total=t, view=v):
        return ctx.lib.c5_render_flux(ctx._h, api.C.byref(view), channels, rows, total, None)

    def flux_submit(ctx, channels=0, rows=r, total=t, view=v):
        return ctx.lib.c5_render_flux_submit(ctx._h, api.C.byref(view), channels, rows, total, api.C.byref(ticket))

    with api.Context(devices=(0,), lib=lib) as ctx:
        assert flux(ctx) == api.E_STATE                                     # no mesh
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        for call in (flux, flux_submit):
            assert call(ctx, rows=None, total=None) == api.E_INVALID       # both outputs NULL
            assert call(ctx, channels=2) == api.E_INVALID
            assert call(ctx, channels=-1) == api.E_INVALID
        assert flux(ctx, channels=1) == api.E_STATE                         # no channels uploaded
        assert flux_submit(ctx, channels=1) == api.E_STATE
        assert flux(ctx, rows=None) == api.OK and flux(ctx, total=None) == api.OK
        ctx.upload_channels(alpha, q)
        v32 = view_of(lib, (64, 48), dict(X=0.3, Y=0.2), precision=32)
        assert flux(ctx, channels=1, view=v32) == api.E_INVALID
        assert flux_submit(ctx, channels=1, view=v32) == api.E_INVALID
        assert flux(ctx, channels=0, view=v32) == api.OK
        sib = ctx.sibling()
        try:
            assert flux_submit(sib) == api.E_STATE                          # submit: not on a sibling ...
            want, want_total, _ = ctx.render_flux(v, channels=True)
            got, got_total, _ = sib.render_flux(v, channels=True)          # ... but the blocking call works
            assert np.array_equal(got, want) and np.array_equal(got_total, want_total)
        finally:
            sib.close()
        # one submit more than lanes; a flux view in flight blocks c5_upload_channels
        ctx.set_views_in_flight(2)
        a, _, _ = ctx.render_flux_submit(v)
        b, _, _ = ctx.render_flux_submit(v, channels=True)
        with pytest.raises(api.C5Error) as e:
            ctx.render_flux_submit(v)
        assert e.value.code == api.E_STATE
        with pytest.raises(api.C5Error) as e:
            ctx.upload_channels(alpha, q)
        assert e.value.code == api.E_STATE
        ctx.render_wait(b)
        ctx.render_wait(a)
        ctx.upload_channels(alpha, q)
    with make_context(lib, mesh, devices=(0, 0)) as many:
        assert flux_submit(many) == api.E_STATE                             # not on a multi-device context


def test_flux_tickets_interleave_with_image_tickets(lib):
    mesh = synth.kuhn_cube(8, seed=38)
    alpha, q = fields(mesh, 2, seed=20)
    views = [view_of(lib, (120, 90), dict(X=0.4, Y=y)) for y in (0.0, 0.3, 0.6, 0.9, 1.2)]
    with make_context(lib, mesh, channels=(alpha, q)) as ctx:
        want_img = [ctx.render_raw(v).image for v in views]
        want_flux = [ctx.render_flux(v, channels=True)[:2] for v in views]
        ctx.set_views_in_flight(4)
        images = [np.full((90, 120, 2), -1.0) for _ in views]
        for order in ([0, 1, 2, 3], [3, 1, 0, 2], [2, 3, 1, 0]):
            pending = []
            for k, v in enumerate(views[:4]):
                if k % 2:
                    pending.append(("flux", k, ctx.render_flux_submit(v, channels=True)))
                else:
                    pending.append(("image", k, ctx.render_submit(v, images[k])))
            for i in order:
                kind, k, handle = pending[i]
                if kind == "flux":
                    ticket, rows, total = handle
                    ctx.render_wait(ticket)
                    assert np.array_equal(rows, want_flux[k][0]) and np.array_equal(total, want_flux[k][1])
                else:
                    ctx.render_wait(handle)
                    assert np.array_equal(images[k], want_img[k])


def test_flux_launches_one_kernel_more(lib):
    mesh = synth.kuhn_cube(8, seed=39)
    alpha, q = fields(mesh, 3, seed=21)
    with make_context(lib, mesh, channels=(alpha, q), solids=reference_solids(0.0)) as ctx:
        for over in (dict(), dict(row_begin=20, row_end=70)):
            v = view_of(lib, (120, 90), dict(X=0.4, Y=0.3), **over)
            for channels in (False, True):
                ctx.render_flux(v, channels=channels)           # warm: lazily built tables and buffers
                before = ctx.kernel_launches()
                ctx.render_channels(v) if channels else ctx.render_raw(v)
                image_launches = ctx.kernel_launches() - before
                before = ctx.kernel_launches()
                ctx.render_flux(v, channels=channels)
                assert ctx.kernel_launches() - before == image_launches + 1


# ---- course --light_curve ----------------------------------------------------------------------------

def test_course_light_curve_flag_parsing():
    from course5_b200 import hostlib
    base = ["-f", "a.vtk", "-d", "curve.csv"]
    assert hostlib.parse_cli(base + ["--light_curve"])[0] == 0
    r, text, _ = hostlib.parse_cli(base + ["--channels", "A1:Q1", "--frames", "4"])
    assert r == 2 and "Error!" in text
    assert hostlib.parse_cli(base + ["--channels", "A1:Q1", "--frames", "4", "--light_curve"])[0] == 0
    assert hostlib.parse_cli(base + ["--light_curve", "--frames", "4", "--sweep_y_to", "1"])[0] == 0
    r, text, _ = hostlib.parse_cli(["--help"])
    assert "--light_curve" in text


@pytest.mark.gpu
def test_course_light_curve_end_to_end(gpu_lib, tmp_path):
    """`course --light_curve` over 4 frames with two --channels pairs: every CSV value parses back to
    exactly what render_flux gives for the same views."""
    import csv
    import subprocess
    from course5_b200 import hostlib
    mesh = synth.kuhn_cube(12, seed=61)
    alpha, q = fields(mesh, 2, seed=26)
    src = str(tmp_path / "grid.vtk")
    synth.write_legacy_vtk(src, mesh)
    with open(src, "ab") as f:
        for name, values in {"A1": alpha[0], "Q1": q[0], "A2": alpha[1], "Q2": q[1]}.items():
            f.write(f"SCALARS {name} double 1\nLOOKUP_TABLE default\n".encode())
            np.savetxt(f, values, fmt="%.17g")
    dst = str(tmp_path / "curve.csv")
    p = subprocess.run([hostlib.COURSE_EXE, "-f", src, "-d", dst, "-x", "320", "-y", "240", "-X", "0.4", "-Y", "0.3",
                        "-D", "0.1", "-I", "-0.03", "--alpha_limit", "2.0", "--frames", "4", "--sweep_y_to", "1.1",
                        "--light_curve", "--channels", "A1:Q1,A2:Q2"], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    with open(dst) as f:
        table = list(csv.reader(f))
    assert table[0] == ["frame", "Y_pi", "hit_pixels", "solid_pixels", "tau_sum", "I_sum",
                        "A1:Q1_tau_sum", "A1:Q1_I_sum", "A2:Q2_tau_sum", "A2:Q2_I_sum"]
    assert len(table) == 5
    views = sweep.sweep_views(320, 240, X=0.4, I=-0.03, alpha_limit=2.0, y_from=0.3, y_to=1.1, frames=4)
    with make_context(gpu_lib, mesh, channels=(alpha, q), solids=reference_solids(0.1)) as ctx:
        for k, (row, v) in enumerate(zip(table[1:], views)):
            _, total, st = ctx.render_flux(v)
            _, ch_total, _ = ctx.render_flux(v, channels=True)
            assert int(row[0]) == k and float(row[1]) == 0.3 + (1.1 - 0.3) * k / 4
            assert int(row[2]) == st["hit_pixels"] and int(row[3]) == st["solid_pixels"]
            got = [float(x) for x in row[4:]]
            want = [total[0, 0], total[0, 1]] + [ch_total[c, w] for c in range(2) for w in range(2)]
            assert got == want, k
