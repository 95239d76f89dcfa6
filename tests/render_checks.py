"""Checks of the C-ABI render path against the oracle, written once and run twice:
  * tests/test_hostsim.py  — the device functions compiled for the host (CPU container, logic only)
  * tests/test_gpu_parity.py (-m gpu) — the CUDA library on a B200: the parity tests proper.
Every function takes the loaded library (a ctypes CDLL typed by course5_b200.api)."""
import numpy as np
import pytest

from cases import golden_case, reference_solids, view_kwargs
from course5_b200 import api, synth
from parity import ABS_FLOOR_FP32, REL_TOL_FP32, assert_image_parity, assert_same_hits


def render_raw(lib, mesh, res_x, res_y, *, solids=None, raw=True, debug=None, **flags):
    """debug: {key: value} for c5_debug_set (tests shrink list sizes / search budgets to reach the
    overflow paths on small meshes)."""
    with api.Context(devices=(0,), lib=lib) as ctx:
        for key, value in (debug or {}).items():
            ctx.debug_set(key, value)
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        if solids is not None:
            ctx.upload_solids(solids[0], True)
            ctx.upload_solids(solids[1], False)
        view = api.make_view(res_x, res_y, lib=lib, round_through_float=0 if raw else 1, **flags)
        return ctx.render_raw(view)


def check_golden(lib, name):
    mesh, meta, gold = golden_case(name)
    solids = None
    if meta["solids"]:
        solids = reference_solids(meta["flags"]["D"])
        if solids is None:
            pytest.skip("solids need oracle/_ref")
    img = render_raw(lib, mesh, meta["res_x"], meta["res_y"], solids=solids, **view_kwargs(meta))
    assert np.array_equal(img.solid, gold["solid"]), "solid (NaN) mask differs"
    assert_same_hits(img.steps, gold["steps"], what=name + ": ")
    assert_image_parity(img.tau, img.inten, gold["tau"], gold["inten"], what=name + ": ")
    assert img.stats["tet_steps"] == meta["total_steps"]
    assert np.array_equal(img.steps, gold["steps"])
    assert img.stats["walk_errors"] == 0
    assert img.stats["solid_pixels"] == int(gold["solid"].sum())
    assert img.stats["hit_pixels"] == int((gold["steps"] > 0).sum())


def check_against_port(lib, port, mesh, res_x, res_y, flags, *, solids=None, steps_exact=True, debug=None):
    img = render_raw(lib, mesh, res_x, res_y, solids=solids, debug=debug, **flags)
    want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=res_x, res_y=res_y,
                       solid_rot=None if solids is None else solids[0],
                       solid_static=None if solids is None else solids[1], **flags)
    assert want.anomalies == 0
    assert np.array_equal(img.solid, want.solid)
    assert_same_hits(img.steps, want.steps)
    assert_image_parity(img.tau, img.inten, want.tau, want.inten)
    if steps_exact:
        assert np.array_equal(img.steps, want.steps)
    assert img.stats["tet_steps"] == want.total_steps
    return img, want


def check_row_bands_equal_full_image(lib):
    mesh = synth.kuhn_cube(7, seed=31)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        full_view = api.make_view(150, 110, X=0.4, Y=0.9, lib=lib, round_through_float=0)
        full, st_full = ctx.render(full_view)
        cost = ctx.last_row_cost(110)
        assert int(cost.sum()) == st_full["tet_steps"]
        bands = api.balanced_bands(cost, 3, base_cost=1.0)
        out = np.full_like(full, -1.0)
        steps = 0
        for lo, hi in bands:
            v = api.make_view(150, 110, X=0.4, Y=0.9, lib=lib, round_through_float=0, row_begin=lo, row_end=hi)
            _, st = ctx.render(v, out=out)
            steps += st["tet_steps"]
            assert st["pixels"] == (hi - lo) * 150
        assert np.array_equal(out, full)          # bit-identical, bands are independent
        assert steps == st_full["tet_steps"]


def check_round_through_float(lib):
    mesh = synth.kuhn_cube(6, seed=32)
    raw = render_raw(lib, mesh, 100, 80, X=0.45, Y=0.3, raw=True)
    cast = render_raw(lib, mesh, 100, 80, X=0.45, Y=0.3, raw=False)
    assert np.array_equal(cast.image, raw.image.astype(np.float32).astype(np.float64))


def check_out_of_window_geometry_is_background(lib):
    """The reference aborts on geometry outside the window (README known problem 2); the B200 path
    must stay finite: pixels that see the mesh get values, the rest background."""
    mesh = synth.kuhn_cube(5, seed=33, centre=(2.1, 0.8, 0.0))     # pokes out of the top-right corner
    img = render_raw(lib, mesh, 120, 90, X=0.0, Y=0.0)
    assert np.isfinite(img.image).all()
    assert img.hit.sum() > 0 and (~img.hit).sum() > 0
    assert np.all(img.image[~img.hit] == 0.0)
    far = synth.kuhn_cube(3, seed=34, centre=(10.0, 10.0, 0.0))    # entirely outside
    img = render_raw(lib, far, 64, 48)
    assert img.hit.sum() == 0 and np.all(img.image == 0.0)


def check_topology_errors(lib):
    mesh = synth.kuhn_cube(3, seed=35)
    with api.Context(devices=(0,), lib=lib) as ctx:
        dup = np.concatenate([mesh.tets, mesh.tets[40:41]])            # an interior tet twice
        with pytest.raises(api.C5Error) as e:
            ctx.upload_mesh(mesh.points, dup, np.append(mesh.alpha, 1.0), np.append(mesh.q, 1.0))
        assert e.value.code == api.E_TOPOLOGY
        bad = mesh.tets.copy()
        bad[5, 2] = mesh.n_points + 7                                  # out-of-range vertex id
        with pytest.raises(api.C5Error) as e:
            ctx.upload_mesh(mesh.points, bad, mesh.alpha, mesh.q)
        assert e.value.code == api.E_INVALID
        v = api.make_view(32, 24, lib=lib)
        with pytest.raises(api.C5Error) as e:
            ctx.render(v)                                              # nothing valid uploaded
        assert e.value.code == api.E_STATE
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)    # the context recovers
        img, st = ctx.render(v)
        assert st["tet_steps"] > 0
        with pytest.raises(api.C5Error):
            ctx.render(api.make_view(1, 24, lib=lib))                  # res = 1 -> step = inf in the reference


def check_single_tet_and_tiny_meshes(lib, port):
    pts = np.array([[0.8, -0.2, 0.0], [1.3, -0.1, 0.1], [1.0, 0.35, -0.05], [1.05, 0.0, 0.6]])
    tets = np.array([[0, 1, 2, 3]], dtype=np.int32)
    mesh = synth.TetMesh(pts, tets, np.array([1.25]), np.array([0.5]))
    check_against_port(lib, port, mesh, 90, 70, dict(X=0.1, Y=0.2))
    two = synth.TetMesh(np.vstack([pts, [[1.1, 0.05, -0.7]]]), np.array([[0, 1, 2, 3], [0, 2, 1, 4]], dtype=np.int32),
                        np.array([1.25, 3.5]), np.array([0.5, 0.1]))
    check_against_port(lib, port, two, 90, 70, dict(X=0.3, Y=1.4, alpha_limit=2.0))


def check_uniform_medium_kat(lib, n=6, res=(96, 72)):
    mesh = synth.kuhn_cube(n, seed=8, scalars="const")
    for limit in (2.5, 0.9):
        img = render_raw(lib, mesh, res[0], res[1], X=0.35, Y=0.8, alpha_limit=limit)
        hit = img.hit
        a_hat = min(1.5, limit)
        want = 0.75 / a_hat * (1.0 - np.exp(-a_hat * img.tau[hit] / 1.5))
        assert np.allclose(img.inten[hit], want, rtol=1e-11, atol=1e-14)


def check_scaling_properties(lib, mesh, res_x, res_y, flags):
    """Size-independent properties: tau is linear in alpha and I is linear in Q, and scaling by a
    power of two is exact in binary floating point, so both hold BIT FOR BIT."""
    with api.Context(devices=(0,), lib=lib) as ctx:
        view = api.make_view(res_x, res_y, lib=lib, round_through_float=0, **flags)
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        base = ctx.render_raw(view)
        again = ctx.render_raw(view)
        assert np.array_equal(base.image, again.image), "render is not deterministic"
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, 4.0 * mesh.q)
        q4 = ctx.render_raw(view)
        assert np.array_equal(q4.inten, 4.0 * base.inten)
        assert np.array_equal(q4.tau, base.tau)
        ctx.upload_mesh(mesh.points, mesh.tets, 0.5 * mesh.alpha, mesh.q)
        view_half = api.make_view(res_x, res_y, lib=lib, round_through_float=0,
                                  **dict(flags, alpha_limit=1e30))
        view_full = api.make_view(res_x, res_y, lib=lib, round_through_float=0,
                                  **dict(flags, alpha_limit=1e30))
        a_half = ctx.render_raw(view_half)
        assert np.array_equal(a_half.tau, 0.5 * base.tau)
        assert np.array_equal(a_half.steps, base.steps)
        assert int(ctx.last_row_cost(res_y).sum()) == a_half.stats["tet_steps"]
        del view_full
    return base


def check_multi_device_context(lib, devices):
    """One context over several devices: each device renders a cost-balanced row band into its rows
    of the caller's buffers, which must give the single-device image."""
    mesh = synth.kuhn_cube(8, seed=36)
    solids = reference_solids(0.0)
    views = [api.make_view(160, 120, X=0.4, Y=y, lib=lib, round_through_float=0) for y in (0.1, 0.8, 0.8)]
    with api.Context(devices=(devices[0],), lib=lib) as one:
        one.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        one.upload_solids(solids[0], True)
        one.upload_solids(solids[1], False)
        want = [one.render_raw(v) for v in views]
        one.debug_set("query_budget", 1)     # nearly every ray goes to the grazing-ray kernel
        want_budget = one.render_raw(views[0])
    assert want_budget.stats["grazing_rays"] > want[0].stats["grazing_rays"]
    with api.Context(devices=devices, lib=lib) as many:
        many.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        many.upload_solids(solids[0], True)
        many.upload_solids(solids[1], False)
        for v, w in zip(views, want):        # 1st view: equal bands; later ones: cut by the previous view's cost
            got = many.render_raw(v)
            assert np.array_equal(got.image, w.image, equal_nan=True)
            assert np.array_equal(got.steps, w.steps) and np.array_equal(got.solid, w.solid)
            assert got.stats["tet_steps"] == w.stats["tet_steps"]
            assert got.stats["n_devices"] == len(devices)
            assert int(many.last_row_cost(120).sum()) == w.stats["tet_steps"]
        pinned = np.full((120, 160, 2), -7.0)
        many.host_register(pinned)           # page-locked: on GPUs every device stores its band in place
        try:
            many.render(views[1], out=pinned)
        finally:
            many.host_unregister(pinned)
        assert np.array_equal(pinned, want[1].image, equal_nan=True)
        many.debug_set("query_budget", 1)    # must reach every device
        got = many.render_raw(views[0])
        assert np.array_equal(got.image, want_budget.image, equal_nan=True)
        assert got.stats["grazing_rays"] == want_budget.stats["grazing_rays"]


def check_fp32_variant(lib, port, mesh, res_x, res_y, flags):
    """precision = 32: geometry in single precision, entry search and accumulators in double.
    Gate: <= 1e-4 relative per pixel and the SAME hit/miss set as the reference."""
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        v32 = api.make_view(res_x, res_y, lib=lib, round_through_float=0, precision=32, **flags)
        v64 = api.make_view(res_x, res_y, lib=lib, round_through_float=0, precision=64, **flags)
        got = ctx.render_raw(v32)
        ref64 = ctx.render_raw(v64)
    want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=res_x, res_y=res_y, **flags)
    assert_same_hits(got.steps, want.steps, what="fp32: ")
    assert_image_parity(got.tau, got.inten, want.tau, want.inten, rel=REL_TOL_FP32, floor=ABS_FLOOR_FP32, what="fp32: ")
    # the two precisions walk (almost always) the same tets
    assert abs(int(got.stats["tet_steps"]) - int(ref64.stats["tet_steps"])) <= 1e-3 * ref64.stats["tet_steps"]
    assert not np.array_equal(got.image, ref64.image)      # it really is a different arithmetic
    return got


def check_solid_mask_high_resolution(lib, port, res=(1200, 900), views=((0.4, 0.3, 0.0), (0.5, 1.3, 0.1))):
    """The NaN mask of the reference's 652 802 solid tets at full resolution, bit for bit (the scanline
    arithmetic is restated with Markstein-exact division, so this is the test that would catch it)."""
    mesh = synth.kuhn_cube(3, seed=37)
    for X, Y, D in views:
        solids = reference_solids(D)
        got = render_raw(lib, mesh, res[0], res[1], solids=solids, X=X, Y=Y)
        want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=res[0], res_y=res[1], X=X, Y=Y,
                           solid_rot=solids[0], solid_static=solids[1])
        assert want.solid.sum() > 1000
        assert np.array_equal(got.solid, want.solid)
        assert np.array_equal(np.isnan(got.tau), want.solid.astype(bool))


def check_static_solid_mask_cache(lib, port, res=(400, 300)):
    """Solids that do not follow the view are scan-converted once per pixel grid (launch_solid_mask);
    the cached footprint must give the masks the uncached path gives — across views, row bands cut
    at odd rows, a change of resolution, a change of window and a second upload of static solids —
    and those must be the oracle's."""
    mesh = synth.kuhn_cube(3, seed=11)
    roche, sphere = reference_solids(0.1)
    extra = sphere[: len(sphere) // 7].copy()
    extra[:, :, 0] += 0.35            # a second static solid, shifted so that its footprint is new
    extra[:, :, 1] += 0.2

    def masks(ctx, views):
        out = []
        for kw in views:
            v = api.make_view(lib=lib, round_through_float=0, **kw)
            out.append(ctx.render_raw(v).solid.copy())
        return out

    views = [dict(res_x=res[0], res_y=res[1], X=0.4, Y=0.3),
             dict(res_x=res[0], res_y=res[1], X=0.5, Y=1.3),
             dict(res_x=res[0], res_y=res[1], X=0.5, Y=1.3, row_begin=res[1] // 2 - 13, row_end=res[1] // 2 + 29),
             dict(res_x=res[0] + 8, res_y=res[1] - 6, X=0.1, Y=0.2),
             dict(res_x=res[0], res_y=res[1], X=0.4, Y=0.3, window=(2.0, -0.1, 0.8, -0.85)),
             dict(res_x=res[0], res_y=res[1], X=0.4, Y=0.3)]
    got = {}
    for cached in (True, False):
        with api.Context(devices=(0,), lib=lib) as ctx:
            if not cached:
                ctx.debug_set("no_static_mask", 1)
            ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
            ctx.upload_solids(roche, True)
            ctx.upload_solids(sphere, False)
            first = masks(ctx, views)
            ctx.upload_solids(extra, False)                      # must invalidate the cached footprint
            second = masks(ctx, views[:2])
            ctx.clear_solids()
            ctx.upload_solids(roche, True)
            third = masks(ctx, views[:1])                        # no static solid left: nothing of it may remain
            got[cached] = first + second + third
    for a, b in zip(got[True], got[False]):
        assert np.array_equal(a, b)
    assert got[True][6].sum() > got[True][0].sum() > got[True][8].sum() > 0
    for k in (0, 1):
        kw = views[k]
        want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=kw["res_x"], res_y=kw["res_y"], X=kw["X"], Y=kw["Y"],
                           solid_rot=roche, solid_static=sphere)
        assert np.array_equal(got[True][k], want.solid)
    band = views[2]
    inside = got[True][2][band["row_begin"]: band["row_end"]]
    assert np.array_equal(inside, got[True][1][band["row_begin"]: band["row_end"]])


def check_solid_mask_tile_sizes(lib, port, res=(320, 240), tiles=(801, 804, 1608, 3216, 6499)):
    """The mask must not depend on the size of the "tile already solid" flags (c5_debug_set "mask_tile" =
    100 w + h): one-row tiles make every row of a tall face an item of its own (hundreds of items per
    warp, the 64-entry list of rows still to be drawn overflows and is drained in the middle of a batch),
    huge tiles are never full, so every tall face is drawn in full."""
    mesh = synth.kuhn_cube(3, seed=12)
    solids = reference_solids(0.1)
    kw = dict(X=0.45, Y=0.8)
    want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=res[0], res_y=res[1],
                       solid_rot=solids[0], solid_static=solids[1], **kw)
    assert want.solid.sum() > 500
    for tile in tiles:
        for cached in (0, 1):
            got = render_raw(lib, mesh, res[0], res[1], solids=solids, debug={"mask_tile": tile, "no_static_mask": 1 - cached}, **kw)
            assert np.array_equal(got.solid, want.solid), f"mask_tile={tile}, static footprint cached={cached}"


def check_grazing_rays(lib, port, *, n=12, res=(240, 180), debug_key="serial_list", debug_value=5):
    """Views that look along a lattice axis see the jittered side walls edge-on: rays there leave
    and re-enter the mesh once per cell. The pixel kernel hands them to the grazing-ray kernel
    (c5_stats.grazing_rays); the result must still match the oracle, and must not depend on how many
    entry faces one collection can hold (the overflow path keeps the lowest part and asks again)."""
    mesh = synth.kuhn_cube(n, seed=48)
    for flags in (dict(X=0.5, Y=0.0), dict(X=0.0, Y=0.5)):
        img, _ = check_against_port(lib, port, mesh, res[0], res[1], flags)
        assert img.stats["grazing_rays"] > 0
        small = render_raw(lib, mesh, res[0], res[1], debug={debug_key: debug_value}, **flags)
        assert small.stats["grazing_rays"] == img.stats["grazing_rays"]
        assert np.array_equal(small.image, img.image)
        assert np.array_equal(small.steps, img.steps)


def check_sibling_context(lib, stream_of=None):
    """c5_create_sibling: same images as the parent, follows the parent's uploads, refuses its own."""
    solids_a = synth.kuhn_cube(2, seed=3, side=0.2, centre=(1.0, 0.1, 0.0)).tet_points()
    mesh = synth.kuhn_cube(7, seed=52)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(solids_a, True)
        sib = ctx.sibling()
        try:
            assert sib.mesh_info().n_tets in (0, mesh.n_tets)        # filled in at the first render
            for flags in (dict(X=0.4, Y=0.2), dict(X=0.5, Y=0.0, alpha_limit=1.1)):
                v = api.make_view(120, 90, lib=lib, **flags)
                a, sa = ctx.render(v)
                b, sb = sib.render(v)
                assert np.array_equal(a, b, equal_nan=True) and sa["tet_steps"] == sb["tet_steps"]
                assert sa["solid_pixels"] == sb["solid_pixels"] > 0
            assert sib.mesh_info().n_tets == mesh.n_tets
            with pytest.raises(api.C5Error):
                sib.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
            with pytest.raises(api.C5Error):
                sib.clear_solids()
            # a new mesh through the parent reaches the sibling at its next render
            mesh2 = synth.kuhn_cube(5, seed=53)
            ctx.upload_mesh(mesh2.points, mesh2.tets, mesh2.alpha, mesh2.q)
            ctx.clear_solids()
            v = api.make_view(120, 90, X=0.3, Y=0.6, lib=lib)
            a, sa = ctx.render(v)
            b, sb = sib.render(v)
            assert np.array_equal(a, b) and sb["solid_pixels"] == 0 and sb["tet_steps"] == sa["tet_steps"] > 0
        finally:
            sib.close()


def check_search_budget(lib, port, *, n=10, res=(200, 150)):
    """A BVH search that exceeds its node budget hands the ray to the grazing-ray kernel (also before
    its first step). With a budget of a few nodes nearly every ray goes that way; the image must
    still match the oracle, hit counts and step counts included."""
    mesh = synth.kuhn_cube(n, seed=55, scalars="sphere", carve_sphere=True)   # a cavity: rays re-enter
    flags = dict(X=0.3, Y=0.4)
    base = render_raw(lib, mesh, res[0], res[1], **flags)
    for budget in (3, 12):
        img, want = check_against_port(lib, port, mesh, res[0], res[1], flags, debug={"query_budget": budget})
        assert img.stats["grazing_rays"] > base.stats["grazing_rays"]
        assert img.stats["hit_pixels"] == base.stats["hit_pixels"] == int(want.hit.sum())


def check_submit_wait(lib, pinned=None):
    """c5_render_submit / c5_render_wait: several views in flight on lanes that share the mesh give the
    images one-at-a-time c5_render gives, tickets can be waited for in any order, one submit too many
    is C5_E_STATE, and stats / row costs belong to the ticket waited for. `pinned(shape)` makes a
    page-locked array on a GPU box (the walk then stores in place); pageable arrays otherwise."""
    alloc = pinned or (lambda shape: np.zeros(shape))
    mesh = synth.kuhn_cube(9, seed=64)
    solid = synth.kuhn_cube(2, seed=3, side=0.2, centre=(1.0, 0.1, 0.0)).tet_points()
    views_flags = [dict(X=0.5, Y=0.0), dict(X=0.4, Y=0.3), dict(X=0.0, Y=0.5, alpha_limit=1.1), dict(X=0.45, Y=1.2),
                   dict(X=0.3, Y=1.7)]
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.upload_solids(solid, True)
        views = [api.make_view(160, 120, lib=lib, **f) for f in views_flags]
        want = [ctx.render(v) for v in views]
        ctx.set_views_in_flight(3)
        outs = [alloc((120, 160, 2)) for _ in views]
        for o in outs:
            o[:] = -7.0
        t = [ctx.render_submit(views[k], outs[k]) for k in range(3)]
        with pytest.raises(api.C5Error) as e:
            ctx.render_submit(views[3], outs[3])                       # three lanes, three views in flight
        assert e.value.code == api.E_STATE
        with pytest.raises(api.C5Error) as e:
            ctx.render_device(views[0], 16, 0)                         # lane 0 is busy
        assert e.value.code == api.E_STATE
        st1 = ctx.render_wait(t[1])                                    # any order
        assert st1["tet_steps"] == want[1][1]["tet_steps"] and st1["solid_pixels"] == want[1][1]["solid_pixels"]
        assert int(ctx.last_row_cost(120).sum()) == st1["tet_steps"]
        t.append(ctx.render_submit(views[3], outs[3]))                 # the freed lane
        st0 = ctx.render_wait(t[0])
        t.append(ctx.render_submit(views[4], outs[4]))
        stats = {0: st0, 1: st1}
        for k in (2, 3, 4):
            stats[k] = ctx.render_wait(t[k])
        with pytest.raises(api.C5Error):
            ctx.render_wait(t[2])                                      # once each
        for k in range(5):
            assert np.array_equal(outs[k], want[k][0], equal_nan=True), f"view {k}"
            assert stats[k]["tet_steps"] == want[k][1]["tet_steps"]
        assert len({*t}) == 5 and all(x > 0 for x in t)
        assert ctx.kernel_launches() > 0
        # a sweep: two views ahead, bands too
        ctx.set_views_in_flight(2)
        band = [api.make_view(160, 120, lib=lib, row_begin=30, row_end=90, **f) for f in views_flags]
        out = [alloc((120, 160, 2)) for _ in range(2)]
        tick = [ctx.render_submit(band[0], out[0])]
        for k in range(1, 5):
            tick.append(ctx.render_submit(band[k], out[k % 2]))
            ctx.render_wait(tick[k - 1])
            assert np.array_equal(out[(k - 1) % 2][30:90], want[k - 1][0][30:90], equal_nan=True)
        ctx.render_wait(tick[4])
        assert np.array_equal(out[0][30:90], want[4][0][30:90], equal_nan=True)
        with pytest.raises(api.C5Error):
            ctx.set_views_in_flight(api.MAX_IN_FLIGHT + 1)
        # a sibling has no lanes of its own
        sib = ctx.sibling()
        try:
            with pytest.raises(api.C5Error) as e:
                sib.render_submit(views[0], outs[0])
            assert e.value.code == api.E_INVALID
        finally:
            sib.close()


def check_output_alignment(lib, device_buffer=None):
    """Pixels are stored as one 128-bit word: a device buffer that is not 16-byte aligned is refused
    (C5_E_INVALID, not a misaligned-address fault), a host buffer that is not takes the copy path."""
    mesh = synth.kuhn_cube(5, seed=65)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        v = api.make_view(64, 48, X=0.4, Y=0.2, lib=lib)
        want, _ = ctx.render(v)
        backing = np.zeros(64 * 48 * 2 + 1)
        odd = backing[1:] if backing.ctypes.data % 16 == 0 else backing[:-1]     # 8-byte aligned only
        assert odd.ctypes.data % 16 == 8
        got, _ = ctx.render(v, out=odd.reshape(48, 64, 2))
        assert np.array_equal(got, want)
        if device_buffer is not None:
            ptr = device_buffer(64 * 48 * 16 + 16)
            with pytest.raises(api.C5Error) as e:
                ctx.render_device(v, ptr + 8, 0)
            assert e.value.code == api.E_INVALID
            ctx.render_device(v, ptr, 0)


# ---- the UNMODIFIED reference at the benchmarked sizes -------------------------------------------

def reference_process(name, overrides, out_path, timeout=1500):
    """oracle/_ref (where it was built, else the C restatement: tests/ref_runner.py) on configuration
    `name` (one view per dict of flag overrides) in a process of its own (the reference reports a
    degenerate ray by std::terminate). Returns the saved arrays."""
    import json
    import os
    import subprocess
    import sys
    runner = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_runner.py")
    p = subprocess.run([sys.executable, runner, name, str(out_path), json.dumps(overrides)],
                       capture_output=True, text=True, timeout=timeout)
    assert p.returncode == 0, f"the reference did not finish on {name} {overrides}: rc {p.returncode}\n{p.stderr[-2000:]}"
    return np.load(str(out_path))


def assert_matches_reference(img, r, k, what=""):
    """The whole parity gate against view k of a reference_process() result: solid masks and hit sets
    identical, per-pixel tets crossed identical, tau and I within 1e-9 relative (+1e-13) of the
    reference's pre-cast doubles."""
    assert np.array_equal(img.solid, r[f"solid{k}"]), f"{what}solid (NaN) masks differ"
    assert_same_hits(img.steps, r[f"steps{k}"], what=what)
    assert np.array_equal(img.steps, r[f"steps{k}"]), f"{what}per-pixel tets crossed differ"
    assert img.stats["tet_steps"] == int(r[f"total_steps{k}"])
    assert img.stats["walk_errors"] == 0
    assert_image_parity(img.tau, img.inten, r[f"tau{k}"], r[f"inten{k}"], what=what)
