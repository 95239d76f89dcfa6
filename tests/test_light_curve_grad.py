"""c5_render_flux_grad_device: the gradient of a light curve in one device call, the views on the lanes.

Held to the exact gradients (tests/exact_grad.py, the gate of DESIGN.md §5c) with each view's upstream pair
spread over its band's pixels, and to the sum over views of c5_render_grad_device against g filled with that
view's pair. On the host-loop build numpy arrays stand in for device memory (as in test_gradients_device.py);
on the GPU they are torch CUDA tensors.
"""
import ctypes as C

import numpy as np
import pytest

import exact_grad
import test_gradients as tg
from course5_b200 import api, synth
from test_gradients_device import CASES, Mem, band_of, grad_device

RES = tg.RES


@pytest.fixture(params=tg.LIBS)
def env(request):
    return request.getfixturevalue(request.param), Mem(request.param == "gpu_lib")


@pytest.fixture(scope="module")
def oracle_port(port):
    return port


def flux_grad(ctx, mem, views, g, *, alpha=True, q=True, stats=True):
    """c5_render_flux_grad_device of g, (n_views, 2) {g_tau, g_I}."""
    d_g = mem.put(np.asarray(g).reshape(-1, 2))
    ga = mem.empty(ctx.n_tets) if alpha else None
    gq = mem.empty(ctx.n_tets) if q else None
    st = ctx.render_flux_grad_device(views, mem.ptr(d_g), mem.ptr(ga), mem.ptr(gq), stats=stats)
    return mem.get(ga), mem.get(gq), st


def per_view(ctx, mem, views, g):
    """Sum over the views of c5_render_grad_device against the view's band filled with its pair."""
    sums = [np.zeros(ctx.n_tets), np.zeros(ctx.n_tets)]
    for v, gk in zip(views, g):
        full = np.zeros((v.res_y, v.res_x, 2))
        rb, re = band_of(v)
        full[rb:re] = gk
        ga, gq, _, _ = grad_device(ctx, mem, v, full)
        sums[0] += ga
        sums[1] += gq
    return sums


def close(got, want, rel):
    for a, b in zip(got, want):
        scale = np.abs(b).max()
        assert scale > 0
        assert np.allclose(a, b, rtol=0.0, atol=rel * scale), float(np.abs(a - b).max() / scale)


def with_rows(view, rows):
    v = api.View.from_buffer_copy(view)
    v.row_begin, v.row_end = rows
    return v


# ---- against the exact gradients --------------------------------------------------------------------------

BAND = (20, 50)


@pytest.mark.parametrize("case", list(CASES))
def test_exact(env, oracle_port, record_property, case):
    """Two views (the whole image and a row band of it) on two lanes; the exact gradient is the per-pixel one
    with g_0 in every pixel plus g_1 in the band's, 0 under the solid mask."""
    lib, mem = env
    c = dict(CASES[case])
    debug = c.pop("debug", None)
    with_solids = c.get("with_solids", False)
    mesh = tg.mesh_of(*c["mesh_key"])
    alpha, q = tg.FIELDS[c["field"]](mesh)
    g = np.random.default_rng(31).normal(size=(2, 2))
    (start, tet, dz), solid = tg.segments_of(oracle_port, c["mesh_key"], c["view"], with_solids)
    g_pix = np.zeros((RES[1], RES[0], 2))
    g_pix[:] = g[0]
    g_pix[BAND[0]:BAND[1]] += g[1]
    g_pix[solid] = 0.0
    exact = exact_grad.vjp(start, tet, dz, alpha, q, tg.NO_LIMIT, g_pix.reshape(-1, 2), mesh.n_tets)
    with api.Context(devices=(0,), lib=lib) as ctx:
        for k, v in (debug or {}).items():
            ctx.debug_set(k, v)
        ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
        if with_solids:
            ctx.upload_solids(tg.solids()[0], True)
            ctx.upload_solids(tg.solids()[1], False)
        ctx.set_views_in_flight(2)
        view = api.make_view(RES[0], RES[1], lib=lib, alpha_limit=tg.NO_LIMIT, round_through_float=0,
                             **tg.VIEWS[c["view"]])
        ga, gq, st = flux_grad(ctx, mem, [view, with_rows(view, BAND)], g)
    assert st["walk_errors"] == 0
    assert st["pixels"] == RES[0] * RES[1] + RES[0] * (BAND[1] - BAND[0])
    if debug and "query_budget" in debug:
        assert st["grazing_rays"] > st["hit_pixels"] // 2
    tg.check_grads(record_property, f"light curve {case}", (ga, gq), exact)


# ---- against the per-view device gradient ------------------------------------------------------------------

def _mixed_views(lib, ctx):
    """Two resolutions, solids on and off, row bands, and a band the mesh does not reach."""
    generic = api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, **tg.VIEWS["generic"])
    steps = ctx.render_raw(generic).steps
    empty = np.flatnonzero(steps.sum(axis=1) == 0)
    assert empty.size and empty[0] == 0
    views = [generic,
             api.make_view(64, 48, lib=lib, round_through_float=0, use_solids=0, **tg.VIEWS["axis"]),
             with_rows(api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, **tg.VIEWS["axis"]), (10, 40)),
             with_rows(generic, (0, int(empty[0]) + 1)),
             api.make_view(48, 40, lib=lib, round_through_float=0, X=0.2, Y=1.3, I=0.1),
             with_rows(api.make_view(64, 48, lib=lib, round_through_float=0, use_solids=0, X=0.7, Y=0.4), (30, 48))]
    g = np.random.default_rng(5).normal(size=(len(views), 2))
    return views, g


def test_per_view_path_and_lanes(env):
    """Mixed views on 1 - 4 lanes equal the per-view sum to 1e-12 of the largest gradient; the counts are the
    views' render_raw counts summed."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    with ctx:
        views, g = _mixed_views(lib, ctx)
        want = per_view(ctx, mem, views, g)
        raws = [ctx.render_raw(v).stats for v in views]
        for lanes in (1, 2, 3, 4):
            ctx.set_views_in_flight(lanes)
            ga, gq, st = flux_grad(ctx, mem, views, g)
            close((ga, gq), want, 1e-12)
            for key in ("pixels", "tet_steps", "hit_pixels", "solid_pixels", "grazing_rays", "walk_errors"):
                assert st[key] == sum(r[key] for r in raws), key
            assert st["ms_rotate"] == st["ms_walk"] == st["ms_d2h"] == 0.0


def test_one_view_one_lane_is_the_device_gradient(hostsim_lib):
    """On the host-loop build (one thread adds in a fixed order) one view on one lane is c5_render_grad_device
    with g filled with the view's pair, bit for bit: the per-view policy is the per-pixel one."""
    mem = Mem(False)
    ctx, mesh, view = tg.small_ctx(hostsim_lib, n=7)
    with ctx:
        ctx.set_views_in_flight(1)
        for v, gk in ((view, (0.7, -1.3)), (with_rows(api.make_view(RES[0], RES[1], lib=hostsim_lib, round_through_float=0,
                                                                    **tg.VIEWS["axis"]), BAND), (0.0, 2.0))):
            ga, gq, st = flux_grad(ctx, mem, [v], [gk])
            want = per_view(ctx, mem, [v], [gk])
            assert np.array_equal(ga, want[0]) and np.array_equal(gq, want[1])
            assert np.abs(gq).max() > 0


# ---- invariance ---------------------------------------------------------------------------------------------

def test_permutation_lanes_and_null_outputs(env):
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    with ctx:
        views, g = _mixed_views(lib, ctx)
        ctx.set_views_in_flight(3)
        ref = flux_grad(ctx, mem, views, g)[:2]
        perm = np.random.default_rng(2).permutation(len(views))
        for lanes in (1, 4):
            ctx.set_views_in_flight(lanes)
            close(flux_grad(ctx, mem, [views[k] for k in perm], g[perm])[:2], ref, 1e-13)
        ctx.set_views_in_flight(3)
        ga, _, _ = flux_grad(ctx, mem, views, g, q=False)
        _, gq, _ = flux_grad(ctx, mem, views, g, alpha=False)
        if mem.gpu:
            close((ga, gq), ref, 1e-13)
        else:
            assert np.array_equal(ga, ref[0]) and np.array_equal(gq, ref[1])


# ---- launches -----------------------------------------------------------------------------------------------

def test_launch_count(env):
    """Sum over the views of c5_render_grad_device's launches, less n_views - 1: one scatter per call."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    with ctx:
        views, g = _mixed_views(lib, ctx)
        ctx.set_views_in_flight(3)
        flux_grad(ctx, mem, views, g)  # lanes made, cells prepared, permutation resident
        per = 0
        for v, gk in zip(views, g):
            n0 = ctx.kernel_launches()
            per_view(ctx, mem, [v], [gk])
            per += ctx.kernel_launches() - n0
        n0 = ctx.kernel_launches()
        flux_grad(ctx, mem, views, g, stats=False)
        assert ctx.kernel_launches() - n0 == per - (len(views) - 1)


# ---- errors -------------------------------------------------------------------------------------------------

def test_errors(env):
    lib, mem = env
    vp = C.c_void_p
    ctx, mesh, view = tg.small_ctx(lib)
    n = mesh.n_tets
    ga, gq = mem.empty(n), mem.empty(n)
    g = mem.put(np.ones((2, 2)))
    pg, pa, pq = mem.ptr(g), mem.ptr(ga), mem.ptr(gq)

    def call(c, views=(view, view), n_views=None, gg=pg, a=pa, q=pq):
        arr = (api.View * max(len(views), 1))(*views) if views is not None else None
        return lib.c5_render_flux_grad_device(c._h, arr, len(views or ()) if n_views is None else n_views,
                                              vp(gg or None), vp(a or None), vp(q or None), None, None)

    with api.Context(devices=(0,), lib=lib) as empty:
        assert call(empty) == api.E_STATE
    with ctx:
        assert call(ctx) == api.OK
        bad = []
        for kw in (dict(n_views=0), dict(views=None, n_views=1), dict(gg=0), dict(a=0, q=0), dict(gg=pg + 4),
                   dict(a=pa + 4), dict(q=pq + 4)):
            bad.append((kw, call(ctx, **kw)))
        for key, val in (("precision", 32), ("round_through_float", 1)):
            v = api.View.from_buffer_copy(view)
            setattr(v, key, val)
            bad.append((key, call(ctx, views=(view, v))))
        for what, rc in bad:
            assert rc == api.E_INVALID, what
            assert call(ctx) == api.OK  # usable after each error
        assert call(ctx, a=0) == api.OK and call(ctx, q=0) == api.OK
        sib = ctx.sibling()
        try:
            assert call(sib) == api.E_STATE
        finally:
            sib.close()
        ctx.set_views_in_flight(2)
        for lane in range(2):  # a view in flight on the context itself, then on its lane
            tickets = [ctx.render_submit(view, np.zeros((RES[1], RES[0], 2))) for _ in range(lane + 1)]
            if lane:
                ctx.render_wait(tickets.pop(0))
            try:
                assert call(ctx) == api.E_STATE
            finally:
                for t in tickets:
                    ctx.render_wait(t)
        assert call(ctx) == api.OK
    with api.Context(devices=(0, 0), lib=lib) as two:
        two.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        assert call(two) == api.E_INVALID
    mem.get(ga)


# ---- ordering without host synchronisation (GPU) ----------------------------------------------------------------

@pytest.mark.gpu
def test_lanes_made_after_a_field_update(gpu_lib):
    """A field update on a torch side stream, held back by a long kernel, then views submitted on lanes that did
    not exist yet: every image is a fresh upload's, bit for bit."""
    import torch
    mesh = tg.mesh_of(8)
    alpha2, q2 = tg.FIELDS["mixed"](mesh)
    views = [api.make_view(RES[0], RES[1], lib=gpu_lib, round_through_float=0, X=0.4, Y=0.1 * k, I=-0.03)
             for k in range(8)]
    fresh = api.Context(devices=(0,), lib=gpu_lib)
    ctx = api.Context(devices=(0,), lib=gpu_lib)
    with fresh, ctx:
        for c, (a, q) in ((fresh, (alpha2, q2)), (ctx, (mesh.alpha, mesh.q))):
            c.upload_mesh(mesh.points, mesh.tets, a, q)
            c.upload_solids(tg.solids()[0], True)
        want = [fresh.render_raw(v).image for v in views]
        ctx.set_views_in_flight(1)
        ctx.render_raw(views[0])
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            a = torch.tensor(alpha2, device="cuda")
            b = torch.tensor(q2, device="cuda")
            torch.cuda._sleep(200_000_000)  # ~0.1 s of device time before the gather
            ctx.update_fields_device(a.data_ptr(), b.data_ptr(), side.cuda_stream)
        ctx.set_views_in_flight(4)
        images = [np.zeros((RES[1], RES[0], 2)) for _ in views]
        tickets = [ctx.render_submit(v, img) for v, img in zip(views[:4], images[:4])]
        for t in tickets:
            ctx.render_wait(t)
        for v, img in zip(views[4:], images[4:]):
            ctx.render_wait(ctx.render_submit(v, img))
        for got, ref in zip(images, want):
            assert np.array_equal(got, ref, equal_nan=True)


@pytest.mark.gpu
def test_no_stats_then_torch_on_the_same_stream(gpu_lib):
    """The call without stats on a side stream (after a long kernel and the write of g there), then a torch
    reduction on that stream, equals the synchronised result."""
    import torch
    mem = Mem(True)
    ctx, mesh, _ = tg.small_ctx(gpu_lib, n=8)
    with ctx:
        views, g = _mixed_views(gpu_lib, ctx)
        ctx.set_views_in_flight(4)
        want = flux_grad(ctx, mem, views, g)[:2]
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            ga = torch.empty(mesh.n_tets, dtype=torch.float64, device="cuda")
            gq = torch.empty_like(ga)
            torch.cuda._sleep(200_000_000)
            d_g = torch.tensor(g, device="cuda") * 1.0  # written on the side stream after the long kernel
            ctx.render_flux_grad_device(views, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=side.cuda_stream,
                                        stats=False)
            sums = torch.stack([ga.abs().sum(), gq.abs().sum(), (ga - torch.tensor(want[0], device="cuda")).abs().max(),
                                (gq - torch.tensor(want[1], device="cuda")).abs().max()]).cpu().numpy()
        for k in range(2):
            scale = np.abs(want[k]).max()
            assert abs(sums[k] - np.abs(want[k]).sum()) <= 1e-12 * np.abs(want[k]).sum()
            assert sums[2 + k] <= 1e-12 * scale


# ---- autograd (GPU) -------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [2, 4])
def test_light_curve_gradcheck_on_lanes(gpu_lib, lanes):
    import torch
    from course5_b200 import autograd
    mesh = synth.kuhn_cube(3, seed=7)
    with api.Context(devices=(0,), lib=gpu_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        ctx.set_views_in_flight(lanes)
        views = [api.make_view(24, 18, lib=gpu_lib, alpha_limit=tg.NO_LIMIT, use_solids=0, X=0.4, Y=0.25 * k, I=-0.03)
                 for k in range(5)]
        alpha = torch.tensor(mesh.alpha, device="cuda", requires_grad=True)
        q = torch.tensor(mesh.q, device="cuda", requires_grad=True)
        assert torch.autograd.gradcheck(lambda a, b: autograd.light_curve(ctx, views, a, b), (alpha, q),
                                        eps=1e-6, atol=1e-6, rtol=1e-5, nondet_tol=1e-12)
