"""c5_render_flux_device and c5_render_flux_jvp_device: a light curve and its J v in one device call, the views on
the lanes.

The totals are held to c5_render_flux bit for bit. The curve's J v is held, bit for bit, to each view's
c5_render_jvp tangent image summed in the documented flux order (tests/test_flux.py: contract_rows, then
sequential_total) outside render_raw's solid mask, which ties it to the exact per-pixel tangents of
tests/test_jvp.py. The adjoint identity ties it to c5_render_flux_grad_device. On the host-loop build numpy arrays
stand in for device memory (as in test_gradients_device.py); on the GPU they are torch CUDA tensors.
"""
import ctypes as C

import numpy as np
import pytest

import test_gradients as tg
from course5_b200 import api, synth
from test_flux import PORT_VIEWS, contract_rows, fields, sequential_total
from test_gradients import c3  # noqa: F401  (C3 at 2400 x 1800 with the reference's solids)
from test_gradients_device import Mem
from test_jvp import direction
from test_light_curve_grad import _mixed_views, flux_grad, with_rows

RES = tg.RES
COUNTS = ("pixels", "tet_steps", "hit_pixels", "solid_pixels", "grazing_rays", "walk_errors")


@pytest.fixture(params=tg.LIBS)
def env(request):
    return request.getfixturevalue(request.param), Mem(request.param == "gpu_lib")


def flux_device(ctx, mem, views, *, channels=False, stats=True):
    """c5_render_flux_device: ((n_views, n, 2) totals, stats)."""
    n = ctx.n_channels if channels else 1
    total = mem.empty((len(views), n, 2))
    st = ctx.render_flux_device(views, mem.ptr(total), channels=channels, stats=stats)
    return mem.get(total), st


def jvp_device(ctx, mem, views, va, vq, *, total=True, stats=True):
    """c5_render_flux_jvp_device: ((n_views, 2) tangent, (n_views, 2) totals or None, stats)."""
    d_va = None if va is None else mem.put(va)
    d_vq = None if vq is None else mem.put(vq)
    t = mem.empty((len(views), 2))
    tot = mem.empty((len(views), 2)) if total else None
    st = ctx.render_flux_jvp_device(views, mem.ptr(d_va), mem.ptr(d_vq), mem.ptr(t), mem.ptr(tot), stats=stats)
    return mem.get(t), mem.get(tot), st


def curve_tangent(ctx, view, va, vq):
    """The view's render_jvp tangent summed outside render_raw's solid mask, in the documented flux order."""
    tangent = ctx.render_jvp(view, va, vq)
    solid = ctx.render_raw(view).solid
    return sequential_total(contract_rows(tangent[:, :, None, :], solid))[0]


def flux_totals(ctx, views):
    return np.stack([ctx.render_flux(v)[1][0] for v in views])


# ---- the totals --------------------------------------------------------------------------------------------

def test_flux_totals(env):
    """Mixed resolutions, row bands, solids on and off, an empty band, the PORT_VIEWS of test_flux with the float
    cast and an FP32 view; the cells' own fields and the uploaded channels; 1 - 4 lanes and a permuted order: every
    total is render_flux's, bit for bit, and the counts are its counts summed."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    with ctx:
        ctx.upload_channels(*fields(mesh, 3, seed=17))
        base, _ = _mixed_views(lib, ctx)
        base += [api.make_view(RES[0], RES[1], lib=lib, round_through_float=1, **f) for f in PORT_VIEWS]
        fp32 = api.make_view(80, 60, lib=lib, precision=32, **tg.VIEWS["generic"])
        for channels in (False, True):
            views = base + ([] if channels else [fp32])
            want = [ctx.render_flux(v, channels=channels) for v in views]
            perm = np.random.default_rng(3).permutation(len(views))
            for lanes in (1, 2, 3, 4):
                ctx.set_views_in_flight(lanes)
                got, st = flux_device(ctx, mem, views, channels=channels)
                assert got.shape == (len(views), 3 if channels else 1, 2)
                for k, (_, total, _) in enumerate(want):
                    assert np.array_equal(got[k], total), (channels, lanes, k)
                for key in COUNTS:
                    assert st[key] == sum(w[2][key] for w in want), key
                assert st["ms_rotate"] == st["ms_walk"] == st["ms_d2h"] == 0.0
                shuffled, _ = flux_device(ctx, mem, [views[k] for k in perm], channels=channels, stats=False)
                assert np.array_equal(shuffled, got[perm])


# ---- the J v of a curve ------------------------------------------------------------------------------------

@pytest.mark.parametrize("dirs", ["alpha", "q", "both"])
def test_jvp_contract(env, dirs):
    """The tangent is each view's tangent image summed in the flux order, bit for bit, and the totals are
    render_flux's; 1 - 4 lanes, a permuted order and no totals give the same bits."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    va, vq = direction(mesh.alpha, mesh.q)
    va, vq = {"alpha": (va, None), "q": (None, vq), "both": (va, vq)}[dirs]
    with ctx:
        views, _ = _mixed_views(lib, ctx)
        totals = flux_totals(ctx, views)
        raws = [ctx.render_raw(v).stats for v in views]
        want = np.stack([curve_tangent(ctx, v, va, vq) for v in views])
        assert np.abs(want).max() > 0
        for lanes in (1, 2, 3, 4):
            ctx.set_views_in_flight(lanes)
            t, tot, st = jvp_device(ctx, mem, views, va, vq)
            assert np.array_equal(t, want), lanes
            assert np.array_equal(tot, totals), lanes
            for key in COUNTS:
                assert st[key] == sum(r[key] for r in raws), key
        perm = np.random.default_rng(4).permutation(len(views))
        t, tot, _ = jvp_device(ctx, mem, [views[k] for k in perm], va, vq, total=False, stats=False)
        assert tot is None and np.array_equal(t, want[perm])


def test_special_direction(env):
    """v_alpha = alpha, v_Q = 0: the tau tangent is the tau total, bit for bit (dtau == tau in every pixel)."""
    lib, mem = env
    mesh = tg.mesh_of(8)
    alpha, q = tg.FIELDS["decade_1"](mesh)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
        ctx.upload_solids(tg.solids()[0], True)
        ctx.upload_solids(tg.solids()[1], False)
        views, _ = _mixed_views(lib, ctx)
        ctx.set_views_in_flight(3)
        t, tot, _ = jvp_device(ctx, mem, views, alpha, None)
    assert np.array_equal(t[:, 0], tot[:, 0])
    assert np.abs(tot[:, 0]).max() > 0 and np.abs(t[:, 1]).max() > 0


def test_adjoint_identity(env):
    """<g, J v> = <c5_render_flux_grad_device(g), v>, and J^T J v from the tangent passed straight in as g
    satisfies <v, J^T J v> = |J v|^2, both to 1e-12 of the sum of absolute terms."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    va, vq = direction(mesh.alpha, mesh.q, seed=9)
    with ctx:
        views, g = _mixed_views(lib, ctx)
        ctx.set_views_in_flight(3)
        t, _, _ = jvp_device(ctx, mem, views, va, vq, total=False)
        ga, gq, _ = flux_grad(ctx, mem, views, g)
        lhs_terms, rhs_terms = g * t, np.concatenate([ga * va, gq * vq])
        size = np.abs(lhs_terms).sum() + np.abs(rhs_terms).sum()
        assert abs(lhs_terms.sum() - rhs_terms.sum()) <= 1e-12 * size, (lhs_terms.sum(), rhs_terms.sum())
        # J^T J v: two calls, nothing in between
        d_va, d_vq = mem.put(va), mem.put(vq)
        d_t = mem.empty((len(views), 2))
        jtj = mem.empty(mesh.n_tets), mem.empty(mesh.n_tets)
        ctx.render_flux_jvp_device(views, mem.ptr(d_va), mem.ptr(d_vq), mem.ptr(d_t), stats=False)
        ctx.render_flux_grad_device(views, mem.ptr(d_t), mem.ptr(jtj[0]), mem.ptr(jtj[1]), stats=False)
        jv, ja, jq = mem.get(d_t), mem.get(jtj[0]), mem.get(jtj[1])
    assert np.array_equal(jv, t)
    lhs_terms, rhs_terms = np.concatenate([va * ja, vq * jq]), jv * jv
    size = np.abs(lhs_terms).sum() + rhs_terms.sum()
    assert abs(lhs_terms.sum() - rhs_terms.sum()) <= 1e-12 * size, (lhs_terms.sum(), rhs_terms.sum())


# ---- launches and memory ------------------------------------------------------------------------------------

def _launch_views(lib):
    """Solids only on the one grid, so that every lane's cached static-solid mask holds for all of its views."""
    v = api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, **tg.VIEWS["generic"])
    return [v, with_rows(api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, **tg.VIEWS["axis"]), (10, 40)),
            api.make_view(64, 48, lib=lib, round_through_float=0, use_solids=0, **tg.VIEWS["axis"]),
            api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, X=0.2, Y=1.3, I=0.1),
            with_rows(v, (30, 72))]


def test_launch_counts_and_device_bytes(env):
    """The flux call launches what render_flux launches for each view plus one total per view; the J v call the
    same plus one gather. The tangent field (16 bytes per tet) counts in device_bytes once, at the first J v call."""
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    va, vq = direction(mesh.alpha, mesh.q)
    with ctx:
        ctx.upload_channels(*fields(mesh, 2, seed=19))
        views = _launch_views(lib)
        ctx.set_views_in_flight(3)
        flux_grad(ctx, mem, views, np.ones((len(views), 2)))  # lanes made, cells prepared, permutation resident
        before = ctx.mesh_info().device_bytes
        for channels in (False, True):
            flux_device(ctx, mem, views, channels=channels)  # warm: tables and buffers of every lane
            per = 0
            for v in views:
                n0 = ctx.kernel_launches()
                ctx.render_flux(v, channels=channels)
                per += ctx.kernel_launches() - n0
            n0 = ctx.kernel_launches()
            flux_device(ctx, mem, views, channels=channels, stats=False)
            assert ctx.kernel_launches() - n0 == per + len(views), channels
            if not channels:
                per_plain = per
        assert ctx.mesh_info().device_bytes == before
        for k in range(2):
            jvp_device(ctx, mem, views, va, vq)
            assert ctx.mesh_info().device_bytes == before + 16 * mesh.n_tets, k
        n0 = ctx.kernel_launches()
        jvp_device(ctx, mem, views, va, None, total=False, stats=False)
        assert ctx.kernel_launches() - n0 == per_plain + len(views) + 1


# ---- errors -------------------------------------------------------------------------------------------------

def test_errors(env):
    lib, mem = env
    vp = C.c_void_p
    ctx, mesh, view = tg.small_ctx(lib)
    da, dq = mem.put(mesh.alpha), mem.put(mesh.q)
    dt, dtot = mem.empty((2, 2)), mem.empty((2, 2))
    pa, pq, pt, ptot = mem.ptr(da), mem.ptr(dq), mem.ptr(dt), mem.ptr(dtot)

    def arr(views):
        return (api.View * max(len(views), 1))(*views) if views is not None else None

    def flux(c, views=(view, view), n_views=None, total=ptot, channels=0):
        return lib.c5_render_flux_device(c._h, arr(views), len(views or ()) if n_views is None else n_views, channels,
                                         vp(total or None), None, None)

    def jvp(c, views=(view, view), n_views=None, a=pa, q=pq, t=pt, total=ptot):
        return lib.c5_render_flux_jvp_device(c._h, arr(views), len(views or ()) if n_views is None else n_views,
                                             vp(a or None), vp(q or None), vp(t or None), vp(total or None), None, None)

    with api.Context(devices=(0,), lib=lib) as empty:
        assert flux(empty) == api.E_STATE and jvp(empty) == api.E_STATE
    with ctx:
        assert flux(ctx) == api.OK and jvp(ctx) == api.OK
        bad = []
        for kw in (dict(n_views=0), dict(views=None, n_views=1), dict(total=0), dict(total=ptot + 4),
                   dict(channels=2), dict(channels=-1)):
            bad.append((("flux", kw), flux(ctx, **kw)))
        for kw in (dict(n_views=0), dict(views=None, n_views=1), dict(t=0), dict(t=pt + 4), dict(total=ptot + 4),
                   dict(a=0, q=0), dict(a=pa + 4), dict(q=pq + 4)):
            bad.append((("jvp", kw), jvp(ctx, **kw)))
        for key, val in (("precision", 32), ("round_through_float", 1)):
            v = api.View.from_buffer_copy(view)
            setattr(v, key, val)
            bad.append(((key,), jvp(ctx, views=(view, v))))
            assert flux(ctx, views=(view, v)) == api.OK  # the flux call takes what render_flux takes
        for what, rc in bad:
            assert rc == api.E_INVALID, what
            assert flux(ctx) == api.OK and jvp(ctx) == api.OK  # usable after each error
        assert jvp(ctx, a=0) == api.OK and jvp(ctx, q=0) == api.OK and jvp(ctx, total=0) == api.OK
        assert flux(ctx, channels=1) == api.E_STATE  # no channels uploaded
        ctx.upload_channels(*fields(mesh, 2, seed=23))
        flux_ch = mem.empty((2, 2, 2))
        assert flux(ctx, channels=1, total=mem.ptr(flux_ch)) == api.OK
        v32 = api.View.from_buffer_copy(view)
        v32.precision = 32
        assert flux(ctx, views=(view, v32), channels=1, total=mem.ptr(flux_ch)) == api.E_INVALID
        sib = ctx.sibling()
        try:
            assert flux(sib) == api.E_STATE and jvp(sib) == api.E_STATE
        finally:
            sib.close()
        ctx.set_views_in_flight(2)
        for lane in range(2):  # a view in flight on the context itself, then on its lane
            tickets = [ctx.render_submit(view, np.zeros((RES[1], RES[0], 2))) for _ in range(lane + 1)]
            if lane:
                ctx.render_wait(tickets.pop(0))
            try:
                assert flux(ctx) == api.E_STATE and jvp(ctx) == api.E_STATE
            finally:
                for t in tickets:
                    ctx.render_wait(t)
        assert flux(ctx) == api.OK and jvp(ctx) == api.OK
        mem.get(flux_ch)
    with api.Context(devices=(0, 0), lib=lib) as two:
        two.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        assert flux(two) == api.E_INVALID and jvp(two) == api.E_INVALID
    mem.get(dt), mem.get(dtot)


# ---- ordering without host synchronisation (GPU) ------------------------------------------------------------

def _phase_views(lib, n=6):
    """Orbital phases of one grid, solids on."""
    return [api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, X=0.4, Y=0.25 * k, I=-0.03) for k in range(n)]


@pytest.mark.gpu
def test_ordering_on_streams(gpu_lib):
    """A field update and the direction written on a torch side stream behind a long kernel, then both calls
    without stats on that stream (on lanes made after the update) and a torch reduction there: the synchronised
    results of a context uploaded with the new fields."""
    import torch
    mesh = tg.mesh_of(8)
    alpha2, q2 = tg.FIELDS["mixed"](mesh)
    va, vq = direction(alpha2, q2)
    views = _phase_views(gpu_lib)
    mem = Mem(True)
    with api.Context(devices=(0,), lib=gpu_lib) as fresh, api.Context(devices=(0,), lib=gpu_lib) as ctx:
        for c, (a, q) in ((fresh, (alpha2, q2)), (ctx, (mesh.alpha, mesh.q))):
            c.upload_mesh(mesh.points, mesh.tets, a, q)
            c.upload_solids(tg.solids()[0], True)
            c.upload_solids(tg.solids()[1], False)
        want_total = flux_totals(fresh, views)
        want_t = np.stack([curve_tangent(fresh, v, va, vq) for v in views])
        ctx.set_views_in_flight(1)
        flux_device(ctx, mem, views)
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            a, b = torch.tensor(alpha2, device="cuda"), torch.tensor(q2, device="cuda")
            d_va0, d_vq0 = torch.tensor(va, device="cuda"), torch.tensor(vq, device="cuda")
            total = torch.full((len(views), 2), float("nan"), dtype=torch.float64, device="cuda")
            tangent = torch.full_like(total, float("nan"))
            total2 = torch.full_like(total, float("nan"))
            torch.cuda._sleep(200_000_000)  # ~0.1 s of device time before the gather
            ctx.update_fields_device(a.data_ptr(), b.data_ptr(), side.cuda_stream)
            d_va, d_vq = d_va0 * 1.0, d_vq0 * 1.0  # written on the side stream after the long kernel
            ctx.set_views_in_flight(4)
            ctx.render_flux_device(views, total.data_ptr(), side.cuda_stream, stats=False)
            ctx.render_flux_jvp_device(views, d_va.data_ptr(), d_vq.data_ptr(), tangent.data_ptr(), total2.data_ptr(),
                                       side.cuda_stream, stats=False)
            gaps = torch.stack([(total - torch.tensor(want_total, device="cuda")).abs().max(),
                                (total2 - total).abs().max(),
                                (tangent - torch.tensor(want_t, device="cuda")).abs().max()]).cpu().numpy()
        assert np.array_equal(gaps, np.zeros(3)), gaps
        side.synchronize()
        assert np.array_equal(total.cpu().numpy(), want_total) and np.array_equal(tangent.cpu().numpy(), want_t)


@pytest.mark.gpu
def test_autograd_without_host_wait(gpu_lib):
    """With the views warmed up, the light_curve forward and its forward_ad tangent on CUDA tensors return while a
    long kernel still holds the current stream; the forward is render_flux's totals and the tangent
    render_flux_jvp_device's, bit for bit."""
    import torch
    import torch.autograd.forward_ad as fwAD
    from course5_b200 import autograd
    ctx, mesh, _ = tg.small_ctx(gpu_lib, n=8)
    va, vq = direction(mesh.alpha, mesh.q)
    views = _phase_views(gpu_lib) + [with_rows(_phase_views(gpu_lib, 1)[0], (10, 50))]
    mem = Mem(True)
    with ctx:
        ctx.set_views_in_flight(3)
        t = lambda x: torch.tensor(x, device="cuda")  # noqa: E731
        a, q, ta, tq = t(mesh.alpha), t(mesh.q), t(va), t(vq)

        def run():
            with fwAD.dual_level():
                out = fwAD.unpack_dual(autograd.light_curve(ctx, views, fwAD.make_dual(a, ta), fwAD.make_dual(q, tq)))
                return out.primal, out.tangent

        run()
        torch.cuda.synchronize()
        torch.cuda._sleep(200_000_000)
        primal, tangent = run()
        busy = not torch.cuda.current_stream().query()
        torch.cuda.synchronize()
        assert busy, "the forward or its tangent waited for the device"
        assert np.array_equal(primal.cpu().numpy(), flux_totals(ctx, views))
        want, _, _ = jvp_device(ctx, mem, views, va, vq, total=False)
        assert np.array_equal(tangent.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [2, 4])
def test_gradcheck_forward_ad_on_lanes(gpu_lib, lanes):
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
        assert torch.autograd.gradcheck(lambda a, b: autograd.light_curve(ctx, views, a, b), (alpha, q), eps=1e-6,
                                        atol=1e-6, rtol=1e-5, nondet_tol=1e-12, check_forward_ad=True)


# ---- full size (GPU) ----------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_full_size(c3):  # noqa: F811
    """C3 at 2400 x 1800 with solids, 8 views: a central difference of the curve along a random alpha direction
    agrees with J v to 1e-6, and the adjoint identity holds to 1e-12."""
    ctx, mesh, view = c3
    kw = dict(synth.CONFIGS["C3"]["view"])
    y0 = kw.pop("Y", 0.0)
    views = [api.make_view(view.res_x, view.res_y, lib=ctx.lib, round_through_float=0, Y=y0 + 0.1 * k, **kw)
             for k in range(8)]
    mem = Mem(True)
    rng = np.random.default_rng(17)
    d = rng.normal(size=mesh.n_tets) * mesh.alpha
    # the clamp is a kink of I(alpha): cells within reach of it would put the central difference across it
    d[np.abs(mesh.alpha - view.alpha_limit) < 1e-2 * view.alpha_limit] = 0.0
    ctx.set_views_in_flight(3)
    jv, tot, st = jvp_device(ctx, mem, views, d, None)
    assert st["solid_pixels"] > 0 and st["grazing_rays"] > 0
    assert np.array_equal(tot, flux_totals(ctx, views))
    # a curve total sums ~4e6 pixels: its rounding (~1e-16 of the sum of |I|) over 2h must stay far below the
    # 1e-6 gate of a tangent that cancels across pixels, and at h = 1e-4 the O(h^2) term is still ~1e-8
    h = 1e-4
    try:
        ctx.update_fields(mesh.alpha + h * d, mesh.q)
        plus = flux_device(ctx, mem, views)[0][:, 0]
        ctx.update_fields(mesh.alpha - h * d, mesh.q)
        minus = flux_device(ctx, mem, views)[0][:, 0]
    finally:
        ctx.update_fields(mesh.alpha, mesh.q)
    fd = (plus - minus) / (2 * h)
    for k in range(len(views)):
        for c, name in ((0, "tau"), (1, "I")):
            assert tg.rel_close(fd[k, c], jv[k, c], 1e-6), (k, name, fd[k, c], jv[k, c])
    print(f"C3 curve central difference vs J v, view 0: {fd[0]} vs {jv[0]}")
    vq = rng.normal(size=mesh.n_tets) * mesh.q
    jv, _, _ = jvp_device(ctx, mem, views, d, vq, total=False)
    g = rng.normal(size=(len(views), 2))
    ga, gq, _ = flux_grad(ctx, mem, views, g)
    lhs_terms, rhs_terms = g * jv, np.concatenate([ga * d, gq * vq])
    size = np.abs(lhs_terms).sum() + np.abs(rhs_terms).sum()
    assert abs(lhs_terms.sum() - rhs_terms.sum()) <= 1e-12 * size, (lhs_terms.sum(), rhs_terms.sum(), size)
    print(f"C3 curve adjoint: <g, J v> {lhs_terms.sum():.12e} vs <J^T g, v> {rhs_terms.sum():.12e}")
