"""c5_render_jvp and c5_render_jvp_device: the Jacobian-vector product of a view along a field direction.

The tangent images are held to an exact forward-mode differentiation (tests/exact_jvp.py) of the integration
along the segments of the C restatement of the reference (oracle/c5_oracle.c, c5o_render_segments), in
decimal arithmetic, over the case matrix of tests/test_gradients.py. Gate per pixel, for dtau and dI each:
|got - exact| <= 1e-10 |exact| + 1e-12 S_p, S_p the pixel's sum of absolute terms. Each case records its worst
|got - exact| / (1e-10 |exact| + 1e-12 S_p) as a user property (printed with -s).
The adjoint identity <g, J v> = <J^T g, v> ties the tangent to c5_render_grad. Every check runs on the
host-loop build and, with -m gpu, on the CUDA library; stream ordering and the full-size checks on the GPU only.
"""
import ctypes as C

import numpy as np
import pytest

import exact_jvp
import test_gradients as tg
from course5_b200 import api, synth
from test_gradients import c3  # noqa: F401  (C3 at 2400 x 1800 with the reference's solids)
from test_gradients_device import Mem, band_of

RES = tg.RES
REL, FLOOR = 1e-10, 1e-12


@pytest.fixture(params=tg.LIBS)
def env(request):
    return request.getfixturevalue(request.param), Mem(request.param == "gpu_lib")


@pytest.fixture(scope="module")
def oracle_port(port):
    assert hasattr(port.lib, "c5o_render_segments")
    return port


def direction(alpha, q, seed=31):
    """Random signs and sizes on the scale of each tet's own fields (unit size where a field is 0)."""
    rng = np.random.default_rng(seed)
    va = rng.normal(size=alpha.shape) * np.where(alpha != 0.0, np.abs(alpha), 1.0)
    vq = rng.normal(size=q.shape) * np.where(q != 0.0, np.abs(q), 1.0)
    return va, vq


def jvp_device(ctx, mem, view, va, vq, *, out=False, stats=True):
    """c5_render_jvp_device: (tangent, out or None, stats), the view's band only."""
    rb, re = band_of(view)
    d_va = None if va is None else mem.put(va)
    d_vq = None if vq is None else mem.put(vq)
    t = mem.empty((re - rb, view.res_x, 2))
    o = mem.empty((re - rb, view.res_x, 2)) if out else None
    st = ctx.render_jvp_device(view, mem.ptr(d_va), mem.ptr(d_vq), mem.ptr(t), mem.ptr(o), stats=stats)
    return mem.get(t), mem.get(o), st


def make_ctx(lib, mesh, alpha, q, *, debug=None, with_solids=False, devices=(0,)):
    ctx = api.Context(devices=devices, lib=lib)
    for k, v in (debug or {}).items():
        ctx.debug_set(k, v)
    ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
    if with_solids:
        ctx.upload_solids(tg.solids()[0], True)
        ctx.upload_solids(tg.solids()[1], False)
    return ctx


def make_view(lib, view, limit=tg.NO_LIMIT, **over):
    return api.make_view(RES[0], RES[1], lib=lib, alpha_limit=limit, round_through_float=0, **tg.VIEWS[view], **over)


# ---- against the exact tangent ----------------------------------------------------------------------------

_EXACT = {}


def exact_tangent(port, mesh_key, field, view, limit, with_solids):
    key = (mesh_key, field, view, limit, with_solids)
    if key not in _EXACT:
        (start, tet, dz), solid = tg.segments_of(port, mesh_key, view, with_solids)
        alpha, q = tg.FIELDS[field](tg.mesh_of(*mesh_key))
        va, vq = direction(alpha, q)
        t, s = exact_jvp.jvp(start, tet, dz, alpha, q, limit, va, vq)
        _EXACT[key] = (t.reshape(RES[1], RES[0], 2), s.reshape(RES[1], RES[0], 2), solid)
    return _EXACT[key]


def check_tangent(record_property, what, got, exact, scale, solid):
    assert np.isnan(got[solid]).all(), f"{what}: a pixel under the solid mask is not NaN"
    live = ~solid
    g, x, s = got[live], exact[live], scale[live]
    assert np.isfinite(g).all(), f"{what}: a pixel outside the solid mask is not finite"
    tol = REL * np.abs(x) + FLOOR * s
    err = np.abs(g - x)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(tol > 0, err / np.where(tol > 0, tol, 1.0), np.where(err > 0, np.inf, 0.0))
    worst = float(ratio.max())
    record_property("worst_ratio_jvp", worst)
    print(f"{what}: worst |got - exact| / (1e-10 |exact| + 1e-12 S_p) = {worst:.2e}")
    assert worst <= 1.0, f"{what}: {int((ratio > 1).sum())} values outside the gate, worst ratio {worst:.2e}"


def run_case(lib, mem, port, record_property, *, mesh_key, field, view, limit=tg.NO_LIMIT, debug=None,
             with_solids=False, what=""):
    """The host form against the exact tangent; its image is render_raw's and the device form gives its bits."""
    exact, scale, solid = exact_tangent(port, mesh_key, field, view, limit, with_solids)
    mesh = tg.mesh_of(*mesh_key)
    alpha, q = tg.FIELDS[field](mesh)
    va, vq = direction(alpha, q)
    with make_ctx(lib, mesh, alpha, q, debug=debug, with_solids=with_solids) as ctx:
        v = make_view(lib, view, limit)
        raw = ctx.render_raw(v)
        tangent, img = ctx.render_jvp(v, va, vq, image=True)
        st = ctx.last_stats
        d_tangent, d_img, _ = jvp_device(ctx, mem, v, va, vq, out=True)
    assert st["walk_errors"] == 0
    assert np.array_equal(img, raw.image, equal_nan=True)
    assert np.array_equal(np.isnan(tangent[..., 0]), raw.solid.astype(bool))
    assert np.array_equal(d_tangent, tangent, equal_nan=True) and np.array_equal(d_img, img, equal_nan=True)
    check_tangent(record_property, what, tangent, exact, scale, solid)
    return st


@pytest.mark.parametrize("view", list(tg.VIEWS))
@pytest.mark.parametrize("a0", tg.DECADES, ids=[f"{a:g}" for a in tg.DECADES])
def test_decades(env, oracle_port, record_property, a0, view):
    lib, mem = env
    i = tg.DECADES.index(a0)
    n = 5 + i % 3 if view == "generic" else 8 + i % 3
    st = run_case(lib, mem, oracle_port, record_property, mesh_key=(n, False), field=f"decade_{a0:g}", view=view,
                  what=f"alpha {a0:g} {view}")
    if view == "axis":
        assert st["grazing_rays"] > 0  # the grazing-ray fold of the tangent is exercised


@pytest.mark.parametrize("path", ["pixel", "budget", "graze_list"])
@pytest.mark.parametrize("view", list(tg.VIEWS))
def test_mixed(env, oracle_port, record_property, view, path):
    """Zero, DBL_EPSILON, the double below it and negative alpha; search-budget deferrals; the grazing-ray
    collection at its minimum list."""
    lib, mem = env
    debug = {"budget": {"query_budget": 3}, "graze_list": {"graze_list": 128, "serial_list": 2}}.get(path)
    st = run_case(lib, mem, oracle_port, record_property, mesh_key=(8, False), field="mixed", view=view, debug=debug,
                  what=f"mixed {view} {path}")
    if path == "budget":
        assert st["grazing_rays"] > st["hit_pixels"] // 2


@pytest.mark.parametrize("limit", ["at_cell", "below_cell", "thin"])
def test_alpha_limit_edges(env, oracle_port, record_property, limit):
    lib, mem = env
    run_case(lib, mem, oracle_port, record_property, mesh_key=(6, False), field="decade_1", view="generic",
             limit=tg.clamp_limits()[limit], what=f"limit {limit}")


@pytest.mark.parametrize("field", ["decade_0.01", "mixed"])
def test_cavity(env, oracle_port, record_property, field):
    lib, mem = env
    run_case(lib, mem, oracle_port, record_property, mesh_key=(10, True), field=field, view="generic",
             what=f"cavity {field}")


def test_reference_solids(env, oracle_port, record_property):
    lib, mem = env
    run_case(lib, mem, oracle_port, record_property, mesh_key=(8, False), field="decade_1", view="generic",
             with_solids=True, what="solids")


# ---- the adjoint identity and special directions --------------------------------------------------------------

def adjoint_gap(tangent, g, ga, gq, va, vq):
    """(<g, J v>, <J^T g, v>, the sum of the absolute terms of both)."""
    live = ~np.isnan(tangent[..., 0])
    terms = g[live] * tangent[live]
    rhs_terms = np.concatenate([ga * va, gq * vq])
    return float(terms.sum()), float(rhs_terms.sum()), float(np.abs(terms).sum() + np.abs(rhs_terms).sum())


@pytest.mark.parametrize("g_kind", ["full", "tau_only", "I_only"])
def test_adjoint_identity(env, g_kind):
    """<g, J v> equals <c5_render_grad(g), v> to 1e-12 of the sum of absolute terms, solids on."""
    lib, mem = env
    mesh = tg.mesh_of(8)
    alpha, q = tg.FIELDS["decade_1"](mesh)
    va, vq = direction(alpha, q, seed=5)
    g = tg.upstream(g_kind)
    with make_ctx(lib, mesh, alpha, q, with_solids=True) as ctx:
        for view in tg.VIEWS:
            v = make_view(lib, view, 2.5)
            tangent = ctx.render_jvp(v, va, vq)
            ga, gq = ctx.render_grad(v, g)
            lhs, rhs, size = adjoint_gap(tangent, g, ga, gq, va, vq)
            assert np.isnan(tangent).any()
            assert abs(lhs - rhs) <= 1e-12 * size, (view, lhs, rhs, size)


def test_special_directions(env):
    """v_alpha = alpha gives dtau == tau bit for bit; v_Q = Q gives dI = I (I is linear in Q); J (2 v) == 2 J v bit
    for bit; J (v + w) = J v + J w to rounding. The axis view has grazing rays, so the fold is in all four."""
    lib, mem = env
    mesh = tg.mesh_of(8)
    alpha, q = tg.FIELDS["decade_1"](mesh)  # alpha, Q > 0
    v1, w1 = direction(alpha, q, seed=1)
    v2, w2 = direction(alpha, q, seed=2)
    with make_ctx(lib, mesh, alpha, q, with_solids=True) as ctx:
        v = make_view(lib, "axis", 2.5)
        raw = ctx.render_raw(v)
        assert raw.stats["grazing_rays"] > 0
        t_a = ctx.render_jvp(v, alpha, None)
        assert np.array_equal(t_a[..., 0], raw.tau, equal_nan=True)
        t_q = ctx.render_jvp(v, None, q)
        live = ~raw.solid.astype(bool)
        assert not t_q[..., 0][live].any()
        assert np.all(np.abs(t_q[..., 1][live] - raw.inten[live]) <= 1e-13 * np.abs(raw.inten[live]))
        j1 = ctx.render_jvp(v, v1, w1)
        assert np.array_equal(ctx.render_jvp(v, 2.0 * v1, 2.0 * w1), 2.0 * j1, equal_nan=True)
        j2 = ctx.render_jvp(v, v2, w2)
        j12 = ctx.render_jvp(v, v1 + v2, w1 + w2)
        scale = np.abs(j1[live]) + np.abs(j2[live])
        assert np.all(np.abs(j12[live] - (j1[live] + j2[live])) <= 1e-12 * scale + 1e-300)


# ---- determinism ----------------------------------------------------------------------------------------------

def test_bit_reproducible(env):
    """Two calls, two row bands pieced together, a (0, 0) context, a sibling, one device, and the device form
    with band-sized buffers: all the same bits."""
    lib, mem = env
    mesh = tg.mesh_of(8)
    alpha, q = tg.FIELDS["mixed"](mesh)
    va, vq = direction(alpha, q)
    debug = {"graze_list": 128, "serial_list": 2}
    with make_ctx(lib, mesh, alpha, q, debug=debug, with_solids=True) as one, \
            make_ctx(lib, mesh, alpha, q, debug=debug, with_solids=True, devices=(0, 0)) as two:
        v = make_view(lib, "axis", 2.5)
        want, img = one.render_jvp(v, va, vq, image=True)
        assert one.last_stats["grazing_rays"] > 0
        assert np.array_equal(one.render_jvp(v, va, vq), want, equal_nan=True)
        pieced = np.zeros_like(want)
        for rows in ((0, 29), (29, RES[1])):
            b = api.View.from_buffer_copy(v)
            b.row_begin, b.row_end = rows
            part = one.render_jvp(b, va, vq)
            assert not part[:rows[0]].any() and not part[rows[1]:].any()
            pieced[rows[0]:rows[1]] = part[rows[0]:rows[1]]
            d_part, d_img, _ = jvp_device(one, mem, b, va, vq, out=True)
            assert np.array_equal(d_part, want[rows[0]:rows[1]], equal_nan=True)
            assert np.array_equal(d_img, img[rows[0]:rows[1]], equal_nan=True)
        assert np.array_equal(pieced, want, equal_nan=True)
        got2, img2 = two.render_jvp(v, va, vq, image=True)
        assert two.last_stats["n_devices"] == 2
        assert np.array_equal(got2, want, equal_nan=True) and np.array_equal(img2, img, equal_nan=True)
        sib = one.sibling()
        try:
            assert np.array_equal(sib.render_jvp(v, va, vq), want, equal_nan=True)
            assert np.array_equal(jvp_device(sib, mem, v, va, vq)[0], want, equal_nan=True)
        finally:
            sib.close()


# ---- the call's surface -------------------------------------------------------------------------------------

def test_launch_counts_and_device_bytes(env):
    """Both forms launch what render_raw launches plus one gather; the tangent field (16 bytes per tet) and the
    device permutation (4 bytes per tet) count in device_bytes from the first call; a new mesh drops both."""
    lib, mem = env
    ctx, mesh, view = tg.small_ctx(lib)
    va, vq = direction(mesh.alpha, mesh.q)
    with ctx:
        ctx.render_raw(view)  # cells prepared for the view's alpha_limit
        n0 = ctx.kernel_launches()
        ctx.render_raw(view)
        n_raw = ctx.kernel_launches() - n0
        before = ctx.mesh_info().device_bytes
        n0 = ctx.kernel_launches()
        ctx.render_jvp(view, va, vq)
        assert ctx.kernel_launches() - n0 == n_raw + 1
        assert ctx.mesh_info().device_bytes == before + 20 * mesh.n_tets
        n0 = ctx.kernel_launches()
        jvp_device(ctx, mem, view, va, None)
        assert ctx.kernel_launches() - n0 == n_raw + 1
        assert ctx.mesh_info().device_bytes == before + 20 * mesh.n_tets
        n0 = ctx.kernel_launches()
        ctx.render_raw(view)
        assert ctx.kernel_launches() - n0 == n_raw
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        plain = ctx.mesh_info().device_bytes
        ctx.render_jvp(view, None, vq)
        assert ctx.mesh_info().device_bytes == plain + 20 * mesh.n_tets


def test_errors(env):
    lib, mem = env
    vp = C.c_void_p
    dp = C.POINTER(C.c_double)
    ctx, mesh, view = tg.small_ctx(lib)
    ha, hq = direction(mesh.alpha, mesh.q)
    ht = np.zeros((RES[1], RES[0], 2))
    da, dq = mem.put(ha), mem.put(hq)
    dt, do = mem.empty((RES[1], RES[0], 2)), mem.empty((RES[1], RES[0], 2))
    pa, pq, pt, po = mem.ptr(da), mem.ptr(dq), mem.ptr(dt), mem.ptr(do)

    def host(c, v=view, a=ha, q=hq, t=ht):
        return lib.c5_render_jvp(c._h, C.byref(v), None if a is None else a.ctypes.data_as(dp),
                                 None if q is None else q.ctypes.data_as(dp),
                                 None if t is None else t.ctypes.data_as(dp), None, None)

    def dev(c, v=view, a=pa, q=pq, t=pt, o=po):
        return lib.c5_render_jvp_device(c._h, C.byref(v), vp(a or None), vp(q or None), vp(t or None), vp(o or None),
                                        None, None)

    with api.Context(devices=(0,), lib=lib) as empty:
        assert host(empty) == api.E_STATE and dev(empty) == api.E_STATE
    with ctx:
        assert host(ctx) == api.OK and dev(ctx) == api.OK
        assert host(ctx, t=None) == api.E_INVALID and dev(ctx, t=0) == api.E_INVALID
        assert host(ctx, a=None, q=None) == api.E_INVALID and dev(ctx, a=0, q=0) == api.E_INVALID
        assert host(ctx, a=None) == api.OK and host(ctx, q=None) == api.OK
        with pytest.raises(ValueError):
            ctx.render_jvp(view, None, None)
        with pytest.raises(ValueError):
            ctx.render_jvp(view, ha[:-1], None)
        assert dev(ctx, a=0, o=0) == api.OK and dev(ctx, q=0) == api.OK
        for key, val in (("precision", 32), ("round_through_float", 1)):
            bad = api.View.from_buffer_copy(view)
            setattr(bad, key, val)
            assert host(ctx, v=bad) == api.E_INVALID and dev(ctx, v=bad) == api.E_INVALID
        for kw in (dict(a=pa + 4), dict(q=pq + 4), dict(t=pt + 8), dict(o=po + 8)):
            assert dev(ctx, **kw) == api.E_INVALID, kw
        sib = ctx.sibling()
        try:
            assert host(sib) == api.OK and dev(sib) == api.OK
        finally:
            sib.close()
        ctx.set_views_in_flight(2)
        t = ctx.render_submit(view, np.zeros((RES[1], RES[0], 2)))
        try:
            assert host(ctx) == api.E_STATE and dev(ctx) == api.E_STATE
        finally:
            ctx.render_wait(t)
    with api.Context(devices=(0, 0), lib=lib) as two:
        two.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        assert host(two) == api.OK
        assert dev(two) == api.E_INVALID
    mem.get(dt)


@pytest.mark.gpu
def test_ordering_on_streams(gpu_lib):
    """A: a field update on a torch side stream, held back by a long kernel, then render_jvp_device on that stream
    without stats: the tangent is that of the new fields. B: render_jvp_device held back on a side stream, then a
    blocking render_raw on the context's own stream, which reuses the scratch the call copies from: the tangent
    is still the synchronised one."""
    import torch
    mesh = tg.mesh_of(8)
    alpha2, q2 = tg.FIELDS["mixed"](mesh)
    va, vq = direction(alpha2, q2)
    view = make_view(gpu_lib, "generic", 2.5)
    with make_ctx(gpu_lib, mesh, alpha2, q2, with_solids=True) as fresh, \
            make_ctx(gpu_lib, mesh, mesh.alpha, mesh.q, with_solids=True) as ctx:
        want = fresh.render_jvp(view, va, vq)
        want_img = fresh.render_raw(view).image
        ctx.render_raw(view)
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            a, b = torch.tensor(alpha2, device="cuda"), torch.tensor(q2, device="cuda")
            d_va, d_vq = torch.tensor(va, device="cuda"), torch.tensor(vq, device="cuda")
            tangent = torch.full((RES[1], RES[0], 2), float("nan"), dtype=torch.float64, device="cuda")
            torch.cuda._sleep(200_000_000)  # ~0.1 s of device time before the gather
            ctx.update_fields_device(a.data_ptr(), b.data_ptr(), side.cuda_stream)
            ctx.render_jvp_device(view, d_va.data_ptr(), d_vq.data_ptr(), tangent.data_ptr(), stream=side.cuda_stream,
                                  stats=False)
            got = tangent.cpu().numpy()
        assert np.array_equal(got, want, equal_nan=True)
        with torch.cuda.stream(side):
            tangent2 = torch.full_like(tangent, float("nan"))
            torch.cuda._sleep(200_000_000)
            ctx.render_jvp_device(view, d_va.data_ptr(), d_vq.data_ptr(), tangent2.data_ptr(), stream=side.cuda_stream,
                                  stats=False)
        assert np.array_equal(ctx.render_raw(view).image, want_img, equal_nan=True)
        side.synchronize()
        assert np.array_equal(tangent2.cpu().numpy(), want, equal_nan=True)


# ---- torch ---------------------------------------------------------------------------------------------------

def _devices(mem):
    return ("cpu", "cuda") if mem.gpu else ("cpu",)


def test_forward_ad(env):
    """forward_ad tangents of autograd.render and autograd.light_curve equal render_jvp and its per-view sums
    over the pixels outside the solid mask (solids and a row band included)."""
    torch = pytest.importorskip("torch")
    import torch.autograd.forward_ad as fwAD
    from course5_b200 import autograd
    lib, mem = env
    ctx, mesh, view = tg.small_ctx(lib, n=6)
    va, vq = direction(mesh.alpha, mesh.q)
    band = api.View.from_buffer_copy(view)
    band.row_begin, band.row_end = 10, 50
    views = [view, band]
    with ctx:
        want = [ctx.render_jvp(v, va, vq) for v in views]
        for dev in _devices(mem):
            t = lambda x: torch.tensor(x, device=dev)  # noqa: E731
            with fwAD.dual_level():
                a = fwAD.make_dual(t(mesh.alpha), t(va))
                q = fwAD.make_dual(t(mesh.q), t(vq))
                for v, w in zip(views, want):
                    out = fwAD.unpack_dual(autograd.render(ctx, v, a, q))
                    assert out.tangent.device.type == dev
                    assert np.array_equal(out.tangent.cpu().numpy(), w, equal_nan=True)
                lc = fwAD.unpack_dual(autograd.light_curve(ctx, views, a, q)).tangent.cpu().numpy()
                # only v_Q moves
                only_q = fwAD.unpack_dual(autograd.render(ctx, view, t(mesh.alpha), q)).tangent.cpu().numpy()
            assert np.array_equal(only_q, ctx.render_jvp(view, None, vq), equal_nan=True)
            for k, w in enumerate(want):
                sums = np.nansum(w, axis=(0, 1))
                assert np.allclose(lc[k], sums, rtol=1e-13, atol=1e-13 * np.nansum(np.abs(w), axis=(0, 1)).max())


def test_gradcheck_forward_ad(env):
    torch = pytest.importorskip("torch")
    from course5_b200 import autograd
    lib, mem = env
    mesh = synth.kuhn_cube(3, seed=7)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        view = api.make_view(24, 18, lib=lib, alpha_limit=tg.NO_LIMIT, use_solids=0, **tg.VIEWS["generic"])
        views = [view, api.make_view(24, 18, lib=lib, alpha_limit=tg.NO_LIMIT, use_solids=0, **tg.VIEWS["axis"])]
        for dev in _devices(mem):
            alpha = torch.tensor(mesh.alpha, device=dev, requires_grad=True)
            q = torch.tensor(mesh.q, device=dev, requires_grad=True)
            kw = dict(eps=1e-6, atol=1e-6, rtol=1e-5, check_forward_ad=True, nondet_tol=1e-12 if mem.gpu else 0.0)
            assert torch.autograd.gradcheck(lambda a, b: autograd.render(ctx, view, a, b), (alpha, q), fast_mode=True,
                                            **kw)
            assert torch.autograd.gradcheck(lambda a, b: autograd.light_curve(ctx, views, a, b), (alpha, q), **kw)


# ---- full size (GPU) ----------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_full_size(c3):  # noqa: F811
    """C3 at 2400 x 1800 with solids: a central difference along a random alpha direction, through
    update_fields and render_raw, agrees with J v summed over the live pixels to 1e-6; the adjoint identity
    holds to 1e-12; the device form gives the host form's bits."""
    import torch
    ctx, mesh, view = c3
    rng = np.random.default_rng(13)
    raw = ctx.render_raw(view)
    assert raw.solid.sum() > 0 and raw.stats["grazing_rays"] > 0
    live = ~raw.solid.astype(bool)
    d = rng.normal(size=mesh.n_tets) * mesh.alpha
    # the clamp is a kink of I(alpha): cells within reach of it would put the central difference across it
    d[np.abs(mesh.alpha - view.alpha_limit) < 1e-3 * view.alpha_limit] = 0.0
    tangent, img = ctx.render_jvp(view, d, None, image=True)
    assert np.array_equal(img, raw.image, equal_nan=True)
    dev = torch.full((view.res_y, view.res_x, 2), float("nan"), dtype=torch.float64, device="cuda")
    ctx.render_jvp_device(view, torch.tensor(d, device="cuda").data_ptr(), 0, dev.data_ptr())
    assert np.array_equal(dev.cpu().numpy(), tangent, equal_nan=True)
    h = 1e-6
    try:
        ctx.update_fields(mesh.alpha + h * d, mesh.q)
        plus = ctx.render_raw(view).image
        ctx.update_fields(mesh.alpha - h * d, mesh.q)
        minus = ctx.render_raw(view).image
    finally:
        ctx.update_fields(mesh.alpha, mesh.q)
    for c, name in ((0, "tau"), (1, "I")):
        fd = float(np.sum((plus[..., c] - minus[..., c])[live]) / (2 * h))
        an = float(np.sum(tangent[..., c][live]))
        assert tg.rel_close(fd, an, 1e-6), (name, fd, an)
        print(f"C3 central difference of sum {name}: {fd:.9e} vs J v {an:.9e}")
    vq = rng.normal(size=mesh.n_tets) * mesh.q
    tangent = ctx.render_jvp(view, d, vq)
    g = rng.normal(size=(view.res_y, view.res_x, 2))
    ga, gq = ctx.render_grad(view, np.where(live[..., None], g, np.nan))
    lhs, rhs, size = adjoint_gap(tangent, g, ga, gq, d, vq)
    assert abs(lhs - rhs) <= 1e-12 * size, (lhs, rhs, size)
    print(f"C3 adjoint: <g, J v> {lhs:.12e} vs <J^T g, v> {rhs:.12e}")
