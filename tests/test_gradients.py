"""c5_render_grad and c5_update_fields.

The gradients are held to an exact reverse-mode differentiation (tests/exact_grad.py) of the integration
along the segments of the C restatement of the reference (oracle/c5_oracle.c, c5o_render_segments), in
decimal arithmetic: a different formulation (adjoint backwards from the viewer) from the kernel's (forward,
with T = exp(-(lam_ray - lam_through))). Gate per tet, for grad_alpha and grad_q each:
|got - exact| <= 1e-10 |exact| + 1e-12 max|exact|. Each test records its worst
|err| / (|exact| + floor / rel * max|exact|) (a user property; printed with -s).
Every check runs on the host-loop build (tests/hostsim) and, with -m gpu, on the CUDA library; the
full-size identities and the multi-device checks run on the GPU only.
"""
import numpy as np
import pytest

import exact_grad
from course5_b200 import api, hostlib, synth
from parity import exact_margin

LIBS = [pytest.param("hostsim_lib", id="hostsim"), pytest.param("gpu_lib", id="gpu", marks=pytest.mark.gpu)]
RES = (96, 72)
VIEWS = {"generic": dict(X=0.4, Y=0.7, I=-0.03), "axis": dict(X=0.5, Y=0.0)}
DECADES = [1e-15, 1e-12, 1e-8, 1e-4, 1e-2, 1.0, 1e2, 1e3]
NO_LIMIT = 1e30
DBL_EPSILON = np.finfo(np.float64).eps
REL, FLOOR = 1e-10, 1e-12


@pytest.fixture(params=LIBS)
def lib(request):
    return request.getfixturevalue(request.param)


@pytest.fixture(scope="module")
def oracle_port(port):
    assert hasattr(port.lib, "c5o_render_segments")
    return port


# ---- meshes, fields, upstream gradients -----------------------------------------------------------------

_MESHES = {}


def mesh_of(n, carve=False):
    key = (n, carve)
    if key not in _MESHES:
        _MESHES[key] = (synth.kuhn_cube(n, seed=55, scalars="sphere", carve_sphere=True) if carve
                        else synth.kuhn_cube(n, seed=7))
    return _MESHES[key]


def decade_field(mesh, a0, seed):
    rng = np.random.default_rng(seed)
    return a0 * rng.uniform(0.5, 1.5, mesh.n_tets), rng.uniform(0.1, 4.0, mesh.n_tets)


def mixed_field(mesh, seed):
    """log10 alpha ~ U(-15, 3), log10 Q ~ U(-3, 3); Q = 0 in one tet of 13; one tet in 17 has alpha
    exactly 0, DBL_EPSILON, the double below it, or a negative alpha."""
    rng = np.random.default_rng(seed)
    alpha = 10.0 ** rng.uniform(-15.0, 3.0, mesh.n_tets)
    q = 10.0 ** rng.uniform(-3.0, 3.0, mesh.n_tets)
    q[::13] = 0.0
    special = np.arange(5, mesh.n_tets, 17)
    kinds = np.array([0.0, DBL_EPSILON, np.nextafter(DBL_EPSILON, 0.0), -1.0])
    alpha[special] = kinds[np.arange(special.size) % 4]
    neg = special[np.arange(special.size) % 4 == 3]
    alpha[neg] = -(10.0 ** rng.uniform(-15.0, 1.0, neg.size))
    return alpha, q


FIELDS = {f"decade_{a0:g}": (lambda mesh, a0=a0, i=i: decade_field(mesh, a0, 500 + i)) for i, a0 in enumerate(DECADES)}
FIELDS["mixed"] = lambda mesh: mixed_field(mesh, 600)


def upstream(kind, seed=11):
    """{g_tau, g_I} per pixel: normal with a tenth of the values 0, or one of the two only."""
    rng = np.random.default_rng(seed)
    g = rng.normal(size=(RES[1], RES[0], 2))
    g[rng.uniform(size=g.shape) < 0.1] = 0.0
    if kind == "tau_only":
        g[..., 1] = 0.0
    elif kind == "I_only":
        g[..., 0] = 0.0
    return g


# ---- the exact gradients, each computed once per module ------------------------------------------------

_SEGMENTS = {}
_EXACT = {}
_SOLIDS = []


def solids():
    if not _SOLIDS:
        _SOLIDS.append(hostlib.make_solids(0.0))
    return _SOLIDS[0]


def segments_of(port, mesh_key, view, with_solids):
    key = (mesh_key, view, with_solids)
    if key not in _SEGMENTS:
        mesh = mesh_of(*mesh_key)
        kw = dict(VIEWS[view])
        if with_solids:
            kw.update(solid_rot=solids()[0], solid_static=solids()[1])
        want = port.render(mesh.tet_points(), mesh.alpha, mesh.q, res_x=RES[0], res_y=RES[1], **kw)
        assert want.anomalies == 0
        seg = port.segments(mesh.tet_points(), mesh.alpha, mesh.q, res_x=RES[0], res_y=RES[1], steps=want.steps, **kw)
        solid = np.isnan(want.tau)
        _SEGMENTS[key] = (seg, solid)
    return _SEGMENTS[key]


def exact_grads(port, mesh_key, field, view, limit, g_kind, with_solids=False):
    key = (mesh_key, field, view, limit, g_kind, with_solids)
    if key not in _EXACT:
        (start, tet, dz), solid = segments_of(port, mesh_key, view, with_solids)
        mesh = mesh_of(*mesh_key)
        alpha, q = FIELDS[field](mesh)
        g = upstream(g_kind).copy()
        g[solid] = 0.0
        _EXACT[key] = exact_grad.vjp(start, tet, dz, alpha, q, limit, g.reshape(-1, 2), mesh.n_tets)
    return _EXACT[key]


def render_grad(lib, mesh, alpha, q, view, limit, g, *, debug=None, with_solids=False, rows=None):
    with api.Context(devices=(0,), lib=lib) as ctx:
        for k, v in (debug or {}).items():
            ctx.debug_set(k, v)
        ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
        if with_solids:
            ctx.upload_solids(solids()[0], True)
            ctx.upload_solids(solids()[1], False)
        over = dict(round_through_float=0)
        if rows is not None:
            over.update(row_begin=rows[0], row_end=rows[1])
        v = api.make_view(RES[0], RES[1], lib=lib, alpha_limit=limit, **VIEWS[view], **over)
        ga, gq = ctx.render_grad(v, g)
        return ga, gq, ctx.last_stats


def check_grads(record_property, what, got, exact):
    report = []
    for name, a, b in (("alpha", got[0], exact[0]), ("q", got[1], exact[1])):
        assert np.isfinite(a).all(), f"{what}: grad_{name} is not finite"
        m = exact_margin(a, b, rel=REL, floor=FLOOR)
        worst = float(m.max()) * REL
        record_property(f"worst_rel_grad_{name}", worst)
        report.append(f"{name} {worst:.1e}")
        bad = m > 1.0
        assert not bad.any(), (f"{what}: grad_{name}: {int(bad.sum())} of {int((b != 0).sum())} tets outside "
                               f"{REL:g} |exact| + {FLOOR:g} max|exact|, worst relative error {worst:.2e}")
    print(f"{what}: worst relative error " + ", ".join(report))


def run_case(lib, port, record_property, *, mesh_key, field, view, limit=NO_LIMIT, g_kind="full", debug=None,
             with_solids=False, what=""):
    exact = exact_grads(port, mesh_key, field, view, limit, g_kind, with_solids)
    mesh = mesh_of(*mesh_key)
    alpha, q = FIELDS[field](mesh)
    g = upstream(g_kind)
    if with_solids:  # whatever g holds under the solid mask is not read
        g = g.copy()
        g[segments_of(port, mesh_key, view, True)[1]] = np.nan
    ga, gq, st = render_grad(lib, mesh, alpha, q, view, limit, g, debug=debug, with_solids=with_solids)
    assert st["walk_errors"] == 0
    check_grads(record_property, what, (ga, gq), exact)
    return st


# ---- against the exact gradient ------------------------------------------------------------------------

@pytest.mark.parametrize("view", list(VIEWS))
@pytest.mark.parametrize("a0", DECADES, ids=[f"{a:g}" for a in DECADES])
def test_decades(lib, oracle_port, record_property, a0, view):
    i = DECADES.index(a0)
    n = 5 + i % 3 if view == "generic" else 8 + i % 3   # the axis view sees side walls edge-on from n = 8 on
    st = run_case(lib, oracle_port, record_property, mesh_key=(n, False), field=f"decade_{a0:g}", view=view,
                  what=f"alpha {a0:g} {view}")
    if view == "axis":
        assert st["grazing_rays"] > 0      # the grazing-ray gradient (fold, then re-walk) is exercised


@pytest.mark.parametrize("path", ["pixel", "budget", "graze_list"])
@pytest.mark.parametrize("view", list(VIEWS))
def test_mixed(lib, oracle_port, record_property, view, path):
    """Zero, DBL_EPSILON, the double below it and negative alpha; search-budget deferrals; the grazing-ray
    collection at its minimum list, so that its overflow path runs."""
    debug = {"budget": {"query_budget": 3}, "graze_list": {"graze_list": 128, "serial_list": 2}}.get(path)
    st = run_case(lib, oracle_port, record_property, mesh_key=(8, False), field="mixed", view=view, debug=debug,
                  what=f"mixed {view} {path}")
    if path == "budget":
        assert st["grazing_rays"] > st["hit_pixels"] // 2


def clamp_limits():
    alpha, _ = FIELDS["decade_1"](mesh_of(6))
    cell = float(alpha[123])
    return {"at_cell": cell, "below_cell": float(np.nextafter(cell, 0.0)), "thin": 1e-12}


@pytest.mark.parametrize("limit", ["at_cell", "below_cell", "thin"])
def test_alpha_limit_edges(lib, oracle_port, record_property, limit):
    """At a cell's alpha dI/dalpha flows through it; one ulp below it is 0; at 1e-12 every cell is clamped."""
    value = clamp_limits()[limit]
    run_case(lib, oracle_port, record_property, mesh_key=(6, False), field="decade_1", view="generic", limit=value,
             what=f"limit {limit}")


@pytest.mark.parametrize("field", ["decade_0.01", "mixed"])
def test_cavity(lib, oracle_port, record_property, field):
    """Rays leave the carved sphere and re-enter: I and lam cross several crossings."""
    run_case(lib, oracle_port, record_property, mesh_key=(10, True), field=field, view="generic",
             what=f"cavity {field}")


@pytest.mark.parametrize("g_kind", ["full", "tau_only", "I_only"])
def test_upstream_kinds(lib, oracle_port, record_property, g_kind):
    run_case(lib, oracle_port, record_property, mesh_key=(7, False), field="decade_1", view="axis", g_kind=g_kind,
             what=f"g {g_kind}")


def test_reference_solids(lib, oracle_port, record_property):
    """Pixels under the solids hold NaN in g: they are not read and add nothing."""
    run_case(lib, oracle_port, record_property, mesh_key=(8, False), field="decade_1", view="generic",
             with_solids=True, what="solids")


# ---- the call's surface ----------------------------------------------------------------------------------

def small_ctx(lib, n=5, solids_too=True):
    mesh = mesh_of(n)
    ctx = api.Context(devices=(0,), lib=lib)
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    if solids_too:
        ctx.upload_solids(solids()[0], True)
        ctx.upload_solids(solids()[1], False)
    view = api.make_view(RES[0], RES[1], lib=lib, round_through_float=0, **VIEWS["generic"])
    return ctx, mesh, view


def test_render_grad_errors(lib):
    import ctypes as C
    _, mesh, view = small_ctx(lib)
    n_pix = RES[0] * RES[1]
    g = np.zeros(2 * n_pix)
    ga = np.zeros(mesh.n_tets)
    dp = C.POINTER(C.c_double)
    with api.Context(devices=(0,), lib=lib) as empty:
        rc = lib.c5_render_grad(empty._h, C.byref(view), g.ctypes.data_as(dp), ga.ctypes.data_as(dp), None, None, None)
        assert rc == api.E_STATE
        assert lib.c5_update_fields(empty._h, ga.ctypes.data_as(dp), ga.ctypes.data_as(dp)) == api.E_STATE
    ctx, mesh, view = small_ctx(lib)
    with ctx:
        def call(v=view, gg=g, a=ga, q=None):
            return lib.c5_render_grad(ctx._h, C.byref(v), None if gg is None else gg.ctypes.data_as(dp),
                                      None if a is None else a.ctypes.data_as(dp),
                                      None if q is None else q.ctypes.data_as(dp), None, None)
        assert call() == api.OK
        assert call(gg=None) == api.E_INVALID
        assert call(a=None, q=None) == api.E_INVALID
        for key, val in (("precision", 32), ("round_through_float", 1)):
            bad = api.View.from_buffer_copy(view)
            setattr(bad, key, val)
            assert call(v=bad) == api.E_INVALID
        assert lib.c5_update_fields(ctx._h, None, ga.ctypes.data_as(dp)) == api.E_INVALID
        sib = ctx.sibling()
        try:
            assert lib.c5_update_fields(sib._h, ga.ctypes.data_as(dp), ga.ctypes.data_as(dp)) == api.E_STATE
        finally:
            sib.close()
        ctx.set_views_in_flight(2)
        t = ctx.render_submit(view, np.zeros((RES[1], RES[0], 2)))
        try:
            assert lib.c5_update_fields(ctx._h, ga.ctypes.data_as(dp), ga.ctypes.data_as(dp)) == api.E_STATE
            assert call() == api.E_STATE
        finally:
            ctx.render_wait(t)


def test_out_is_render_raw_and_launch_count(lib):
    """out of render_grad is render_raw's image bit for bit; render_grad launches exactly two kernels more
    than render_raw of the same view (the gradient pass's pixel and grazing-ray kernels), and render_raw
    launches what it did before (its count does not move after a gradient render)."""
    ctx, mesh, view = small_ctx(lib)
    with ctx:
        raw = ctx.render_raw(view)                      # cells prepared for the view's alpha_limit
        n0 = ctx.kernel_launches()
        raw = ctx.render_raw(view)
        n_raw = ctx.kernel_launches() - n0
        g = upstream("full")
        n0 = ctx.kernel_launches()
        ga, gq, img = ctx.render_grad(view, g, image=True)
        n_grad = ctx.kernel_launches() - n0
        n0 = ctx.kernel_launches()
        again = ctx.render_raw(view)
        assert ctx.kernel_launches() - n0 == n_raw
        assert n_grad == n_raw + 2
        assert np.array_equal(img, raw.image, equal_nan=True)
        assert np.array_equal(again.image, raw.image, equal_nan=True)
        assert raw.solid.sum() > 0
        assert ctx.last_stats["tet_steps"] == raw.stats["tet_steps"]
        assert ctx.last_stats["solid_pixels"] == raw.stats["solid_pixels"]


def test_row_bands_add_up(lib):
    ctx, mesh, view = small_ctx(lib, n=6)
    g = upstream("full")
    with ctx:
        whole = ctx.render_grad(view, g)
        parts = []
        for rows in ((0, 29), (29, RES[1])):
            v = api.View.from_buffer_copy(view)
            v.row_begin, v.row_end = rows
            parts.append(ctx.render_grad(v, g))
    for k in range(2):
        summed = parts[0][k] + parts[1][k]
        assert np.allclose(summed, whole[k], rtol=1e-13, atol=1e-13 * np.abs(whole[k]).max())


# ---- c5_update_fields ------------------------------------------------------------------------------------

def test_update_fields_matches_a_fresh_upload(lib):
    """Across an alpha_limit change, through a sibling, with channels and solids kept."""
    mesh = mesh_of(6)
    alpha2, q2 = FIELDS["mixed"](mesh)
    ch_a = np.stack([mesh.alpha * 0.5, mesh.alpha * 2.0])
    ch_q = np.stack([mesh.q, mesh.q * 3.0])
    with api.Context(devices=(0,), lib=lib) as fresh, api.Context(devices=(0,), lib=lib) as upd:
        fresh.upload_mesh(mesh.points, mesh.tets, alpha2, q2)
        upd.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        for c in (fresh, upd):
            c.upload_solids(solids()[0], True)
            c.upload_solids(solids()[1], False)
            c.upload_channels(ch_a, ch_q)
        sib = upd.sibling()
        try:
            for limit in (2.5, 1.0):  # the first render prepares cells for 2.5 before the update
                v = api.make_view(RES[0], RES[1], lib=lib, alpha_limit=limit, round_through_float=0, **VIEWS["axis"])
                if limit == 2.5:
                    upd.render_raw(v)
                    sib.render_raw(v)
                    upd.update_fields(alpha2, q2)
                want = fresh.render_raw(v)
                want_ch = fresh.render_channels(v)[0]
                for c in (upd, sib):
                    got = c.render_raw(v)
                    assert np.array_equal(got.image, want.image, equal_nan=True)
                    assert np.array_equal(got.steps, want.steps) and np.array_equal(got.solid, want.solid)
                    assert np.array_equal(c.render_channels(v)[0], want_ch, equal_nan=True)
        finally:
            sib.close()


# ---- torch ---------------------------------------------------------------------------------------------

def test_torch_gradcheck(hostsim_lib):
    torch = pytest.importorskip("torch")
    from course5_b200 import autograd
    mesh = synth.kuhn_cube(3, seed=7)
    with api.Context(devices=(0,), lib=hostsim_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        view = api.make_view(24, 18, lib=hostsim_lib, alpha_limit=NO_LIMIT, use_solids=0, **VIEWS["generic"])
        alpha = torch.tensor(mesh.alpha, dtype=torch.float64, requires_grad=True)
        q = torch.tensor(mesh.q, dtype=torch.float64, requires_grad=True)
        assert torch.autograd.gradcheck(lambda a, b: autograd.render(ctx, view, a, b), (alpha, q), fast_mode=True,
                                        eps=1e-6, atol=1e-6, rtol=1e-5)


def test_torch_loss_with_solids_and_two_forwards(lib):
    torch = pytest.importorskip("torch")
    from course5_b200 import autograd
    ctx, mesh, view = small_ctx(lib)
    with ctx:
        a1 = torch.tensor(mesh.alpha, requires_grad=True)
        q1 = torch.tensor(mesh.q, requires_grad=True)
        img1 = autograd.render(ctx, view, a1, q1)
        solid = torch.isnan(img1[..., 0])
        assert solid.any()
        loss1 = torch.where(solid, 0.0, img1[..., 1]).pow(2).sum() + torch.where(solid, 0.0, img1[..., 0]).sum()
        # a second forward with other fields runs before the first backward
        a2 = torch.tensor(mesh.alpha * 3.0, requires_grad=True)
        q2 = torch.tensor(mesh.q * 0.5, requires_grad=True)
        loss2 = torch.where(solid, 0.0, autograd.render(ctx, view, a2, q2)[..., 1]).sum()
        loss1.backward()
        loss2.backward()
        assert torch.isfinite(a1.grad).all() and torch.isfinite(q1.grad).all()
        assert a1.grad.abs().sum() > 0 and q1.grad.abs().sum() > 0
        # the same gradient from a context that only ever saw the first fields
        g = np.zeros((RES[1], RES[0], 2))
        raw = np.where(solid.numpy(), 0.0, img1[..., 1].detach().numpy())
        g[..., 1] = 2.0 * raw
        g[..., 0] = np.where(solid.numpy(), 0.0, 1.0)
        ctx.update_fields(mesh.alpha, mesh.q)
        ga, gq = ctx.render_grad(view, g)
        assert np.allclose(a1.grad.numpy(), ga, rtol=1e-12, atol=1e-14 * np.abs(ga).max())
        assert np.allclose(q1.grad.numpy(), gq, rtol=1e-12, atol=1e-14 * np.abs(gq).max())


# ---- full size, devices, siblings (GPU) -------------------------------------------------------------------

@pytest.fixture(scope="module")
def c3(gpu_lib):
    """C3 at 2400 x 1800 with the reference's solids."""
    mesh, view_kw = synth.make_config("C3")
    ctx = api.Context(devices=(0,), lib=gpu_lib)
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    roche, sphere = solids()
    ctx.upload_solids(roche, True)
    ctx.upload_solids(sphere, False)
    res_x, res_y = view_kw.pop("res_x"), view_kw.pop("res_y")
    view = api.make_view(res_x, res_y, lib=gpu_lib, round_through_float=0, **view_kw)
    yield ctx, mesh, view
    ctx.close()


def rel_close(a, b, rel):
    return abs(a - b) <= rel * max(abs(a), abs(b))


@pytest.mark.gpu
def test_full_size_identities(c3):
    """I is linear in Q and tau in alpha: sum_t grad_q q = sum_p g_I I, and with g_I = 0,
    sum_t grad_alpha alpha = sum_p g_tau tau; a central difference along a random alpha direction, taken
    through update_fields and render_raw, agrees with <grad_alpha, v>."""
    ctx, mesh, view = c3
    rng = np.random.default_rng(3)
    raw = ctx.render_raw(view)
    assert raw.solid.sum() > 0 and raw.stats["grazing_rays"] > 0
    live = ~raw.solid.astype(bool)
    g = rng.normal(size=(view.res_y, view.res_x, 2))
    g[~live] = np.nan
    ga, gq, img = ctx.render_grad(view, g, image=True)
    assert np.array_equal(img, raw.image, equal_nan=True)
    lhs, rhs = float(np.dot(gq, mesh.q)), float(np.sum(g[..., 1][live] * raw.inten[live]))
    assert rel_close(lhs, rhs, 1e-12), (lhs, rhs)
    g_tau = g.copy()
    g_tau[..., 1] = 0.0
    ga_tau, _ = ctx.render_grad(view, g_tau, q=False)
    lhs, rhs = float(np.dot(ga_tau, mesh.alpha)), float(np.sum(g[..., 0][live] * raw.tau[live]))
    assert rel_close(lhs, rhs, 1e-12), (lhs, rhs)
    g0 = np.where(np.isnan(g), 0.0, g)
    d = rng.normal(size=mesh.n_tets) * mesh.alpha
    # the clamp is a kink of I(alpha): cells within reach of it would put the central difference across it
    d[np.abs(mesh.alpha - view.alpha_limit) < 1e-3 * view.alpha_limit] = 0.0
    h = 1e-6
    try:
        ctx.update_fields(mesh.alpha + h * d, mesh.q)
        plus = ctx.render_raw(view).image
        ctx.update_fields(mesh.alpha - h * d, mesh.q)
        minus = ctx.render_raw(view).image
    finally:
        ctx.update_fields(mesh.alpha, mesh.q)
    fd = float(np.sum(np.where(live[..., None], (plus - minus) / (2 * h) * g0, 0.0)))
    an = float(np.dot(ga, d))
    assert rel_close(fd, an, 1e-6), (fd, an)
    print(f"C3 identities: Q {lhs:.6e}; central difference {fd:.9e} vs {an:.9e}")


def test_bands_devices_and_siblings(lib, request):
    """Two row bands add up to the whole view; a context over devices (0, 0) and a sibling equal a
    single device; update_fields reaches the parts and the sibling."""
    gpu = "gpu" in request.node.callspec.id
    mesh = mesh_of(10 if gpu else 6)
    alpha2, q2 = FIELDS["mixed"](mesh)
    res_x, res_y = (480, 360) if gpu else RES
    view = api.make_view(res_x, res_y, lib=lib, round_through_float=0, **VIEWS["axis"])
    rng = np.random.default_rng(5)
    g = rng.normal(size=(res_y, res_x, 2))
    roche, sphere = solids()

    def close(a, b):
        for x, y in zip(a, b):
            assert np.allclose(x, y, rtol=1e-13, atol=1e-13 * np.abs(y).max())

    with api.Context(devices=(0,), lib=lib) as one, api.Context(devices=(0, 0), lib=lib) as two, \
            api.Context(devices=(0,), lib=lib) as fresh:
        for c in (one, two):
            c.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
            c.upload_solids(roche, True)
            c.upload_solids(sphere, False)
            c.render_raw(view)
            c.update_fields(alpha2, q2)
        fresh.upload_mesh(mesh.points, mesh.tets, alpha2, q2)
        fresh.upload_solids(roche, True)
        fresh.upload_solids(sphere, False)
        want = fresh.render_raw(view).image
        whole = one.render_grad(view, g)
        parts = []
        for rows in ((0, res_y // 2 - 7), (res_y // 2 - 7, res_y)):
            v = api.View.from_buffer_copy(view)
            v.row_begin, v.row_end = rows
            parts.append(one.render_grad(v, g))
        close((parts[0][0] + parts[1][0], parts[0][1] + parts[1][1]), whole)
        ga2, gq2, img2 = two.render_grad(view, g, image=True)
        assert two.last_stats["n_devices"] == 2
        assert np.array_equal(img2, want, equal_nan=True)
        assert np.array_equal(two.render_raw(view).image, want, equal_nan=True)
        close((ga2, gq2), whole)
        sib = one.sibling()
        try:
            ga3, gq3, img3 = sib.render_grad(view, g, image=True)
            assert np.array_equal(img3, want, equal_nan=True)
            close((ga3, gq3), whole)
        finally:
            sib.close()
