"""c5_update_fields_device, c5_render_grad_device, autograd on CUDA tensors and autograd.light_curve.

The device forms are held to the exact gradients of tests/test_gradients.py (same cases, same gate) and to
the host forms: bit for bit on the host-loop build (one thread adds in a fixed order), within 1e-12 of the
largest gradient on the GPU (FP64 atomics add in any order). On the host-loop build "device" memory is host
memory, so numpy arrays stand in for device buffers there; on the GPU they are torch CUDA tensors.
"""
import numpy as np
import pytest

import test_gradients as tg
from course5_b200 import api, synth

RES = tg.RES


class Mem:
    """Buffers the device forms read and write: CUDA tensors for the GPU library, numpy arrays for the
    host-loop build."""

    def __init__(self, gpu):
        self.gpu = gpu
        if gpu:
            import torch
            self.torch = torch

    def put(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        return self.torch.tensor(a, device="cuda") if self.gpu else a.copy()

    def empty(self, shape):
        if self.gpu:
            shape = shape if isinstance(shape, tuple) else (shape,)
            return self.torch.full(shape, float("nan"), dtype=self.torch.float64, device="cuda")
        return np.full(shape, np.nan)

    def ptr(self, x):
        if x is None:
            return 0
        return x.data_ptr() if self.gpu else x.ctypes.data

    def get(self, x):
        if x is None or not self.gpu:
            return x
        self.torch.cuda.synchronize()
        return x.cpu().numpy()


@pytest.fixture(params=tg.LIBS)
def env(request):
    return request.getfixturevalue(request.param), Mem(request.param == "gpu_lib")


@pytest.fixture(scope="module")
def oracle_port(port):
    return port


def band_of(view):
    return (0, view.res_y) if view.row_begin == 0 and view.row_end == 0 else (view.row_begin, view.row_end)


def grad_device(ctx, mem, view, g, *, alpha=True, q=True, out=False, stats=True):
    """c5_render_grad_device of g (the WHOLE image's upstream gradient; its band is handed over)."""
    rb, re = band_of(view)
    d_g = mem.put(np.asarray(g)[rb:re])
    ga = mem.empty(ctx.n_tets) if alpha else None
    gq = mem.empty(ctx.n_tets) if q else None
    o = mem.empty((re - rb, view.res_x, 2)) if out else None
    st = ctx.render_grad_device(view, mem.ptr(d_g), mem.ptr(ga), mem.ptr(gq), mem.ptr(o), stats=stats)
    return mem.get(ga), mem.get(gq), mem.get(o), st


def update_device(ctx, mem, alpha, q):
    a, b = mem.put(alpha), mem.put(q)
    ctx.update_fields_device(mem.ptr(a), mem.ptr(b))
    return a, b  # alive until the gather has run


def same_as_host(mem, got, want):
    """Bit for bit on the host-loop build, within 1e-12 max|want| on the GPU."""
    for a, b in zip(got, want):
        if mem.gpu:
            assert np.allclose(a, b, rtol=0.0, atol=1e-12 * np.abs(b).max())
        else:
            assert np.array_equal(a, b)


# ---- against the exact gradients and the host form -----------------------------------------------------

CASES = {  # meshes as in test_gradients, so that its exact gradients are shared
    "generic_1e-08": dict(mesh_key=(7, False), field="decade_1e-08", view="generic"),
    "generic_1": dict(mesh_key=(7, False), field="decade_1", view="generic"),
    "generic_1000": dict(mesh_key=(6, False), field="decade_1000", view="generic"),
    "axis_1": dict(mesh_key=(10, False), field="decade_1", view="axis"),
    "mixed_generic": dict(mesh_key=(8, False), field="mixed", view="generic"),
    "mixed_axis": dict(mesh_key=(8, False), field="mixed", view="axis"),
    "mixed_budget": dict(mesh_key=(8, False), field="mixed", view="axis", debug={"query_budget": 3}),
    "mixed_graze_list": dict(mesh_key=(8, False), field="mixed", view="axis",
                             debug={"graze_list": 128, "serial_list": 2}),
    "solids": dict(mesh_key=(8, False), field="decade_1", view="generic", with_solids=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_exact_and_host_form(env, oracle_port, record_property, case):
    lib, mem = env
    c = dict(CASES[case])
    debug = c.pop("debug", None)
    with_solids = c.get("with_solids", False)
    exact = tg.exact_grads(oracle_port, c["mesh_key"], c["field"], c["view"], tg.NO_LIMIT, "full", with_solids)
    mesh = tg.mesh_of(*c["mesh_key"])
    alpha, q = tg.FIELDS[c["field"]](mesh)
    g = tg.upstream("full")
    if with_solids:  # whatever g holds under the solid mask is not read
        g = g.copy()
        g[tg.segments_of(oracle_port, c["mesh_key"], c["view"], True)[1]] = np.nan
    with api.Context(devices=(0,), lib=lib) as ctx:
        for k, v in (debug or {}).items():
            ctx.debug_set(k, v)
        ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
        if with_solids:
            ctx.upload_solids(tg.solids()[0], True)
            ctx.upload_solids(tg.solids()[1], False)
        view = api.make_view(RES[0], RES[1], lib=lib, alpha_limit=tg.NO_LIMIT, round_through_float=0,
                             **tg.VIEWS[c["view"]])
        ga, gq, _, st = grad_device(ctx, mem, view, g)
        host = ctx.render_grad(view, g)
    assert st["walk_errors"] == 0
    if debug and "query_budget" in debug:
        assert st["grazing_rays"] > st["hit_pixels"] // 2
    tg.check_grads(record_property, f"device {case}", (ga, gq), exact)
    same_as_host(mem, (ga, gq), host)


def test_out_and_launch_counts(env):
    """d_out is render_raw's image bit for bit; the device gradient launches three kernels more than
    render_raw of the same view (the gradient pass's two and the scatter), the field update one."""
    lib, mem = env
    ctx, mesh, view = tg.small_ctx(lib)
    with ctx:
        ctx.render_raw(view)  # cells prepared for the view's alpha_limit
        n0 = ctx.kernel_launches()
        raw = ctx.render_raw(view)
        n_raw = ctx.kernel_launches() - n0
        g = tg.upstream("full")
        grad_device(ctx, mem, view, g)  # the resident permutation is made here
        n0 = ctx.kernel_launches()
        ga, gq, out, _ = grad_device(ctx, mem, view, g, out=True)
        assert ctx.kernel_launches() - n0 == n_raw + 3
        assert np.array_equal(out, raw.image, equal_nan=True)
        assert raw.solid.sum() > 0
        ga1, _, _, _ = grad_device(ctx, mem, view, g, q=False)
        _, gq1, _, _ = grad_device(ctx, mem, view, g, alpha=False)
        same_as_host(mem, (ga1, gq1), (ga, gq))
        n0 = ctx.kernel_launches()
        keep = update_device(ctx, mem, mesh.alpha, mesh.q)
        assert ctx.kernel_launches() - n0 == 1
        del keep


def test_row_bands_and_sibling(env):
    """Band-sized g and out: the bands' gradients add up to the whole view's and each band's out is its
    rows of the full image; a sibling gives the same gradients."""
    lib, mem = env
    ctx, mesh, view = tg.small_ctx(lib, n=6)
    g = tg.upstream("full")
    with ctx:
        raw = ctx.render_raw(view)
        whole = grad_device(ctx, mem, view, g)
        parts = []
        for rows in ((0, 29), (29, RES[1])):
            v = api.View.from_buffer_copy(view)
            v.row_begin, v.row_end = rows
            ga, gq, out, _ = grad_device(ctx, mem, v, g, out=True)
            assert np.array_equal(out, raw.image[rows[0]:rows[1]], equal_nan=True)
            parts.append((ga, gq))
        for k in range(2):
            summed = parts[0][k] + parts[1][k]
            assert np.allclose(summed, whole[k], rtol=1e-13, atol=1e-13 * np.abs(whole[k]).max())
        sib = ctx.sibling()
        try:
            ga, gq, out, _ = grad_device(sib, mem, view, g, out=True)
            assert np.array_equal(out, raw.image, equal_nan=True)
            same_as_host(mem, (ga, gq), whole[:2])
        finally:
            sib.close()


# ---- c5_update_fields_device ------------------------------------------------------------------------------

def test_update_fields_device_matches_a_fresh_upload(env):
    """render_raw, render_flux, render_channels, a submitted view and a sibling's render after the device
    update equal those of a fresh upload; device_bytes grows by 4 bytes per tet at the first device call only."""
    lib, mem = env
    mesh = tg.mesh_of(6)
    alpha2, q2 = tg.FIELDS["mixed"](mesh)
    ch_a = np.stack([mesh.alpha * 0.5, mesh.alpha * 2.0])
    ch_q = np.stack([mesh.q, mesh.q * 3.0])
    with api.Context(devices=(0,), lib=lib) as fresh, api.Context(devices=(0,), lib=lib) as upd:
        fresh.upload_mesh(mesh.points, mesh.tets, alpha2, q2)
        upd.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        for c in (fresh, upd):
            c.upload_solids(tg.solids()[0], True)
            c.upload_solids(tg.solids()[1], False)
            c.upload_channels(ch_a, ch_q)
        sib = upd.sibling()
        try:
            v = api.make_view(RES[0], RES[1], lib=lib, alpha_limit=2.5, round_through_float=0, **tg.VIEWS["axis"])
            upd.render_raw(v)
            sib.render_raw(v)
            before = upd.mesh_info().device_bytes
            keep = update_device(upd, mem, alpha2, q2)
            assert upd.mesh_info().device_bytes == before + 4 * mesh.n_tets
            keep2 = update_device(upd, mem, alpha2, q2)
            assert upd.mesh_info().device_bytes == before + 4 * mesh.n_tets
            want = fresh.render_raw(v)
            want_flux = fresh.render_flux(v)
            want_ch = fresh.render_channels(v)[0]
            for c in (upd, sib):
                got = c.render_raw(v)
                assert np.array_equal(got.image, want.image, equal_nan=True)
                assert np.array_equal(got.steps, want.steps) and np.array_equal(got.solid, want.solid)
                assert np.array_equal(c.render_channels(v)[0], want_ch, equal_nan=True)
                flux = c.render_flux(v)
                assert np.array_equal(flux[0], want_flux[0]) and np.array_equal(flux[1], want_flux[1])
            img = np.zeros((RES[1], RES[0], 2))
            upd.render_wait(upd.render_submit(v, img))
            assert np.array_equal(img, want.image, equal_nan=True)
            # a new mesh drops the device permutation; the next device call makes it again
            upd.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
            plain = upd.mesh_info().device_bytes
            update_device(upd, mem, alpha2, q2)
            assert upd.mesh_info().device_bytes == plain + 4 * mesh.n_tets
            del keep, keep2
        finally:
            sib.close()


# ---- ordering without host synchronisation (GPU) -------------------------------------------------------------

def _fresh_ctx(lib, mesh, alpha, q):
    ctx = api.Context(devices=(0,), lib=lib)
    ctx.upload_mesh(mesh.points, mesh.tets, alpha, q)
    ctx.upload_solids(tg.solids()[0], True)
    ctx.upload_solids(tg.solids()[1], False)
    return ctx


@pytest.mark.gpu
def test_ordering_on_streams(gpu_lib):
    """A: an update on a torch side stream, held back by a long kernel, is seen by render_raw on the library's
    stream. B: render_grad_device without stats on a side stream, then a torch reduction on that stream, gives
    the synchronised result. C: update -> grad -> update -> grad on one stream gives each step's gradients."""
    import torch
    mesh = tg.mesh_of(8)
    alpha2, q2 = tg.FIELDS["mixed"](mesh)
    view = api.make_view(RES[0], RES[1], lib=gpu_lib, round_through_float=0, **tg.VIEWS["generic"])
    g = tg.upstream("full")
    with _fresh_ctx(gpu_lib, mesh, alpha2, q2) as fresh, _fresh_ctx(gpu_lib, mesh, mesh.alpha, mesh.q) as ctx:
        want = fresh.render_raw(view).image
        want_a, want_q = fresh.render_grad(view, g)
        ctx.render_raw(view)
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        # A
        with torch.cuda.stream(side):
            a = torch.tensor(alpha2, device="cuda")
            b = torch.tensor(q2, device="cuda")
            torch.cuda._sleep(200_000_000)  # ~0.1 s of device time before the gather
            ctx.update_fields_device(a.data_ptr(), b.data_ptr(), side.cuda_stream)
        assert np.array_equal(ctx.render_raw(view).image, want, equal_nan=True)
        # B
        with torch.cuda.stream(side):
            d_g = torch.tensor(g, device="cuda")
            ga = torch.empty(mesh.n_tets, dtype=torch.float64, device="cuda")
            gq = torch.empty_like(ga)
            torch.cuda._sleep(200_000_000)
            ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=side.cuda_stream,
                                   stats=False)
            sums = torch.stack([ga.abs().sum(), gq.abs().sum()]).cpu().numpy()
        for got, ref in zip(sums, (want_a, want_q)):
            assert abs(got - np.abs(ref).sum()) <= 1e-12 * np.abs(ref).sum()
        # C
        fields = [(mesh.alpha, mesh.q), (alpha2, q2)]
        wants = []
        for fa, fq in fields:
            with _fresh_ctx(gpu_lib, mesh, fa, fq) as f:
                wants.append(f.render_grad(view, g))
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            outs, keep = [], []
            for fa, fq in fields:
                a, b = torch.tensor(fa, device="cuda"), torch.tensor(fq, device="cuda")
                keep.append((a, b))
                ctx.update_fields_device(a.data_ptr(), b.data_ptr(), side.cuda_stream)
                ga = torch.empty(mesh.n_tets, dtype=torch.float64, device="cuda")
                gq = torch.empty_like(ga)
                ctx.render_grad_device(view, d_g.data_ptr(), ga.data_ptr(), gq.data_ptr(), stream=side.cuda_stream,
                                       stats=False)
                outs.append((ga, gq))
        side.synchronize()
        for (ga, gq), (wa, wq) in zip(outs, wants):
            assert np.allclose(ga.cpu().numpy(), wa, rtol=0.0, atol=1e-12 * np.abs(wa).max())
            assert np.allclose(gq.cpu().numpy(), wq, rtol=0.0, atol=1e-12 * np.abs(wq).max())


# ---- errors -----------------------------------------------------------------------------------------------

def test_errors(env):
    import ctypes as C
    lib, mem = env
    vp = C.c_void_p
    n = tg.mesh_of(5).n_tets
    ga, gq = mem.empty(n), mem.empty(n)
    g = mem.put(np.zeros((RES[1], RES[0], 2)))
    out = mem.empty((RES[1], RES[0], 2))
    pg, pa, pq, po = mem.ptr(g), mem.ptr(ga), mem.ptr(gq), mem.ptr(out)

    def upd(ctx, a=pa, q=pq):
        return lib.c5_update_fields_device(ctx._h, vp(a or None), vp(q or None), None)

    def grad(ctx, view, gg=pg, a=pa, q=pq, o=po):
        return lib.c5_render_grad_device(ctx._h, C.byref(view), vp(gg or None), vp(a or None), vp(q or None),
                                         vp(o or None), None, None)

    ctx, mesh, view = tg.small_ctx(lib)
    with api.Context(devices=(0,), lib=lib) as empty:
        assert upd(empty) == api.E_STATE
        assert grad(empty, view) == api.E_STATE
    with ctx:
        assert grad(ctx, view) == api.OK
        assert upd(ctx) == api.OK
        assert grad(ctx, view, gg=0) == api.E_INVALID
        assert grad(ctx, view, a=0, q=0) == api.E_INVALID
        assert grad(ctx, view, a=0) == api.OK and grad(ctx, view, q=0, o=0) == api.OK
        for kw in (dict(gg=pg + 4), dict(a=pa + 4), dict(q=pq + 4), dict(o=po + 4)):
            assert grad(ctx, view, **kw) == api.E_INVALID, kw
        for key, val in (("precision", 32), ("round_through_float", 1)):
            bad = api.View.from_buffer_copy(view)
            setattr(bad, key, val)
            assert grad(ctx, bad) == api.E_INVALID
        assert upd(ctx, a=0) == api.E_INVALID and upd(ctx, q=0) == api.E_INVALID
        assert upd(ctx, a=pa + 4) == api.E_INVALID and upd(ctx, q=pq + 4) == api.E_INVALID
        sib = ctx.sibling()
        try:
            assert upd(sib) == api.E_STATE
            assert grad(sib, view) == api.OK
        finally:
            sib.close()
        ctx.set_views_in_flight(2)
        t = ctx.render_submit(view, np.zeros((RES[1], RES[0], 2)))
        try:
            assert upd(ctx) == api.E_STATE
            assert grad(ctx, view) == api.E_STATE
        finally:
            ctx.render_wait(t)
    with api.Context(devices=(0, 0), lib=lib) as two:
        two.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        assert upd(two) == api.E_INVALID
        assert grad(two, view) == api.E_INVALID
    mem.get(ga)


# ---- autograd on CUDA tensors (GPU) ----------------------------------------------------------------------------

def _loss(img, solid):
    import torch
    return torch.where(solid, 0.0, img[..., 1]).pow(2).sum() + torch.where(solid, 0.0, img[..., 0]).sum()


@pytest.mark.gpu
def test_autograd_render_on_cuda(gpu_lib):
    """Forward equals render_raw bit for bit; backward equals the CPU-tensor path; two forwards before one
    backward; a row-band view."""
    import torch
    from course5_b200 import autograd
    ctx, mesh, view = tg.small_ctx(gpu_lib)
    with ctx:
        want = ctx.render_raw(view).image
        grads = {}
        for dev in ("cpu", "cuda"):
            a1 = torch.tensor(mesh.alpha, device=dev, requires_grad=True)
            q1 = torch.tensor(mesh.q, device=dev, requires_grad=True)
            img1 = autograd.render(ctx, view, a1, q1)
            assert img1.device.type == dev
            assert np.array_equal(img1.detach().cpu().numpy(), want, equal_nan=True)
            solid = torch.isnan(img1[..., 0])
            loss1 = _loss(img1, solid)
            a2 = torch.tensor(mesh.alpha * 3.0, device=dev, requires_grad=True)
            q2 = torch.tensor(mesh.q * 0.5, device=dev, requires_grad=True)
            loss2 = torch.where(solid, 0.0, autograd.render(ctx, view, a2, q2)[..., 1]).sum()
            loss1.backward()
            loss2.backward()
            grads[dev] = [t.grad.cpu().numpy() for t in (a1, q1, a2, q2)]
        for got, ref in zip(grads["cuda"], grads["cpu"]):
            assert np.isfinite(got).all() and np.abs(ref).max() > 0
            assert np.allclose(got, ref, rtol=0.0, atol=1e-12 * np.abs(ref).max())
        band = api.View.from_buffer_copy(view)
        band.row_begin, band.row_end = 20, 50
        a = torch.tensor(mesh.alpha, device="cuda", requires_grad=True)
        q = torch.tensor(mesh.q, device="cuda", requires_grad=True)
        img = autograd.render(ctx, band, a, q)
        assert np.array_equal(img[20:50].detach().cpu().numpy(), want[20:50], equal_nan=True)
        assert not img[:20].any() and not img[50:].any()
        _loss(img, torch.isnan(img[..., 0])).backward()
        g = np.zeros((RES[1], RES[0], 2))
        solid = np.isnan(want[..., 0])
        g[..., 1] = np.where(solid, 0.0, 2.0 * want[..., 1])
        g[..., 0] = np.where(solid, 0.0, 1.0)
        ctx.update_fields(mesh.alpha, mesh.q)
        wa, wq = ctx.render_grad(band, g)
        assert np.allclose(a.grad.cpu().numpy(), wa, rtol=0.0, atol=1e-12 * np.abs(wa).max())
        assert np.allclose(q.grad.cpu().numpy(), wq, rtol=0.0, atol=1e-12 * np.abs(wq).max())
        with pytest.raises(ValueError):
            autograd.render(ctx, view, a.detach().cpu(), q.detach())


@pytest.mark.gpu
def test_autograd_gradcheck_on_cuda(gpu_lib):
    import torch
    from course5_b200 import autograd
    mesh = synth.kuhn_cube(3, seed=7)
    with api.Context(devices=(0,), lib=gpu_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        view = api.make_view(24, 18, lib=gpu_lib, alpha_limit=tg.NO_LIMIT, use_solids=0, **tg.VIEWS["generic"])
        alpha = torch.tensor(mesh.alpha, device="cuda", requires_grad=True)
        q = torch.tensor(mesh.q, device="cuda", requires_grad=True)
        # the GPU adds the gradients with atomics: two backwards agree to rounding, not bit for bit
        assert torch.autograd.gradcheck(lambda a, b: autograd.render(ctx, view, a, b), (alpha, q), fast_mode=True,
                                        eps=1e-6, atol=1e-6, rtol=1e-5, nondet_tol=1e-12)


# ---- light curves -------------------------------------------------------------------------------------------

def _devices(mem):
    return ("cpu", "cuda") if mem.gpu else ("cpu",)


def _lc_views(lib, limit=2.5, use_solids=1):
    band = dict(row_begin=10, row_end=50)
    return [api.make_view(RES[0], RES[1], lib=lib, alpha_limit=limit, use_solids=use_solids, **tg.VIEWS["generic"]),
            api.make_view(RES[0], RES[1], lib=lib, alpha_limit=limit, use_solids=use_solids, **tg.VIEWS["axis"],
                          **band)]


def test_light_curve_forward_and_backward(env):
    """The forward is render_flux's totals bit for bit (solids and a row band included); the backward is the sum
    over views of render_grad against g filled with grad_output[k]."""
    import torch
    from course5_b200 import autograd
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=6)
    views = _lc_views(lib)
    w = np.random.default_rng(8).normal(size=(len(views), 2))
    with ctx:
        for dev in _devices(mem):
            a = torch.tensor(mesh.alpha, device=dev, requires_grad=True)
            q = torch.tensor(mesh.q, device=dev, requires_grad=True)
            lc = autograd.light_curve(ctx, views, a, q)
            assert lc.shape == (len(views), 2) and lc.device.type == dev
            (lc * torch.tensor(w, device=dev)).sum().backward()
            want_a, want_q = np.zeros(mesh.n_tets), np.zeros(mesh.n_tets)
            for k, v in enumerate(views):
                raw = api.View.from_buffer_copy(v)
                raw.round_through_float = 0
                assert np.array_equal(lc[k].detach().cpu().numpy(), ctx.render_flux(raw)[1][0])
                rb, re = band_of(raw)
                g = np.zeros((RES[1], RES[0], 2))
                g[rb:re] = w[k]
                ga, gq = ctx.render_grad(raw, g)
                want_a += ga
                want_q += gq
            for got, ref in ((a.grad, want_a), (q.grad, want_q)):
                assert np.abs(ref).max() > 0
                assert np.allclose(got.cpu().numpy(), ref, rtol=0.0, atol=1e-12 * np.abs(ref).max())


def test_light_curve_central_difference(env):
    """Along a random alpha and Q direction the totals' central difference agrees with <grad, v>."""
    import torch
    from course5_b200 import autograd
    lib, mem = env
    ctx, mesh, _ = tg.small_ctx(lib, n=5)
    views = _lc_views(lib, limit=tg.NO_LIMIT)
    rng = np.random.default_rng(21)
    w = rng.normal(size=(len(views), 2))
    da = rng.normal(size=mesh.n_tets) * mesh.alpha
    dq = rng.normal(size=mesh.n_tets) * mesh.q
    h = 1e-6
    with ctx:
        for dev in _devices(mem):
            t = lambda x: torch.tensor(x, device=dev)  # noqa: E731
            a = torch.tensor(mesh.alpha, device=dev, requires_grad=True)
            q = torch.tensor(mesh.q, device=dev, requires_grad=True)
            (autograd.light_curve(ctx, views, a, q) * t(w)).sum().backward()
            an = float(np.dot(a.grad.cpu().numpy(), da) + np.dot(q.grad.cpu().numpy(), dq))
            plus = autograd.light_curve(ctx, views, t(mesh.alpha + h * da), t(mesh.q + h * dq)).cpu().numpy()
            minus = autograd.light_curve(ctx, views, t(mesh.alpha - h * da), t(mesh.q - h * dq)).cpu().numpy()
            fd = float(np.sum(w * (plus - minus) / (2 * h)))
            assert abs(fd - an) <= 1e-6 * max(abs(fd), abs(an)), (dev, fd, an)


def test_light_curve_gradcheck(env):
    import torch
    from course5_b200 import autograd
    lib, mem = env
    mesh = synth.kuhn_cube(3, seed=7)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        views = [api.make_view(24, 18, lib=lib, alpha_limit=tg.NO_LIMIT, use_solids=0, **tg.VIEWS[k])
                 for k in ("generic", "axis")]
        for dev in _devices(mem):
            alpha = torch.tensor(mesh.alpha, device=dev, requires_grad=True)
            q = torch.tensor(mesh.q, device=dev, requires_grad=True)
            assert torch.autograd.gradcheck(lambda a, b: autograd.light_curve(ctx, views, a, b), (alpha, q),
                                            eps=1e-6, atol=1e-6, rtol=1e-5, nondet_tol=1e-12 if mem.gpu else 0.0)
