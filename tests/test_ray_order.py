"""The pixel kernels take each region's rays in an order sorted by the tet-steps the previous view took at each
pixel (order_rays in c5_walk.cu). Only the map from pixels to threads changes, so every image, per-pixel step
count, counter and per-row cost must be the same bits as with c5_debug_set("no_ray_order", 1) (the Morton order),
whichever view the order was made from; gradients, summed with atomics, agree to rounding.
The order itself (c5_debug_ray_order, on the host) is a stable sort by (bucket, Morton index)."""
import numpy as np
import pytest

from course5_b200 import api, hostlib, synth

COUNTS = ("tet_steps", "hit_pixels", "solid_pixels", "walk_errors", "grazing_rays")


def ray_order(lib, cost):
    """(order, bucket) of one region whose pixels cost cost[y, x] steps."""
    side = int(np.sqrt(cost.size))
    cost = np.ascontiguousarray(cost, dtype=np.uint16)
    order = np.zeros(side * side, dtype=np.uint16)
    bucket = np.zeros(side * side, dtype=np.int32)
    rc = lib.c5_debug_ray_order(cost.ctypes.data, order.ctypes.data, bucket.ctypes.data)
    assert rc == side
    return order, bucket


def morton_xy(m):
    m = np.asarray(m, dtype=np.int64)
    x = sum(((m >> (2 * b)) & 1) << b for b in range(8))
    y = sum(((m >> (2 * b + 1)) & 1) << b for b in range(8))
    return x, y


def region_side(lib):
    zeros = np.zeros(64 * 64, dtype=np.uint16)           # larger than any region
    order = np.zeros(64 * 64, dtype=np.uint16)
    bucket = np.zeros(64 * 64, dtype=np.int32)
    return lib.c5_debug_ray_order(zeros.ctypes.data, order.ctypes.data, bucket.ctypes.data)


def stable_sort(bucket):
    return np.lexsort((np.arange(bucket.size), bucket)).astype(np.uint16)


def warp_steps(cost_m, order):
    """The sum over warps of the order of the most steps a ray of the warp takes."""
    return int(cost_m[order].reshape(-1, 32).max(axis=1).sum())


@pytest.mark.parametrize("kind", ["equal", "zero", "even", "lattice", "random", "wide", "saturated"])
def test_order_is_morton_or_a_stable_sort_by_bucket(hostsim_lib, kind):
    side = region_side(hostsim_lib)
    assert side * side % 128 == 0
    rng = np.random.default_rng(5)
    y, x = np.mgrid[0:side, 0:side]
    cost = {
        "equal": np.full((side, side), 361),
        "zero": np.zeros((side, side)),
        "even": 356 + (rng.random((side, side)) < 0.02),                      # a sort saves < 1 % of the warp steps
        "lattice": np.where((x % 9 < 2) | (y % 9 < 3), 400 + 7 * (x % 3), 356) * (x + y > 6),
        "random": rng.integers(0, 500, size=(side, side)),
        "wide": rng.integers(0, 65536, size=(side, side)),
        "saturated": np.where(rng.random((side, side)) < 0.5, 65535, 300),
    }[kind].astype(np.uint16)
    order, bucket = ray_order(hostsim_lib, cost)
    assert np.array_equal(np.sort(order), np.arange(side * side))      # a permutation of the local Morton indices
    # the bucket is a non-decreasing function of the cost, and cost 0 is alone in bucket 0
    mx, my = morton_xy(np.arange(side * side))
    c_m = cost[my, mx].astype(np.int64)
    by_cost = np.lexsort((bucket, c_m))
    assert np.all(np.diff(bucket[by_cost]) >= 0)
    assert np.all((bucket == 0) == (c_m == 0))
    morton = np.arange(side * side, dtype=np.uint16)
    ranked = stable_sort(bucket)                                        # buckets ascend, Morton order inside one
    assert np.array_equal(order, morton) or np.array_equal(order, ranked)
    if not np.array_equal(order, morton):                               # sorted only where it saves warp steps
        assert warp_steps(c_m, ranked) < warp_steps(c_m, morton)
    if kind in ("equal", "zero", "even"):                               # nothing to gain: the Morton order ...
        assert np.array_equal(order, morton)
        ox, oy = morton_xy(order)                                        # ... warps of 8 x 4, blocks of 16 x 8
        assert (ox[:32].max() + 1, oy[:32].max() + 1) == (8, 4)
        assert (ox[:128].max() + 1, oy[:128].max() + 1) == (16, 8)
    if kind in ("random", "saturated"):                                 # much to gain: the sort
        assert np.array_equal(order, ranked)


# ---- on the GPU: the same bits with and without the order ---------------------------------------------------

@pytest.fixture(scope="module")
def scene():
    mesh = synth.kuhn_cube(24, seed=11)
    roche, sphere = hostlib.make_solids(0.0)
    return mesh, roche, sphere


def two_contexts(gpu_lib, scene, *, solids=True):
    mesh, roche, sphere = scene
    out = []
    for no_order in (0, 1):
        ctx = api.Context(devices=(0,), lib=gpu_lib)
        ctx.debug_set("no_ray_order", no_order)
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        if solids:
            ctx.upload_solids(roche, True)
            ctx.upload_solids(sphere, False)
        out.append(ctx)
    return out


def same_raw(a, b, view):
    assert np.array_equal(a.image.view(np.uint64), b.image.view(np.uint64))
    assert np.array_equal(a.steps, b.steps)
    assert np.array_equal(a.solid, b.solid)
    assert {k: a.stats[k] for k in COUNTS} == {k: b.stats[k] for k in COUNTS}


def views_sequence(gpu_lib):
    """Views whose orders come from a different view each time: turning, a band that moves, a new resolution."""
    seq = []
    for k, (X, Y) in enumerate([(0.4, 0.3), (0.45, 0.32), (0.1, 0.7), (0.5, 0.0), (0.5, 0.0)]):
        seq.append(api.make_view(400, 300, X=X, Y=Y, I=-0.03, alpha_limit=2.5, round_through_float=0, lib=gpu_lib))
    seq.append(api.make_view(400, 300, X=0.5, Y=0.0, alpha_limit=2.5, round_through_float=0, lib=gpu_lib,
                             row_begin=40, row_end=170))
    seq.append(api.make_view(400, 300, X=0.5, Y=0.0, alpha_limit=2.5, round_through_float=0, lib=gpu_lib,
                             row_begin=120, row_end=300))
    seq.append(api.make_view(333, 251, X=0.42, Y=0.31, alpha_limit=2.5, round_through_float=0, lib=gpu_lib))
    seq.append(api.make_view(400, 300, X=0.42, Y=0.31, alpha_limit=2.5, round_through_float=0, lib=gpu_lib))
    return seq


@pytest.mark.gpu
@pytest.mark.parametrize("solids", [True, False])
def test_images_do_not_depend_on_the_order(gpu_lib, scene, solids):
    with_order, without = two_contexts(gpu_lib, scene, solids=solids)
    try:
        for view in views_sequence(gpu_lib):
            a, b = with_order.render_raw(view), without.render_raw(view)
            same_raw(a, b, view)
            assert a.stats["tet_steps"] > 0
            assert np.array_equal(with_order.last_row_cost(view.res_y), without.last_row_cost(view.res_y))
    finally:
        with_order.close()
        without.close()


@pytest.mark.gpu
def test_fp32_channels_depth_and_jvp_do_not_depend_on_the_order(gpu_lib, scene):
    mesh = scene[0]
    rng = np.random.default_rng(3)
    ch_a = np.stack([mesh.alpha, mesh.alpha * rng.uniform(0.5, 2.0, size=mesh.alpha.shape)])
    ch_q = np.stack([mesh.q, mesh.q * rng.uniform(0.5, 2.0, size=mesh.q.shape)])
    va = rng.normal(size=mesh.alpha.shape) * mesh.alpha
    vq = rng.normal(size=mesh.q.shape) * mesh.q
    with_order, without = two_contexts(gpu_lib, scene)
    try:
        for ctx in (with_order, without):
            ctx.upload_channels(ch_a, ch_q)
        for view in (views_sequence(gpu_lib)[k] for k in (0, 2, 5, 7)):   # turning, a band, a new resolution
            v32 = api.make_view(view.res_x, view.res_y, X=0.0, Y=0.0, lib=gpu_lib)
            v32.rot, v32.n_rot, v32.precision = view.rot, view.n_rot, 32
            v32.row_begin, v32.row_end = view.row_begin, view.row_end
            a, b = with_order.render_raw(v32), without.render_raw(v32)
            same_raw(a, b, v32)
            ca, cb = with_order.render_channels(view, raw=True), without.render_channels(view, raw=True)
            assert np.array_equal(ca[0].view(np.uint64), cb[0].view(np.uint64))
            assert np.array_equal(ca[1], cb[1])
            assert {k: ca[3][k] for k in COUNTS} == {k: cb[3][k] for k in COUNTS}
            ta, ia = with_order.render_jvp(view, va, vq, image=True)
            tb, ib = without.render_jvp(view, va, vq, image=True)
            assert np.array_equal(ta.view(np.uint64), tb.view(np.uint64))
            assert np.array_equal(ia.view(np.uint64), ib.view(np.uint64))
            g = rng.normal(size=(view.res_y, view.res_x, 2))
            ga_a, gq_a, img_a = with_order.render_grad(view, g, image=True)    # the depth pass's image ...
            ga_b, gq_b, img_b = without.render_grad(view, g, image=True)
            assert np.array_equal(img_a.view(np.uint64), img_b.view(np.uint64))
            assert {k: with_order.last_stats[k] for k in COUNTS} == {k: without.last_stats[k] for k in COUNTS}
            for x, y in ((ga_a, ga_b), (gq_a, gq_b)):                          # ... and gradients to rounding
                scale = np.abs(y).max()
                assert scale > 0
                assert np.abs(x - y).max() <= 1e-12 * scale
    finally:
        with_order.close()
        without.close()


@pytest.mark.gpu
def test_lanes_keep_their_own_order(gpu_lib, scene):
    """render_submit deals consecutive views to the lanes, each of which orders by the view it rendered last."""
    with_order, without = two_contexts(gpu_lib, scene)
    try:
        views = views_sequence(gpu_lib)[:5]
        results = []
        for ctx in (with_order, without):
            ctx.set_views_in_flight(2)
            imgs = [np.zeros((v.res_y, v.res_x, 2)) for v in views]
            tickets = [ctx.render_submit(v, img) for v, img in zip(views[:2], imgs[:2])]
            for k in range(2, len(views)):                    # one view in flight beside the one waited for
                counts = ctx.render_wait(tickets[k - 2])
                assert counts["tet_steps"] > 0
                tickets.append(ctx.render_submit(views[k], imgs[k]))
            for t in tickets[-2:]:
                ctx.render_wait(t)
            results.append(imgs)
        for x, y in zip(*results):
            assert np.array_equal(x.view(np.uint64), y.view(np.uint64))
    finally:
        with_order.close()
        without.close()


@pytest.mark.gpu
def test_device_order_is_the_host_order(gpu_lib, scene):
    """order_rays on the device deals every region as the host form does from the same step counts, and some
    regions of a view close to a lattice axis are sorted."""
    mesh, roche, sphere = scene
    ctx = api.Context(devices=(0,), lib=gpu_lib)
    try:
        ctx.debug_set("query_budget", 1 << 20)   # no ray deferred: the map holds each ray's whole step count
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        view = api.make_view(400, 300, X=0.45, Y=0.05, alpha_limit=2.5, lib=gpu_lib)   # no wall seen edge-on
        first = ctx.render_raw(view)
        assert first.stats["grazing_rays"] == 0
        ctx.render_raw(view)                     # ordered by the first render's steps
        cost = np.minimum(first.steps, 65535).astype(np.uint16)
        side = region_side(gpu_lib)
        order = np.zeros(side * side, dtype=np.uint16)
        origin = np.zeros(2, dtype=np.int32)
        n = np.zeros(1, dtype=np.int32)
        sorted_regions = 0
        r = 0
        while True:
            rc = gpu_lib.c5_debug_ray_order_read(ctx._h, r, order.ctypes.data, origin.ctypes.data_as(api._i32p),
                                                 n.ctypes.data_as(api._i32p))
            assert rc == api.OK
            x0, y0 = origin
            patch = np.zeros((side, side), dtype=np.uint16)   # pixels past the image cost 0
            c = cost[y0:y0 + side, x0:x0 + side]
            patch[:c.shape[0], :c.shape[1]] = c
            want, _ = ray_order(gpu_lib, patch)
            assert np.array_equal(order, want), (r, x0, y0)
            sorted_regions += not np.array_equal(order, np.arange(side * side))
            r += 1
            if r == n[0]:
                break
        assert n[0] > 50 and sorted_regions > 0
    finally:
        ctx.close()
