"""Views in flight on several lanes: each view's prologue (rotation, BVH refit, solid mask, ray order) and grazing-ray
kernel run on the lane's high-priority side stream, its pixel kernel on the lane's own stream (enqueue_view). Views
that differ in angle, band and pixel grid, dealt to 2 and 4 lanes, must give the same bits as the same views rendered
one at a time: a grazing-ray kernel that read the next view's rotated vertices or BVH boxes, or a pixel kernel that
started before its mask or ray order, would change pixels, counters or per-row costs."""
import numpy as np
import pytest

from course5_b200 import api, hostlib, synth

COUNTS = ("tet_steps", "hit_pixels", "solid_pixels", "walk_errors", "grazing_rays")


@pytest.fixture(scope="module")
def scene():
    mesh = synth.kuhn_cube(40, seed=3)
    roche, sphere = hostlib.make_solids(0.0)
    return mesh, roche, sphere


def context(gpu_lib, scene):
    mesh, roche, sphere = scene
    ctx = api.Context(devices=(0,), lib=gpu_lib)
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    ctx.upload_solids(roche, True)
    ctx.upload_solids(sphere, False)
    return ctx


def views(gpu_lib):
    """Consecutive views differ: the angle turns, the band moves, one has another pixel grid."""
    out = []
    for k in range(12):
        band = {} if k % 3 == 0 else dict(row_begin=40 * (k % 4), row_end=480 - 30 * (k % 5))
        res = (512, 384) if k == 7 else (640, 480)
        if band and band["row_end"] > res[1]:
            band["row_end"] = res[1]
        out.append(api.make_view(*res, X=0.3 + 0.04 * k, Y=0.1 + 0.05 * (k % 5), I=-0.03, alpha_limit=2.5,
                                 round_through_float=0, lib=gpu_lib, **band))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [2, 4])
def test_views_in_flight_match_views_one_at_a_time(gpu_lib, scene, lanes):
    seq = views(gpu_lib)
    single = context(gpu_lib, scene)
    piped = context(gpu_lib, scene)
    try:
        want = []
        for v in seq:
            img, st = single.render(v)
            want.append((img, {k: st[k] for k in COUNTS}, single.last_row_cost(v.res_y)))
        piped.set_views_in_flight(lanes)
        imgs = [np.zeros((v.res_y, v.res_x, 2)) for v in seq]
        tickets, got = [], []
        for k, v in enumerate(seq):
            if k >= lanes:                                  # keep `lanes` views in flight
                st = piped.render_wait(tickets[k - lanes])
                got.append(({c: st[c] for c in COUNTS}, piped.last_row_cost(seq[k - lanes].res_y)))
            tickets.append(piped.render_submit(v, imgs[k]))
        for k in range(len(seq) - lanes, len(seq)):
            st = piped.render_wait(tickets[k])
            got.append(({c: st[c] for c in COUNTS}, piped.last_row_cost(seq[k].res_y)))
        for k, (v, (img, counts, rows)) in enumerate(zip(seq, want)):
            assert counts["tet_steps"] > 0 and counts["solid_pixels"] > 0, k
            assert np.array_equal(imgs[k].view(np.uint64), img.view(np.uint64)), f"view {k}: image"
            assert got[k][0] == counts, f"view {k}: counters"
            assert np.array_equal(got[k][1], rows), f"view {k}: row costs"
    finally:
        piped.close()
        single.close()
