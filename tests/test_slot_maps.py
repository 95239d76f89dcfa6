"""The walk's connectivity (c5_types.h): per tet a 32-byte Conn whose apex word for face k carries, besides
the neighbour's new vertex, the slots in the neighbour of this tet's vertices at slots (k + 1) & 3,
(k + 2) & 3 and (k + 3) & 3; per boundary face the slots in its tet of the face's vertices. The walk
tracks these slots instead of comparing vertex ids. Checked on the host-loop build against a brute-force
search of the tets' vertex ids, on the synthetic meshes and on a mesh whose tets list their vertices in
random order; and the upload's refusal of a mesh with more points than the packing holds."""
import ctypes as C

import numpy as np
import pytest

import render_checks as rc
from course5_b200 import api, synth

ID_BITS = 26
C5_MAX_POINTS = 1 << ID_BITS


def permuted(mesh, seed):
    """The same mesh with its points, its tets and the vertex order inside every tet shuffled."""
    rng = np.random.default_rng(seed)
    n_pts, n_tets = mesh.n_points, mesh.n_tets
    pt_perm = rng.permutation(n_pts)            # new point i is old point pt_perm[i]
    old_to_new = np.empty(n_pts, dtype=np.int64)
    old_to_new[pt_perm] = np.arange(n_pts)
    tet_perm = rng.permutation(n_tets)
    tets = old_to_new[mesh.tets[tet_perm]]
    slot_perm = np.argsort(rng.random((n_tets, 4)), axis=1)
    tets = np.take_along_axis(tets, slot_perm, axis=1).astype(np.int32)
    return synth.TetMesh(points=np.ascontiguousarray(mesh.points[pt_perm]), tets=tets,
                         alpha=np.ascontiguousarray(mesh.alpha[tet_perm]), q=np.ascontiguousarray(mesh.q[tet_perm]))


def topology(lib, mesh):
    lib.c5_hostsim_topology.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    with api.Context(devices=(0,), lib=lib) as ctx:
        info = ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        conn = np.zeros((mesh.n_tets, 8), dtype=np.int32)
        bfaces = np.zeros((info.n_boundary_faces, 8), dtype=np.int32)
        tperm = np.zeros(mesh.n_tets, dtype=np.uint32)
        assert lib.c5_hostsim_topology(ctx._h, conn.ctypes.data, bfaces.ctypes.data, tperm.ctypes.data) == 0
    return conn, bfaces, tperm


def check_slot_maps(lib, mesh):
    conn, bfaces, tperm = topology(lib, mesh)
    v = mesh.tets[tperm.astype(np.int64)]      # vertex ids (file numbering) of every tet, in Morton order
    nbr = conn[:, :4]
    apex = conn[:, 4:].view(np.uint32)
    ids = apex & np.uint32((1 << ID_BITS) - 1)
    maps = apex >> np.uint32(ID_BITS)
    file_to_dev = {}

    def same_vertex(file_id, dev_id):            # one device id per file id and back
        assert file_to_dev.setdefault(int(file_id), int(dev_id)) == int(dev_id)

    interior = 0
    for t in range(mesh.n_tets):
        for k in range(4):
            u = nbr[t, k]
            if u < 0:
                continue
            interior += 1
            face = {int(v[t, (k + j) & 3]) for j in (1, 2, 3)}
            assert len(set(int(x) for x in v[u]) & face) == 3, (t, k, u)
            for j in (1, 2, 3):
                slot = (int(maps[t, k]) >> (2 * (j - 1))) & 3
                want = [s for s in range(4) if v[u, s] == v[t, (k + j) & 3]]
                assert want == [slot], (t, k, j)
            apex_slot = [s for s in range(4) if int(v[u, s]) not in face]
            assert len(apex_slot) == 1
            same_vertex(v[u, apex_slot[0]], ids[t, k])
            assert nbr[u, apex_slot[0]] == t     # u reaches t back through the face opposite its apex
    assert interior > 0
    n_b = 0
    for bf in bfaces:
        a, b, c, tet, apex_id, slots = (int(x) for x in bf[:6])
        sa, sc, sb = slots & 3, (slots >> 2) & 3, (slots >> 4) & 3    # the walk's order a, c, b
        assert len({sa, sb, sc}) == 3 and slots >> 6 == 0
        for dev_id, s in ((a, sa), (b, sb), (c, sc)):
            same_vertex(v[tet, s], dev_id)
        k = 6 - sa - sb - sc
        same_vertex(v[tet, k], apex_id)
        assert nbr[tet, k] < 0                   # the face opposite the apex is on the boundary
        n_b += 1
    assert n_b + interior == 4 * mesh.n_tets
    assert len(set(file_to_dev.values())) == len(file_to_dev)


@pytest.mark.parametrize("make", [
    lambda: synth.kuhn_cube(5, seed=7),
    lambda: synth.kuhn_cube(6, seed=43, grade_beta=1.5),
    lambda: synth.kuhn_cube(7, seed=42, scalars="sphere", carve_sphere=True),
], ids=["kuhn", "graded", "cavity"])
def test_slot_maps_synthetic(hostsim_lib, make):
    check_slot_maps(hostsim_lib, make())


def test_slot_maps_random_permutation(hostsim_lib):
    check_slot_maps(hostsim_lib, permuted(synth.kuhn_cube(6, seed=11), seed=5))


def test_walk_on_randomly_ordered_tets(hostsim_lib, port):
    """Every slot order a tet can list its vertices in, through the walk, against the oracle."""
    mesh = permuted(synth.kuhn_cube(10, seed=41), seed=9)
    rc.check_against_port(hostsim_lib, port, mesh, 160, 120, dict(X=0.3, Y=0.2))


def test_upload_refuses_more_points_than_the_ids_hold(hostsim_lib):
    """C5_MAX_POINTS + 1 points are refused before any array is read, so the arrays can be tiny; the
    points beyond the first few do not exist."""
    mesh = synth.kuhn_cube(2, seed=3)
    lib = hostsim_lib
    with api.Context(devices=(0,), lib=lib) as ctx:
        for n_pts in (C5_MAX_POINTS + 1, 1 << 31):
            code = lib.c5_upload_mesh(ctx._h, mesh.points.ctypes.data_as(api._dp), n_pts,
                                      mesh.tets.ctypes.data_as(api._i32p), mesh.n_tets,
                                      mesh.alpha.ctypes.data_as(api._dp), mesh.q.ctypes.data_as(api._dp))
            assert code == api.E_INVALID
            assert b"C5_MAX_POINTS" in lib.c5_last_error(ctx._h)
        info = ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)  # the context is still usable
        assert info.n_points == mesh.n_points
