"""Logic of the device functions on CPU: tests/hostsim/libc5hostsim.so is the product's own
translation units compiled with -DC5_HOSTSIM (kernel bodies as host loops). It is never loaded by
the package and is not a fallback; it lets the container without a GPU check the walk, the BVH,
the topology build and the C ABI plumbing against the oracle. The parity tests proper are the
`-m gpu` ones in test_gpu_parity.py."""
import numpy as np
import pytest

import render_checks as rc
from cases import GOLDEN_CASES
from course5_b200 import synth


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden(hostsim_lib, name):
    rc.check_golden(hostsim_lib, name)


@pytest.mark.parametrize("flags", [dict(X=0.0, Y=0.0), dict(X=0.4, Y=0.7, I=-0.03, alpha_limit=1.2),
                                   dict(X=0.5, Y=1.9, I=0.3)])
def test_against_port(hostsim_lib, port, flags):
    rc.check_against_port(hostsim_lib, port, synth.kuhn_cube(10, seed=41), 200, 150, flags)


def test_cavity_reentry(hostsim_lib, port):
    mesh = synth.kuhn_cube(12, seed=42, scalars="sphere", carve_sphere=True)
    img, want = rc.check_against_port(hostsim_lib, port, mesh, 160, 120, dict(X=0.2, Y=0.3))
    assert want.steps.max() > 0


def test_grazing_rays(hostsim_lib, port):
    rc.check_grazing_rays(hostsim_lib, port)


def test_search_budget(hostsim_lib, port):
    rc.check_search_budget(hostsim_lib, port)


def test_submit_wait_lanes(hostsim_lib):
    rc.check_submit_wait(hostsim_lib)


def test_misaligned_output_is_rejected_or_copied(hostsim_lib):
    rc.check_output_alignment(hostsim_lib)


def test_graded_mesh(hostsim_lib, port):
    rc.check_against_port(hostsim_lib, port, synth.kuhn_cube(9, seed=43, grade_beta=1.5), 160, 120,
                          dict(X=0.45, Y=1.2))


def test_row_bands(hostsim_lib):
    rc.check_row_bands_equal_full_image(hostsim_lib)


def test_round_through_float(hostsim_lib):
    rc.check_round_through_float(hostsim_lib)


def test_out_of_window(hostsim_lib):
    rc.check_out_of_window_geometry_is_background(hostsim_lib)


def test_topology_errors(hostsim_lib):
    rc.check_topology_errors(hostsim_lib)


def test_tiny_meshes(hostsim_lib, port):
    rc.check_single_tet_and_tiny_meshes(hostsim_lib, port)


def test_uniform_medium(hostsim_lib):
    rc.check_uniform_medium_kat(hostsim_lib)


def test_scaling_properties(hostsim_lib):
    rc.check_scaling_properties(hostsim_lib, synth.kuhn_cube(6, seed=44), 100, 76, dict(X=0.4, Y=0.5))


def test_multi_device_context(hostsim_lib):
    rc.check_multi_device_context(hostsim_lib, (0, 0, 0))


@pytest.mark.parametrize("flags", [dict(X=0.0, Y=0.0), dict(X=0.4, Y=0.7, I=-0.03, alpha_limit=1.2)])
def test_fp32_variant(hostsim_lib, port, flags):
    rc.check_fp32_variant(hostsim_lib, port, synth.kuhn_cube(12, seed=47), 240, 180, flags)


def test_solid_mask_high_resolution(hostsim_lib, port):
    rc.check_solid_mask_high_resolution(hostsim_lib, port, res=(800, 600), views=((0.4, 0.3, 0.0),))


def test_solid_mask_tile_sizes(hostsim_lib, port):
    rc.check_solid_mask_tile_sizes(hostsim_lib, port)


def test_static_solid_mask_cache(hostsim_lib, port):
    rc.check_static_solid_mask_cache(hostsim_lib, port)


def test_debug_set_rejects_unknown_keys(hostsim_lib):
    """Keys c5gpu.h does not list return C5_E_INVALID instead of being ignored; the first three
    selected kernel variants and a second stream that have been removed."""
    from course5_b200 import api
    with api.Context(lib=hostsim_lib) as ctx:
        for key in ("prep_priority", "graze_blocks", "mask_per_face", "no_such_key"):
            with pytest.raises(api.C5Error) as e:
                ctx.debug_set(key, 1)
            assert e.value.code == api.E_INVALID, key
        ctx.debug_set("query_budget", 0)  # a listed key is still accepted


def test_image_handles_and_host_register(hostsim_lib):
    """c5_image_create / open / close and c5_host_register bookkeeping (the CUDA IPC mapping itself
    needs two processes and two GPUs: test_gpu_dist.py)."""
    import ctypes as C
    from course5_b200 import api
    mesh = synth.kuhn_cube(6, seed=51)
    with api.Context(lib=hostsim_lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        v = api.make_view(64, 48, X=0.4, Y=0.2, lib=hostsim_lib)
        full, _ = ctx.render(v)
        ptr, handle = ctx.image_create(64 * 48 * 16)
        assert len(handle) == api.IPC_HANDLE_BYTES
        alias = ctx.image_open(handle)             # hostsim: the same process may "open" its own image
        band = api.View.from_buffer_copy(v)
        band.row_begin, band.row_end = 10, 30
        ctx.render_device(band, alias + 10 * 64 * 16, 0)
        got = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_double)), shape=(48, 64, 2))
        assert np.array_equal(got[10:30], full[10:30])
        ctx.image_close(alias)
        ctx.image_close(ptr)
        with pytest.raises(api.C5Error):
            ctx.image_close(ptr)
        out = np.zeros((48, 64, 2))
        ctx.host_register(out)
        ctx.render(band, out=out)
        assert np.array_equal(out[10:30], full[10:30]) and not out[:10].any()
        ctx.host_unregister(out)
        with pytest.raises(api.C5Error):
            ctx.host_unregister(out)


def test_sibling_context_shares_the_mesh(hostsim_lib):
    rc.check_sibling_context(hostsim_lib)
