"""Multi-channel rendering (c5_upload_channels / c5_render_channels): several pairs of cell fields
integrated along each ray in one walk. Every check runs on the host-loop build of the device code
(tests/hostsim) and, with -m gpu, on the CUDA library; the full-size checks are GPU only.

Channel c must be the image a plain render gives for a mesh uploaded with (alpha_c, q_c): the same
rays, hit set, solid mask and steps, values within the parity gate of tests/parity.py."""
import numpy as np
import pytest

from cases import reference_solids
from course5_b200 import api, synth
from parity import assert_image_parity, assert_same_hits

LIBS = [pytest.param("hostsim_lib", id="hostsim"), pytest.param("gpu_lib", id="gpu", marks=pytest.mark.gpu)]
PORT_VIEWS = [dict(X=0.0, Y=0.0), dict(X=0.4, Y=0.7, I=-0.03, alpha_limit=1.2), dict(X=0.5, Y=1.9, I=0.3)]


@pytest.fixture(params=LIBS)
def lib(request):
    return request.getfixturevalue(request.param)


def fields(mesh, n, seed):
    """n seeded channel pairs (alpha in [0, 4), some below DBL_EPSILON and some above any limit)."""
    rng = np.random.default_rng(seed)
    alpha = rng.uniform(0.0, 4.0, (n, mesh.n_tets))
    alpha[:, ::17] = 0.0
    q = rng.uniform(0.1, 4.0, (n, mesh.n_tets))
    return alpha, q


def channel_context(lib, mesh, alpha, q, *, solids=None, debug=None, devices=(0,)):
    ctx = api.Context(devices=devices, lib=lib)
    for key, value in (debug or {}).items():
        ctx.debug_set(key, value)
    ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
    if solids is not None:
        ctx.upload_solids(solids[0], True)
        ctx.upload_solids(solids[1], False)
    ctx.upload_channels(alpha, q)
    return ctx


def view_of(lib, res, flags, **over):
    return api.make_view(res[0], res[1], lib=lib, **{"round_through_float": 0, **flags, **over})


def check_channels_against_port(port, mesh, alpha, q, img, steps, solid, stats, res, flags, solids=None):
    for c in range(alpha.shape[0]):
        want = port.render(mesh.tet_points(), alpha[c], q[c], res_x=res[0], res_y=res[1],
                           solid_rot=None if solids is None else solids[0],
                           solid_static=None if solids is None else solids[1], **flags)
        assert want.anomalies == 0
        assert np.array_equal(solid, want.solid), f"channel {c}: solid mask"
        assert_same_hits(steps, want.steps, what=f"channel {c}: ")
        assert np.array_equal(steps, want.steps), f"channel {c}: steps"
        assert_image_parity(img[:, :, c, 0], img[:, :, c, 1], want.tau, want.inten, what=f"channel {c}: ")
    assert stats["tet_steps"] == int(steps.sum())
    assert stats["walk_errors"] == 0


def plain_render(lib, mesh, a, q, view, *, solids=None, debug=None):
    with api.Context(devices=(0,), lib=lib) as one:
        for key, value in (debug or {}).items():
            one.debug_set(key, value)
        one.upload_mesh(mesh.points, mesh.tets, a, q)
        if solids is not None:
            one.upload_solids(solids[0], True)
            one.upload_solids(solids[1], False)
        return one.render_raw(view)


# ---- parity with the oracle ------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 3, 8])
def test_channels_against_port(lib, port, n):
    mesh = synth.kuhn_cube(10, seed=41)
    alpha, q = fields(mesh, n, seed=100 + n)
    res = (200, 150)
    with channel_context(lib, mesh, alpha, q) as ctx:
        for flags in PORT_VIEWS:
            img, steps, solid, st = ctx.render_channels(view_of(lib, res, flags), raw=True)
            assert img.shape == (150, 200, n, 2)
            check_channels_against_port(port, mesh, alpha, q, img, steps, solid, st, res, flags)


def test_channels_equal_plain_renders(lib):
    """Channel c against c5_render_raw of a context uploaded with (alpha_c, q_c): the same steps,
    mask and counts, and the same bits (both walks evaluate the same expressions in the same order)."""
    mesh = synth.kuhn_cube(9, seed=42)
    alpha, q = fields(mesh, 3, seed=7)
    alpha[1], q[1] = mesh.alpha, mesh.q
    v = view_of(lib, (160, 120), dict(X=0.4, Y=0.7, I=-0.03, alpha_limit=1.2))
    with channel_context(lib, mesh, alpha, q) as ctx:
        img, steps, solid, st = ctx.render_channels(v, raw=True)
        own = ctx.render_raw(v)
    assert np.array_equal(own.image, img[:, :, 1])
    for c in range(3):
        want = plain_render(lib, mesh, alpha[c], q[c], v)
        assert np.array_equal(steps, want.steps) and np.array_equal(solid, want.solid)
        for key in ("tet_steps", "hit_pixels", "solid_pixels", "grazing_rays", "pixels"):
            assert st[key] == want.stats[key], key
        assert_image_parity(img[:, :, c, 0], img[:, :, c, 1], want.tau, want.inten, what=f"channel {c}: ")
        assert np.array_equal(img[:, :, c], want.image), f"channel {c} is not bitwise equal to a plain render"


def test_channels_grazing_rays_and_cavities(lib, port, request):
    """Deferred rays (edge-on jittered walls; a tiny search budget on a carved cavity) carry their
    channel values through the grazing-ray kernel's queue; shrinking its lists changes no bit."""
    gpu = "gpu" in request.node.callspec.id
    small = {"graze_list": 128} if gpu else {"serial_list": 5}
    mesh = synth.kuhn_cube(12, seed=48)
    alpha, q = fields(mesh, 3, seed=11)
    res = (240, 180)
    for flags in (dict(X=0.5, Y=0.0), dict(X=0.0, Y=0.5)):
        v = view_of(lib, res, flags)
        with channel_context(lib, mesh, alpha, q) as ctx:
            img, steps, solid, st = ctx.render_channels(v, raw=True)
        assert st["grazing_rays"] > 0
        check_channels_against_port(port, mesh, alpha, q, img, steps, solid, st, res, flags)
        with channel_context(lib, mesh, alpha, q, debug=small) as ctx:
            img2, steps2, _, st2 = ctx.render_channels(v, raw=True)
        assert st2["grazing_rays"] == st["grazing_rays"]
        assert np.array_equal(img2, img) and np.array_equal(steps2, steps)

    mesh = synth.kuhn_cube(10, seed=55, scalars="sphere", carve_sphere=True)
    alpha, q = fields(mesh, 2, seed=12)
    res, flags = (200, 150), dict(X=0.3, Y=0.4)
    with channel_context(lib, mesh, alpha, q) as ctx:
        base = ctx.render_channels(view_of(lib, res, flags), raw=True)[3]
    for budget in (3, 12):
        with channel_context(lib, mesh, alpha, q, debug={"query_budget": budget}) as ctx:
            img, steps, solid, st = ctx.render_channels(view_of(lib, res, flags), raw=True)
        assert st["grazing_rays"] > base["grazing_rays"]
        assert st["hit_pixels"] == base["hit_pixels"]
        check_channels_against_port(port, mesh, alpha, q, img, steps, solid, st, res, flags)


def test_channels_follow_alpha_limit(lib, port):
    mesh = synth.kuhn_cube(8, seed=43)
    alpha, q = fields(mesh, 3, seed=13)
    res = (120, 90)
    with channel_context(lib, mesh, alpha, q) as ctx:
        for limit in (1.2, 3.0, 1.2):
            flags = dict(X=0.4, Y=0.3, alpha_limit=limit)
            img, steps, solid, st = ctx.render_channels(view_of(lib, res, flags), raw=True)
            check_channels_against_port(port, mesh, alpha, q, img, steps, solid, st, res, flags)


def test_channel_row_bands(lib):
    mesh = synth.kuhn_cube(7, seed=31)
    alpha, q = fields(mesh, 3, seed=14)
    flags = dict(X=0.4, Y=0.9)
    with channel_context(lib, mesh, alpha, q) as ctx:
        full, st_full = ctx.render_channels(view_of(lib, (150, 110), flags))
        for lo, hi in ((0, 37), (37, 80), (80, 110), (50, 51)):
            out = np.full_like(full, -1.0)
            _, st = ctx.render_channels(view_of(lib, (150, 110), flags, row_begin=lo, row_end=hi), out=out)
            assert np.array_equal(out[lo:hi], full[lo:hi])
            assert np.all(out[:lo] == -1.0) and np.all(out[hi:] == -1.0)
            assert st["pixels"] == (hi - lo) * 150


def test_channel_solids_background_and_float_cast(lib):
    mesh = synth.kuhn_cube(6, seed=32)
    solids = reference_solids(0.0)
    alpha, q = fields(mesh, 4, seed=15)
    flags = dict(X=0.45, Y=0.3)
    with channel_context(lib, mesh, alpha, q, solids=solids) as ctx:
        raw, steps, solid, st = ctx.render_channels(view_of(lib, (100, 80), flags), raw=True)
        cast, _ = ctx.render_channels(view_of(lib, (100, 80), flags, round_through_float=1))
    assert solid.sum() > 0 and st["solid_pixels"] == int(solid.sum())
    assert np.isnan(raw[solid.astype(bool)]).all()
    background = (steps == 0) & ~solid.astype(bool)
    assert background.sum() > 0 and np.all(raw[background] == 0.0)
    assert not np.isnan(raw[~solid.astype(bool)]).any()
    assert np.array_equal(cast, raw.astype(np.float32).astype(np.float64), equal_nan=True)


def test_channel_errors(lib):
    mesh = synth.kuhn_cube(5, seed=35)
    alpha, q = fields(mesh, 2, seed=16)
    v = view_of(lib, (64, 48), dict(X=0.3, Y=0.2))
    with api.Context(devices=(0,), lib=lib) as ctx:
        with pytest.raises(api.C5Error) as e:                               # no mesh
            ctx.upload_channels(alpha, q)
        assert e.value.code == api.E_STATE
        with pytest.raises(api.C5Error) as e:
            ctx.render_channels(v)
        assert e.value.code == api.E_STATE
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        with pytest.raises(api.C5Error) as e:                               # no channels
            ctx.render_channels(v)
        assert e.value.code == api.E_STATE
        d = alpha.ctypes.data_as(api._dp)
        assert ctx.lib.c5_upload_channels(ctx._h, None, d, 2) == api.E_INVALID
        assert ctx.lib.c5_upload_channels(ctx._h, d, None, 2) == api.E_INVALID
        assert ctx.lib.c5_upload_channels(ctx._h, d, d, -1) == api.E_INVALID
        assert ctx.lib.c5_upload_channels(ctx._h, d, d, api.MAX_CHANNELS + 1) == api.E_INVALID
        bytes_mesh = ctx.mesh_info().device_bytes
        ctx.upload_channels(alpha, q)
        assert ctx.mesh_info().device_bytes > bytes_mesh
        v32 = view_of(lib, (64, 48), dict(X=0.3, Y=0.2), precision=32)
        with pytest.raises(api.C5Error) as e:
            ctx.render_channels(v32)
        assert e.value.code == api.E_INVALID
        sib = ctx.sibling()
        try:
            with pytest.raises(api.C5Error) as e:                           # uploads go through the parent
                sib.upload_channels(alpha, q)
            assert e.value.code == api.E_STATE
            want, _ = ctx.render_channels(v)
            got, _ = sib.render_channels(v)                                 # the parent's channels
            assert np.array_equal(got, want)
            alpha2, q2 = fields(mesh, 3, seed=17)                           # ... also after a re-upload
            ctx.upload_channels(alpha2, q2)
            want, _ = ctx.render_channels(v)
            got, _ = sib.render_channels(v)
            assert got.shape[2] == 3 and np.array_equal(got, want)
        finally:
            sib.close()
        # a submitted view blocks the upload
        ctx.set_views_in_flight(1)
        out = np.zeros((48, 64, 2))
        t = ctx.render_submit(v, out)
        with pytest.raises(api.C5Error) as e:
            ctx.upload_channels(alpha, q)
        assert e.value.code == api.E_STATE
        ctx.render_wait(t)
        ctx.upload_channels(alpha[:0], q[:0])                               # n = 0 removes them
        assert ctx.mesh_info().device_bytes == bytes_mesh
        with pytest.raises(api.C5Error) as e:
            ctx.render_channels(v)
        assert e.value.code == api.E_STATE
        ctx.upload_channels(alpha, q)
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)        # a new mesh drops them
        assert ctx.n_channels == 0
        assert ctx.lib.c5_render_channels(ctx._h, api.C.byref(v), np.zeros(64 * 48 * 4).ctypes.data_as(api._dp),
                                          None, None, None) == api.E_STATE


def test_plain_renders_unaffected(lib):
    mesh = synth.kuhn_cube(7, seed=44)
    alpha, q = fields(mesh, 4, seed=18)
    v = api.make_view(120, 90, X=0.4, Y=0.2, lib=lib)
    with api.Context(devices=(0,), lib=lib) as ctx:
        ctx.upload_mesh(mesh.points, mesh.tets, mesh.alpha, mesh.q)
        before, st_before = ctx.render(v)
        ctx.upload_channels(alpha, q)
        ctx.render_channels(v)
        after, st_after = ctx.render(v)
    assert np.array_equal(before, after)
    assert st_before["tet_steps"] == st_after["tet_steps"]


def test_multi_device_channels(lib):
    """A context over several devices (here (0, 0): two parts on one device) cuts row bands as for a
    plain render and gives the one-device image."""
    mesh = synth.kuhn_cube(8, seed=36)
    alpha, q = fields(mesh, 3, seed=19)
    views = [view_of(lib, (160, 120), dict(X=0.4, Y=y)) for y in (0.1, 0.8)]
    with channel_context(lib, mesh, alpha, q) as one:
        want = [one.render_channels(v, raw=True) for v in views]
    with channel_context(lib, mesh, alpha, q, devices=(0, 0)) as many:
        for v, w in zip(views, want):
            got = many.render_channels(v, raw=True)
            assert np.array_equal(got[0], w[0]) and np.array_equal(got[1], w[1]) and np.array_equal(got[2], w[2])
            assert got[3]["tet_steps"] == w[3]["tet_steps"] and got[3]["n_devices"] == 2


# ---- GPU only: benchmark sizes, page-locked images, distinct devices ---------------------------------

@pytest.mark.gpu
def test_config_c1_channels_with_reference_solids(gpu_lib, port):
    mesh, view = synth.make_config("C1")
    solids = reference_solids(view["D"])
    flags = dict(X=view["X"], Y=view["Y"], I=view["I"], alpha_limit=view["alpha_limit"])
    res = (view["res_x"], view["res_y"])
    alpha, q = fields(mesh, 4, seed=21)
    with channel_context(gpu_lib, mesh, alpha, q, solids=solids) as ctx:
        img, steps, solid, st = ctx.render_channels(view_of(gpu_lib, res, flags), raw=True)
    assert solid.sum() > 0
    check_channels_against_port(port, mesh, alpha, q, img, steps, solid, st, res, flags, solids=solids)


@pytest.mark.gpu
def test_config_c3_channels(gpu_lib):
    """C3 at 2400 x 1800: channel 0 = the mesh's own fields against c5_render_raw of the same context
    (equal stats counts); channels 1..3 each against a context uploaded with that pair."""
    mesh, view = synth.make_config("C3")
    flags = dict(X=view["X"], Y=view["Y"], I=view["I"], alpha_limit=view["alpha_limit"])
    alpha, q = fields(mesh, 4, seed=22)
    alpha[0], q[0] = mesh.alpha, mesh.q
    v = view_of(gpu_lib, (view["res_x"], view["res_y"]), flags)
    with channel_context(gpu_lib, mesh, alpha, q) as ctx:
        img, steps, solid, st = ctx.render_channels(v, raw=True)
        own = ctx.render_raw(v)
    assert st["walk_errors"] == 0 and st["tet_steps"] > 3e8
    for key in ("tet_steps", "hit_pixels", "solid_pixels", "grazing_rays", "walk_errors", "pixels"):
        assert st[key] == own.stats[key], key
    assert np.array_equal(steps, own.steps)
    assert_image_parity(img[:, :, 0, 0], img[:, :, 0, 1], own.tau, own.inten, what="channel 0: ")
    assert np.array_equal(img[:, :, 0], own.image)
    del own
    for c in (1, 2, 3):
        want = plain_render(gpu_lib, mesh, alpha[c], q[c], v)
        assert np.array_equal(steps, want.steps)
        assert_image_parity(img[:, :, c, 0], img[:, :, c, 1], want.tau, want.inten, what=f"channel {c}: ")


@pytest.mark.gpu
def test_channels_page_locked_out(gpu_lib):
    torch = pytest.importorskip("torch")
    mesh = synth.kuhn_cube(9, seed=64)
    alpha, q = fields(mesh, 3, seed=23)
    v = view_of(gpu_lib, (160, 120), dict(X=0.4, Y=0.3))
    with channel_context(gpu_lib, mesh, alpha, q) as ctx:
        pageable, _ = ctx.render_channels(v)
        pinned = torch.zeros((120, 160, 3, 2), dtype=torch.float64).pin_memory().numpy()
        ctx.render_channels(v, out=pinned)
        assert np.array_equal(pinned, pageable)
        band = torch.full((120, 160, 3, 2), -1.0, dtype=torch.float64).pin_memory().numpy()
        ctx.render_channels(view_of(gpu_lib, (160, 120), dict(X=0.4, Y=0.3), row_begin=30, row_end=70), out=band)
        assert np.array_equal(band[30:70], pageable[30:70]) and np.all(band[:30] == -1.0) and np.all(band[70:] == -1.0)


@pytest.mark.gpu
def test_channels_distinct_devices(gpu_lib):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mesh = synth.kuhn_cube(8, seed=37)
    alpha, q = fields(mesh, 2, seed=24)
    v = view_of(gpu_lib, (160, 120), dict(X=0.4, Y=0.5))
    with channel_context(gpu_lib, mesh, alpha, q) as one:
        want = one.render_channels(v, raw=True)
    with channel_context(gpu_lib, mesh, alpha, q, devices=(0, 1)) as many:
        got = many.render_channels(v, raw=True)
    assert all(np.array_equal(g, w) for g, w in zip(got[:3], want[:3]))


# ---- course --channels: the .vti arrays and the command line ----------------------------------------

def write_vtk_with_channels(path, mesh, named):
    """The legacy grid of synth.write_legacy_vtk plus further CELL_DATA scalars {name: values}."""
    synth.write_legacy_vtk(path, mesh)
    with open(path, "ab") as f:
        for name, values in named.items():
            f.write(f"SCALARS {name} double 1\nLOOKUP_TABLE default\n".encode())
            np.savetxt(f, values, fmt="%.17g")


@pytest.mark.parametrize("mode", [dict(), dict(compress=True), dict(compress=True, base64=True)])
def test_vti_extra_arrays_decode_to_the_rendered_channels(hostsim_lib, tmp_path, mode):
    from course5_b200 import hostlib
    mesh = synth.kuhn_cube(6, seed=46)
    alpha, q = fields(mesh, 3, seed=25)
    v = view_of(hostsim_lib, (90, 70), dict(X=0.4, Y=0.3), round_through_float=1)
    with channel_context(hostsim_lib, mesh, alpha, q) as ctx:
        image, _ = ctx.render(v)
        chans, _ = ctx.render_channels(v)
    names = [f"a{c}:q{c}" for c in range(3)]
    plain, extra = str(tmp_path / "plain.vti"), str(tmp_path / "extra.vti")
    hostlib.write_vti(plain, image, **mode)
    hostlib.write_vti(extra, image, extra={n: chans[:, :, c] for c, n in enumerate(names)}, **mode)
    assert np.array_equal(hostlib.read_vti(extra).tobytes(), hostlib.read_vti(plain).tobytes())
    for c, n in enumerate(names):
        got = hostlib.read_vti(extra, n)
        assert got.shape == (70, 90, 2)
        assert np.array_equal(got, chans[:, :, c], equal_nan=True)
    with pytest.raises(RuntimeError):
        hostlib.read_vti(extra, "missing:array")


def test_course_channels_flag_errors(tmp_path):
    import subprocess
    from course5_b200 import hostlib
    r, _, _ = hostlib.parse_cli(["-f", "a.vtk", "-d", "b.vti", "--channels", "A1:Q1,A2:Q2"])
    assert r == 0
    for bad in (["--channels", "A1"], ["--channels", "A1:Q1,"], ["--channels", ":Q"],
                ["--channels", ",".join(f"A{k}:Q{k}" for k in range(9))],
                ["--channels", "A1:Q1", "--frames", "3"]):
        r, text, _ = hostlib.parse_cli(["-f", "a.vtk", "-d", "b.vti"] + bad)
        assert r == 2 and "Error!" in text, bad
    # a missing array is reported with the array and the file, before any device work
    mesh = synth.kuhn_cube(3, seed=47)
    src = str(tmp_path / "grid.vtk")
    write_vtk_with_channels(src, mesh, {"A1": mesh.alpha, "Q1": mesh.q})
    p = subprocess.run([hostlib.COURSE_EXE, "-f", src, "-d", str(tmp_path / "o.vti"), "-x", "40", "-y", "30",
                        "--channels", "A1:Q1,A1:NoSuchQ"], capture_output=True, text=True)
    assert p.returncode != 0
    assert "NoSuchQ" in p.stderr and src in p.stderr


@pytest.mark.gpu
def test_course_channels_end_to_end(gpu_lib, tmp_path):
    """`course --channels`: ImageScalars byte-identical to a run without the flag, and each A:Q array
    equal to the channel render of that pair."""
    import subprocess
    from course5_b200 import hostlib
    mesh = synth.kuhn_cube(12, seed=61)
    alpha, q = fields(mesh, 2, seed=26)
    src = str(tmp_path / "grid.vtk")
    write_vtk_with_channels(src, mesh, {"A1": alpha[0], "Q1": q[0], "A2": alpha[1], "Q2": q[1]})
    args = ["-f", src, "-j4", "-x", "320", "-y", "240", "-X", "0.4", "-Y", "0.3", "-D", "0.1", "-I", "-0.03",
            "--alpha_limit", "2.0"]
    plain, chan = str(tmp_path / "plain.vti"), str(tmp_path / "chan.vti")
    p = subprocess.run([hostlib.COURSE_EXE, "-d", plain] + args, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    p = subprocess.run([hostlib.COURSE_EXE, "-d", chan, "--channels", "A1:Q1,AbsorpCoef:radEnLooseRate,A2:Q2"] + args,
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    image = hostlib.read_vti(chan)
    assert image.tobytes() == hostlib.read_vti(plain).tobytes()
    assert np.array_equal(hostlib.read_vti(chan, "AbsorpCoef:radEnLooseRate"), image, equal_nan=True)
    roche, sphere = reference_solids(0.1)
    v = api.make_view(320, 240, X=0.4, Y=0.3, I=-0.03, alpha_limit=2.0, lib=gpu_lib)
    with channel_context(gpu_lib, mesh, alpha, q, solids=(roche, sphere)) as ctx:
        want, _ = ctx.render_channels(v)
    from parity import float_ulp_distance
    for c, name in enumerate(("A1:Q1", "A2:Q2")):   # the gate of test_course_cli_end_to_end
        got = hostlib.read_vti(chan, name)
        nan = np.isnan(want[:, :, c])
        assert np.array_equal(np.isnan(got), nan)
        ulps = float_ulp_distance(got[~nan], want[:, :, c][~nan])
        assert ulps.max() <= 1 and (ulps > 0).mean() <= 1e-4, name
