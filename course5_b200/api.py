"""ctypes binding of include/c5gpu.h and a small host-side mirror of the reference's objects.

The product path is CUDA only: :func:`load_library` opens ``course5_b200/libc5gpu.so`` and raises
if it is missing; :class:`Context` raises if no CUDA device is usable. There is no CPU fallback.

``Context`` wraps one ``c5_ctx``: ``upload_mesh`` / ``upload_solids`` are what main() builds before
its timed region (/root/reference/project/src/main.cpp:96-123: the grid from the VTK file, the
solid Roche lobe and sphere); ``render(view)`` is plane ctor + find_intersections + trace_rays
(main.cpp:127-129) for one set of CLI flags and returns the ``ImageScalars`` array the .vti holds
(object2d.cpp:7-29): shape (res_y, res_x, 2), component 0 = tau, component 1 ('Y') = I.
The C++ mirror of the reference's classes (plane, object3d_*, object2d) lives in
course5_b200/host/; this module is the binding tests and bench.py use.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# C5GPU_LIBRARY: another build of the same library (A/B runs of two builds in one process-per-build experiment)
DEFAULT_SO = os.environ.get("C5GPU_LIBRARY") or os.path.join(HERE, "libc5gpu.so")
C5_MAX_ROT = 8
MAX_CHANNELS = 8       # C5_MAX_CHANNELS
PI = 3.14159265358979323846  # config.hpp:45

OK, E_INVALID, E_CUDA, E_NOMEM, E_TOPOLOGY, E_STATE, E_WALK, E_NCCL = 0, -1, -2, -3, -4, -5, -6, -7


class C5Error(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"c5gpu error {code}: {text}")
        self.code = code


class Rotation(C.Structure):
    _fields_ = [("axis", C.c_int32), ("reserved", C.c_int32), ("angle", C.c_double), ("x0", C.c_double)]


class View(C.Structure):
    _fields_ = [("res_x", C.c_int32), ("res_y", C.c_int32), ("window", C.c_double * 4),
                ("n_rot", C.c_int32), ("reserved0", C.c_int32), ("rot", Rotation * C5_MAX_ROT),
                ("alpha_limit", C.c_double), ("precision", C.c_int32), ("round_through_float", C.c_int32),
                ("use_solids", C.c_int32), ("row_begin", C.c_int32), ("row_end", C.c_int32),
                ("reserved1", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("pixels", C.c_uint64), ("tet_steps", C.c_uint64), ("hit_pixels", C.c_uint64),
                ("solid_pixels", C.c_uint64), ("walk_errors", C.c_uint64), ("ms_rotate", C.c_float),
                ("ms_bvh", C.c_float), ("ms_mask", C.c_float), ("ms_walk", C.c_float),
                ("ms_gather", C.c_float), ("ms_d2h", C.c_float), ("ms_total", C.c_float),
                ("n_devices", C.c_int32), ("grazing_rays", C.c_int32), ("ms_graze", C.c_float),
                ("reserved", C.c_int32)]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_ if name != "reserved"}


class MeshInfo(C.Structure):
    _fields_ = [("n_points", C.c_int64), ("n_tets", C.c_int64), ("n_boundary_faces", C.c_int64),
                ("n_bvh_nodes", C.c_int64), ("n_solid_tets", C.c_int64), ("device_bytes", C.c_int64)]


_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)
_u8p = C.POINTER(C.c_uint8)
_u64p = C.POINTER(C.c_uint64)

# every symbol include/c5gpu.h declares: (restype, argtypes)
SYMBOLS = {
    "c5_abi_version": (C.c_int, []),
    "c5_view_from_flags": (None, [C.POINTER(View), C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                                  C.c_double]),
    "c5_create": (C.c_int, [_i32p, C.c_int32, C.POINTER(C.c_void_p)]),
    "c5_create_sibling": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "c5_destroy": (None, [C.c_void_p]),
    "c5_last_error": (C.c_char_p, [C.c_void_p]),
    "c5_upload_mesh": (C.c_int, [C.c_void_p, _dp, C.c_int64, _i32p, C.c_int64, _dp, _dp]),
    "c5_upload_solids": (C.c_int, [C.c_void_p, _dp, C.c_int64, C.c_int32]),
    "c5_clear_solids": (C.c_int, [C.c_void_p]),
    "c5_mesh_info_get": (C.c_int, [C.c_void_p, C.POINTER(MeshInfo)]),
    "c5_render": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, C.POINTER(Stats)]),
    "c5_render_raw": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, _u32p, _u8p, C.POINTER(Stats)]),
    "c5_upload_channels": (C.c_int, [C.c_void_p, _dp, _dp, C.c_int32]),
    "c5_render_channels": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, _u32p, _u8p, C.POINTER(Stats)]),
    "c5_render_flux": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, _dp, _dp, C.POINTER(Stats)]),
    "c5_render_flux_submit": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, _dp, _dp, _u64p]),
    "c5_update_fields": (C.c_int, [C.c_void_p, _dp, _dp]),
    "c5_render_grad": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, _dp, _dp, _dp, C.POINTER(Stats)]),
    "c5_update_fields_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "c5_render_grad_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.POINTER(Stats)]),
    "c5_render_flux_grad_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "c5_render_jvp": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, _dp, _dp, _dp, C.POINTER(Stats)]),
    "c5_render_jvp_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.POINTER(Stats)]),
    "c5_render_flux_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.POINTER(Stats)]),
    "c5_render_flux_jvp_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "c5_render_device": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "c5_last_row_cost": (C.c_int, [C.c_void_p, _u64p, C.c_int32]),
    "c5_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "c5_render_submit": (C.c_int, [C.c_void_p, C.POINTER(View), _dp, _u64p]),
    "c5_render_wait": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(Stats)]),
    "c5_set_views_in_flight": (C.c_int, [C.c_void_p, C.c_int32]),
    "c5_debug_set": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "c5_debug_ray_order": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "c5_debug_ray_order_read": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, _i32p, _i32p]),
    "c5_timeline_read": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_int32, _i32p]),
    "c5_image_create": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), _u8p]),
    "c5_image_open": (C.c_int, [C.c_void_p, _u8p, C.POINTER(C.c_void_p)]),
    "c5_image_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "c5_host_register": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "c5_host_unregister": (C.c_int, [C.c_void_p, C.c_void_p]),
}
IPC_HANDLE_BYTES = 80
MAX_IN_FLIGHT = 8
ABI_VERSION = 9        # C5_ABI_VERSION of include/c5gpu.h this binding was written against
TIMELINE_PHASES = 6


def load_library(path: str | None = None) -> C.CDLL:
    """Opens the C-ABI library and types every symbol. No fallback: a missing .so is an error."""
    path = path or DEFAULT_SO
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). course5_b200 has no CPU path.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


def _ptr(a, typ):
    return None if a is None else a.ctypes.data_as(typ)


def make_view(res_x: int, res_y: int, *, X: float = 0.0, Y: float = 0.0, I: float = 0.0,
              alpha_limit: float = 2.5, lib: C.CDLL | None = None, **overrides) -> View:
    """The view main.cpp:83-107 derives from the CLI flags -x -y -X -Y -I --alpha_limit
    (angles in units of pi). D (the donor angle) acts on the Roche lobe at generation time,
    not on the view."""
    v = View()
    (lib or load_library()).c5_view_from_flags(C.byref(v), res_x, res_y, X, Y, I, alpha_limit)
    for k, val in overrides.items():
        setattr(v, k, val)
    return v


@dataclass
class RawImage:
    image: np.ndarray   # (rows, res_x, 2) float64
    steps: np.ndarray   # (rows, res_x) uint32
    solid: np.ndarray   # (rows, res_x) uint8
    stats: dict

    @property
    def tau(self):
        return self.image[..., 0]

    @property
    def inten(self):
        return self.image[..., 1]

    @property
    def hit(self):
        return self.steps > 0


class Context:
    """Owns one c5_ctx (device memory, stream, kernels)."""

    def __init__(self, devices=(0,), lib: C.CDLL | None = None):
        self.lib = lib or load_library()
        devs = (C.c_int32 * len(devices))(*devices)
        handle = C.c_void_p()
        rc = self.lib.c5_create(devs, len(devices), C.byref(handle))
        if rc != OK:
            raise C5Error(rc, (self.lib.c5_last_error(None) or b"").decode())
        self._h = handle
        self.devices = tuple(devices)
        self.n_devices = len(devices)
        self._views_in_flight = 3  # c5_create's default

    def sibling(self) -> "Context":
        """A context on the same device that shares this one's mesh and solids and owns only per-view
        state: rendering alternate views through the two, on two streams, lets consecutive views
        overlap on the device (c5_create_sibling). Close it before this context."""
        handle = C.c_void_p()
        self._check(self.lib.c5_create_sibling(self._h, C.byref(handle)))
        sib = Context.__new__(Context)
        sib.lib, sib._h, sib.n_devices, sib._parent = self.lib, handle, 1, self
        sib.devices = self.devices
        return sib

    def debug_set(self, key: str, value: int):
        """Diagnostics knob of include/c5gpu.h (tests, profiling scripts): graze_list, query_budget,
        serial_list, no_zero_copy, timeline."""
        self._check(self.lib.c5_debug_set(self._h, key.encode(), int(value)))

    def timeline(self, origin_event: int, max_views: int = 4096) -> np.ndarray:
        """(n, 6) milliseconds since `origin_event` (a cudaEvent_t handle, e.g. torch.cuda.Event.cuda_event)
        for the last views this context rendered: start, rotated, refitted, mask done, pixel kernel
        done, grazing-ray kernel done (after debug_set("timeline", n))."""
        out = np.zeros((max_views, TIMELINE_PHASES), dtype=np.float32)
        n = C.c_int32(0)
        self._check(self.lib.c5_timeline_read(self._h, C.c_void_p(origin_event), out.ctypes.data_as(C.POINTER(C.c_float)),
                                              max_views, C.byref(n)))
        return out[: n.value].copy()

    def set_views_in_flight(self, n: int):
        self._check(self.lib.c5_set_views_in_flight(self._h, n))
        self._views_in_flight = n

    @property
    def views_in_flight(self) -> int:
        """The lanes of render_submit, render_flux_submit and the light-curve device calls (render_flux_device,
        render_flux_jvp_device, render_flux_grad_device; set_views_in_flight)."""
        return self._views_in_flight

    def _check(self, rc: int):
        if rc != OK:
            raise C5Error(rc, (self.lib.c5_last_error(self._h) or b"").decode())

    def close(self):
        if getattr(self, "_h", None):
            self.lib.c5_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- uploads ------------------------------------------------------------------------------
    def upload_mesh(self, points, tets, alpha, q) -> MeshInfo:
        points = np.ascontiguousarray(points, dtype=np.float64)
        tets = np.ascontiguousarray(tets, dtype=np.int32)
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        if points.ndim != 2 or points.shape[1] != 3 or tets.ndim != 2 or tets.shape[1] != 4:
            raise ValueError("points must be (n,3) and tets (m,4)")
        if alpha.shape != (tets.shape[0],) or q.shape != (tets.shape[0],):
            raise ValueError("alpha and q must have one value per tet")
        self._n_channels = 0  # a new mesh drops the channels, also when its upload fails
        self._fields_version = self.fields_version + 1
        self._check(self.lib.c5_upload_mesh(self._h, _ptr(points, _dp), points.shape[0], _ptr(tets, _i32p),
                                            tets.shape[0], _ptr(alpha, _dp), _ptr(q, _dp)))
        return self.mesh_info()

    def upload_solids(self, tet_points, follows_view: bool):
        tet_points = np.ascontiguousarray(tet_points, dtype=np.float64)
        if tet_points.size and tet_points.shape[1:] != (4, 3):
            raise ValueError("tet_points must be (n,4,3)")
        self._check(self.lib.c5_upload_solids(self._h, _ptr(tet_points, _dp), tet_points.shape[0],
                                              1 if follows_view else 0))

    def clear_solids(self):
        self._check(self.lib.c5_clear_solids(self._h))

    def mesh_info(self) -> MeshInfo:
        info = MeshInfo()
        self._check(self.lib.c5_mesh_info_get(self._h, C.byref(info)))
        return info

    # -- rendering ----------------------------------------------------------------------------
    def render(self, view: View, out: np.ndarray | None = None):
        """Full image (res_y, res_x, 2) in a host array; returns (image, stats dict)."""
        if out is None:
            out = np.zeros((view.res_y, view.res_x, 2), dtype=np.float64)
        st = Stats()
        self._check(self.lib.c5_render(self._h, C.byref(view), _ptr(out, _dp), C.byref(st)))
        return out, st.as_dict()

    def upload_channels(self, alpha, q):
        """Several pairs of cell fields for render_channels: alpha and q of shape (n, n_tets), tets in
        the order given to upload_mesh (c5_upload_channels). n = 0 removes them."""
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        if alpha.ndim != 2 or alpha.shape != q.shape:
            raise ValueError("alpha and q must both have shape (n_channels, n_tets)")
        n_tets = self.mesh_info().n_tets  # 0 before upload_mesh: the library reports that
        if n_tets and alpha.shape[0] and alpha.shape[1] != n_tets:
            raise ValueError("alpha and q need one value per tet of the uploaded mesh")
        self._n_channels = 0  # a failed upload leaves no channels
        self._check(self.lib.c5_upload_channels(self._h, alpha.ctypes.data_as(_dp), q.ctypes.data_as(_dp),
                                                alpha.shape[0]))
        self._n_channels = alpha.shape[0]

    @property
    def n_channels(self) -> int:
        """Channels uploaded through this context (a sibling's are its parent's)."""
        owner = getattr(self, "_parent", None) or self
        return getattr(owner, "_n_channels", 0)

    def render_channels(self, view: View, out: np.ndarray | None = None, *, raw: bool = False):
        """All uploaded channels of one view in one walk (c5_render_channels): returns (image, stats)
        with image of shape (res_y, res_x, n, 2), [..., c, 0] = tau and [..., c, 1] = I of channel c;
        with raw=True (image, steps, solid mask, stats)."""
        shape = (view.res_y, view.res_x, self.n_channels, 2)
        if out is None:
            out = np.zeros(shape, dtype=np.float64)
        if out.dtype != np.float64 or not out.flags["C_CONTIGUOUS"] or out.shape != shape:
            raise ValueError(f"out must be a C-contiguous float64 array of shape {shape}")
        steps = np.zeros((view.res_y, view.res_x), dtype=np.uint32) if raw else None
        solid = np.zeros((view.res_y, view.res_x), dtype=np.uint8) if raw else None
        st = Stats()
        self._check(self.lib.c5_render_channels(self._h, C.byref(view), _ptr(out, _dp), _ptr(steps, _u32p),
                                                _ptr(solid, _u8p), C.byref(st)))
        if raw:
            return out, steps, solid, st.as_dict()
        return out, st.as_dict()

    def render_submit(self, view: View, out: np.ndarray) -> int:
        """Enqueues the view and returns a ticket at once (c5_render_submit); `out` must stay alive and
        untouched until render_wait(ticket). Page-locked `out` (torch pin_memory, host_register) is
        written in place by the walk kernel; up to set_views_in_flight() views overlap on the device."""
        if out.dtype != np.float64 or not out.flags["C_CONTIGUOUS"] or out.size != view.res_y * view.res_x * 2:
            raise ValueError("out must be a C-contiguous float64 array of res_y * res_x * 2")
        ticket = C.c_uint64(0)
        self._check(self.lib.c5_render_submit(self._h, C.byref(view), _ptr(out, _dp), C.byref(ticket)))
        return int(ticket.value)

    def render_wait(self, ticket: int) -> dict:
        st = Stats()
        try:
            self._check(self.lib.c5_render_wait(self._h, ticket, C.byref(st)))
        finally:
            getattr(self, "_flux_in_flight", {}).pop(ticket, None)
        return st.as_dict()

    def _flux_arrays(self, view: View, channels: bool):
        n = self.n_channels if channels else 1
        return np.zeros((view.res_y, n, 2), dtype=np.float64), np.zeros((n, 2), dtype=np.float64)

    def render_flux(self, view: View, *, channels: bool = False):
        """Row sums of one view, reduced on the device (c5_render_flux): returns (rows, total, stats) with
        rows of shape (res_y, n, 2) and total of shape (n, 2), [c, 0] = sum of tau and [c, 1] = sum of I
        over the pixels outside the solid mask; n = 1 for the cells' own fields, n = n_channels with
        channels=True. Rows outside the view's band are 0."""
        rows, total = self._flux_arrays(view, channels)
        st = Stats()
        self._check(self.lib.c5_render_flux(self._h, C.byref(view), 1 if channels else 0, _ptr(rows, _dp),
                                            _ptr(total, _dp), C.byref(st)))
        return rows, total, st.as_dict()

    def render_flux_submit(self, view: View, *, channels: bool = False):
        """The pipelined form (c5_render_flux_submit): returns (ticket, rows, total) at once; render_wait(ticket)
        fills the two arrays. The context keeps them alive until then."""
        rows, total = self._flux_arrays(view, channels)
        ticket = C.c_uint64(0)
        self._check(self.lib.c5_render_flux_submit(self._h, C.byref(view), 1 if channels else 0, _ptr(rows, _dp),
                                                   _ptr(total, _dp), C.byref(ticket)))
        if not hasattr(self, "_flux_in_flight"):
            self._flux_in_flight = {}
        self._flux_in_flight[int(ticket.value)] = (rows, total)
        return int(ticket.value), rows, total

    def update_fields(self, alpha, q):
        """Replaces the cells' own alpha and Q (one value per tet, in the order given to upload_mesh)
        without rebuilding topology or BVH (c5_update_fields)."""
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        n_tets = self.mesh_info().n_tets  # 0 before upload_mesh: the library reports that
        if alpha.ndim != 1 or alpha.shape != q.shape or (n_tets and alpha.shape[0] != n_tets):
            raise ValueError("alpha and q need one value per tet of the uploaded mesh")
        self._fields_version = self.fields_version + 1
        self._check(self.lib.c5_update_fields(self._h, _ptr(alpha, _dp), _ptr(q, _dp)))

    @property
    def fields_version(self) -> int:
        """Counts the uploads of the cells' own fields (upload_mesh, update_fields) through this context
        (a sibling's are its parent's): autograd.render compares it to know whether its fields are still
        the context's."""
        owner = getattr(self, "_parent", None) or self
        return getattr(owner, "_fields_version", 0)

    def render_grad(self, view: View, g, *, image: bool = False, alpha: bool = True, q: bool = True):
        """Vector-Jacobian product of the pre-cast image against g, shape (res_y, res_x, 2) with {g_tau, g_I}
        per pixel (c5_render_grad; the view needs round_through_float = 0). Returns (grad_alpha, grad_q),
        each of shape (n_tets,) in the order given to upload_mesh (None for one that was not asked for),
        and with image=True also the (res_y, res_x, 2) {tau, I} image of render_raw. Gradients are summed
        with atomics: equal to rounding, not bit for bit, from run to run."""
        g = np.ascontiguousarray(g, dtype=np.float64)
        if g.size != view.res_y * view.res_x * 2:
            raise ValueError("g must hold res_y * res_x * 2 doubles")
        n_tets = self.n_tets
        ga = np.empty(n_tets, dtype=np.float64) if alpha else None
        gq = np.empty(n_tets, dtype=np.float64) if q else None
        out = np.zeros((view.res_y, view.res_x, 2), dtype=np.float64) if image else None
        st = Stats()
        self._check(self.lib.c5_render_grad(self._h, C.byref(view), _ptr(g, _dp), _ptr(ga, _dp), _ptr(gq, _dp),
                                            _ptr(out, _dp), C.byref(st)))
        self.last_stats = st.as_dict()
        return (ga, gq, out) if image else (ga, gq)

    @property
    def n_tets(self) -> int:
        """Tets of the uploaded mesh (0 before upload_mesh). A sibling reports its parent's: its own mesh
        info is filled in only once it has rendered."""
        owner = getattr(self, "_parent", None) or self
        return int(owner.mesh_info().n_tets)

    def update_fields_device(self, alpha_ptr: int, q_ptr: int, stream: int = 0):
        """update_fields from DEVICE memory (c5_update_fields_device): alpha_ptr and q_ptr point to n_tets
        doubles each on the context's device (e.g. tensor.data_ptr()), in the order given to upload_mesh.
        The gather is enqueued on `stream` (a cudaStream_t handle, 0 = the legacy default stream) without a
        host synchronisation; the library's later renders and later work on `stream` see the new fields.
        The arrays must stay valid until the gather has run on `stream`."""
        self._fields_version = self.fields_version + 1
        self._check(self.lib.c5_update_fields_device(self._h, C.c_void_p(alpha_ptr), C.c_void_p(q_ptr),
                                                     C.c_void_p(stream)))

    def render_grad_device(self, view: View, g_ptr: int, grad_alpha_ptr: int, grad_q_ptr: int, out_ptr: int = 0,
                           stream: int = 0, *, stats: bool = True) -> dict:
        """render_grad on DEVICE memory (c5_render_grad_device), enqueued on `stream`. g_ptr: the view's row
        band only, (row_end - row_begin) * res_x * 2 doubles {g_tau, g_I}; out_ptr (0 = none): the same size,
        receives that band of render_raw's image; grad_alpha_ptr / grad_q_ptr (0 = not wanted, not both):
        n_tets doubles each, overwritten. stats=False: enqueue only (no readback, no synchronisation, a ray
        stopped by the step cap is not reported); returns {}."""
        st = Stats() if stats else None
        self._check(self.lib.c5_render_grad_device(self._h, C.byref(view), C.c_void_p(g_ptr),
                                                   C.c_void_p(grad_alpha_ptr or None), C.c_void_p(grad_q_ptr or None),
                                                   C.c_void_p(out_ptr or None), C.c_void_p(stream),
                                                   C.byref(st) if stats else None))
        self.last_stats = st.as_dict() if stats else {}
        return self.last_stats

    def render_jvp(self, view: View, v_alpha, v_q, *, image: bool = False):
        """Jacobian-vector product of the pre-cast image along the field direction (v_alpha, v_q), each of
        shape (n_tets,) in the order given to upload_mesh or None for zero, not both (c5_render_jvp; the view
        needs round_through_float = 0). Returns the (res_y, res_x, 2) tangent image {dtau, dI} per pixel, and
        with image=True also render_raw's (res_y, res_x, 2) {tau, I} image. One walk, no atomics: bit for
        bit the same from run to run, for any row band and device count. Rows outside the band are 0."""
        n_tets = self.n_tets
        if v_alpha is None and v_q is None:
            raise ValueError("v_alpha and v_q are both None")
        dirs = []
        for d in (v_alpha, v_q):
            if d is not None:
                d = np.ascontiguousarray(d, dtype=np.float64)
                if d.shape != (n_tets,):
                    raise ValueError("v_alpha and v_q need one value per tet of the uploaded mesh")
            dirs.append(d)
        tangent = np.zeros((view.res_y, view.res_x, 2), dtype=np.float64)
        out = np.zeros((view.res_y, view.res_x, 2), dtype=np.float64) if image else None
        st = Stats()
        self._check(self.lib.c5_render_jvp(self._h, C.byref(view), _ptr(dirs[0], _dp), _ptr(dirs[1], _dp),
                                           _ptr(tangent, _dp), _ptr(out, _dp), C.byref(st)))
        self.last_stats = st.as_dict()
        return (tangent, out) if image else tangent

    def render_jvp_device(self, view: View, v_alpha_ptr: int, v_q_ptr: int, tangent_ptr: int, out_ptr: int = 0,
                          stream: int = 0, *, stats: bool = True) -> dict:
        """render_jvp on DEVICE memory (c5_render_jvp_device), enqueued on `stream`. v_alpha_ptr / v_q_ptr:
        n_tets doubles each, file order (0 = zero, not both); tangent_ptr and out_ptr (0 = none): the view's row
        band only, (row_end - row_begin) * res_x * 2 doubles, 16-byte aligned. stats=False: enqueue only (no
        readback, no synchronisation); returns {}."""
        st = Stats() if stats else None
        self._check(self.lib.c5_render_jvp_device(self._h, C.byref(view), C.c_void_p(v_alpha_ptr or None),
                                                  C.c_void_p(v_q_ptr or None), C.c_void_p(tangent_ptr or None),
                                                  C.c_void_p(out_ptr or None), C.c_void_p(stream),
                                                  C.byref(st) if stats else None))
        self.last_stats = st.as_dict() if stats else {}
        return self.last_stats

    def render_flux_grad_device(self, views, g_ptr: int, grad_alpha_ptr: int, grad_q_ptr: int, stream: int = 0, *,
                                stats: bool = True) -> dict:
        """The gradient of sum_k g_k . total_k, total_k the {sum tau, sum I} of render_flux for views[k]
        (round_through_float = 0), on DEVICE memory (c5_render_flux_grad_device), enqueued on `stream`. g_ptr:
        len(views) * 2 doubles {g_tau_k, g_I_k}; grad_alpha_ptr / grad_q_ptr as for render_grad_device. The
        views run on the context's views_in_flight lanes. stats=False: enqueue only; returns {}. With stats, the
        counts are summed over the views and ms_total is the call's span on `stream`."""
        views = list(views)
        arr = (View * max(len(views), 1))(*views)
        st = Stats() if stats else None
        self._check(self.lib.c5_render_flux_grad_device(self._h, arr if views else None, len(views), C.c_void_p(g_ptr),
                                                        C.c_void_p(grad_alpha_ptr or None), C.c_void_p(grad_q_ptr or None),
                                                        C.c_void_p(stream), C.byref(st) if stats else None))
        self.last_stats = st.as_dict() if stats else {}
        return self.last_stats

    def render_flux_device(self, views, total_ptr: int, stream: int = 0, *, channels: bool = False,
                           stats: bool = True) -> dict:
        """The totals of render_flux for every view, on DEVICE memory (c5_render_flux_device), enqueued on `stream`:
        total_ptr receives len(views) * n * 2 doubles, view k's (n, 2) total at k * n * 2, bit for bit render_flux's;
        n = 1, or n_channels with channels=True. The views run on the context's views_in_flight lanes.
        stats=False: enqueue only; returns {}. With stats, the counts are summed over the views and ms_total is
        the call's span on `stream`."""
        views = list(views)
        arr = (View * max(len(views), 1))(*views)
        st = Stats() if stats else None
        self._check(self.lib.c5_render_flux_device(self._h, arr if views else None, len(views), 1 if channels else 0,
                                                   C.c_void_p(total_ptr or None), C.c_void_p(stream),
                                                   C.byref(st) if stats else None))
        self.last_stats = st.as_dict() if stats else {}
        return self.last_stats

    def render_flux_jvp_device(self, views, v_alpha_ptr: int, v_q_ptr: int, tangent_ptr: int, total_ptr: int = 0,
                               stream: int = 0, *, stats: bool = True) -> dict:
        """The J v of a light curve on DEVICE memory (c5_render_flux_jvp_device), enqueued on `stream`: tangent_ptr
        receives len(views) * 2 doubles, {sum dtau, sum dI} of each view's render_jvp tangent over the pixels
        outside its solid mask, in render_flux's summation order; total_ptr (0 = none) the same size, the views'
        render_flux totals bit for bit. v_alpha_ptr / v_q_ptr as for render_jvp_device (0 = zero, not both). The
        views (FP64, round_through_float = 0) run on the context's views_in_flight lanes. The tangent is laid out
        as render_flux_grad_device's g. stats as for render_flux_device."""
        views = list(views)
        arr = (View * max(len(views), 1))(*views)
        st = Stats() if stats else None
        self._check(self.lib.c5_render_flux_jvp_device(self._h, arr if views else None, len(views),
                                                       C.c_void_p(v_alpha_ptr or None), C.c_void_p(v_q_ptr or None),
                                                       C.c_void_p(tangent_ptr or None), C.c_void_p(total_ptr or None),
                                                       C.c_void_p(stream), C.byref(st) if stats else None))
        self.last_stats = st.as_dict() if stats else {}
        return self.last_stats

    def render_raw(self, view: View) -> RawImage:
        out = np.zeros((view.res_y, view.res_x, 2), dtype=np.float64)
        steps = np.zeros((view.res_y, view.res_x), dtype=np.uint32)
        solid = np.zeros((view.res_y, view.res_x), dtype=np.uint8)
        st = Stats()
        self._check(self.lib.c5_render_raw(self._h, C.byref(view), _ptr(out, _dp), _ptr(steps, _u32p),
                                           _ptr(solid, _u8p), C.byref(st)))
        return RawImage(out, steps, solid, st.as_dict())

    def render_device(self, view: View, device_ptr: int, stream: int = 0, *, stats: bool = True) -> dict:
        """Renders the view's row band into caller-owned DEVICE memory (e.g. tensor.data_ptr()).
        stats=False: enqueue only (no readback, no synchronisation); returns {}."""
        if not stats:
            self._check(self.lib.c5_render_device(self._h, C.byref(view), C.c_void_p(device_ptr),
                                                  C.c_void_p(stream), None))
            return {}
        st = Stats()
        self._check(self.lib.c5_render_device(self._h, C.byref(view), C.c_void_p(device_ptr),
                                              C.c_void_p(stream), C.byref(st)))
        return st.as_dict()

    # -- one image, several processes (include/c5gpu.h) ----------------------------------------
    def image_create(self, nbytes: int) -> tuple[int, bytes]:
        """Device image other processes can map: returns (device pointer, opaque handle bytes)."""
        ptr = C.c_void_p()
        handle = (C.c_uint8 * IPC_HANDLE_BYTES)()
        self._check(self.lib.c5_image_create(self._h, nbytes, C.byref(ptr), handle))
        return int(ptr.value), bytes(handle)

    def image_open(self, handle: bytes) -> int:
        """Maps an image created by ANOTHER process (CUDA IPC over NVLink); returns the device pointer."""
        ptr = C.c_void_p()
        buf = (C.c_uint8 * IPC_HANDLE_BYTES).from_buffer_copy(handle)
        self._check(self.lib.c5_image_open(self._h, buf, C.byref(ptr)))
        return int(ptr.value)

    def image_close(self, ptr: int):
        self._check(self.lib.c5_image_close(self._h, C.c_void_p(ptr)))

    def host_register(self, array: np.ndarray):
        """Pins `array`'s memory (e.g. a shared-memory image) so c5_render writes bands into it in place."""
        self._check(self.lib.c5_host_register(self._h, C.c_void_p(array.ctypes.data), array.nbytes))

    def host_unregister(self, array: np.ndarray):
        self._check(self.lib.c5_host_unregister(self._h, C.c_void_p(array.ctypes.data)))

    def last_row_cost(self, n_rows: int) -> np.ndarray:
        rows = np.zeros(n_rows, dtype=np.uint64)
        self._check(self.lib.c5_last_row_cost(self._h, _ptr(rows, _u64p), n_rows))
        return rows

    def kernel_launches(self) -> int:
        return int(self.lib.c5_kernel_launches(self._h))


def balanced_bands(row_cost: np.ndarray, n_bands: int, *, base_cost: float = 0.0) -> list[tuple[int, int]]:
    """Cuts [0, n_rows) into n_bands contiguous row bands of equal estimated cost.

    row_cost: tet-steps per row from a previous (or coarser) render; base_cost: fixed cost added
    per row (empty rows are not free). Contiguous bands are contiguous spans of the x-fastest
    output buffer (object2d.cpp:17-21), so one gather assembles the image."""
    cost = np.asarray(row_cost, dtype=np.float64) + float(base_cost)
    n_rows = cost.shape[0]
    if n_bands <= 1:
        return [(0, n_rows)]
    csum = np.concatenate(([0.0], np.cumsum(cost)))
    total = csum[-1]
    cuts = [0]
    for b in range(1, n_bands):
        target = total * b / n_bands
        j = int(np.searchsorted(csum, target, side="left"))
        j = max(j, cuts[-1] + 1)
        j = min(j, n_rows - (n_bands - b))
        cuts.append(j)
    cuts.append(n_rows)
    return [(cuts[i], cuts[i + 1]) for i in range(n_bands)]


def time_weighted_row_cost(row_steps: np.ndarray, band: tuple[int, int], band_ms: float, *, base_cost: float = 0.0) -> np.ndarray:
    """Spreads the device time one band took over ITS rows (zeros elsewhere), in proportion to their
    tet-steps plus a per-row constant. Summed over the ranks (bands are disjoint) this is a per-row
    time estimate in milliseconds: cutting it into equal parts (``balanced_bands(cost, n)``, no extra
    base cost) gives bands that would have taken equal time at the rates just observed — a band of
    short silhouette rays, or one that also carries the solid mask, runs at a lower rate per tet-step
    than a band of long central rays and gets fewer rows."""
    steps = np.asarray(row_steps, dtype=np.float64)
    lo, hi = band
    weight = np.zeros_like(steps)
    weight[lo:hi] = steps[lo:hi] + float(base_cost)
    total = float(weight.sum())
    return weight * (float(band_ms) / total) if total > 0.0 else weight
