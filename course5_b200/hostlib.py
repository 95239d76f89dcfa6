"""ctypes binding of libc5host.so: the host-side C++ pieces of the `course` executable that do
not touch the GPU — the Roche-lobe / sphere generators (object3d_base.cpp:84-196,
object3d_roche_lobe.cpp:20-49, object3d_sphere.cpp:11-18 restated), the legacy-VTK reader, the
.vti writer/reader and the command-line parser."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
HOST_SO = os.path.join(HERE, "libc5host.so")
COURSE_EXE = os.path.join(HERE, "bin", "course")

_dp = C.POINTER(C.c_double)
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(HOST_SO):
            raise FileNotFoundError(f"{HOST_SO} not built (make -C course5_b200/host)")
        l = C.CDLL(HOST_SO)
        l.c5host_last_error.restype = C.c_char_p
        l.c5host_solids_make.restype = C.c_longlong
        l.c5host_solids_make.argtypes = [C.c_int, C.c_double]
        l.c5host_solids_copy.argtypes = [C.c_int, _dp]
        l.c5host_read_vtk.restype = C.c_longlong
        l.c5host_read_vtk.argtypes = [C.c_char_p]
        l.c5host_grid_points.restype = C.c_longlong
        l.c5host_grid_has_scalar.argtypes = [C.c_char_p]
        l.c5host_grid_copy.argtypes = [_dp, C.POINTER(C.c_int32), C.c_char_p, _dp, C.c_char_p, _dp]
        l.c5host_write_vti.restype = C.c_longlong
        l.c5host_write_vti.argtypes = [C.c_char_p, _dp, C.c_longlong, C.c_longlong, C.c_int]
        l.c5host_read_vti.restype = C.c_longlong
        l.c5host_read_vti.argtypes = [C.c_char_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong),
                                      C.POINTER(C.c_longlong), _dp]
        l.c5host_write_vti_arrays.restype = C.c_longlong
        l.c5host_write_vti_arrays.argtypes = [C.c_char_p, _dp, C.c_longlong, C.c_longlong, C.c_int, C.c_int,
                                              C.POINTER(C.c_char_p), C.POINTER(_dp)]
        l.c5host_read_vti_array.restype = C.c_longlong
        l.c5host_read_vti_array.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong),
                                            C.POINTER(C.c_longlong), _dp]
        l.c5host_parse_cli.restype = C.c_int
        l.c5host_parse_cli.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_char_p, C.c_int, _dp, C.c_char_p,
                                       C.c_char_p, C.c_int]
        _lib = l
    return _lib


def _err():
    return (lib().c5host_last_error() or b"").decode()


def make_solids(donor_angle_pi: float = 0.0):
    """(roche (n,4,3), sphere (m,4,3)): the reference's solid objects in the pre-view frame."""
    out = []
    for which in (0, 1):
        n = lib().c5host_solids_make(which, donor_angle_pi)
        if n < 0:
            raise RuntimeError(_err())
        a = np.zeros((n, 4, 3))
        lib().c5host_solids_copy(which, a.ctypes.data_as(_dp))
        out.append(a)
    return out[0], out[1]


def read_vtk(path: str, alpha_name="AbsorpCoef", q_name="radEnLooseRate"):
    n = lib().c5host_read_vtk(path.encode())
    if n < 0:
        raise RuntimeError(_err())
    n_pts = lib().c5host_grid_points()
    pts = np.zeros((n_pts, 3)); tets = np.zeros((n, 4), dtype=np.int32)
    alpha = np.zeros(n); q = np.zeros(n)
    for name in (alpha_name, q_name):
        if not lib().c5host_grid_has_scalar(name.encode()):
            raise KeyError(f"{path}: no cell scalar {name!r}")
    lib().c5host_grid_copy(pts.ctypes.data_as(_dp), tets.ctypes.data_as(C.POINTER(C.c_int32)), alpha_name.encode(),
                           alpha.ctypes.data_as(_dp), q_name.encode(), q.ctypes.data_as(_dp))
    return pts, tets, alpha, q


def write_vti(path: str, image: np.ndarray, compress=False, base64=False, extra: dict | None = None):
    """compress: vtkZLibDataCompressor blocks; base64 (with compress): the appended section as base64
    streams — together what vtkXMLImageDataWriter writes by default. extra: {name: (res_y, res_x, 2)
    array} written as further PointData arrays beside ImageScalars."""
    image = np.ascontiguousarray(image, dtype=np.float64)
    res_y, res_x, comps = image.shape
    assert comps == 2
    mode = 2 if (compress and base64) else 1 if compress else 0
    if not extra:
        rc = lib().c5host_write_vti(path.encode(), image.ctypes.data_as(_dp), res_x, res_y, mode)
    else:
        arrays = [np.ascontiguousarray(a, dtype=np.float64) for a in extra.values()]
        assert all(a.shape == image.shape for a in arrays)
        names = (C.c_char_p * len(arrays))(*[n.encode() for n in extra])
        data = (_dp * len(arrays))(*[a.ctypes.data_as(_dp) for a in arrays])
        rc = lib().c5host_write_vti_arrays(path.encode(), image.ctypes.data_as(_dp), res_x, res_y, mode, len(arrays),
                                           names, data)
    if rc < 0:
        raise RuntimeError(_err())


def read_vti(path: str, name: str | None = None) -> np.ndarray:
    """The PointData array `name` (default: the first, ImageScalars) as (res_y, res_x, components)."""
    x, y, c = C.c_longlong(), C.c_longlong(), C.c_longlong()
    nm = name.encode() if name else None
    n = lib().c5host_read_vti_array(path.encode(), nm, C.byref(x), C.byref(y), C.byref(c), None)
    if n < 0:
        raise RuntimeError(_err())
    out = np.zeros((y.value, x.value, c.value))
    lib().c5host_read_vti_array(path.encode(), nm, C.byref(x), C.byref(y), C.byref(c), out.ctypes.data_as(_dp))
    return out


def parse_cli(argv: list[str]):
    """(result, printed text, values dict): result 0 run / 1 exit 0 / 2 error."""
    args = [b"course"] + [a.encode() for a in argv]
    arr = (C.c_char_p * len(args))(*args)
    text = C.create_string_buffer(8192)
    vals = np.zeros(8)
    f = C.create_string_buffer(1024); d = C.create_string_buffer(1024)
    r = lib().c5host_parse_cli(len(args), arr, text, 8192, vals.ctypes.data_as(_dp), f, d, 1024)
    keys = ("res_x", "res_y", "X", "Y", "D", "I", "alpha_limit", "threads")
    v = dict(zip(keys, vals.tolist()))
    v["file"], v["destination"] = f.value.decode(), d.value.decode()
    return r, text.value.decode(), v
