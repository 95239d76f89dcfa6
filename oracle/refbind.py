"""ctypes bindings for the parity oracles.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module; nothing under course5_b200/ does.

  * ``Ref``   -> oracle/_ref/libc5ref.so : the UNMODIFIED reference sources driven by
                 oracle/ref_harness.cpp (built here by `make -C oracle ref`; the .so
                 travels to the GPU box, /root/reference does not).
  * ``Port``  -> oracle/libc5oracle.so   : the plain-C restatement (oracle/c5_oracle.c).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libc5ref.so")
PORT_SO = os.path.join(HERE, "libc5oracle.so")

_dp = C.POINTER(C.c_double)
_u32p = C.POINTER(C.c_uint32)
_u8p = C.POINTER(C.c_uint8)


def _ptr(a, typ):
    return None if a is None else a.ctypes.data_as(typ)


@dataclass
class OracleImage:
    tau: np.ndarray        # (res_y, res_x) float64
    inten: np.ndarray      # (res_y, res_x) float64
    steps: np.ndarray      # (res_y, res_x) uint32, records per pixel (0 under solids)
    solid: np.ndarray      # (res_y, res_x) uint8
    total_steps: int
    timings: dict          # seconds: rotate, ctor, find, trace

    @property
    def hit(self) -> np.ndarray:
        return self.steps > 0


def build(which: str = "all") -> None:
    """Compile the oracle libraries (the reference one only where /root/reference exists)."""
    subprocess.run(["make", "-C", HERE, which], check=True, stdout=subprocess.DEVNULL)


class Ref:
    """The reference's own code (hot path: plane.cpp / line.cpp / tetra.cpp)."""

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(f"{REF_SO} missing: run `make -C oracle ref` where /root/reference exists")
        lib = C.CDLL(REF_SO)
        lib.c5ref_render.restype = C.c_int
        lib.c5ref_render.argtypes = [_dp, _dp, _dp, C.c_longlong, C.c_int, _dp, C.c_longlong, C.c_int, C.c_int,
                                     C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                                     C.c_int, _dp, _dp, _u32p, _u8p, _dp, C.POINTER(C.c_ulonglong)]
        lib.c5ref_solids.restype = C.c_longlong
        lib.c5ref_solids.argtypes = [C.c_double, _dp, C.c_longlong, C.POINTER(C.c_longlong),
                                     C.POINTER(C.c_longlong)]
        lib.c5ref_pixel_coords.restype = None
        lib.c5ref_pixel_coords.argtypes = [C.c_int, C.c_int, _dp, _dp]
        lib.c5ref_run_files.restype = C.c_int
        lib.c5ref_run_files.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_double, C.c_double,
                                        C.c_double, C.c_double, C.c_double, C.c_int]
        self.lib = lib

    def render(self, tet_pts, alpha, q, *, res_x, res_y, X=0.0, Y=0.0, D=0.0, I=0.0, alpha_limit=2.5,
               threads=None, solids=0, solid_pts=None, raw=True) -> OracleImage:
        tet_pts = np.ascontiguousarray(tet_pts, dtype=np.float64)
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        n = tet_pts.shape[0]
        threads = threads or min(32, os.cpu_count() or 1)
        tau = np.zeros((res_y, res_x)); inten = np.zeros((res_y, res_x))
        steps = np.zeros((res_y, res_x), dtype=np.uint32)
        solid = np.zeros((res_y, res_x), dtype=np.uint8)
        tm = np.zeros(4); total = C.c_ulonglong(0)
        n_solid = 0
        if solid_pts is not None:
            solid_pts = np.ascontiguousarray(solid_pts, dtype=np.float64)
            n_solid = solid_pts.shape[0]
            solids = 2
        rc = self.lib.c5ref_render(_ptr(tet_pts, _dp), _ptr(alpha, _dp), _ptr(q, _dp), n, solids,
                                   _ptr(solid_pts, _dp), n_solid, res_x, res_y, X, Y, D, I, alpha_limit,
                                   threads, 1 if raw else 0, _ptr(tau, _dp), _ptr(inten, _dp),
                                   _ptr(steps, _u32p), _ptr(solid, _u8p), _ptr(tm, _dp), C.byref(total))
        if rc != 0:
            raise RuntimeError(f"c5ref_render failed rc={rc}")
        return OracleImage(tau, inten, steps, solid, int(total.value),
                           dict(rotate=tm[0], ctor=tm[1], find=tm[2], trace=tm[3]))

    def solids(self, D=0.0):
        """(roche_pts (n,4,3), sphere_pts (m,4,3)) in the pre-view frame."""
        nr = C.c_longlong(0); ns = C.c_longlong(0)
        n = self.lib.c5ref_solids(D, None, 0, C.byref(nr), C.byref(ns))
        out = np.zeros((n, 4, 3))
        self.lib.c5ref_solids(D, _ptr(out, _dp), n, None, None)
        return out[: nr.value].copy(), out[nr.value:].copy()

    def pixel_coords(self, res_x, res_y):
        xs = np.zeros(res_x); ys = np.zeros(res_y)
        self.lib.c5ref_pixel_coords(res_x, res_y, _ptr(xs, _dp), _ptr(ys, _dp))
        return xs, ys

    def run_files(self, src, dst, *, res_x, res_y, X=0.0, Y=0.0, D=0.0, I=0.0, alpha_limit=2.5, threads=8):
        return self.lib.c5ref_run_files(src.encode(), dst.encode(), res_x, res_y, X, Y, D, I, alpha_limit,
                                        threads)


class _View(C.Structure):
    _fields_ = [("res_x", C.c_int), ("res_y", C.c_int), ("window", C.c_double * 4),
                ("alpha_limit", C.c_double), ("threads", C.c_int)]


WINDOW = (2.2, -0.2, 0.9, -0.9)   # x_max, x_min, y_max, y_min — main.cpp:83
ACC_X0 = 1.0                      # config.hpp:55


class Port:
    """The plain-C restatement (oracle/c5_oracle.c)."""

    def __init__(self, so=PORT_SO):
        if so == PORT_SO and not os.path.exists(PORT_SO):
            build("port")
        lib = C.CDLL(so)
        lib.c5o_render.restype = C.c_int
        lib.c5o_render.argtypes = [_dp, _dp, _dp, C.c_int64, _dp, C.c_int64, C.POINTER(_View), _dp, _dp,
                                   _u32p, _u8p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        lib.c5o_rotate_points.restype = None
        lib.c5o_rotate_points.argtypes = [_dp, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double]
        lib.c5o_rotate_axis.restype = None
        lib.c5o_rotate_axis.argtypes = [_dp, C.c_int64, C.c_int, C.c_double, C.c_double]
        lib.c5o_pixel_coords.restype = None
        lib.c5o_pixel_coords.argtypes = [C.POINTER(_View), _dp, _dp]
        if hasattr(lib, "c5o_render_segments"):   # absent from a library built before it existed
            lib.c5o_render_segments.restype = C.c_int
            lib.c5o_render_segments.argtypes = [_dp, _dp, _dp, C.c_int64, _dp, C.c_int64, C.POINTER(_View),
                                                C.POINTER(C.c_int64), C.POINTER(C.c_int32), _dp]
        self.lib = lib

    def rotate(self, pts, X=0.0, Y=0.0, I=0.0):
        """View rotations on a copy of pts (any shape (...,3))."""
        out = np.ascontiguousarray(pts, dtype=np.float64).copy()
        self.lib.c5o_rotate_points(_ptr(out, _dp), out.size // 3, X, Y, I, ACC_X0)
        return out

    def pixel_coords(self, res_x, res_y, window=WINDOW):
        v = _View(res_x, res_y, (C.c_double * 4)(*window), 2.5, 1)
        xs = np.zeros(res_x); ys = np.zeros(res_y)
        self.lib.c5o_pixel_coords(C.byref(v), _ptr(xs, _dp), _ptr(ys, _dp))
        return xs, ys

    def render(self, tet_pts, alpha, q, *, res_x, res_y, X=0.0, Y=0.0, D=0.0, I=0.0, alpha_limit=2.5,
               threads=None, solid_rot=None, solid_static=None, window=WINDOW) -> OracleImage:
        """tet_pts (n,4,3) in the FILE frame; solid_rot follows the view rotations
        (the Roche lobe, main.cpp:112-114), solid_static does not (the sphere, main.cpp:116)."""
        import time
        threads = threads or (os.cpu_count() or 1)
        t0 = time.perf_counter()
        pts = self.rotate(tet_pts, X, Y, I)
        sol = []
        if solid_rot is not None and len(solid_rot):
            sol.append(self.rotate(solid_rot, X, Y, I))
        if solid_static is not None and len(solid_static):
            sol.append(np.ascontiguousarray(solid_static, dtype=np.float64))
        sol = np.concatenate(sol) if sol else None
        t_rot = time.perf_counter() - t0
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        v = _View(res_x, res_y, (C.c_double * 4)(*window), alpha_limit, threads)
        tau = np.zeros((res_y, res_x)); inten = np.zeros((res_y, res_x))
        steps = np.zeros((res_y, res_x), dtype=np.uint32)
        solid = np.zeros((res_y, res_x), dtype=np.uint8)
        total = C.c_uint64(0); odd = C.c_uint64(0)
        t0 = time.perf_counter()
        rc = self.lib.c5o_render(_ptr(pts, _dp), _ptr(alpha, _dp), _ptr(q, _dp), pts.shape[0],
                                 _ptr(sol, _dp), 0 if sol is None else sol.shape[0], C.byref(v),
                                 _ptr(tau, _dp), _ptr(inten, _dp), _ptr(steps, _u32p), _ptr(solid, _u8p),
                                 C.byref(total), C.byref(odd))
        if rc != 0:
            raise RuntimeError(f"c5o_render failed rc={rc}")
        img = OracleImage(tau, inten, steps, solid, int(total.value),
                          dict(rotate=t_rot, ctor=0.0, find=0.0, trace=time.perf_counter() - t0))
        img.anomalies = int(odd.value)
        return img

    def segments(self, tet_pts, alpha, q, *, res_x, res_y, X=0.0, Y=0.0, I=0.0, alpha_limit=2.5, threads=None,
                 solid_rot=None, solid_static=None, window=WINDOW, steps=None):
        """Each pixel's ordered segments, as the I recurrence takes them (the lowest first): pixel
        j * res_x + i crosses tets seg_tet[seg_start[p]:seg_start[p + 1]] over depths seg_dz[...].
        Returns (seg_start (n_pix + 1,) int64, seg_tet int32, seg_dz float64). `steps`: the per-pixel
        step counts of a render() of the same arguments, if already at hand."""
        if steps is None:
            steps = self.render(tet_pts, alpha, q, res_x=res_x, res_y=res_y, X=X, Y=Y, I=I,
                                alpha_limit=alpha_limit, threads=threads, solid_rot=solid_rot,
                                solid_static=solid_static, window=window).steps
        threads = threads or (os.cpu_count() or 1)
        pts = self.rotate(tet_pts, X, Y, I)
        sol = []
        if solid_rot is not None and len(solid_rot):
            sol.append(self.rotate(solid_rot, X, Y, I))
        if solid_static is not None and len(solid_static):
            sol.append(np.ascontiguousarray(solid_static, dtype=np.float64))
        sol = np.concatenate(sol) if sol else None
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        q = np.ascontiguousarray(q, dtype=np.float64)
        seg_start = np.zeros(res_x * res_y + 1, dtype=np.int64)
        np.cumsum(np.asarray(steps, dtype=np.int64).ravel(), out=seg_start[1:])
        seg_tet = np.zeros(max(int(seg_start[-1]), 1), dtype=np.int32)
        seg_dz = np.zeros(max(int(seg_start[-1]), 1))
        v = _View(res_x, res_y, (C.c_double * 4)(*window), alpha_limit, threads)
        rc = self.lib.c5o_render_segments(_ptr(pts, _dp), _ptr(alpha, _dp), _ptr(q, _dp), pts.shape[0],
                                          _ptr(sol, _dp), 0 if sol is None else sol.shape[0], C.byref(v),
                                          _ptr(seg_start, C.POINTER(C.c_int64)), _ptr(seg_tet, C.POINTER(C.c_int32)),
                                          _ptr(seg_dz, _dp))
        if rc != 0:
            raise RuntimeError(f"c5o_render_segments failed rc={rc}")
        n = int(seg_start[-1])
        return seg_start, seg_tet[:n], seg_dz[:n]
