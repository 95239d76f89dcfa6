"""The parity gate, in one place (BASELINE.json north_star / SURVEY.md §7 'hard parts').

FP64 path: per pixel |got - want| <= 1e-9 * |want| + 1e-13 on the PRE-float-cast doubles, and
identical hit/miss sets. The absolute floor covers pixels that graze the silhouette: their path
length (hence tau, I) goes to 0 while the rounding noise of a face-plane z (coordinates ~1) stays
~1e-16, so a purely relative bound is meaningless below ~1e-6. The reference's own noise floor
under a vertex-order permutation is 3.6e-14 relative (SURVEY.md §8c).
"""
import numpy as np

REL_TOL_FP64 = 1e-9
ABS_FLOOR = 1e-13
# FP32 variant (BASELINE.json north_star: <= 1e-4 relative). Per-step geometry is single precision on
# coordinates relative to the pixel / entry depth; depths relative to the entry point reach ~1, so a float depth carries ~1e-7 of absolute noise: the floor (1e-6) covers silhouette-grazing pixels whose tau and I are themselves ~1e-4.
REL_TOL_FP32 = 1e-4
ABS_FLOOR_FP32 = 1e-6
# Against the exact integration of the same segments (tests/exact_ray.py, tests/test_optical_depth.py):
# |got - exact| <= REL_TOL_EXACT |exact| + FLOOR_EXACT max|exact|, the max over the image, for tau and I
# separately. The floor scales with the image, so thin media are held to it instead of hidden under an
# absolute 1e-13. The FP64 walk's step I - (s - I) expm1(-a dz) stays within 1e-14 relative for alpha in
# [1e-15, 1] and 2e-13 at alpha = 1e3, on 96 x 72 views of n = 5..10 meshes, silhouette and grazing pixels
# included; 1e-11 leaves room for longer rays, while the step s - (s - I) exp() it replaced is past it
# from alpha = 1e-4 on (a constant medium: 1e-12 relative at alpha = 1e-2, 8e-11 at 1e-4). The FP32 variant is held to
# its documented gate (REL_TOL_FP32) with the floor ABS_FLOOR_FP32 scaled the same way.
REL_TOL_EXACT = 1e-11
FLOOR_EXACT = 1e-13


def exact_margin(got, want, *, rel=REL_TOL_EXACT, floor=FLOOR_EXACT):
    """Per pixel |got - want| / (rel |want| + floor max|want|): the gate holds where this is <= 1."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    scale = np.abs(want).max() if want.size else 0.0
    tol = rel * np.abs(want) + floor * scale
    err = np.abs(got - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(tol > 0, err / np.where(tol > 0, tol, 1.0), np.where(err > 0, np.inf, 0.0))


def assert_image_parity(got_tau, got_I, want_tau, want_I, *, rel=REL_TOL_FP64, floor=ABS_FLOOR, what=""):
    for got, want, name in ((got_tau, want_tau, "tau"), (got_I, want_I, "I")):
        got = np.asarray(got)
        want = np.asarray(want)
        assert got.shape == want.shape, f"{what}{name}: shape {got.shape} vs {want.shape}"
        nan_g, nan_w = np.isnan(got), np.isnan(want)
        assert np.array_equal(nan_g, nan_w), f"{what}{name}: NaN (solid) masks differ"
        err = np.abs(np.where(nan_w, 0.0, got - want))
        tol = rel * np.abs(np.where(nan_w, 0.0, want)) + floor
        bad = err > tol
        assert not bad.any(), (f"{what}{name}: {int(bad.sum())} pixels out of tolerance, "
                               f"max abs err {err.max():.3e}")


def assert_same_hits(got_steps, want_steps, what=""):
    got_hit = np.asarray(got_steps) > 0
    want_hit = np.asarray(want_steps) > 0
    diff = int((got_hit != want_hit).sum())
    assert diff == 0, f"{what}hit/miss sets differ on {diff} pixels"


def float_ulp_distance(a, b):
    """ULP distance of two arrays of doubles that hold float-rounded values."""
    fa = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    fb = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.abs(fa - fb)
