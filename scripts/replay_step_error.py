#!/usr/bin/env python
"""Replays the per-step I recurrence on synthetic rays, CPU only, and prints the worst relative error of I
against a 50-digit decimal integration, per alpha decade and per form of the step:

    python scripts/replay_step_error.py

For each alpha: 20 rays of 300 steps, dz ~ U(0.001, 0.005) (tets of config C3), Q ~ U(0.1, 4), alpha
times U(0.5, 1.5) per step, no clamp. Forms: the reference's (Q - (Q - a I) e) / a; s - (s - I) e in
double (the walk before expm1); the same with a float exp of a float product (the FP32 walk before);
I - (s - I) expm1 in double and with expm1f. A step with alpha < DBL_EPSILON leaves I unchanged.
"""
import decimal
import math

import numpy as np

EPS = 2.0 ** -52


def expm1f(x):
    # single precision, like the device's expm1f (numpy's float32 expm1 is the C library's expm1f)
    return float(np.expm1(np.float32(x)))


def step(form, I, a, q, dz):
    s = q / a
    if form == "reference":
        return (q - (q - a * I) * math.exp(-a * dz)) / a
    if form == "fp64 exp":
        return s - (s - I) * math.exp(-a * dz)
    if form == "fp32 expf":
        return s - (s - I) * float(np.exp(np.float32(-np.float32(a) * np.float32(dz))))
    if form == "fp64 expm1":
        return I - (s - I) * math.expm1(-a * dz)
    return I - (s - I) * expm1f(np.float32(-np.float32(a) * np.float32(dz)))


def main():
    forms = ["reference", "fp64 exp", "fp32 expf", "fp64 expm1", "fp32 expm1f"]
    rng = np.random.default_rng(2026)
    print("alpha    " + "  ".join(f"{f:>11}" for f in forms))
    for a0 in (1e3, 1.0, 0.1, 1e-2, 1e-4, 1e-6, 1e-8, 1e-12, 1e-14):
        worst = dict.fromkeys(forms, 0.0)
        for _ in range(20):
            a = a0 * rng.uniform(0.5, 1.5, 300)
            q = rng.uniform(0.1, 4.0, 300)
            dz = rng.uniform(0.001, 0.005, 300)
            with decimal.localcontext() as ctx:
                ctx.prec = 50
                exact = decimal.Decimal(0)
                for k in range(300):
                    if a[k] >= EPS:
                        da = decimal.Decimal(a[k])
                        s = decimal.Decimal(q[k]) / da
                        exact = s - (s - exact) * (-da * decimal.Decimal(dz[k])).exp()
                exact = float(exact)
            for f in forms:
                I = 0.0
                for k in range(300):
                    if a[k] >= EPS:
                        I = step(f, I, a[k], q[k], dz[k])
                worst[f] = max(worst[f], abs(I - exact) / abs(exact))
        print(f"{a0:<8g} " + "  ".join(f"{worst[f]:11.1e}" for f in forms))


if __name__ == "__main__":
    main()
