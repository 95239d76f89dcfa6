"""tau and I along given ray segments, integrated in 60-digit decimal arithmetic.

This is what the walk's per-step recurrence approximates, with the reference's rules (line.cpp:176-227):
  * tau = sum of alpha * dz, alpha not clamped;
  * I <- s - (s - I) exp(-a^ dz), s = Q / a^, a^ = min(alpha, alpha_limit), from I = 0 at the entry;
  * a step with a^ < DBL_EPSILON leaves I unchanged (kept on purpose: it is the reference's defined
    behaviour, pinned by test_kat_transparent_cells_leave_I_unchanged).
Every alpha, Q, limit and dz enters as its exact binary value (Decimal(float)), so the only error is the
decimal rounding. The subtraction s - (s - I) e loses about log10(1 / (a^ dz)) digits, at most about 19
(a^ = DBL_EPSILON, dz = 1e-3); 60 digits leave more than 40, far below the double result's rounding.

Plain Python on purpose: no numpy arithmetic touches the values.
"""
import decimal
from decimal import Decimal

import numpy as np

PREC = 60
DBL_EPSILON = 2.0 ** -52


def integrate(seg_start, seg_tet, seg_dz, alpha, q, alpha_limit):
    """Per pixel (seg_start[p] .. seg_start[p + 1] of the segment arrays, in the order I is integrated,
    entry first): returns (tau, inten), float64 arrays of n_pix values, each the correctly rounded
    double of the 60-digit result. Pixels without segments get 0."""
    ctx = decimal.Context(prec=PREC)
    limit = float(alpha_limit)
    # per tet: exact alpha, and (a^, s) where a^ >= DBL_EPSILON, else None (the step leaves I alone)
    cells = {}
    for t in set(int(x) for x in np.unique(seg_tet)):
        a = float(alpha[t])
        a_hat = a if a <= limit else limit
        if a_hat < DBL_EPSILON:
            cells[t] = (Decimal(a), None, None)
        else:
            da = Decimal(a_hat)
            cells[t] = (Decimal(a), da, ctx.divide(Decimal(float(q[t])), da))
    starts = [int(x) for x in seg_start]
    tets = [int(x) for x in seg_tet]
    dzs = [Decimal(float(x)) for x in seg_dz]
    n_pix = len(starts) - 1
    tau = np.zeros(n_pix)
    inten = np.zeros(n_pix)
    with decimal.localcontext(ctx):
        for p in range(n_pix):
            b, e = starts[p], starts[p + 1]
            if b == e:
                continue
            t_sum = Decimal(0)
            i_val = Decimal(0)
            for k in range(b, e):
                a, a_hat, s = cells[tets[k]]
                dz = dzs[k]
                t_sum += a * dz
                if a_hat is not None:
                    i_val = s - (s - i_val) * (-(a_hat * dz)).exp()
            tau[p] = float(t_sum)
            inten[p] = float(i_val)
    return tau, inten
