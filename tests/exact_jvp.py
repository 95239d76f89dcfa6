"""The tangent image of a Jacobian-vector product along given ray segments, in decimal arithmetic.

The function differentiated is the one tests/exact_ray.py integrates (the reference's rules): tau = sum of
alpha dz with alpha not clamped; I <- s - (s - I) e, e = exp(-a^ dz), s = Q / a^, a^ = min(alpha, alpha_limit),
skipped where a^ < DBL_EPSILON. Here it is differentiated in forward mode along (v_alpha, v_Q), per pixel and
in the ray's order, with the partials of tests/exact_grad.py:
    dtau  += v_alpha dz                                                        (every segment)
    dI    <- e dI + (1 - e) / a^ v_Q + (-I_in dz e + Q / a^2 ((1 + x) e - 1)) v_alpha,  x = a^ dz
where the v_alpha term is dropped where alpha > alpha_limit. Alongside, S, the sum of the absolute values of
the terms (carried through e like dI itself), sets the scale of the rounding a double computation may leave.
(1 + x) e - 1 cancels to about x^2 / 2: the precision is raised with the smallest x of the call so that at
least 25 digits survive it, as in tests/exact_grad.py.

Plain Python on purpose: no numpy arithmetic touches the values.
"""
import decimal
import math
from decimal import Decimal

import numpy as np

DBL_EPSILON = 2.0 ** -52
MIN_DIGITS = 60


def jvp(seg_start, seg_tet, seg_dz, alpha, q, alpha_limit, v_alpha, v_q):
    """Returns (tangent, scale): (n_pix, 2) float64 arrays, {dtau, dI} per pixel (the correctly rounded double
    of the decimal value) and {S_tau, S_I}, the sums of absolute terms. Pixels without segments get 0."""
    limit = float(alpha_limit)
    starts = [int(x) for x in seg_start]
    tets = [int(x) for x in seg_tet]
    dz_f = [float(x) for x in seg_dz]
    min_x = math.inf
    cells = {}
    for t in set(tets):
        a = float(alpha[t])
        a_hat = a if a <= limit else limit
        cells[t] = (a_hat if a_hat >= DBL_EPSILON else None, float(q[t]), a <= limit, float(v_alpha[t]), float(v_q[t]))
    for t, dz in zip(tets, dz_f):
        a_hat = cells[t][0]
        if a_hat is not None and a_hat * dz > 0:
            min_x = min(min_x, a_hat * dz)
    digits = MIN_DIGITS
    if min_x < 1.0:
        digits = max(digits, 25 + 2 * math.ceil(-math.log10(min_x)) + 5)
    ctx = decimal.Context(prec=digits)
    dec = {t: (None if ah is None else Decimal(ah), Decimal(qq), flows, Decimal(va), Decimal(vq))
           for t, (ah, qq, flows, va, vq) in cells.items()}
    n_pix = len(starts) - 1
    tangent = np.zeros((n_pix, 2))
    scale = np.zeros((n_pix, 2))
    with decimal.localcontext(ctx):
        for p in range(n_pix):
            b, e_ = starts[p], starts[p + 1]
            if b == e_:
                continue
            i_val = d_tau = s_tau = d_i = s_i = Decimal(0)
            for k in range(b, e_):
                a_hat, qq, flows, va, vq = dec[tets[k]]
                dz = Decimal(dz_f[k])
                d_tau += va * dz
                s_tau += abs(va * dz)
                if a_hat is None:
                    continue
                e = (-(a_hat * dz)).exp()
                t_q = (1 - e) / a_hat * vq
                t_i = t_s = Decimal(0)
                if flows:
                    x = a_hat * dz
                    t_i = -i_val * dz * e * va
                    t_s = qq / (a_hat * a_hat) * ((1 + x) * e - 1) * va
                d_i = e * d_i + t_q + t_i + t_s
                s_i = e * s_i + abs(t_q) + abs(t_i) + abs(t_s)
                i_val = qq / a_hat - (qq / a_hat - i_val) * e
            tangent[p] = (float(d_tau), float(d_i))
            scale[p] = (float(s_tau), float(s_i))
    return tangent, scale
