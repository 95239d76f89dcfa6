"""grad_alpha and grad_q of an image's vector-Jacobian product along given ray segments, in decimal arithmetic.

The function differentiated is the one tests/exact_ray.py integrates (the reference's rules): tau = sum of
alpha dz with alpha not clamped; I <- s - (s - I) e, e = exp(-a^ dz), s = Q / a^, a^ = min(alpha, alpha_limit),
skipped where a^ < DBL_EPSILON. Here it is differentiated in reverse mode, which is not how the walk does it
(the walk goes forward with T = exp(-(lam_ray - lam_through))): per pixel, I is integrated forward, then an
adjoint a_ = g_I starts at the viewer and runs backwards over the segments,
    dI/dQ_t     += a_ (1 - e) / a^
    dI/dalpha_t += a_ (-I_in dz e + Q / a^2 ((1 + x) e - 1)),  x = a^ dz   (only where alpha_t <= alpha_limit)
    a_          <- a_ e
and every segment adds g_tau dz to dtau/dalpha_t. (1 + x) e - 1 cancels to about x^2 / 2: the precision
is raised with the smallest x of the call so that at least 25 digits survive it.

Plain Python on purpose: no numpy arithmetic touches the values.
"""
import decimal
import math
from decimal import Decimal

import numpy as np

DBL_EPSILON = 2.0 ** -52
MIN_DIGITS = 60


def vjp(seg_start, seg_tet, seg_dz, alpha, q, alpha_limit, g, n_tets):
    """g: (n_pix, 2) {g_tau, g_I} per pixel (pixels to leave out must have g = 0). Returns
    (grad_alpha, grad_q), float64 arrays of n_tets, each the correctly rounded double of the decimal sum."""
    limit = float(alpha_limit)
    starts = [int(x) for x in seg_start]
    tets = [int(x) for x in seg_tet]
    dz_f = [float(x) for x in seg_dz]
    g = np.asarray(g, dtype=np.float64).reshape(-1, 2)
    min_x = math.inf
    cells = {}
    for t in set(tets):
        a = float(alpha[t])
        a_hat = a if a <= limit else limit
        cells[t] = (a, a_hat if a_hat >= DBL_EPSILON else None, float(q[t]), a <= limit)
    for t, dz in zip(tets, dz_f):
        a_hat = cells[t][1]
        if a_hat is not None and a_hat * dz > 0:
            min_x = min(min_x, a_hat * dz)
    digits = MIN_DIGITS
    if min_x < 1.0:
        digits = max(digits, 25 + 2 * math.ceil(-math.log10(min_x)) + 5)
    ctx = decimal.Context(prec=digits)
    dec = {t: (Decimal(a), None if ah is None else Decimal(ah), Decimal(qq), flows)
           for t, (a, ah, qq, flows) in cells.items()}
    ga = {}
    gq = {}
    with decimal.localcontext(ctx):
        for p in range(len(starts) - 1):
            b, e_ = starts[p], starts[p + 1]
            g_tau, g_I = float(g[p, 0]), float(g[p, 1])
            if b == e_ or (g_tau == 0.0 and g_I == 0.0):
                continue
            d_tau, d_I = Decimal(g_tau), Decimal(g_I)
            # forward: I entering each segment and its e
            fwd = []
            i_val = Decimal(0)
            for k in range(b, e_):
                t = tets[k]
                a, a_hat, qq, _ = dec[t]
                dz = Decimal(dz_f[k])
                if a_hat is None:
                    fwd.append((t, dz, None, None))
                    continue
                e = (-(a_hat * dz)).exp()
                fwd.append((t, dz, i_val, e))
                i_val = qq / a_hat - (qq / a_hat - i_val) * e
            # backward
            adj = d_I
            for t, dz, i_in, e in reversed(fwd):
                if d_tau:
                    ga[t] = ga.get(t, Decimal(0)) + d_tau * dz
                if e is None:
                    continue
                a, a_hat, qq, flows = dec[t]
                gq[t] = gq.get(t, Decimal(0)) + adj * (1 - e) / a_hat
                if flows:
                    x = a_hat * dz
                    d_out = -i_in * dz * e + qq / (a_hat * a_hat) * ((1 + x) * e - 1)
                    ga[t] = ga.get(t, Decimal(0)) + adj * d_out
                adj = adj * e
    out_a = np.zeros(n_tets)
    out_q = np.zeros(n_tets)
    for t, v in ga.items():
        out_a[t] = float(v)
    for t, v in gq.items():
        out_q[t] = float(v)
    return out_a, out_q
