"""TEST INFRASTRUCTURE ONLY -- restatement of the product's production-mode nuisance step
(instagraal_b200/csrc/ig_k_nuis.cuh: k_nuis_propose, nuis_dmax_root, k_nuis_accept) in NumPy/Python.

The reference's step_nuisance_parameters (cuda_lib_gl_single.py:2961-3051) draws choice(4), one normal and one uniform
from NumPy's stream and solves for d_max with scipy's fsolve.  The device draws them from Philox4x32-10 (key = the chain's
seed, counters (t, cycle, 0x80000000, 0) and (t, cycle, 0x80000001, 0), a domain the neighbour draws never use) and finds
d_max as the root of rippe(x) = y (deviation D3).  The proposal arithmetic is the float32 arithmetic of
sampler._nuisance_finish under NumPy's promotion rules.  Only tests import this module."""
import math

import numpy as np

from oracle.device_rng import philox4x32_10

MASK = 0xFFFFFFFF
F32 = np.float32


def _u53(hi, lo):
    return float(((hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0)


def counters(t, cycle):
    """the two Philox counters of nuisance step t of `cycle` (the neighbour draws use draw indices < IG_MAX_CANDS)"""
    return (t, cycle, 0x80000000, 0), (t, cycle, 0x80000001, 0)


def draws(t, cycle, seed):
    """-> (id_modif, u, z): the parameter to move, the acceptance draw and the standard normal of step t"""
    key = (seed & MASK, (seed >> 32) & MASK)
    ca, cb = counters(t, cycle)
    a = philox4x32_10(ca, key)
    b = philox4x32_10(cb, key)
    u1, u2 = _u53(b[0], b[1]), _u53(b[2], b[3])
    z = math.sqrt(-2.0 * math.log(1.0 - u1)) * math.cos(2.0 * math.pi * u2)
    return a[0] >> 30, _u53(a[1], a[2]), z


def sigma(v):
    """10 ** (log10(v) - 2) as _nuisance_draws computes it in float32, each operation rounded once"""
    if not v > 0:
        return F32(0.0) if v == 0 else F32(np.nan)
    l = F32(math.log10(float(v)))
    return F32(10.0 ** float(F32(l - F32(2.0))))


def draw_of(id_modif, z, p8):
    """the normal draw of _nuisance_draws for live parameters p8 (None: id 3 with d_nuc <= 0)"""
    if id_modif == 0:
        return float(sigma(p8[6])) * z
    if id_modif == 1:
        return 0.005 * z
    if id_modif == 2:
        return 100.0 * z
    s = sigma(p8[7])
    return float(s) * z if s > 0 else None


def dmax_root(kuhn, lm, slope, dd, A, y):
    """x > 0 with A 0.53 kuhn^-3 (lm x / kuhn)^slope exp((dd - 2) / ((lm x / kuhn)^2 + dd)) = y, or None (no root).
    dd == 2: closed form; otherwise safeguarded Newton in log x inside a sign-change bracket (nuis_dmax_root)."""
    kuhn, lm, slope, dd, A, y = (float(v) for v in (kuhn, lm, slope, dd, A, y))
    vals = (kuhn, lm, slope, dd, A, y)
    if not all(math.isfinite(v) for v in vals) or not (A > 0 and y > 0 and slope < 0 and kuhn > 0 and lm > 0):
        return None
    c = A * 0.53 * kuhn ** -3.0
    try:
        x0 = (kuhn / lm) * (y / c) ** (1.0 / slope)
    except OverflowError:
        x0 = math.inf
    if dd == 2.0:
        return x0 if (math.isfinite(x0) and x0 > 0) else None
    k = lm / kuhn
    lk, lc, ly = math.log(k), math.log(c), math.log(y)

    def g(L):
        return lc + slope * (lk + L) + (dd - 2.0) / (k * k * math.exp(2.0 * L) + dd) - ly

    def dg(L):
        q2 = k * k * math.exp(2.0 * L)
        return slope - (dd - 2.0) * 2.0 * q2 / ((q2 + dd) * (q2 + dd))

    L = math.log(x0) if (math.isfinite(x0) and x0 > 0) else 0.0
    a = b = L
    ga = gb = g(L)
    if ga == 0.0:
        return math.exp(L)
    s = 1.0
    while not ((ga > 0 and gb < 0) or (ga < 0 and gb > 0)):
        if s > 1400.0:
            return None
        a, b = max(L - s, -700.0), min(L + s, 700.0)
        ga, gb = g(a), g(b)
        if not (math.isfinite(ga) and math.isfinite(gb)):
            return None
        s *= 2.0
    rising = gb > 0
    for _ in range(200):
        gl = g(L)
        if gl == 0.0:
            break
        if (gl > 0) == rising:
            b = L
        else:
            a = L
        Ln = L - gl / dg(L)
        if not (a < Ln < b):
            Ln = 0.5 * (a + b)
        step = abs(Ln - L)
        L = Ln
        if step <= 1e-14 * max(1.0, abs(L)) or b - a <= 1e-14 * max(1.0, abs(L)):
            break
    x = math.exp(L)
    return x if (math.isfinite(x) and x > 0) else None


def _c1(kuhn, lm, slope):
    return F32((0.53 * np.power(lm / kuhn, slope)) * np.power(kuhn, -3))


def propose(p8, id_modif, draw):
    """-> (p_test float32[8], valid): sampler._nuisance_finish's arithmetic with d_max from dmax_root (NaN: no root)"""
    kuhn, lm, c1, slope, d, d_max, fact, d_nuc = (F32(v) for v in p8)
    root = None
    with np.errstate(all="ignore"):
        if id_modif == 0:
            fact = fact + draw
            root = dmax_root(kuhn, lm, slope, d, fact, d_nuc)
        elif id_modif == 1:
            slope = slope + draw
            root = dmax_root(kuhn, lm, slope, d, fact, d_nuc)
        elif id_modif == 2:
            d_max = d_max + draw
            # opti.peval(new_d_max, [kuhn, lm, slope, d, fact]): param[3] = d as the amplitude (quirk Q7), exp term 1
            d_nuc = d * (0.53 * (kuhn ** -3.0) * np.power((lm * d_max / kuhn), slope) * np.exp((2 - 2) / (np.power((lm * d_max / kuhn), 2) + 2)))
        else:
            d_nuc = d_nuc if draw is None else d_nuc + draw
            root = dmax_root(kuhn, lm, slope, d, fact, d_nuc)
        if id_modif != 2:
            d_max = F32(np.nan) if root is None else F32(root)
        c1 = _c1(kuhn, lm, slope)
    p = np.array([kuhn, lm, c1, slope, d, d_max, fact, d_nuc], dtype=np.float32)
    valid = bool(np.all(np.isfinite(p)) and (id_modif == 2 or root is not None) and p[6] > 0 and p[3] < 0 and p[5] > 0 and p[7] > 0)
    return p, valid


def step(p8, t, cycle, seed):
    """-> (id_modif, u, draw (NaN: none), p_test, valid) of nuisance step t for live parameters p8"""
    id_modif, u, z = draws(t, cycle, seed)
    draw = draw_of(id_modif, z, p8)
    p, valid = propose(p8, id_modif, draw)
    return id_modif, u, (math.nan if draw is None else draw), p, valid
