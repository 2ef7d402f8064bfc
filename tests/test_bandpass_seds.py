"""Bandpass-integrated SEDs against an extended-precision reference (CPU part).

Every SED type of the reference is restated here from its formulas (src/dang_component_mod.f90 evaluate_*,
src/dang_bp_mod.f90 a2t / compute_bnu_prime_RJ, as cited in dang_b200/csrc/common.cuh) and summed over the FULL
bandpass table, sum_i tau_i g(nu_i) with nu_i = 0 skipped as the reference skips it.  Terms are evaluated in
np.longdouble (64-bit mantissa) and summed exactly (math.fsum over a double-double split of each term), so the
reference -- a long double, which keeps a lognormal's far tail below the double range -- is good to ~1e-18
relative wherever the formula itself is well conditioned; test_reference_agrees_with_mpmath certifies it against
40-digit mpmath.  Nothing here uses the oracle's code.

test_eight_node_rule_domain records where the library's 8-node Gauss rule (dang_gpu_bandpass_quadrature) is NOT
enough for 1e-14: the 'cmb' SED at high frequency and narrow lognormals near nu_p.  The library verifies every rule
against the SEDs on its handle before using it (tests/test_gpu_bandpass_seds.py checks what the device does).
"""
import math

import numpy as np
import pytest

LD = np.longdouble
# src/dang_util_mod.f90:12-13 as the reference's double-precision constants (dang_b200.synth / common.cuh DG_H, DG_KB)
H = float(1.0545726691251021e-34 * 2.0 * np.pi)
KB = 1.3806503e-23
C_LIGHT = 2.99792458e8
SQRT3_PI = np.sqrt(LD(3)) / LD("3.14159265358979323846264338327950288")

TYPES = ("power-law", "mbb", "freefree", "lognormal", "cmb", "T_cmb", "hi_fit")
NU_REF = {"power-law": 30e9, "mbb": 353e9, "freefree": 40e9, "lognormal": 22e9, "cmb": 100e9, "T_cmb": 100e9,
          "hi_fit": 353e9}
# parameter boxes (SURVEY.md's parameter files name no wider ranges): power-law beta; mbb (beta, T_d [K]);
# freefree T_e [K]; lognormal (nu_p [GHz], w_ame); 'cmb' T_CMB [K]; 'T_cmb' T [K]; hi_fit T_d [K]
BOXES = {"power-law": [(-4.5, -1.5)], "mbb": [(0.5, 3.0), (5.0, 50.0)], "freefree": [(1e3, 2e4)],
         "lognormal": [(10.0, 60.0), (0.1, 1.0)], "cmb": [(2.6, 2.8)], "T_cmb": [(2.6, 2.8)], "hi_fit": [(5.0, 50.0)]}


# ------------------------------------------------------------------ the reference
def _terms(kind, nu, th, nu_ref):
    """g(nu) of one SED type in long double; nu (n,) [Hz], th: tuple of parameter arrays broadcast against nu."""
    nu = np.asarray(nu, dtype=LD)
    nr = LD(nu_ref)
    if kind == "power-law":
        return (nu / nr) ** LD(th[0])
    if kind == "mbb":
        z = LD(H) / (LD(KB) * LD(th[1]))
        return np.expm1(z * nr) / np.expm1(z * nu) * (nu / nr) ** (LD(th[0]) + 1)
    if kind == "freefree":
        def gaunt(v):
            return np.log(np.exp(LD(5.960) - SQRT3_PI * np.log(v / LD(1e9) * (LD(th[0]) / LD(1e4)) ** LD(-1.5)))
                          + LD(2.71828))
        return gaunt(nu) / gaunt(nr) * (nr / nu) ** 2
    if kind == "lognormal":
        t = np.log(nu / (LD(th[0]) * LD(1e9))) / LD(th[1])
        return np.exp(-0.5 * t * t) * (nr / nu) ** 2
    if kind == "cmb":   # the summand of a2t; y uses the GHz/Hz rule of a2t (nu0 <= 1e7 is read as GHz)
        y = np.where(nu > 1e7, LD(H) * nu, LD(H) * nu * LD(1e9)) / (LD(KB) * LD(th[0]))
        return np.expm1(y) ** 2 / (y * y * np.exp(y))
    if kind in ("T_cmb", "hi_fit"):   # B_nu(T) / compute_bnu_prime_RJ(nu) = h nu / (k (e^y - 1)), times 1e6
        y = LD(H) * nu / (LD(KB) * LD(th[0]))
        return LD(H) * nu / (LD(KB) * np.expm1(y)) * LD(1e6)
    raise ValueError(kind)


def _exact_sum(x):
    """Exact sum of long-double terms along the last axis, as a long double.  Each row is scaled by a power of two
    into the double range (a lognormal's far tail reaches 1e-500), split into two doubles and summed by math.fsum."""
    x = x.reshape(-1, x.shape[-1])
    scale = np.ldexp(LD(1), -np.frexp(np.max(np.abs(x), axis=1))[1].astype(np.int64))[:, None]
    scale[~np.isfinite(scale)] = 1
    y = x * scale
    hi = y.astype(np.float64)
    lo = (y - hi.astype(LD)).astype(np.float64)
    out = np.array([math.fsum(np.concatenate([a, b])) for a, b in zip(hi, lo)], dtype=LD)
    return out / scale[:, 0]


def ref_sed(kind, nu_c, nu, tau, th, nu_ref=None, t_cmb=2.7255):
    """Bandpass-integrated SED of `kind` for parameter arrays th (each (m,)): full table sum_i tau_i g(nu_i), or
    g(nu_c) for a delta band (nu empty).  'cmb' is 1 / a2t(band) at T_CMB = th[0]."""
    nu_ref = NU_REF[kind] if nu_ref is None else nu_ref
    th = tuple(np.atleast_1d(np.asarray(t, dtype=np.float64))[:, None] for t in th)
    if len(nu) == 0:
        nu, tau = np.array([nu_c]), np.array([1.0])
    keep = np.asarray(nu) != 0.0
    nu, tau = np.asarray(nu)[keep], np.asarray(tau)[keep]
    s = _exact_sum(np.asarray(tau, dtype=LD) * _terms(kind, nu, th, nu_ref))
    return 1 / s if kind == "cmb" else s


def mp_sed(kind, nu_c, nu, tau, th, nu_ref=None):
    """The same at 40 digits (one parameter point)."""
    import mpmath as mp
    mp.mp.dps = 40
    nu_ref = mp.mpf(NU_REF[kind] if nu_ref is None else nu_ref)
    h, kb = mp.mpf(H), mp.mpf(KB)
    th = [mp.mpf(float(t)) for t in th]
    if len(nu) == 0:
        nu, tau = [nu_c], [1.0]

    def g(v):
        if kind == "power-law":
            return (v / nu_ref) ** th[0]
        if kind == "mbb":
            z = h / (kb * th[1])
            return mp.expm1(z * nu_ref) / mp.expm1(z * v) * (v / nu_ref) ** (th[0] + 1)
        if kind == "freefree":
            def gaunt(x):
                return mp.log(mp.exp(mp.mpf(5.960) - mp.sqrt(3) / mp.pi * mp.log(x / 1e9 * (th[0] / 1e4) ** mp.mpf(-1.5)))
                              + mp.mpf(2.71828))
            return gaunt(v) / gaunt(nu_ref) * (nu_ref / v) ** 2
        if kind == "lognormal":
            t = mp.log(v / (th[0] * 1e9)) / th[1]
            return mp.exp(-t * t / 2) * (nu_ref / v) ** 2
        if kind == "cmb":
            y = (h * v if v > 1e7 else h * v * 1e9) / (kb * th[0])
            return mp.expm1(y) ** 2 / (y * y * mp.exp(y))
        y = h * v / (kb * th[0])
        return h * v / (kb * mp.expm1(y)) * 1e6

    s = mp.fsum(mp.mpf(float(t)) * g(mp.mpf(float(v))) for t, v in zip(tau, nu) if v != 0.0)
    return 1 / s if kind == "cmb" else s


# ------------------------------------------------------------------ bands
def tophat(nu_c, hw, n=128):
    """n equal weights log-spaced over nu_c exp([-hw, hw]) (edges pulled in by 1e-12 so that exp / log rounding
    keeps them inside the library's limit |ln(nu / nu_c)| <= 0.25)."""
    hw = hw * (1.0 - 1e-12)
    return nu_c, nu_c * np.exp(np.linspace(-hw, hw, n)), np.full(n, 1.0 / n)


def synth_c3(nu_c):
    from dang_b200.synth import _tabulated_band
    b = _tabulated_band(nu_c / 1e9, 128)
    return nu_c, b.bp_nu_ghz * 1e9, b.bp_tau / b.bp_tau.sum()


def jagged(nu_c, seed=31, n=97):
    """Random weights on unequal spacing over +-12 %, a sample at nu = 0 (skipped) and zero weights."""
    rng = np.random.default_rng(seed)
    nu = np.sort(nu_c * (1.0 + 0.12 * (2.0 * rng.random(n) - 1.0)))
    tau = rng.random(n) ** 3 + 0.01 * (rng.random(n) < 0.3)
    tau[rng.random(n) < 0.1] = 0.0
    nu[0] = 0.0
    return nu_c, nu, tau / tau.sum()


CENTRES_GHZ = (20.0, 30.0, 44.0, 70.0, 100.0, 143.0, 217.0, 353.0, 545.0, 857.0, 1000.0)
SHAPES = {"c3": synth_c3, "hw0.05": lambda c: tophat(c, 0.05), "hw0.15": lambda c: tophat(c, 0.15),
          "hw0.25": lambda c: tophat(c, 0.25), "jagged": jagged, "n17": lambda c: tophat(c, 0.15, 17)}


def grid(kind, n):
    """n points per dimension over the parameter box, corners included."""
    axes = [np.linspace(lo, hi, n) for lo, hi in BOXES[kind]]
    return tuple(a.ravel() for a in np.meshgrid(*axes, indexing="ij"))


def rule(nu_c, nu, tau, nq=8):
    from dang_b200 import _lib
    lib = _lib.load()
    dp = lambda a: a.ctypes.data_as(_lib.c_dp)
    nu, tau = np.ascontiguousarray(nu, dtype=np.float64), np.ascontiguousarray(tau, dtype=np.float64)
    nq_nu, nq_w = np.zeros(nq), np.zeros(nq)
    rc = lib.dang_gpu_bandpass_quadrature(nu_c, len(nu), dp(nu), dp(tau), nq, dp(nq_nu), dp(nq_w))
    return (nq_nu, nq_w) if rc == 0 else None


def expected_samples(nu_c, nu, tau, points, nq0=8, nq_max=32):
    """The samples a handle serves a tabulated band with, restated from the reference: the smallest rule of nq0,
    nq0 + 4, ... nodes whose sum is within 1e-14 (relative) of the full table's at every (kind, th, nu_ref) point;
    n_bp (the table) when no rule can be built first; None when no rule up to nq_max nodes passes (the library tries
    up to n_bp / 2, this restatement up to the 32 nodes dang_gpu_bandpass_quadrature builds)."""
    full = [ref_sed(k, nu_c, nu, tau, th, nu_ref=nr) for k, th, nr in points]
    for nq in range(nq0, nq_max + 1, 4):
        if 2 * nq > len(nu):
            return len(nu)
        q = rule(nu_c, nu, tau, nq)
        if q is None:
            return len(nu)
        if all(np.all(np.abs(ref_sed(k, nu_c, q[0], q[1], th, nu_ref=nr) / f - 1) <= 1e-14)
               for (k, th, nr), f in zip(points, full)):
            return nq
    return None


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("kind", TYPES)
def test_reference_agrees_with_mpmath(kind):
    """The long-double reference against 40-digit mpmath at the corners (and centre) of the parameter box, on
    delta bands and tabulated bands from 20 to 1000 GHz: a few hundred points per type."""
    import mpmath
    pts = [p for p in zip(*grid(kind, 5 if len(BOXES[kind]) == 1 else 3))]
    worst = 0.0
    n = 0
    for nu_ghz in CENTRES_GHZ:
        for band in ((nu_ghz * 1e9, np.zeros(0), np.zeros(0)), tophat(nu_ghz * 1e9, 0.25, 24),
                     jagged(nu_ghz * 1e9, seed=int(nu_ghz), n=24)):
            for p in pts:
                r = ref_sed(kind, band[0], band[1], band[2], p)[0]
                m = LD(mpmath.nstr(mp_sed(kind, band[0], band[1], band[2], p), 25))
                worst = max(worst, float(abs((r - m) / m)))
                n += 1
    print(f"{kind}: {n} points, worst |ref - mpmath| / |mpmath| = {worst:.2e}")
    assert n >= 150
    # ~ 1e-19 per operation; the lognormal's exp(-t^2/2) at t ~ 50 amplifies it by t^2 / 2 ~ 1e3
    assert worst < 1e-15, worst


def test_reference_on_the_c3_bands_matches_the_numpy_sums():
    """The reference restates band_sed (dang_b200.synth) for the c3 types: a float64 sum agrees to ~1e-15."""
    from dang_b200.synth import band_sed, make_config
    cfg = make_config("c3", nside=4)
    for b in cfg.bands:
        nu_c, nu, tau = b.nu_ghz * 1e9, b.bp_nu_ghz * 1e9, b.bp_tau / b.bp_tau.sum()
        assert abs(ref_sed("power-law", nu_c, nu, tau, (-3.1,))[0] / band_sed(b, cfg.comps[0], -3.1) - 1) < 1e-14
        assert abs(ref_sed("mbb", nu_c, nu, tau, (1.55, 19.6))[0] / band_sed(b, cfg.comps[1], 1.55, 19.6) - 1) < 1e-14


def eight_node_errors():
    """worst relative error of the 8-node rule against the full table, per (type, shape, centre)."""
    out = {}
    for shape, make in SHAPES.items():
        for nu_ghz in CENTRES_GHZ:
            nu_c, nu, tau = make(nu_ghz * 1e9)
            q = rule(nu_c, nu, tau)
            assert q is not None, (shape, nu_ghz)
            for kind in TYPES:
                th = grid(kind, 5)
                full = ref_sed(kind, nu_c, nu, tau, th)
                quad = ref_sed(kind, nu_c, q[0], q[1], th)
                out[kind, shape, nu_ghz] = float(np.max(np.abs(quad / full - 1.0)))
    return out


def test_eight_node_rule_domain():
    """Where 8 Gauss nodes reproduce the full table to 1e-14 and where they do not, over every SED type's
    parameter box, band centres 20-1000 GHz, the c3 shape, top-hats of half-width 0.05 / 0.15 / 0.25 in ln nu, a
    jagged table and the shortest table the rule accepts (n_bp = 17)."""
    err = eight_node_errors()
    for shape in SHAPES:
        print(shape.ljust(7), " ".join(f"{k}:{max(err[k, shape, c] for c in CENTRES_GHZ):.0e}" for k in TYPES))
    # the slowly varying SEDs: every shape, every centre, every corner of the box
    for kind in ("power-law", "freefree", "mbb", "hi_fit"):
        assert max(v for (k, _, _), v in err.items() if k == kind) < 1e-14, kind
    # B_nu / RJ at T = 2.6 K is a Wien tail above ~300 GHz: e^{-h nu / kT} spans h nu / kT ~ 10 across a wide band
    assert max(v for (k, s, c), v in err.items() if k == "T_cmb" and c <= 353.0) < 1e-14
    assert err["T_cmb", "hw0.25", 1000.0] > 1e-13
    # 'cmb' is not slowly varying: (e^y - 1)^2 / (y^2 e^y) grows like e^y, y = h nu / kT_CMB = 15 at 857 GHz
    assert 1e-8 < err["cmb", "hw0.25", 857.0] < 1e-7            # 4.0e-8 over T_CMB 2.6-2.8 K
    assert 1e-10 < err["cmb", "hw0.25", 545.0] < 1e-9
    assert 1e-12 < err["cmb", "c3", 857.0] < 1e-10
    assert max(err["cmb", s, c] for s in SHAPES for c in CENTRES_GHZ if c <= 143.0) < 1e-14
    # nor is a narrow lognormal, exp(-ln^2(nu / nu_p) / 2 w^2): at w = 0.1 it changes by e^{-3} across a band of
    # half-width 0.25 near nu_p, and far from nu_p (1e-500 at 1000 GHz) the rule misses by O(1) relative
    assert err["lognormal", "hw0.25", 30.0] > 1e-7
    assert max(v for (k, _, _), v in err.items() if k == "lognormal") > 0.1


def test_expected_samples_of_the_named_cases():
    """The rule sizes the library's verification should settle on: 'cmb' at 857 GHz needs 12 nodes on the c3 shape
    and 16 on a top-hat of half-width 0.25; a lognormal at nu_p = 30 GHz, w = 0.1 on a 30 GHz top-hat of half-width
    0.25 needs 16; the same lognormal 34 widths into its tail at 857 GHz needs more than 32."""
    cmb = [("cmb", ([2.7255],), 100e9)]
    ame = [("lognormal", ([30.0], [0.1]), 22e9)]
    assert expected_samples(*synth_c3(857e9), cmb) == 12
    assert expected_samples(*tophat(857e9, 0.25), cmb) == 16
    assert expected_samples(*tophat(30e9, 0.25), ame + cmb) == 16
    assert expected_samples(*tophat(857e9, 0.25), ame + cmb) is None
    assert expected_samples(*tophat(30e9, 0.25), [("lognormal", ([30.0], [1.0]), 22e9)] + cmb) == 8


def test_lognormal_and_cmb_rows_of_the_domain():
    """The two named cases one parameter point at a time: lognormal nu_p = 30 GHz, w = 0.1 at nu_p (2e-6) and
    w = 0.3 on the c3 shape at 353 GHz (3e-10), both far above 1e-14; 12 nodes bring the second to ~1e-15."""
    nu_c, nu, tau = tophat(30e9, 0.25)
    q = rule(nu_c, nu, tau)
    e = abs(ref_sed("lognormal", nu_c, *q, (30.0, 0.1))[0] / ref_sed("lognormal", nu_c, nu, tau, (30.0, 0.1))[0] - 1)
    assert 5e-7 < e < 1e-5, e
    nu_c, nu, tau = synth_c3(353e9)
    for nq, lo, hi in ((8, 1e-11, 1e-9), (12, 0.0, 1e-14)):
        q = rule(nu_c, nu, tau, nq)
        e = abs(ref_sed("lognormal", nu_c, *q, (30.0, 0.3))[0] / ref_sed("lognormal", nu_c, nu, tau, (30.0, 0.3))[0] - 1)
        assert lo < e < hi, (nq, e)
