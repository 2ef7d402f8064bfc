"""The error budget of the screened per-pixel Metropolis kernel (dang_b200/csrc/kernels_mh_pix.cuh), checked on the CPU.

The kernel decides a proposal from a single-precision evaluation of lnL(theta') - lnL(cur) whenever that value is further
from ln u than an error bound `eps` it carries along; the claim "the decisions are the fp64 kernel's" rests on
|screened difference - exact difference| <= eps for EVERY proposal.  On the GPU the record mode checks exactly that on
the parity cases (tests/test_gpu_parity.py).  This file restates the kernel's single-precision arithmetic step by step
in numpy float32 (state {2P, Q, e_P} per band, degree-9 exp(x) - 1 polynomial, accept update, rescaled Planck factors in
T mode, the growth of e_P / eps_Q / kappa) and compares it with a float64 evaluation from the data over a much wider
range of signal-to-noise ratios, step sizes, band counts and chain lengths than the GPU cases cover.  numpy rounds every
operation where the GPU fuses multiply-adds, so this is the same algorithm with slightly MORE rounding, not the same
bits."""
import numpy as np
import pytest

f32 = np.float32
KAPPA_BETA, KAPPA_T = f32(1.0e-6), f32(1.5e-6)
H_OVER_K = 6.62607015e-34 / 1.380649e-23


def em1_poly(x):
    """k5p_em1: Taylor of exp(x) - 1 to x^9, Horner, float32."""
    x = x.astype(f32)
    p = x * f32(1.0 / 362880.0) + f32(1.0 / 40320.0)
    for c in (1.0 / 5040.0, 1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5, 1.0):
        p = p * x + f32(c)
    return (p * x).astype(f32)


def template_width(B):
    """NB of the mh_perpixel_pix_kernel<NB, MODE> instance host_mh_ppx.cu launches for B bands."""
    return next(nb for nb in (8, 12, 20, 32) if B <= nb)


def run_chains(mode, B, S, npix, nprop, step, snr, seed, NB, accept_rule="metropolis"):
    """B data bands in a kernel instance NB bands wide: bands B..NB-1 are the instance's padding, which the kernel
    runs through every sum (state {0, 0, 0}; frequency factor 0 for beta, the reference's for T, so rho = 0
    exactly) and whose b_j enters b_max; the sum's rounding term is (NB + 4) 2^-24."""
    assert B <= NB
    rng = np.random.default_rng(seed)
    nu = np.exp(np.linspace(np.log(20.0), np.log(857.0), B)) * 1e9
    nu_ref = 353e9
    L = np.log(nu / nu_ref)                                    # float64
    beta0, T0 = 1.5 + 0.1 * rng.standard_normal(npix), 19.0 + 1.5 * rng.standard_normal(npix)

    def sed(beta, T):                                          # mbb, float64: [npix, B]
        z = H_OVER_K / T[:, None]
        return np.expm1(z * nu_ref) / np.expm1(z * nu[None, :]) * np.exp((beta[:, None] + 1.0) * L[None, :])

    amp = snr * (0.2 + rng.random((npix, S))) * rng.choice([-1.0, 1.0], (npix, S))
    sigma = 0.5 + rng.random((npix, B, S))
    truth = sed(beta0 + 0.05 * rng.standard_normal(npix), T0 + 0.5 * rng.standard_normal(npix))
    D = amp[:, None, :] * truth[:, :, None] + sigma * rng.standard_normal((npix, B, S))

    def lnl(beta, T):                                          # exact, float64
        r = (D - amp[:, None, :] * sed(beta, T)[:, :, None]) / sigma
        return -0.5 * np.sum(r * r, axis=(1, 2))

    cur_b, cur_T = beta0.copy(), T0.copy()
    s_cur = sed(cur_b, cur_T)
    t = (D - amp[:, None, :] * s_cur[:, :, None]) / sigma
    g = amp[:, None, :] * s_cur[:, :, None] / sigma
    pad = np.zeros((npix, NB - B), dtype=f32)
    P2 = np.hstack([(2.0 * np.sum(g * t, axis=2)).astype(f32), pad])   # state at the chain's first point: fp64 -> fp32
    Q = np.hstack([np.sum(g * g, axis=2).astype(f32), pad])
    eP = np.hstack([(1.0e-7 * 2.0 * np.sum(np.abs(g * t), axis=2)).astype(f32) + f32(1e-37), pad])
    epsQ = np.full(npix, 1.2e-7, dtype=f32)
    kappa = KAPPA_T if mode == "T" else KAPPA_BETA
    kap = np.full(npix, kappa, dtype=f32)
    c_round = f32((NB + 4) * 5.97e-8)
    if mode == "T":
        cref = f32(H_OVER_K * nu_ref)
        cf = np.concatenate([(H_OVER_K * nu).astype(f32), np.full(NB - B, cref, dtype=f32)])
        kref1 = (1.0 / np.expm1(H_OVER_K * nu_ref / cur_T)).astype(f32)
        kjs = np.hstack([(1.0 / np.expm1(H_OVER_K * nu[None, :] / cur_T[:, None])).astype(f32),
                         np.repeat(kref1[:, None], NB - B, axis=1)])
    else:
        cf = np.concatenate([L.astype(f32), np.zeros(NB - B, dtype=f32)])
    worst, n_checked, n_big = 0.0, 0, 0
    for _ in range(nprop):
        z = rng.standard_normal(npix)
        if mode == "T":
            x = cur_T + step * z
            x = np.where(x < 5.0, cur_T, x)                     # (out of bounds: no move, rho = 0)
            d = ((cur_T - x) / (x * cur_T)).astype(f32)
            e1 = em1_poly(cref * d)
            n1 = (kref1 * e1 + e1).astype(f32)
            arg = np.abs(d)[:, None] * np.maximum(cf, cref)[None, :]
        else:
            x = cur_b + step * z
            d = (x - cur_b).astype(f32)
            arg = np.abs(d)[:, None] * np.abs(cf)[None, :]
        small = np.all(arg < 0.7, axis=1)                       # the hot form's range; others take the general form
        n_big += int((~small).sum())
        lam = np.zeros(npix, dtype=f32); E1 = lam.copy(); W = lam.copy(); SP = lam.copy(); bmax = lam.copy()
        rho_all = np.zeros((npix, NB), dtype=f32)
        for j in range(NB):
            if mode == "T":
                e = em1_poly(cf[j] * d)
                n2 = (kjs[:, j] * e + e).astype(f32)
                inv = (f32(1.0) / (f32(1.0) + n2)).astype(f32)
                rho = ((n1 - n2) * inv).astype(f32)
                b = ((np.abs(n1) + np.abs(n2)) * inv).astype(f32)
            else:
                xx = (d * cf[j]).astype(f32)
                rho = em1_poly(xx)
                b = (np.abs(rho) * np.abs(xx) + np.abs(rho)).astype(f32)
            ar = np.abs(rho)
            m = (ar * Q[:, j] + np.abs(P2[:, j])).astype(f32)
            lam = (rho * (P2[:, j] - rho * Q[:, j]).astype(f32) + lam).astype(f32)
            E1 = (b * m + E1).astype(f32)
            W = (ar * m + W).astype(f32)
            SP = (ar * eP[:, j] + SP).astype(f32)
            bmax = np.maximum(bmax, b)
            rho_all[:, j] = rho
        assert not rho_all[:, B:].any()                          # padding bands: rho = 0 exactly
        eps = (f32(0.55) * (f32(2.0) * kap * E1 + (c_round + epsQ) * W + SP)).astype(np.float64)
        new_b, new_T = (cur_b, x) if mode == "T" else (x, cur_T)
        diff = lnl(new_b, new_T) - lnl(cur_b, cur_T)
        err = np.abs(0.5 * lam.astype(np.float64) - diff)
        scale = np.maximum(1.0, np.abs(lnl(cur_b, cur_T)))
        ok = small & np.isfinite(eps)
        bad = ok & (err > eps + 1e-13 * scale)
        assert not bad.any(), (mode, B, S, step, snr, float(err[bad].max()), float(eps[bad].min()), int(bad.sum()))
        worst = max(worst, float(np.max(np.where(ok & (eps > 0), err / np.maximum(eps, 1e-300), 0.0))))
        n_checked += int(ok.sum())
        # accept: the Metropolis rule on the exact difference, or a coin (walks further from the first point)
        u = rng.random(npix)
        acc = (diff > np.log(u)) if accept_rule == "metropolis" else (u < 0.5)
        acc &= small & (x != (cur_T if mode == "T" else cur_b))
        if not acc.any():
            continue
        a = acc
        kbm = (f32(1.1) * kap * bmax).astype(f32)
        c2 = (f32(1.1) * epsQ).astype(f32)
        if mode == "T":
            inv1 = (f32(1.0) / (f32(1.0) + n1)).astype(f32)
        opmin = np.ones(npix, dtype=f32)
        for j in range(NB):
            rho = rho_all[:, j]
            op = (f32(1.0) + rho).astype(f32)
            q2 = ((rho + rho) * Q[:, j]).astype(f32)
            aq2 = np.abs(q2)
            mm = (np.abs(P2[:, j]) + aq2).astype(f32)
            t1 = (aq2 * c2 + mm * f32(2.2e-7)).astype(f32)
            t2 = (op * (Q[:, j] + Q[:, j]) + mm).astype(f32)
            eP_n = ((op * f32(1.000001)) * eP[:, j] + (kbm * t2 + op * t1)).astype(f32) + f32(1e-37)
            P2_n = (op * (P2[:, j] - q2)).astype(f32)
            Q_n = (op * op * Q[:, j]).astype(f32)
            eP[:, j] = np.where(a, eP_n, eP[:, j])
            P2[:, j] = np.where(a, P2_n, P2[:, j])
            Q[:, j] = np.where(a, Q_n, Q[:, j])
            opmin = np.minimum(opmin, np.where(a, op, f32(1.0)))
            if mode == "T":
                kjs[:, j] = np.where(a, (kjs[:, j] * (op * inv1)).astype(f32), kjs[:, j])
        epsQ = np.where(a, (epsQ + f32(4.0) * kap * bmax + f32(2.5e-7)).astype(f32), epsQ)
        epsQ = np.where(a & ~(opmin > 0.5), f32(np.inf), epsQ)
        if mode == "T":
            kref1 = np.where(a, (kref1 * inv1).astype(f32), kref1)
            kap = np.where(a, (kap + f32(4.0) * kap * bmax + f32(5.0e-7)).astype(f32), kap)
            cur_T = np.where(a, x, cur_T)
        else:
            cur_b = np.where(a, x, cur_b)
    return worst, n_checked, n_big


@pytest.mark.parametrize("accept_rule", ["metropolis", "coin"])
@pytest.mark.parametrize("mode,step", [("beta", 0.01), ("beta", 0.05), ("beta", 0.15), ("T", 0.2), ("T", 0.5), ("T", 1.5)])
# every template width: NB 8 (B 5, 8), NB 12 (B 9, 12), NB 20 (B 20), NB 32 (B 21, 32); padded and full instances
@pytest.mark.parametrize("B,S,snr", [(5, 2, 3.0), (8, 2, 100.0), (20, 2, 1.0e4), (20, 1, 30.0), (9, 2, 30.0),
                                     (12, 1, 1.0e4), (21, 2, 100.0), (32, 2, 1.0e4), (32, 1, 3.0)])
def test_screened_difference_stays_inside_its_bound(mode, step, B, S, snr, accept_rule):
    worst, n, n_big = run_chains(mode, B, S, npix=400, nprop=40, step=step, snr=snr, seed=B * 1000 + S,
                                 NB=template_width(B), accept_rule=accept_rule)
    assert n > 0.5 * 400 * 40          # most proposals are in the hot form's range and were checked
    assert worst <= 1.0, worst


def test_the_bound_is_not_vacuous():
    """The bound is conservative but not absurdly so: the worst observed error is within two orders of magnitude of
    it (measured: err / eps between 0.03 and 0.08 over all cases above), so the fallback stays rare."""
    for mode, step, B, snr in [("beta", 0.05, 8, 100.0), ("T", 0.5, 20, 30.0)]:
        worst, n, _ = run_chains(mode, B, 2, npix=300, nprop=20, step=step, snr=snr, seed=7, NB=template_width(B))
        assert 0.01 < worst <= 1.0, worst
