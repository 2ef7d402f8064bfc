"""Production-mode randomness: every sampler drawing its own deviates, against the Philox definition and against the
exact per-pixel posterior.

Called without `eta` / `z` / `u` (as the Fortran shim's production path and bench.py do), every kernel draws its
deviates from Philox4x32-10.  The definition is common.cuh (`philox_uniform2`, `philox_normal`, the DG_STREAM_*
ids) and DESIGN.md section 4.5; the oracle restates it independently (`ora_philox_*`).  Slots are global pixel
numbers, so a sharded run draws what one GPU draws:

    eta of a CG solve     stream 1, slot s * npix + pix                  (S = 1 for a T, Q or U flag)
    per-pixel z / u       streams 2 / 3, slot l * npix + pix             ('prior' draws: z at slot pix)
    full-sky z / u        streams 2 / 3, slot l
    step-size tuner z / u streams 4 / 5, slot blk * nsample + l
    band gain             stream 6, slot band

Engine's seed schedule of one Gibbs iteration (dang_b200/engine.py) is restated beside it.  The oracle is fed the
arrays this restatement builds, so a wrong slot, stream, uniform or seed in any kernel shows up as a different
decision or amplitude.  tests/multi_gpu_check.py (case 'rng') runs the Gibbs loop on two ring-partitioned ranks.

test_perpixel_chain_keeps_the_exact_posterior does not use the oracle: a Metropolis chain started in its target
distribution stays in it, so the kernels' final indices must pass a Kolmogorov-Smirnov test against the posterior
computed by quadrature.  It pins the accept rule, prior and bounds that kernels and oracle could misread together.

test_every_rng_call_site_is_covered (no GPU) fails when a Philox call site appears under dang_b200/csrc that
RNG_SITES does not map to a test case here."""
import os
import re

import numpy as np
import pytest

from conftest import TOL, rel_err
from helpers import intensity_case, small_case, template_case
from test_gpu_shapes import CSRC, FS_CASES, ODD_RANGE, PP_FAMILIES, ROOT, SED, shape_case

STREAM_ETA, STREAM_MH_Z, STREAM_MH_U, STREAM_TUNE_Z, STREAM_TUNE_U, STREAM_GAIN = 1, 2, 3, 4, 5, 6
TUNE_MAX_BLOCKS = 1000  # what Engine.sample_spectral_parameters passes to the tuner


# ------------------------------------------------------------------ 1. the slot layout, host side
def eta_draw(seed, S, npix):
    """The normals of one CG solve with S planes."""
    from oracle.binding import philox_normals
    return philox_normals(seed, STREAM_ETA, 0, S * npix)


def perpixel_draw(seed, nsample, npix):
    """(z, u) of a per-pixel Metropolis draw, [l][pix]."""
    from oracle.binding import philox_normals, philox_uniforms
    return philox_normals(seed, STREAM_MH_Z, 0, nsample * npix), philox_uniforms(seed, STREAM_MH_U, 0, nsample * npix)


def fullsky_draw(seed, nsample):
    from oracle.binding import philox_normals, philox_uniforms
    return philox_normals(seed, STREAM_MH_Z, 0, nsample), philox_uniforms(seed, STREAM_MH_U, 0, nsample)


def tuner_draw(seed, nsample, max_blocks):
    """(z, u) of tune_spectral_parameter_length, [blk][l]."""
    from oracle.binding import philox_normals, philox_uniforms
    n = nsample * max_blocks
    return philox_normals(seed, STREAM_TUNE_Z, 0, n), philox_uniforms(seed, STREAM_TUNE_U, 0, n)


def gain_draw(seed, band):
    from oracle.binding import philox_normals
    return float(philox_normals(seed, STREAM_GAIN, band, 1)[0])


def cg_seed(seed, it, ig, f):
    """Engine.gibbs_iteration -> sample_cg_groups: solve of (group ig, flag f)."""
    return seed + 2 * it + 1000003 * (3 * ig + f)


def draw_seed(seed, it, ncall):
    """Engine.gibbs_iteration -> sample_spectral_parameters: the ncall-th sample_index_mh of the iteration."""
    return seed + 2 * it + 1 + 7919 * ncall


def tune_seed(seed, it, ncall):
    """... and the step-size tuner run before that call when the index is not tuned yet."""
    return seed + 2 * it + 1 + 104729 * (ncall + 1)


def oracle_gibbs_iteration(ora, cfg, it, seed, tuned):
    """The oracle's side of Engine.gibbs_iteration(it, seed=seed) with the device's deviates: sample_cg_group per
    sampled group, then (it > 1) tune_step where `tuned` says so and sample_index_mh per (component, index, flag).
    Returns (CG iteration counts, chi-square after the amplitudes, acceptances, chi-square after the indices,
    decisions of the last draw)."""
    from dang_b200.config import flag_to_map_n, return_poltype_flag
    n_cg = []
    for ig, g in enumerate(cfg.cg_groups):
        if not g.sample:
            continue
        flags = return_poltype_flag(g.poltype)
        eta = np.concatenate([eta_draw(cg_seed(seed, it, ig, f), 2 if fl & 8 else 1, cfg.npix)
                              for f, fl in enumerate(flags)])
        its, _ = ora.sample_cg_group(ig, 1, eta)
        n_cg += its
    chisq_cg = ora.compute_chisq()[0]
    if it == 1:
        return n_cg, chisq_cg, None, None, None
    nsample, acc, ncall, dec = cfg.nsample, [], 0, None
    for ic, c in enumerate(cfg.comps):
        if not c.indices or not any(s.sample for s in c.indices):
            continue
        for j, s in enumerate(c.indices):
            if not s.sample:
                continue
            for flag in return_poltype_flag(s.poltype):
                map_n = flag_to_map_n(flag)
                if not tuned[ic][j] and s.lnl_type != "prior":
                    z, u = tuner_draw(tune_seed(seed, it, ncall), nsample, TUNE_MAX_BLOCKS)
                    ora.tune_step(ic, j, map_n, nsample, 1, z, u, TUNE_MAX_BLOCKS, perpixel_start=s.region != "fullsky")
                    tuned[ic] = [True] * len(c.indices)
                sd = draw_seed(seed, it, ncall)
                z, u = fullsky_draw(sd, nsample) if s.region == "fullsky" else perpixel_draw(sd, nsample, cfg.npix)
                a, dec, _ = ora.sample_index_mh(ic, j, map_n, nsample, 1, z, u)
                acc.append(a)
                ncall += 1
    ora.update_sky_model()
    return n_cg, chisq_cg, acc, ora.compute_chisq()[0], dec


def test_philox_restatement_is_the_stream_layout():
    """The restatement above against ora_philox_uniform2 slot by slot (no GPU): a slot offset, a stream id or a
    u1 / u2 mix-up in the helpers would make every comparison below vacuous."""
    from oracle.binding import load
    import ctypes as C
    lib = load()

    def u12(seed, stream, slot):
        a, b = C.c_double(), C.c_double()
        lib.ora_philox_uniform2(seed, stream, slot, C.byref(a), C.byref(b))
        return a.value, b.value

    seed, npix, nsample = 987654321012, 48, 5
    z, u = perpixel_draw(seed, nsample, npix)
    for l, pix in ((0, 0), (3, 17), (4, 47)):
        u1, u2 = u12(seed, STREAM_MH_Z, l * npix + pix)
        assert z[l * npix + pix] == np.sqrt(-2.0 * np.log(u1)) * np.sin(2.0 * np.pi * u2)
        assert u[l * npix + pix] == u12(seed, STREAM_MH_U, l * npix + pix)[0]
    assert np.array_equal(fullsky_draw(seed, nsample)[0], perpixel_draw(seed, nsample, 1)[0])
    zt, ut = tuner_draw(seed, nsample, 3)
    assert ut[2 * nsample + 1] == u12(seed, STREAM_TUNE_U, 2 * nsample + 1)[0]
    assert zt.size == 3 * nsample and not np.array_equal(zt, fullsky_draw(seed, 3 * nsample)[0])
    assert gain_draw(seed, 3) == eta_like(seed, STREAM_GAIN, 3)
    eta = eta_draw(seed, 2, npix)
    assert eta[npix + 5] == eta_like(seed, STREAM_ETA, npix + 5)
    # Box-Muller of the definition: roughly standard normal, and the streams are distinct
    big = eta_draw(seed, 1, 200000)
    assert abs(big.mean()) < 0.01 and abs(big.std() - 1.0) < 0.01
    assert len({float(eta_like(seed, s, 7)) for s in range(1, 7)}) == 6
    assert cg_seed(5, 2, 0, 1) == 5 + 4 + 1000003 and draw_seed(5, 2, 1) == 5 + 5 + 7919
    assert tune_seed(5, 2, 0) == 5 + 5 + 104729


def eta_like(seed, stream, slot):
    from oracle.binding import philox_normals
    return float(philox_normals(seed, stream, slot, 1)[0])


# ------------------------------------------------------------------ 2. CG eta in production mode
def _masked(sky, pix_range):
    if pix_range:
        lo, hi = pix_range
        sky.mask[:lo] = 0.0
        sky.mask[hi:] = 0.0


def _cg_device(cfg, sky, options=(), pix_range=None, seeds=(1234567, 7654321), bordered=False, ig=0, flag_n=0):
    """Two consecutive solves (the second warm-starts from the first) with the device's eta against the oracle fed
    the Philox normals.  Bordered groups (template, monopole, hi_fit) are ill-conditioned: as in test_gpu_intensity
    their first residual norms and converged solutions are compared, at 1e-8, not the iteration count.  Only the
    cold start's residual norms: a warm start's r = b - A x0 cancels to a small part of A x0, and the 1e-15 that
    the two x0 differ by comes back amplified (measured on a B200 for monopole + hi_fit at nside 8: 1.5e-8 on the
    first norm of the second solve, against 6e-16 on the first solve's)."""
    from dang_b200.config import return_poltype_flag
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    _masked(sky, pix_range)
    lo, hi = pix_range or (0, cfg.npix)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky, pix_range=pix_range)
    for opt, v in options:
        eng.set_option(opt, v)
    S = 2 if return_poltype_flag(cfg.cg_groups[ig].poltype)[flag_n] & 8 else 1
    tol = 1e-8 if bordered else TOL
    worst = 0.0
    for seed in seeds:
        it_o, _, tr_o = ora.cg_search_trace(ig, flag_n, 1, eta_draw(seed, S, cfg.npix))
        it_g, _ = eng.cg_solve(ig, flag_n, "sample", eta=None, seed=seed)
        tr_g = eng.cg_trace()
        if bordered:
            if seed == seeds[0]:
                assert np.allclose(tr_g[:5], tr_o[:5], rtol=1e-7, atol=0)
        else:
            assert it_g == it_o, (it_g, it_o)
            assert np.allclose(tr_g, tr_o, rtol=1e-7, atol=0)
        for ic, c in enumerate(cfg.comps):
            if c.type in ("template", "monopole", "hi_fit"):
                e = rel_err(eng.template_amplitudes(ic), ora.template_amplitudes(ic))
            else:
                e = rel_err(eng.amplitude(ic)[:, lo:hi], ora.amplitude(ic)[:, lo:hi])
            worst = max(worst, e)
            assert e < tol, (seed, ic, e)
    if not pix_range and not bordered:
        assert rel_err(eng.cg_x(ig, flag_n), ora.cg_x(ig, flag_n)) < TOL
    print(f"worst amplitude error with device eta: {worst:.2e}")
    return worst


# (name, K1 path) -> builder; every eta call site of kernels_cg / kernels_stream / kernels_uni / kernels_tmpl runs
def _cg_case(name):
    from dang_b200.engine import OPT_CG_PERSISTENT, OPT_STREAM_RING, OPT_TMA
    if name == "ring_stream":   # config c2 as configured: ring-stream K1 inside the persistent solve
        cfg, sky = small_case("c2", 16, perturb=False)
        return cfg, sky, {}
    if name == "ring_plain":   # uniform indices without the cp.async ring: the uni K1 with nothing staged
        cfg, sky = small_case("c2", 16, perturb=False)
        return cfg, sky, dict(options=((OPT_STREAM_RING, 0),))
    if name == "tma":
        cfg, sky = small_case("c2", 16, perturb=False)
        return cfg, sky, dict(options=((OPT_TMA, 1),))
    if name in ("uni1", "uni2", "generic"):   # the '_cg' shapes of test_gpu_shapes
        B, varying = {"uni1": (9, ("synch",)), "uni2": (20, ("synch", "dust")), "generic": (21, ("synch", "dust"))}[name]
        cfg, sky = shape_case(B, ("synch", "dust"), varying=varying)
        return cfg, sky, dict(options=((OPT_CG_PERSISTENT, 1),))
    if name in ("plane_Q", "plane_U"):
        cfg, sky = shape_case(13, ("synch", "dust"), poltype=name[-1], varying=("synch",))
        return cfg, sky, {}
    if name == "uni2_odd_range":
        cfg, sky = shape_case(9, ("synch", "dust"), nside=8, varying=("synch", "dust"))
        return cfg, sky, dict(pix_range=ODD_RANGE)
    if name == "template":
        cfg, sky, _ = template_case(8)
        cfg.cg_groups[0].converge, cfg.cg_groups[0].max_iter = 1e-20, 300
        return cfg, sky, dict(bordered=True)
    if name == "monopole_hi_fit":
        from oracle.binding import load
        load().ora_set_T_CMB(2.7255)
        cfg, sky, _, _ = intensity_case(8, with_hi=True)
        cfg.cg_groups[0].converge, cfg.cg_groups[0].max_iter = 1e-22, 2000
        return cfg, sky, dict(bordered=True)
    raise ValueError(name)


CG_DEVICE_CASES = ("ring_stream", "ring_plain", "tma", "uni1", "uni2", "generic", "plane_Q", "plane_U", "uni2_odd_range",
                   "template", "monopole_hi_fit")


@pytest.mark.gpu
@pytest.mark.parametrize("name", CG_DEVICE_CASES)
def test_cg_device_eta(name):
    """The device normals are r * sinpi(2 u2), the oracle's r * sin(2 pi u2): they differ by an ulp or so, which
    leaves the amplitudes well inside TOL = 1e-10 (the printed worst error)."""
    cfg, sky, kw = _cg_case(name)
    _cg_device(cfg, sky, **kw)


# ------------------------------------------------------------------ 3. Metropolis z / u in production mode
def _perpixel_device(family, cfg, sky, ic, nind, map_n, nsample=12, seed=424242, pix_range=None, compare_lnl=True):
    """A per-pixel draw with the device's z / u against the oracle fed the Philox arrays.  Record mode accepts
    device deviates, so decisions are compared too; the split form runs only without recording (its index maps
    and acceptance are compared)."""
    from dang_b200.engine import OPT_PERPIXEL_FAST, OPT_PERPIXEL_SERIAL, OPT_RECORD, Engine
    from oracle.binding import Oracle
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region = True, "per-pixel"
    _masked(sky, pix_range)
    lo, hi = pix_range or (0, cfg.npix)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky, pix_range=pix_range)
    split = family == "split"
    eng.set_option(OPT_RECORD, int(not split))
    eng.set_option(OPT_PERPIXEL_SERIAL, 0 if split else PP_FAMILIES[family]["serial"])
    eng.set_option(OPT_PERPIXEL_FAST, 2 if split else PP_FAMILIES[family]["fast"])
    z, u = perpixel_draw(seed, nsample, cfg.npix)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, map_n, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(ic, nind, map_n, nsample, "sample", seed=seed)
    assert acc_g == acc_o, (acc_g, acc_o)
    if spec.lnl_type != "prior":
        assert 0 < acc_o
    if not split:
        dec_g, lnl_g = eng.decisions(nsample, fullsky=False)
        dec_g, lnl_g = dec_g.reshape(nsample, -1)[:, lo:hi], lnl_g.reshape(nsample, -1)[:, lo:hi]
        dec_o, lnl_o = dec_o.reshape(nsample, -1)[:, lo:hi], lnl_o.reshape(nsample, -1)[:, lo:hi]
        assert np.array_equal(dec_g, dec_o), f"{(dec_g != dec_o).sum()} decisions differ"
        ev = dec_o < 2
        if compare_lnl and ev.any():
            assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL
    assert rel_err(eng.indices(ic)[:, :, lo:hi], ora.indices(ic)[:, :, lo:hi]) < 1e-14
    return eng


# (family, SED mode, S): every per-pixel form, every SED mode, S = 2 and S = 1 on Q or U
PP_DEVICE_CASES = [(f, sed, m) for f in ("pixel", "lane", "fp64", "serial", "split") for sed, m in
                   zip(SED, (-1, 2, 3) if f in ("pixel", "fp64", "split") else (3, -1, 2))]


@pytest.mark.gpu
@pytest.mark.parametrize("family,sed,map_n", PP_DEVICE_CASES)
def test_perpixel_device_deviates(family, sed, map_n):
    ic, nind = SED[sed]
    cfg, sky = shape_case(9)
    _perpixel_device(family, cfg, sky, ic, nind, map_n)


@pytest.mark.gpu
def test_perpixel_device_deviates_odd_pixel_range():
    """Odd pix_lo: a kernel that draws at its local pixel p instead of pix_lo + p differs on every pixel."""
    for family in ("pixel", "lane"):
        cfg, sky = shape_case(17, nside=8)
        _perpixel_device(family, cfg, sky, 0, 0, -1, pix_range=ODD_RANGE)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["marginal", "prior"])
def test_perpixel_device_deviates_strict_variants(variant):
    """The strict kernel's marginal likelihood, and the 'prior' draw whose single normal sits at slot pix."""
    cfg, sky = small_case("c1", 8)
    cfg.comps[0].indices[0].lnl_type = variant
    _perpixel_device("fp64", cfg, sky, 0, 0, -1, nsample=8)


@pytest.mark.gpu
def test_perpixel_device_deviates_bandpass_series():
    """Config c3 (tabulated bandpasses): the moment-series chains."""
    cfg, sky = small_case("c3", 8)
    _perpixel_device("lane", cfg, sky, 0, 0, -1, nsample=16)
    cfg, sky = small_case("c3", 8)
    _perpixel_device("lane", cfg, sky, 1, 0, -1, nsample=16)


def _fs_pick():
    picked = []
    for family in ("ring", "uni", "stream"):
        for ns in (24, 200):
            picked.append(next(c for c in FS_CASES if c[0] == family and c[3] == ns))
    return picked


@pytest.mark.gpu
@pytest.mark.parametrize("family,B,map_n,nsample,ncomp,sed", _fs_pick())
def test_fullsky_device_deviates(family, B, map_n, nsample, ncomp, sed):
    from dang_b200.engine import OPT_FULLSKY_STREAM, OPT_RECORD, OPT_STREAM_RING, Engine
    from oracle.binding import Oracle
    from test_gpu_shapes import COMPS
    ic, nind = SED[sed]
    cfg, sky = shape_case(B, COMPS[:ncomp], varying=())
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region, spec.step = True, "fullsky", (0.002, 0.02)[nind]
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eng.set_option(OPT_STREAM_RING, int(family != "uni"))
    eng.set_option(OPT_FULLSKY_STREAM, int(family == "stream"))
    eng.set_option(OPT_RECORD, 1)
    seed = 31337 + B
    z, u = fullsky_draw(seed, nsample)
    acc_o, dec_o, _ = ora.sample_index_mh(ic, nind, map_n, nsample, 1, z, u)
    acc_g = eng.sample_index_mh(ic, nind, map_n, nsample, "sample", seed=seed)
    dec_g, _ = eng.decisions(nsample, fullsky=True)
    assert np.array_equal(dec_g, dec_o[:nsample]), (dec_g, dec_o[:nsample])
    assert acc_g == acc_o and 0 < acc_o
    assert eng.index_fullsky(ic, nind, 2 if map_n == -1 else map_n) == ora.indices(ic)[nind, 1 if map_n == -1 else map_n - 1, 0]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["marginal", "jeffreys", "prior_draw"])
def test_fullsky_device_deviates_rare_variants(variant):
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 16, perturb=False)
    spec = cfg.comps[0].indices[0]
    spec.sample, spec.region, spec.step = True, "fullsky", 0.01
    if variant == "marginal":
        spec.lnl_type = "marginal"
    elif variant == "jeffreys":
        spec.prior = "jeffreys"
    else:
        spec.lnl_type = "prior"
    rng = np.random.default_rng(17)
    for c in cfg.comps:
        sky.amplitude[c.label][1:3] = sky.truth[c.label][1:3] * (1.0 + 0.05 * rng.standard_normal((2, cfg.npix)))
    nsample, seed = 16, 55
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    z, u = fullsky_draw(seed, nsample)
    acc_o, dec_o, _ = ora.sample_index_mh(0, 0, -1, nsample, 1, z, u)
    acc_g = eng.sample_index_mh(0, 0, -1, nsample, "sample", seed=seed)
    assert acc_g == acc_o
    assert eng.index_fullsky(0, 0, 2) == ora.indices(0)[0, 1, 0]
    if variant == "prior_draw":
        assert ora.indices(0)[0, 1, 0] == spec.gauss[0] + spec.gauss[1] * z[0]
    else:
        dec_g, _ = eng.decisions(nsample, fullsky=True)
        assert np.array_equal(dec_g, dec_o[:nsample]) and 0 < acc_o


@pytest.mark.gpu
@pytest.mark.parametrize("start", ["fullsky", "perpixel"])
def test_tuner_device_deviates(start):
    """tune_spectral_parameter_length on streams 4 / 5: the same blocks and the same step as the oracle."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    nsample, max_blocks, seed = 20, 12, 8086
    if start == "fullsky":
        cfg, sky = small_case("c2", 16, perturb=False)
        ic, step0 = 1, 0.002
    else:
        cfg, sky = small_case("c1", 8)
        ic, step0 = 0, 0.4
    spec = cfg.comps[ic].indices[0]
    spec.step, spec.tune = step0, True
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    z, u = tuner_draw(seed, nsample, max_blocks)
    nb_o, step_o = ora.tune_step(ic, 0, -1, nsample, 1, z, u, max_blocks, perpixel_start=start == "perpixel")
    nb_g, step_g = eng.tune_index(ic, 0, -1, nsample, "sample", seed=seed, max_blocks=max_blocks)
    assert nb_g == nb_o and step_g == step_o and nb_o > 1, (nb_g, nb_o, step_g, step_o)


@pytest.mark.gpu
def test_band_gain_device_deviate():
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 8)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eta = eta_draw(3, 2, cfg.npix)
    ora.sample_cg_group(0, 1, eta)
    eng.cg_solve(0, 0, "sample", eta=None, seed=3)
    chisq_o, _ = ora.compute_chisq()
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o
    seed = 2718281828
    for band in (0, 3):
        g_o = ora.fit_band_gain(2, band, 1, gain_draw(seed, band))
        g_g = eng.fit_band_gain(2, band, "sample", seed=seed)
        assert abs(g_g - g_o) <= TOL * abs(g_o), (band, g_g, g_o)


# ------------------------------------------------------------------ 4. whole Gibbs iterations, as bench.py runs them
def _gibbs_device(name, nside, tune=False, deferred=False, seed=0, n_it=5):
    """eng.gibbs_iteration(it, seed=seed) for it = 1..n_it against oracle_gibbs_iteration.  `tune`: the sampled
    index starts untuned, so the step-size tuner runs once (iteration 2) on its own seed.  `deferred`: from
    iteration 3 on, DANG_OPT_DEFER_SCALARS; each iteration's scalars are read back through its mark."""
    from dang_b200.engine import OPT_DEFER_SCALARS, Engine
    from oracle.binding import Oracle
    cfg, sky = small_case(name, nside, perturb=False)
    for c in cfg.comps:
        for s in c.indices:
            s.tune = s.tune or (tune and s.sample)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    tuned = [[not s.tune for s in c.indices] for c in cfg.comps]
    fullsky = [(ic, j) for ic, c in enumerate(cfg.comps) for j, s in enumerate(c.indices) if s.sample and s.region == "fullsky"]
    for it in range(1, n_it + 1):
        n_o, chi_cg_o, acc_o, chi_mh_o, dec_o = oracle_gibbs_iteration(ora, cfg, it, seed, tuned)
        if deferred and it == 3:
            eng.set_option(OPT_DEFER_SCALARS, 1)
        r1, r2 = eng.gibbs_iteration(it, seed=seed)
        if deferred and it >= 3:
            q = eng.iteration_scalars(eng.iteration_mark())
            n_g, chi_cg_g, acc_g, chi_mh_g = [q["n_iter"]], q["chisq_amplitudes"], [q["accept"]], q["chisq_index"]
            ic, j = fullsky[0]
            assert q["index_value"] == ora.indices(ic)[j, 1, 0]
        else:
            n_g, chi_cg_g = [r[0] for r in r1[:-1]], r1[-1]
            acc_g, chi_mh_g = (r2[0], r2[1]) if r2 else (None, None)
        assert n_g == n_o, (it, n_g, n_o)
        assert abs(chi_cg_g - chi_cg_o) <= TOL * chi_cg_o, (it, chi_cg_g, chi_cg_o)
        if it > 1:
            assert acc_g == acc_o, (it, acc_g, acc_o)
            assert abs(chi_mh_g - chi_mh_o) <= TOL * chi_mh_o, (it, chi_mh_g, chi_mh_o)
            if fullsky and not deferred:
                dec_g, _ = eng.decisions(cfg.nsample, fullsky=True)
                assert np.array_equal(dec_g, dec_o[:cfg.nsample]), it
        for ic in range(len(cfg.comps)):
            assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL, (it, ic)
            assert rel_err(eng.indices(ic), ora.indices(ic)) < 1e-14, (it, ic)
    if deferred:
        eng.set_option(OPT_DEFER_SCALARS, 0)
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize("name,nside,tune", [("c2", 16, True), ("c2", 64, False), ("c4", 8, False)])
def test_gibbs_iterations_with_device_deviates(name, nside, tune):
    """c2 is the benchmark's configuration (persistent solve, one statistics pass, full-sky beta_d); at nside 16
    its beta_d starts untuned, so the tuner's seed is checked inside the loop too.  c4 draws beta_d and T_d per pixel."""
    _gibbs_device(name, nside, tune=tune)


@pytest.mark.gpu
def test_gibbs_iterations_with_device_deviates_deferred_scalars():
    """bench.py times c2 with deferred scalars: the same numbers, read back through the iteration marks."""
    _gibbs_device("c2", 16, tune=True, deferred=True)


# ------------------------------------------------------------------ 5. two GPUs
@pytest.mark.gpu
def test_two_gpus_gibbs_iterations_with_device_deviates():
    """tests/multi_gpu_check.py, case 'rng': the c2 Gibbs loop with device deviates on two ring-partitioned ranks;
    each rank's slice must follow the single-process oracle -- the global-slot rule at work -- over NVLink
    mailboxes and NCCL."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, DANG_MGC_CASE="rng", DANG_MGC_NSIDE="32")
    for mailbox in ("1", "0"):
        env["DANG_GPU_MAILBOX"] = mailbox
        p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29541",
                            os.path.join(ROOT, "tests", "multi_gpu_check.py")],
                           env=env, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        assert p.stdout.count("multi-GPU parity ok") == 2


# ------------------------------------------------------------------ 6. stationarity against the exact posterior
KS_C = 1.95  # sqrt(n) D > 1.95 has probability ~1e-3 for n independent draws from the target (Kolmogorov)


def _flat_sky(sed, S, bound, nside):
    """Every pixel holds the same data, noise and amplitudes, so every pixel's index has the same posterior.
    Returns (cfg, sky, ic, nind, loglike(theta grid), log prior(theta grid, prior mean), the sampled IndexSpec)."""
    from dang_b200.synth import band_sed, band_sigma, sed_mbb, sed_powerlaw
    kind = "synch" if sed == "powerlaw" else "dust"
    cfg, sky = shape_case(6, (kind,), nside=nside, varying=())
    comp = cfg.comps[0]
    nind = 0 if sed == "powerlaw" else 1
    spec = comp.indices[nind]
    spec.sample, spec.region = True, "per-pixel"
    if sed == "powerlaw":   # a Gaussian prior twice as wide as the likelihood
        truth, width = -3.1, 0.1
        spec.prior, spec.gauss, spec.step = "gaussian", (-3.05, 0.2), 0.03
        spec.uni = (-3.15, -2.0) if bound else (-4.0, -2.0)
        sed_of = lambda b, t: sed_powerlaw(b.nu_ghz, comp.nu_ref_ghz, t)       # noqa: E731
        other = ()
    else:                   # mbb T with the uniform prior
        truth, width = 19.6, 1.5
        spec.prior, spec.uni, spec.step = "uniform", (10.0, 35.0), 0.5
        sed_of = lambda b, t: sed_mbb(b.nu_ghz, comp.nu_ref_ghz, 1.55, t)      # noqa: E731
        other = (1.55,)
    planes = (1, 2) if S == 2 else (1,)
    sigma = np.array([band_sigma(b.nu_ghz) for b in cfg.bands])
    # the vectorised SED is synth.band_sed on these delta bands
    for b in cfg.bands:
        assert sed_of(b, truth) == band_sed(b, comp, *(other + (truth,)) if other else (truth,))
    d = np.array([(sed_of(b, truth + 1e-6) - sed_of(b, truth - 1e-6)) / 2e-6 for b in cfg.bands])
    amp0 = np.array([0.0, 1.0, -0.6])
    fisher = sum(np.sum((amp0[k] * d / sigma) ** 2) for k in planes)
    amp = amp0 / (width * np.sqrt(fisher))   # likelihood width `width`
    noise = np.random.default_rng(99).standard_normal((cfg.nbands, 3))
    data = np.array([[amp[k] * sed_of(b, truth) + sigma[j] * noise[j, k] for k in range(3)]
                     for j, b in enumerate(cfg.bands)])
    npix = cfg.npix
    sky.mask[:] = 1.0
    sky.sig[:] = data[:, :, None]
    sky.rms[:] = 1.0
    sky.rms[:, 1:3] = sigma[:, None, None]
    sky.amplitude[comp.label][:] = amp[:, None] * np.ones(npix)
    sky.indices[comp.label][:] = np.array([s.init for s in comp.indices])[:, None, None]
    if sed == "mbb_T":
        sky.indices[comp.label][0] = 1.55

    def loglike(theta):
        sed_t = np.array([sed_of(b, theta) for b in cfg.bands])   # [band][theta]
        out = np.zeros_like(theta)
        for k in planes:
            for j in range(cfg.nbands):
                t = (data[j, k] - amp[k] * sed_t[j]) / sigma[j]
                out -= 0.5 * t * t
        return out

    def logprior(theta, mean):
        return -0.5 * ((theta - mean) / spec.gauss[1]) ** 2 if spec.prior == "gaussian" else np.zeros_like(theta)

    return cfg, sky, 0, nind, loglike, logprior, spec


def _cdf(grid, logp):
    p = np.exp(logp - logp.max())
    c = np.concatenate([[0.0], np.cumsum(0.5 * (p[1:] + p[:-1]) * np.diff(grid))])
    return c / c[-1]


def _ks(x, grid, cdf):
    x = np.sort(x)
    n = x.size
    F = np.interp(x, grid, cdf)
    return max(np.max(np.arange(1, n + 1) / n - F), np.max(F - np.arange(n) / n))


STATIONARITY_CASES = [("default", "powerlaw", 2, False), ("fp64", "powerlaw", 1, False), ("strict", "powerlaw", 2, False),
                      ("default", "mbb_T", 2, False), ("strict", "mbb_T", 1, False), ("default", "powerlaw", 1, True),
                      ("fp64", "powerlaw", 2, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,sed,S,bound", STATIONARITY_CASES)
def test_perpixel_chain_keeps_the_exact_posterior(kernel, sed, S, bound):
    """Start every pixel's chain at an independent draw from its exact posterior pi (inverse CDF of a 2^18-point
    quadrature) and run one production draw of 50 proposals: a correct Metropolis kernel for pi leaves the pixels
    distributed as pi, however little it mixes.  The Kolmogorov-Smirnov distance to pi must stay below 1.95 / sqrt(n)
    (p ~ 1e-3; deterministic, the seeds are fixed), and the same samples must fail against two wrong targets: the
    prior mean moved by 0.2 posterior widths (a translation of pi by 0.2 widths under the uniform prior), and the
    likelihood tempered by 1.1.  Their CDFs differ from pi's by 0.010 .. 0.08 at most (measured on exact draws from
    pi), so the maps are nside 256: n = 786432 puts the threshold at 0.0022, and both wrong targets must exceed three
    times that.  (At nside 64 the tempered target would sit within a factor 1.3 of the threshold.)"""
    from dang_b200.engine import OPT_PERPIXEL_FAST, OPT_PERPIXEL_SERIAL, Engine
    nside, nsample = 256, 50
    cfg, sky, ic, nind, loglike, logprior, spec = _flat_sky(sed, S, bound, nside)
    grid = np.linspace(spec.uni[0], spec.uni[1], 2 ** 18 + 1)
    ll = loglike(grid)
    mean = spec.gauss[0] if spec.prior == "gaussian" else 0.0
    cdf = _cdf(grid, ll + logprior(grid, mean))
    mu = np.interp(0.5, cdf, grid)
    width = np.interp(0.8413, cdf, grid) - np.interp(0.1587, cdf, grid)
    width *= 0.5
    assert grid[0] < mu - 3 * width or bound
    if bound:   # pi presses against the lower bound: proposals beyond it are rejected (Q5)
        assert cdf[np.searchsorted(grid, spec.uni[0] + 0.5 * width)] > 0.1
    assert 1.5 * spec.step < width < 8 * spec.step
    n = cfg.npix
    start = np.interp(np.random.default_rng(2024).random(n), cdf, grid)
    idx = sky.indices[cfg.comps[ic].label].copy()
    for k in ((1, 2) if S == 2 else (1,)):
        idx[nind, k] = start
    eng = Engine(cfg, sky)
    eng.set_option(OPT_PERPIXEL_FAST, {"default": 3, "fp64": 0, "strict": 1}[kernel])
    eng.set_option(OPT_PERPIXEL_SERIAL, int(kernel == "strict"))
    eng.set_indices(ic, idx)
    acc = eng.sample_index_mh(ic, nind, -1 if S == 2 else 2, nsample, "sample", seed=77)
    assert 0.2 * n * nsample < acc < 0.9 * n * nsample
    final = eng.indices(ic)[nind, 1]
    if S == 2:
        assert np.array_equal(final, eng.indices(ic)[nind, 2])
    assert np.all(final >= spec.uni[0]) and np.all(final <= spec.uni[1])
    thr = KS_C / np.sqrt(n)
    d_true = _ks(final, grid, cdf)
    if spec.prior == "gaussian":
        wrong_shift = _cdf(grid, ll + logprior(grid, mean + 0.2 * width))
    else:
        wrong_shift = _cdf(grid, np.interp(grid - 0.2 * width, grid, ll))
    d_shift = _ks(final, grid, wrong_shift)
    d_temper = _ks(final, grid, _cdf(grid, 1.1 * ll + logprior(grid, mean)))
    print(f"KS {kernel} {sed} S={S} bound={bound}: D = {d_true:.5f} against pi, {d_shift:.5f} prior moved, "
          f"{d_temper:.5f} tempered; threshold {thr:.5f} (acceptance {acc / (n * nsample):.2f})")
    assert d_true < thr
    assert d_shift > 3 * thr and d_temper > 3 * thr


# ------------------------------------------------------------------ 7. every device-RNG call site is covered (CPU)
# (file, enclosing function) of each philox_normal( / philox_uniform2( call under dang_b200/csrc -> the test that
# reaches it with device deviates
RNG_SITES = {
    ("dang_gpu.cu", "dang_gpu_fit_band_gain"): "test_band_gain_device_deviate",
    ("kernels_stream.cuh", "rhs_blocks_ring_kernel"): "test_cg_device_eta[ring_stream]",
    ("kernels_uni.cuh", "rhs_blocks_uni_kernel"): "test_cg_device_eta[uni1]",
    ("kernels_uni.cuh", "rhs_blocks_tma_kernel"): "test_cg_device_eta[tma]",
    ("kernels_cg.cuh", "rhs_blocks_kernel"): "test_cg_device_eta[generic]",
    ("kernels_tmpl.cuh", "tmpl_rhs_kernel"): "test_cg_device_eta[template]",
    ("kernels_mh_pix.cuh", "mh_perpixel_pix_kernel"): "test_perpixel_device_deviates_odd_pixel_range",
    ("kernels_mh_fast.cuh", "mh_perpixel_fast_kernel"): "test_perpixel_device_deviates[lane-powerlaw-3]",
    ("kernels_mh_fast.cuh", "k5_rng_kernel"): "test_perpixel_device_deviates[split-powerlaw--1]",
    ("kernels_mh.cuh", "mh_perpixel_kernel"): "test_perpixel_device_deviates[fp64-powerlaw--1]",
    ("kernels_mh.cuh", "mh_perpixel_serial_kernel"): "test_perpixel_device_deviates_strict_variants",
    ("kernels_mh.cuh", "mh_draw_z"): "test_fullsky_device_deviates",
    ("kernels_mh.cuh", "mh_draw_u"): "test_fullsky_device_deviates",
    ("kernels_mh.cuh", "mh_suff_tune_kernel"): "test_tuner_device_deviates",
}


def rng_call_sites():
    """{(file, enclosing function): number of Philox calls} under dang_b200/csrc (the definitions in common.cuh
    excluded).  The enclosing function is the last definition that starts in column 0 before the call."""
    sites = {}
    head = re.compile(r"^(?:template\s*<[^>]*>\s*)?(?:[A-Za-z_][\w:<>,*& ]*?\s)?[*&]?(\w+)\s*\(")
    for name in sorted(os.listdir(CSRC)):
        if not name.endswith((".cu", ".cuh", ".inc")):
            continue
        with open(os.path.join(CSRC, name)) as f:
            lines = f.read().split("\n")
        func = None
        for line in lines:
            if re.match(r"[A-Za-z_]", line) and not line.startswith(("return", "else", "if", "for")):
                m = head.match(re.sub(r"__launch_bounds__\([^)]*\)", "", line))
                if m:
                    func = m.group(1)
            code = line.split("//")[0]
            n = len(re.findall(r"\bphilox_(?:normal|uniform2)\(", code))
            if n and not (name == "common.cuh" and func in ("philox_uniform2", "philox_normal")):
                sites[(name, func)] = sites.get((name, func), 0) + n
    return sites


def test_every_rng_call_site_is_covered():
    sites = rng_call_sites()
    missing = sorted(set(sites) - set(RNG_SITES))
    assert not missing, f"device-RNG call sites without a device-deviate test case in RNG_SITES: {missing}"
    stale = sorted(set(RNG_SITES) - set(sites))
    assert not stale, f"RNG_SITES names call sites that no longer exist: {stale}"
    for test in RNG_SITES.values():
        assert callable(globals().get(test.split("[")[0])), test
