"""GPU parity tests: every call goes through the C ABI (dang_b200.engine -> libdang_gpu.so) and
is compared with the CPU oracle on the same seeded inputs and injected deviates.

Bars (BASELINE.json north_star): accept/reject decisions and pixel indexing bit-exact;
amplitude maps, index maps, chi-square and lnL within 1e-10 relative (norm-wise) in fp64.
"""
import numpy as np
import pytest

from conftest import TOL, rel_err
from helpers import clone_sky, deviates, small_case

pytestmark = pytest.mark.gpu


def make_pair(name="c1", nside=16, **kw):
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case(name, nside, **kw)
    return cfg, sky, Oracle(cfg, sky), Engine(cfg, sky)


# ------------------------------------------------------------------ chi-square / sky model
@pytest.mark.parametrize("name,nside", [("c1", 16), ("c2", 16), ("c3", 8), ("c4", 8)])
def test_chisq_and_sky_model(name, nside):
    cfg, sky, ora, eng = make_pair(name, nside)
    ora.update_sky_model()
    chisq_o, planes_o = ora.compute_chisq()
    planes_g, n_unmasked = eng.chisq_planes()
    assert n_unmasked == int((sky.mask != 0).sum())
    assert rel_err(planes_g, planes_o) < TOL
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * abs(chisq_o)
    sky_g, res_g, chi_g = eng.update_sky_model()
    assert rel_err(sky_g, ora.sky_model()) < TOL
    assert rel_err(res_g, ora.res_map()) < TOL
    assert rel_err(chi_g, ora.chi_map()) < TOL
    # pixel indexing: masked pixels carry exactly zero chi-square
    assert np.all(chi_g[:, sky.mask == 0] == 0.0)


def test_chisq_missval_mask_and_ragged_size():
    # nside=4 -> 192 pixels (not a multiple of the 64-pixel plane padding once sliced);
    # mask uses the reference's missval sentinel as well as zeros
    from dang_b200.config import MISSVAL
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 4)
    sky.mask[::7] = MISSVAL
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    ora.update_sky_model()
    chisq_o, planes_o = ora.compute_chisq()
    planes_g, n = eng.chisq_planes()
    assert n == int(((sky.mask != 0) & (sky.mask != MISSVAL)).sum())
    assert rel_err(planes_g, planes_o) < TOL


# ------------------------------------------------------------------ amplitude draw
@pytest.mark.parametrize("name", ["c1", "c2"])  # c1: per-pixel SEDs; c2: tabulated (uniform) SEDs
@pytest.mark.parametrize("form", ["recompute8", "recompute3", "streaming", "two_pass"])
@pytest.mark.parametrize("ml_mode", ["optimize", "sample"])
def test_cg_solve_matches_oracle(name, form, ml_mode):
    """All CG forms (checkpointed recompute, streaming fused pass, classic two-pass) follow the
    oracle's cg_search: same iteration count, same residual trajectory, same amplitudes."""
    from dang_b200.engine import OPT_CG_CHECKPOINT, OPT_CG_TWO_PASS
    cfg, sky, ora, eng = make_pair(name, 16)
    eng.set_option(OPT_CG_TWO_PASS, int(form == "two_pass"))
    eng.set_option(OPT_CG_CHECKPOINT, {"recompute8": 8, "recompute3": 3}.get(form, 0))
    eta = np.random.default_rng(5).standard_normal(2 * cfg.npix)
    it_o, delta_o, trace_o = ora.cg_search_trace(ml_mode=1 if ml_mode == "sample" else 0, eta=eta)
    it_g, delta_g = eng.cg_solve(0, 0, ml_mode, eta=eta)
    trace_g = eng.cg_trace()
    assert it_g == it_o, (it_g, it_o, trace_g, trace_o)
    # the residual norm follows the oracle's trajectory iteration by iteration
    assert np.allclose(trace_g, trace_o, rtol=1e-6, atol=0)
    for ic in range(len(cfg.comps)):
        assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL
    assert rel_err(eng.cg_x(), ora.cg_x()) < TOL
    # masked pixels keep their initial amplitude exactly (zero rows / columns)
    m = sky.mask == 0
    for ic, c in enumerate(cfg.comps):
        assert np.array_equal(eng.amplitude(ic)[:, m], sky.amplitude[c.label][:, m])


def test_tma_staged_k1_matches():
    """DANG_OPT_TMA: K1 fed by cp.async.bulk + mbarrier produces the same bits as the LDG form."""
    from dang_b200.engine import OPT_TMA, Engine
    cfg, sky = small_case("c2", 16, perturb=False)
    eta = np.random.default_rng(4).standard_normal(2 * cfg.npix)
    out = []
    for tma in (0, 1):
        eng = Engine(cfg, sky)
        eng.set_option(OPT_TMA, tma)
        it, delta = eng.cg_solve(0, 0, "sample", eta=eta)
        out.append((it, delta, eng.amplitude(0).copy(), eng.amplitude(1).copy()))
    assert out[0][0] == out[1][0]
    assert rel_err(out[1][2], out[0][2]) < 1e-13 and rel_err(out[1][3], out[0][3]) < 1e-13


def test_cg_sample_vector_quirk_and_fix():
    """SURVEY Q1: with two diffuse components the reference's fluctuation lands in slot 1 only;
    DANG_OPT_FIX_SAMPLE_VECTOR switches to the per-component form.  Both match the oracle."""
    from dang_b200.engine import OPT_FIX_SAMPLE_VECTOR
    eta = np.random.default_rng(6).standard_normal(2 * 12 * 8 * 8)
    res = {}
    for fix in (0, 1):
        cfg, sky, ora, eng = make_pair("c1", 8)
        eng.set_option(OPT_FIX_SAMPLE_VECTOR, fix)
        ora.cg_search_trace(ml_mode=1, eta=eta, fix_q1=bool(fix))
        eng.cg_solve(0, 0, "sample", eta=eta)
        for ic in range(2):
            assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL
        res[fix] = eng.amplitude(1).copy()
    assert rel_err(res[0], res[1]) > 1e-3  # the two conventions really differ


def test_cg_warm_start_across_iterations():
    """Q10: x is seeded from c%amplitude once and then warm-started from the saved x."""
    cfg, sky, ora, eng = make_pair("c1", 8)
    rng = np.random.default_rng(7)
    for it in range(3):
        eta = rng.standard_normal(2 * cfg.npix)
        it_o, _, _ = ora.cg_search_trace(ml_mode=1, eta=eta)
        it_g, _ = eng.cg_solve(0, 0, "sample", eta=eta)
        assert it_g == it_o
        for ic in range(2):
            assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL


@pytest.mark.parametrize("poltype", ["Q", "U", "Q,U"])
def test_cg_single_plane_flags(poltype):
    from dang_b200.config import return_poltype_flag
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 8)
    cfg.cg_groups[0].poltype = poltype
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    rng = np.random.default_rng(8)
    for f, _ in enumerate(return_poltype_flag(poltype)):
        eta = rng.standard_normal(cfg.npix)
        it_o, _, _ = ora.cg_search_trace(flag_n=f, ml_mode=1, eta=eta)
        it_g, _ = eng.cg_solve(0, f, "sample", eta=eta)
        assert it_g == it_o
    for ic in range(2):
        assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL


def test_cg_one_component_with_out_of_group_subtraction():
    """Only synch is solved for; dust is not amplitude-sampled, so its signal is subtracted
    from the data first (compute_rhs :427-443)."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 8)
    cfg.comps[1].amp_sample = False
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eta = np.random.default_rng(9).standard_normal(2 * cfg.npix)
    it_o, _, _ = ora.cg_search_trace(ml_mode=1, eta=eta)
    it_g, _ = eng.cg_solve(0, 0, "sample", eta=eta)
    assert it_g == it_o
    for ic in range(2):
        assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL


def test_cg_recovers_noiseless_sky():
    """Known answer: noiseless data, indices at truth => optimize-mode CG returns the input sky."""
    from dang_b200.engine import Engine
    from dang_b200.synth import TRUE_THETA, make_config, make_sky, band_sed
    cfg = make_config("c1", nside=8)
    sky = make_sky(cfg)
    sky.sig[:] = 0.0
    for c in cfg.comps:
        for k, v in enumerate(TRUE_THETA[c.label]):
            sky.indices[c.label][k][:] = v
        for j, b in enumerate(cfg.bands):
            sky.sig[j, 1:3] += sky.truth[c.label][1:3] * band_sed(b, c, *TRUE_THETA[c.label])
    eng = Engine(cfg, sky)
    eng.cg_solve(0, 0, "optimize")
    m = sky.mask != 0
    for ic, c in enumerate(cfg.comps):
        a = eng.amplitude(ic)
        assert np.max(np.abs(a[1:3][:, m] - sky.truth[c.label][1:3][:, m])) < 1e-6
    assert eng.compute_chisq() < 1e-12


def test_device_rng_eta_matches_philox_definition():
    """eta == NULL: the device draws eta from Philox4x32-10; feeding the oracle the same stream
    (restated independently in oracle/dang_oracle.c) gives the same amplitudes.  The device's normals are
    r * sinpi(2 u2), the oracle's r * sin(2 pi u2): they differ by an ulp or so, and the amplitudes stay within
    TOL (~7e-16 measured on a B200; tests/test_gpu_device_rng.py covers every other call site)."""
    from oracle.binding import philox_normals
    cfg, sky, ora, eng = make_pair("c1", 8)
    seed = 1234567
    eta = philox_normals(seed, 1, 0, 2 * cfg.npix)
    assert abs(eta.mean()) < 0.1 and abs(eta.std() - 1.0) < 0.1
    it_o, _, _ = ora.cg_search_trace(ml_mode=1, eta=eta)
    it_g, _ = eng.cg_solve(0, 0, "sample", eta=None, seed=seed)
    assert it_g == it_o
    for ic in range(2):
        assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL


# ------------------------------------------------------------------ spectral-parameter draw
def run_perpixel(cfg, sky, ic, nind, nsample, ml_mode="sample", seed=11, serial=0, fast=1):
    from dang_b200.engine import OPT_PERPIXEL_FAST, OPT_PERPIXEL_SERIAL, OPT_RECORD, Engine
    from oracle.binding import Oracle
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eng.set_option(OPT_RECORD, 1)
    eng.set_option(OPT_PERPIXEL_SERIAL, serial)
    eng.set_option(OPT_PERPIXEL_FAST, fast)
    z, u = deviates(cfg, nsample, seed=seed)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, -1, nsample, 1 if ml_mode == "sample" else 0, z, u,
                                              want_trace=True)
    acc_g = eng.sample_index_mh(ic, nind, -1, nsample, ml_mode, z, u)
    dec_g, lnl_g = eng.decisions(nsample, fullsky=False)
    return ora, eng, (acc_o, dec_o, lnl_o), (acc_g, dec_g, lnl_g)


# kernels: fp32-screened lane-cooperative (default), fp64 lane-cooperative, strict reference order
# and the one-thread-per-pixel screened form (kernels_mh_pix.cuh)
@pytest.mark.parametrize("kernel", ["screened", "pixel", "fp64", "serial"])
@pytest.mark.parametrize("name,ic,nind,nside", [("c1", 0, 0, 16), ("c3", 1, 0, 4), ("c3", 0, 0, 4), ("c4", 1, 0, 8),
                                                ("c4", 1, 1, 8), ("c2", 1, 1, 8), ("c4", 0, 0, 8)])
def test_perpixel_metropolis_bit_exact_decisions(name, ic, nind, nside, kernel):
    cfg, sky = small_case(name, nside)
    cfg.comps[ic].indices[nind].sample = True
    cfg.comps[ic].indices[nind].region = "per-pixel"
    nsample = 12
    ora, eng, (acc_o, dec_o, lnl_o), (acc_g, dec_g, lnl_g) = run_perpixel(
        cfg, sky, ic, nind, nsample, serial=int(kernel == "serial"), fast={"screened": 1, "pixel": 3}.get(kernel, 0))
    assert np.array_equal(dec_g, dec_o), f"{(dec_g != dec_o).sum()} decisions differ"
    assert acc_g == acc_o
    if kernel in ("screened", "pixel"):  # record mode checks every screened difference against its error bound
        fallbacks, violations = eng.perpixel_stats()
        assert violations == 0, (fallbacks, violations)
        assert fallbacks <= 0.02 * (dec_o < 2).sum(), (fallbacks, (dec_o < 2).sum())
    ev = dec_o < 2
    assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL
    # accepted proposals are stored verbatim => index maps agree to the last bit up to the
    # 1-ulp regrouping of step*z; masked pixels are zeroed exactly as index_map is (:223,:465)
    idx_g, idx_o = eng.indices(ic), ora.indices(ic)
    assert rel_err(idx_g, idx_o) < 1e-14
    assert np.all(idx_g[nind][1:3][:, sky.mask == 0] == 0.0)
    assert np.array_equal(idx_g[nind][0], idx_o[nind][0])  # I plane untouched


@pytest.mark.parametrize("form", [1, 3])
@pytest.mark.parametrize("name,ic,nind", [("c4", 1, 0), ("c4", 1, 1), ("c1", 0, 0)])
def test_perpixel_screened_kernel_takes_the_fp64_decisions(name, ic, nind, form):
    """Production mode (no recording): the fp32-screened kernel and the fp64 kernel leave identical index
    maps and acceptance counts after long chains with big steps, at a size where ~1e6 proposals are
    decided; the fallback rate stays small."""
    from dang_b200.engine import OPT_PERPIXEL_FAST, Engine
    cfg, sky = small_case(name, 64)
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region = True, "per-pixel"
    spec.step *= 3.0
    nsample = 40
    z, u = deviates(cfg, nsample, seed=5)
    a, b = Engine(cfg, sky), Engine(cfg, sky)
    a.set_option(OPT_PERPIXEL_FAST, form)
    b.set_option(OPT_PERPIXEL_FAST, 0)
    acc_a = a.sample_index_mh(ic, nind, -1, nsample, "sample", z, u)
    acc_b = b.sample_index_mh(ic, nind, -1, nsample, "sample", z, u)
    fallbacks, _ = a.perpixel_stats()
    assert acc_a == acc_b and acc_a > 0
    assert np.array_equal(a.indices(ic), b.indices(ic))
    n_unmasked = int((sky.mask != 0).sum())
    # (the one-thread-per-pixel form carries one error bound for all bands of a pixel: with steps three times the
    # configured ones and 40-proposal chains it gives up earlier -- slower there, never wrong)
    assert fallbacks < (0.005 if form == 1 else 0.1) * nsample * n_unmasked, (fallbacks, nsample * n_unmasked)
    # and with the device RNG
    acc_a = a.sample_index_mh(ic, nind, -1, nsample, "sample", seed=99)
    acc_b = b.sample_index_mh(ic, nind, -1, nsample, "sample", seed=99)
    assert acc_a == acc_b
    assert np.array_equal(a.indices(ic), b.indices(ic))


@pytest.mark.parametrize("ic,nind", [(0, 0), (1, 0)])
def test_perpixel_bandpass_moment_series(ic, nind):
    """Config c3 (tabulated bandpasses, n_bp = 128): the moment series about the chain's first point gives the
    oracle's decisions and lnL, and the same chains as summing the bandpass for every proposal -- also with
    steps large enough to push proposals beyond the series' range (direct-sum fallback)."""
    from dang_b200.engine import OPT_PERPIXEL_BP_SERIES, OPT_RECORD, Engine
    from oracle.binding import Oracle
    for step_scale in (1.0, 12.0):
        cfg, sky = small_case("c3", 8)
        spec = cfg.comps[ic].indices[nind]
        spec.sample, spec.region = True, "per-pixel"
        spec.step *= step_scale
        nsample = 16
        z, u = deviates(cfg, nsample, seed=21)
        ora = Oracle(cfg, sky)
        acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, -1, nsample, 1, z, u, want_trace=True)
        res = {}
        for series in (1, 0):
            eng = Engine(cfg, sky)
            eng.set_option(OPT_RECORD, 1)
            eng.set_option(OPT_PERPIXEL_BP_SERIES, series)
            acc = eng.sample_index_mh(ic, nind, -1, nsample, "sample", z, u)
            dec, lnl = eng.decisions(nsample, fullsky=False)
            res[series] = (acc, dec, lnl, eng.indices(ic).copy())
            assert np.array_equal(dec, dec_o) and acc == acc_o, (series, step_scale)
            ev = dec_o < 2
            assert rel_err(lnl[ev], lnl_o[ev]) < TOL
            assert rel_err(eng.indices(ic), ora.indices(ic)) < 1e-14
        assert np.array_equal(res[1][3], res[0][3])
        ev = dec_o < 2
        assert rel_err(res[1][2][ev], res[0][2][ev]) < 1e-12


def test_bandpass_gauss_quadrature_matches_the_full_table():
    """Tabulated bandpasses reach the device as their 8-point Gauss quadrature (DANG_OPT_BP_QUADRATURE): chi-square,
    sky model and CG amplitudes agree with the full 128-sample tables (option 0) to rounding, and with the oracle."""
    from dang_b200.engine import OPT_BP_QUADRATURE, Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c3", 8)
    ora = Oracle(cfg, sky)
    ora.update_sky_model()
    chisq_o, _ = ora.compute_chisq()
    eta = np.random.default_rng(2).standard_normal(2 * cfg.npix)
    its_o, _ = ora.sample_cg_group(0, 1, eta)
    out = {}
    for nq in (8, 0):
        eng = Engine(cfg, sky)
        eng.set_option(OPT_BP_QUADRATURE, nq)
        c0 = eng.compute_chisq()
        sky_g, _, _ = eng.update_sky_model()
        it, _ = eng.cg_solve(0, 0, "sample", eta)
        out[nq] = (c0, sky_g, it, eng.amplitude(0), eng.amplitude(1))
        assert abs(c0 - chisq_o) <= TOL * chisq_o and it == its_o[0]
        assert rel_err(eng.amplitude(0), ora.amplitude(0)) < TOL and rel_err(eng.amplitude(1), ora.amplitude(1)) < TOL
    assert abs(out[8][0] - out[0][0]) <= 1e-13 * out[0][0]
    assert rel_err(out[8][1], out[0][1]) < 1e-13
    assert rel_err(out[8][3], out[0][3]) < 1e-11 and rel_err(out[8][4], out[0][4]) < 1e-11


def test_perpixel_split_form_matches():
    """The split form of the screened kernel (option 12 = 2: rng / state / chain kernels) leaves the same
    index maps and acceptance counts as the default monolithic kernel, with injected and device deviates."""
    from dang_b200.engine import OPT_PERPIXEL_FAST, Engine
    cfg, sky = small_case("c4", 32)
    for ic, nind in ((1, 0), (1, 1)):
        spec = cfg.comps[ic].indices[nind]
        spec.sample, spec.region = True, "per-pixel"
    nsample = 20
    z, u = deviates(cfg, nsample, seed=9)
    a, b = Engine(cfg, sky), Engine(cfg, sky)
    b.set_option(OPT_PERPIXEL_FAST, 2)
    for ic, nind in ((1, 0), (1, 1)):
        assert a.sample_index_mh(ic, nind, -1, nsample, "sample", z, u) == b.sample_index_mh(ic, nind, -1, nsample, "sample", z, u)
        assert a.sample_index_mh(ic, nind, -1, nsample, "sample", seed=5) == b.sample_index_mh(ic, nind, -1, nsample, "sample", seed=5)
        assert np.array_equal(a.indices(ic), b.indices(ic))


def test_perpixel_optimize_mode_and_uniform_prior():
    cfg, sky = small_case("c1", 8)
    cfg.comps[0].indices[0].prior = "uniform"
    cfg.comps[0].indices[0].uni = (-3.2, -2.9)  # tight bounds => many out-of-bounds proposals (Q5)
    ora, eng, (acc_o, dec_o, _), (acc_g, dec_g, _) = run_perpixel(cfg, sky, 0, 0, 16, ml_mode="optimize")
    assert (dec_o == 2).sum() > 0
    assert np.array_equal(dec_g, dec_o)
    assert acc_g == acc_o
    assert rel_err(eng.indices(0), ora.indices(0)) < 1e-14


def test_perpixel_marginal_lnl():
    cfg, sky = small_case("c1", 8)
    cfg.comps[0].indices[0].lnl_type = "marginal"
    ora, eng, (acc_o, dec_o, lnl_o), (acc_g, dec_g, lnl_g) = run_perpixel(cfg, sky, 0, 0, 8)
    assert np.array_equal(dec_g, dec_o)
    ev = dec_o < 2
    assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL


@pytest.mark.parametrize("stream", [0, 1])
@pytest.mark.parametrize("name,ic,nind,others_uniform", [("c2", 1, 0, True), ("c4", 1, 1, True), ("c1", 0, 0, True),
                                                        ("c1", 1, 0, False)])
def test_fullsky_metropolis(stream, name, ic, nind, others_uniform):
    from dang_b200.engine import OPT_FULLSKY_STREAM, Engine
    from oracle.binding import Oracle
    cfg, sky = small_case(name, 16)
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region = True, "fullsky"
    for i2, c in enumerate(cfg.comps):  # the sampled component's indices are uniform maps
        for k, s in enumerate(c.indices):
            if others_uniform or i2 == ic:
                sky.indices[c.label][k][:] = s.init
    spec.step = {0: 0.002, 1: 0.02}[nind]
    nsample = 24
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eng.set_option(OPT_FULLSKY_STREAM, stream)
    rng = np.random.default_rng(13)
    z, u = rng.standard_normal(nsample), rng.random(nsample)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, -1, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(ic, nind, -1, nsample, "sample", z, u)
    dec_g, lnl_g = eng.decisions(nsample, fullsky=True)
    assert np.array_equal(dec_g, dec_o[:nsample]), (dec_g, dec_o[:nsample])
    assert acc_g == acc_o
    ev = dec_o[:nsample] < 2
    assert ev.sum() > 0 and 0 < acc_o < ev.sum()  # a non-trivial chain
    assert rel_err(lnl_g[ev], lnl_o[:nsample][ev]) < TOL
    assert rel_err(eng.indices(ic), ora.indices(ic)) < 1e-14


@pytest.mark.parametrize("variant", ["marginal", "jeffreys", "prior_draw"])
def test_fullsky_metropolis_rare_variants(variant):
    """Full-sky chains with the marginal likelihood (dang_lnl_mod.f90:47-124), the Jeffreys prior
    (:242-304, synchrotron only) and lnl_type 'prior' (a plain draw from the Gaussian prior)."""
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
    # non-zero amplitudes (the Jeffreys term divides by them)
    rng = np.random.default_rng(17)
    for c in cfg.comps:
        sky.amplitude[c.label][1:3] = sky.truth[c.label][1:3] * (1.0 + 0.05 * rng.standard_normal((2, cfg.npix)))
    nsample = 16
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    z, u = rng.standard_normal(nsample), rng.random(nsample)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(0, 0, -1, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(0, 0, -1, nsample, "sample", z, u)
    assert rel_err(eng.indices(0), ora.indices(0)) < 1e-14
    if variant == "prior_draw":
        assert np.all(eng.indices(0)[0, 1] == spec.gauss[0] + spec.gauss[1] * z[0])
        return
    dec_g, lnl_g = eng.decisions(nsample, fullsky=True)
    assert np.array_equal(dec_g, dec_o[:nsample])
    assert acc_g == acc_o
    ev = dec_o[:nsample] < 2
    assert rel_err(lnl_g[ev], lnl_o[:nsample][ev]) < TOL


@pytest.mark.parametrize("step0", [0.2, 0.0005, 0.004])
def test_step_size_tuner(step0):
    """tune_spectral_parameter_length: same blocks, same halving / x1.5 sequence, same final step."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c2", 16, perturb=False)
    spec = cfg.comps[1].indices[0]
    spec.step, spec.tune = step0, True
    nsample, max_blocks = 20, 8
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    rng = np.random.default_rng(31)
    z, u = rng.standard_normal(nsample * max_blocks), rng.random(nsample * max_blocks)
    nb_o, step_o = ora.tune_step(1, 0, -1, nsample, 1, z, u, max_blocks)
    nb_g, step_g = eng.tune_index(1, 0, -1, nsample, "sample", z, u, max_blocks=max_blocks)
    assert nb_g == nb_o and nb_o >= 1
    assert step_g == step_o
    if nb_o == max_blocks:
        return  # never settled inside 0.4..0.6 within max_blocks: the oracle still counts as untuned
    # the tuned step is the one the next draw uses
    z2, u2 = rng.standard_normal(nsample), rng.random(nsample)
    acc_o, dec_o, _ = ora.sample_index_mh(1, 0, -1, nsample, 1, z2, u2)
    acc_g = eng.sample_index_mh(1, 0, -1, nsample, "sample", z2, u2)
    dec_g, _ = eng.decisions(nsample, fullsky=True)
    assert np.array_equal(dec_g, dec_o[:nsample]) and acc_g == acc_o


def test_async_staging_matches_synchronous_calls():
    """dang_gpu_stage_eta / get_*_async / download_wait deliver the same bits as the blocking calls,
    including when a later solve and draw are issued while downloads are still in flight."""
    from dang_b200.engine import Engine
    cfg, sky = small_case("c1", 16)
    rng = np.random.default_rng(41)
    etas = [rng.standard_normal(2 * cfg.npix) for _ in range(3)]
    zs, us = deviates(cfg, 6, ncalls=3)
    a, b = Engine(cfg, sky), Engine(cfg, sky)
    amp_async = [np.zeros((3, cfg.npix)) for _ in cfg.comps]
    idx_async = [np.zeros((len(c.indices), 3, cfg.npix)) for c in cfg.comps]
    snaps = []
    b.stage_eta(etas[0])
    for it in range(3):
        a.sample_cg_groups(eta=etas[it], stats=False)
        b.sample_cg_groups(eta=None, stats=False)
        if it < 2:
            b.stage_eta(etas[it + 1])
        for ic in range(2):
            b.amplitude_async(ic, amp_async[ic])
        z, u = zs[it * 6 * cfg.npix:(it + 1) * 6 * cfg.npix], us[it * 6 * cfg.npix:(it + 1) * 6 * cfg.npix]
        a.sample_spectral_parameters(nsample=6, z=z, u=u, stats=False)
        b.sample_spectral_parameters(nsample=6, z=z, u=u, stats=False)
        b.indices_async(0, 0, idx_async[0])
        if it == 2:
            b.download_wait()
            for ic in range(2):
                assert np.array_equal(amp_async[ic][1:3], a.amplitude(ic)[1:3])
            assert np.array_equal(idx_async[0][0][1:3], a.indices(0)[0][1:3])
    for ic in range(2):
        assert np.array_equal(a.amplitude(ic), b.amplitude(ic))
        assert np.array_equal(a.indices(ic), b.indices(ic))


def test_async_pipeline_two_deep():
    """The bench's end-to-end pattern: the deviates of solve k+1 are staged BEFORE solve k runs (two-slot
    FIFO), every step's amplitudes are downloaded into their own host arrays without ever waiting
    (the next solve unpacks into the second amplitude buffer), and every download holds exactly the
    state of its step."""
    from dang_b200.engine import DangGpuError, Engine
    cfg, sky = small_case("c2", 16)
    rng = np.random.default_rng(43)
    nstep = 5
    etas = [rng.standard_normal(2 * cfg.npix) for _ in range(nstep + 1)]
    a, b = Engine(cfg, sky), Engine(cfg, sky)
    out = [[np.zeros((3, cfg.npix)) for _ in cfg.comps] for _ in range(nstep)]
    ref = []
    b.stage_eta(etas[0])
    for it in range(nstep):
        a.sample_cg_groups(eta=etas[it], stats=False)
        ref.append([a.amplitude(ic).copy() for ic in range(2)])
        b.stage_eta(etas[it + 1])          # queued behind the deviates this solve consumes
        if it == 0:
            with pytest.raises(DangGpuError):
                b.stage_eta(etas[it + 1])  # a third set does not fit
        b.sample_cg_groups(eta=None, stats=False)
        for ic in range(2):
            b.amplitude_async(ic, out[it][ic])
        a.sample_spectral_parameters(stats=True)
        b.sample_spectral_parameters(stats=True)
    b.download_wait()
    for it in range(nstep):
        for ic in range(2):
            assert np.array_equal(out[it][ic][1:3], ref[it][ic][1:3]), (it, ic)
    for ic in range(2):
        assert np.array_equal(a.amplitude(ic), b.amplitude(ic))
        assert np.array_equal(a.indices(ic), b.indices(ic))
    # in-place writers respect a pending download too
    b.amplitude_async(0, out[0][0])
    amp = ref[0][0] * 2.0
    b.set_amplitude(0, amp)
    b.download_wait()
    assert np.array_equal(out[0][0][1:3], a.amplitude(0)[1:3])
    assert np.array_equal(b.amplitude(0), amp)


def test_golden_vectors_through_the_c_abi():
    """The committed fixture tests/golden/c1_nside4.npz (oracle output, made by
    tests/golden/make_golden.py) reproduced on the GPU with the same injected deviates."""
    import os
    from dang_b200.engine import Engine
    from dang_b200.synth import make_config, make_sky
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "c1_nside4.npz"))
    cfg = make_config("c1", nside=4)
    sky = make_sky(cfg)
    eng = Engine(cfg, sky)
    rng = np.random.default_rng(20260103)
    nsample = 10
    for it in (1, 2, 3):
        eta = rng.standard_normal(2 * cfg.npix)
        r = eng.sample_cg_groups(eta=eta)
        assert r[0][0] == int(gold[f"it{it}_n_cg"][0])
        assert abs(r[1] - float(gold[f"it{it}_chisq_cg"])) <= TOL * float(gold[f"it{it}_chisq_cg"])
        if it > 1:
            z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
            _, chisq = eng.sample_spectral_parameters(nsample=nsample, z=z, u=u)
            assert abs(chisq - float(gold[f"it{it}_chisq_mh"])) <= TOL * float(gold[f"it{it}_chisq_mh"])
        assert rel_err(eng.amplitude(0), gold[f"it{it}_amp_synch"]) < TOL
        assert rel_err(eng.amplitude(1), gold[f"it{it}_amp_dust"]) < TOL
        assert rel_err(eng.indices(0), gold[f"it{it}_beta_s"]) < 1e-13


def test_full_gibbs_chain_c1():
    """Three Gibbs iterations of config c1 (CG amplitudes + per-pixel beta_s) with injected
    deviates: amplitudes, indices and chi-square follow the oracle throughout."""
    cfg, sky, ora, eng = make_pair("c1", 8, perturb=False)
    rng = np.random.default_rng(21)
    nsample = 10
    for it in range(1, 4):
        eta = rng.standard_normal(2 * cfg.npix)
        its_o, _ = ora.sample_cg_group(0, 1, eta)
        r = eng.sample_cg_groups(eta=eta)
        assert r[0][0] == its_o[0]
        chisq_o, _ = ora.compute_chisq()
        assert abs(r[1] - chisq_o) <= TOL * chisq_o
        if it > 1:
            z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
            ora.sample_spectral_parameters(nsample, 1, z, u)
            acc, chisq_g = eng.sample_spectral_parameters(nsample=nsample, z=z, u=u)
            chisq_o, _ = ora.compute_chisq()
            assert abs(chisq_g - chisq_o) <= TOL * chisq_o
        for ic in range(2):
            assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL
            assert rel_err(eng.indices(ic), ora.indices(ic)) < 1e-13

@pytest.mark.parametrize("nside,name", [(16, "c2"), (8, "c2")])
def test_full_gibbs_chain_c2_one_statistics_pass(nside, name):
    """Gibbs iterations of the headline config (CG amplitudes + full-sky beta_d): the chi-square after
    the amplitude draw, the full-sky draw and the chi-square after it are served by ONE pass over the
    maps (statistics cache); everything still follows the oracle, and the uncached path agrees."""
    from dang_b200.engine import OPT_STAT_CACHE, Engine
    from oracle.binding import Oracle
    cfg, sky = small_case(name, nside, perturb=False)
    ora, eng, plain = Oracle(cfg, sky), Engine(cfg, sky), Engine(cfg, sky)
    plain.set_option(OPT_STAT_CACHE, 0)
    rng = np.random.default_rng(5)
    nsample = cfg.nsample
    ic = [i for i, c in enumerate(cfg.comps) if any(s.sample for s in c.indices)][0]
    for it in range(1, 5):
        eta = rng.standard_normal(2 * cfg.npix)
        its_o, _ = ora.sample_cg_group(0, 1, eta)
        chisq_o, planes_o = ora.compute_chisq()
        n0 = eng.launch_count(reset=True)
        r = eng.sample_cg_groups(eta=eta)
        rp = plain.sample_cg_groups(eta=eta)
        assert r[0][0] == its_o[0] == rp[0][0]
        assert abs(r[1] - chisq_o) <= TOL * chisq_o
        assert abs(rp[1] - chisq_o) <= TOL * chisq_o
        assert abs(r[1] - rp[1]) <= 1e-13 * chisq_o
        if it > 1:
            z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
            acc_o = ora.sample_spectral_parameters(nsample, 1, z, u)
            eng.kernel_stats(reset=True)
            acc, chisq_g = eng.sample_spectral_parameters(nsample=nsample, z=z, u=u)
            st = eng.kernel_stats()
            # no pass over the maps at all in this block: the statistics were gathered by the chi-square call
            assert st["mh_suffstat_kernel"]["launches"] == 0 and st["chisq_kernel"]["launches"] == 0, st
            accp, chisq_p = plain.sample_spectral_parameters(nsample=nsample, z=z, u=u)
            chisq_o, _ = ora.compute_chisq()
            assert acc == accp
            assert abs(chisq_g - chisq_o) <= TOL * chisq_o
            assert abs(chisq_p - chisq_o) <= TOL * chisq_o
            dec_g, lnl_g = eng.decisions(nsample, fullsky=True)
            dec_p, lnl_p = plain.decisions(nsample, fullsky=True)
            assert np.array_equal(dec_g, dec_p)
            assert eng.index_fullsky(ic, 0, 2) == ora.indices(ic)[0, 1, 0] == eng.index_fullsky(ic, 0, 3)
        for i2 in range(2):
            assert rel_err(eng.amplitude(i2), ora.amplitude(i2)) < TOL
            assert rel_err(eng.indices(i2), ora.indices(i2)) < 1e-13


def test_statistics_cache_is_invalidated_by_state_changes():
    """A chi-square served from cached statistics must never survive a change of the model state."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c2", 8, perturb=False)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    rng = np.random.default_rng(6)
    eta = rng.standard_normal(2 * cfg.npix)
    ora.sample_cg_group(0, 1, eta)
    eng.sample_cg_groups(eta=eta, stats=False)
    c1 = eng.compute_chisq()          # gathers the statistics of the coming beta_d draw
    assert abs(c1 - ora.compute_chisq()[0]) <= TOL * c1
    assert eng.compute_chisq() == c1  # served again (cache or kernel), same state
    amp = eng.amplitude(0)
    amp[1] *= 1.5
    eng.set_amplitude(0, amp)
    ora.amplitude(0)[:] = amp
    ora.update_sky_model()
    c2 = eng.compute_chisq()
    assert abs(c2 - ora.compute_chisq()[0]) <= TOL * c2 and abs(c2 - c1) > 1e-3 * c1
    # a draw after the change uses fresh statistics
    nsample = 12
    z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
    ora.sample_spectral_parameters(nsample, 1, z, u)
    acc, c3 = eng.sample_spectral_parameters(nsample=nsample, z=z, u=u)
    assert abs(c3 - ora.compute_chisq()[0]) <= TOL * c3
    idx = eng.indices(1)
    idx[0] += 0.01
    eng.set_indices(1, idx)
    ora.indices(1)[:] = idx
    ora.update_sky_model()
    c4 = eng.compute_chisq()
    assert abs(c4 - ora.compute_chisq()[0]) <= TOL * c4


def test_freefree_lognormal_cmb_components():
    """The remaining diffuse SED types (evaluate_freefree :1001-1040, evaluate_lognormal :960-999,
    'cmb' = 1/a2t) through chi-square, the CG amplitude draw (5x5 blocks split over two CG groups)
    and a per-pixel draw of the free-free electron temperature."""
    from dang_b200.config import CGGroup, Component, IndexSpec
    from dang_b200.engine import OPT_RECORD, Engine
    from oracle.binding import Oracle
    cfg, sky0 = small_case("c1", 8)
    cfg.comps += [
        Component("ff", "freefree", 40.0, cg_group=2, indices=[
            IndexSpec("T_e", 7000.0, sample=True, region="per-pixel", prior="uniform", uni=(4000.0, 11000.0), step=300.0)]),
        Component("ame", "lognormal", 22.0, cg_group=2, indices=[IndexSpec("NU_P", 21.0), IndexSpec("W_AME", 0.55)]),
        Component("cmb", "cmb", 100.0, cg_group=2, indices=[]),
    ]
    cfg.cg_groups.append(CGGroup(sample=True, max_iter=60, converge=1e-10, poltype="Q+U"))
    from dang_b200.synth import make_sky
    sky = make_sky(cfg)
    rng = np.random.default_rng(23)
    for c in cfg.comps:
        sky.amplitude[c.label][1:3] = rng.normal(0.0, 5.0, size=(2, cfg.npix))
    sky.indices["ff"][0][:] = 7000.0 + 500.0 * rng.standard_normal(cfg.npix)[None, :]
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eng.set_option(OPT_RECORD, 1)
    ora.update_sky_model()
    chisq_o, planes_o = ora.compute_chisq()
    assert rel_err(eng.chisq_planes()[0], planes_o) < TOL
    sky_g, res_g, _ = eng.update_sky_model()
    assert rel_err(sky_g, ora.sky_model()) < TOL
    for ig in (0, 1):
        eta = rng.standard_normal(2 * cfg.npix)
        it_o, _, _ = ora.cg_search_trace(ig=ig, ml_mode=1, eta=eta)
        it_g, _ = eng.cg_solve(ig, 0, "sample", eta=eta)
        assert it_g == it_o
    for ic in range(len(cfg.comps)):
        assert rel_err(eng.amplitude(ic), ora.amplitude(ic)) < TOL
    nsample = 8
    z, u = deviates(cfg, nsample, seed=29)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(2, 0, -1, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(2, 0, -1, nsample, "sample", z, u)
    dec_g, lnl_g = eng.decisions(nsample, fullsky=False)
    assert np.array_equal(dec_g, dec_o) and acc_g == acc_o
    assert rel_err(eng.indices(2), ora.indices(2)) < 1e-14


def test_template_cg_operator_matches_oracle():
    """Right-hand side and matrix-free apply with the template's border rows: the residual norms of the first
    CG iterations agree with the oracle to rounding.  (Later iterations do not, in ANY two implementations:
    the bordered system is ill-conditioned and the CG trajectory amplifies 1e-16 differences by ~1e3 per
    iteration -- the oracle itself changes trajectory with its summation order -- so for this path parity is
    asserted on the operator here and on the converged solution below, not on the iteration count.)"""
    from dang_b200.engine import Engine
    from helpers import template_case
    from oracle.binding import Oracle
    cfg, sky, _ = template_case(16)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eta = np.random.default_rng(1).standard_normal(2 * cfg.npix)
    it_o, delta_o, tr_o = ora.cg_search_trace(0, 0, 1, eta)
    it_g, delta_g = eng.cg_solve(0, 0, "sample", eta)
    tr_g = eng.cg_trace()
    assert np.max(np.abs(tr_g[:5] - tr_o[:5]) / tr_o[:5]) < 1e-12
    assert delta_g <= cfg.cg_groups[0].converge and delta_o <= cfg.cg_groups[0].converge
    assert abs(it_g - it_o) <= 6


@pytest.mark.parametrize("ml_mode", ["optimize", "sample"])
def test_template_component_cg_and_draws(ml_mode):
    """SURVEY 8f-1: a dust TEMPLATE fitted per band next to diffuse synchrotron (the arXiv:2201.03530 set-up).
    The bordered CG (template rows / columns), its warm start, the chi-square / sky model and a full-sky
    beta_s draw whose data have the template removed follow the oracle.  Both sides iterate to a tight
    threshold so that what is compared is the solution of the linear system, not where the CG stopped."""
    from dang_b200.engine import Engine
    from helpers import template_case
    from oracle.binding import Oracle
    cfg, sky, tamp_true = template_case(16)
    cfg.ml_mode = ml_mode
    cfg.cg_groups[0].converge, cfg.cg_groups[0].max_iter = 1e-20, 300
    spec = cfg.comps[0].indices[0]
    spec.sample, spec.region, spec.step = True, "fullsky", 0.002
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    rng = np.random.default_rng(3)
    ml = 1 if ml_mode == "sample" else 0
    tol = 1e-8
    for it in range(1, 4):
        eta = rng.standard_normal(2 * cfg.npix)
        its_o, _ = ora.sample_cg_group(0, ml, eta)
        r = eng.sample_cg_groups(ml_mode=ml_mode, eta=eta)
        assert abs(r[0][0] - its_o[0]) <= 10, (r[0], its_o)
        chisq_o, _ = ora.compute_chisq()
        assert abs(r[1] - chisq_o) <= tol * chisq_o
        assert rel_err(eng.amplitude(0), ora.amplitude(0)) < tol
        ta_g, ta_o = eng.template_amplitudes(1), ora.template_amplitudes(1)
        assert rel_err(ta_g, ta_o) < tol
        assert np.array_equal(ta_g[1], ta_g[2]) and np.all(ta_g[0] == 0.0)
        if it == 1 and ml_mode == "optimize":  # the fit sees the true amplitudes through the noise
            assert np.allclose(ta_g[1], tamp_true, rtol=0.1, atol=2.0)
        nsample = 12
        z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
        ora.sample_spectral_parameters(nsample, ml, z, u)
        acc, chisq_g = eng.sample_spectral_parameters(nsample=nsample, ml_mode=ml_mode, z=z, u=u)
        chisq_o, _ = ora.compute_chisq()
        assert abs(chisq_g - chisq_o) <= tol * chisq_o
        assert rel_err(eng.indices(0), ora.indices(0)) < 1e-14
    sky_g, res_g, chi_g = eng.update_sky_model()
    assert rel_err(sky_g, ora.sky_model()) < tol and rel_err(res_g, ora.res_map()) < tol


def test_template_unsupported_layouts_are_loud():
    from dang_b200.engine import DangGpuError, Engine
    from helpers import template_case
    cfg, sky, _ = template_case(4)
    cfg.cg_groups[0].poltype = "Q"   # the reference sizes b for template rows only in the Q+U branch
    eng = Engine(cfg, sky)
    with pytest.raises(DangGpuError, match="Q\\+U"):
        eng.sample_cg_groups(eta=np.zeros(cfg.npix))


def test_band_gain_fit_intensity():
    """fit_band_gain on a Stokes-I run (TQU = T): gains and offsets enter the data, the fitted
    gain matches the oracle and feeds the next chi-square."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 8)
    cfg.tqu = "T"
    cfg.cg_groups[0].poltype = "T"
    for c in cfg.comps:
        for s in c.indices:
            s.poltype = "T"
    rng = np.random.default_rng(37)
    sky.gain = 1.0 + 0.02 * rng.standard_normal(cfg.nbands)
    sky.offset = rng.normal(0.0, 0.5, cfg.nbands)
    sky.rms[:, 0] = sky.rms[:, 1]
    for c in cfg.comps:
        sky.amplitude[c.label][0] = sky.truth[c.label][1]
        sky.indices[c.label][:, 0] = sky.indices[c.label][:, 1]
    from dang_b200.synth import TRUE_THETA, band_sed
    for j, b in enumerate(cfg.bands):
        sky.sig[j, 0] = sum(sky.truth[c.label][1] * band_sed(b, c, *TRUE_THETA[c.label]) for c in cfg.comps)
        sky.sig[j, 0] = sky.sig[j, 0] * sky.gain[j] + sky.offset[j] + sky.rms[j, 0] * rng.standard_normal(cfg.npix)
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eta = rng.standard_normal(cfg.npix)
    it_o, _, _ = ora.cg_search_trace(ml_mode=1, eta=eta)
    it_g, _ = eng.cg_solve(0, 0, "sample", eta=eta)
    assert it_g == it_o
    ora.update_sky_model()
    chisq_o, _ = ora.compute_chisq()
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o
    for band, z in ((0, 0.3), (3, -1.1)):
        g_o = ora.fit_band_gain(1, band, 1, z)
        g_g = eng.fit_band_gain(1, band, "sample", z)
        assert abs(g_g - g_o) <= TOL * abs(g_o)
    ora.update_sky_model()
    chisq_o, _ = ora.compute_chisq()
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o


def test_ensemble_of_chains_shares_one_copy_of_the_maps():
    """BASELINE config c5 in miniature: independent chains (different deviates) on one GPU that
    borrow one device copy of sig / rms / mask evolve exactly like chains with private copies."""
    from dang_b200.engine import Engine
    cfg, sky = small_case("c2", 16, perturb=False)
    owner = Engine(cfg, sky)
    members = [owner] + [Engine(cfg, sky, share_maps_with=owner) for _ in range(3)]
    private = [Engine(cfg, sky) for _ in range(4)]
    for it in (1, 2, 3):
        for k, (a, b) in enumerate(zip(members, private)):  # interleaved: chains do not disturb each other
            ra = a.gibbs_iteration(it, seed=1000 * k)
            rb = b.gibbs_iteration(it, seed=1000 * k)
            assert ra[0][0] == rb[0][0] and ra[0][1] == rb[0][1]
    for a, b in zip(members, private):
        for ic in range(2):
            assert np.array_equal(a.amplitude(ic), b.amplitude(ic))
            assert np.array_equal(a.indices(ic), b.indices(ic))
    assert not np.array_equal(members[0].amplitude(0), members[1].amplitude(0))  # different chains
    for e in members[1:] + private:
        e.close()


# ------------------------------------------------------------------ error behaviour
def test_errors_are_loud_and_specific():
    """Everything outside the built scope fails with a nonzero code and a message (the Fortran
    shim prints it and stops, like the reference's own `write(*,*) ...; stop`)."""
    import ctypes as C
    from dang_b200 import _lib
    from dang_b200.engine import DangGpuError, Engine
    cfg, sky = small_case("c1", 4)
    # sample_nside /= nside needs HEALPix udgrade_ring (out of scope)
    cfg.comps[0].indices[0].samp_nside = 2
    eng = Engine(cfg, sky)
    with pytest.raises(DangGpuError, match="udgrade"):
        eng.sample_index_mh(0, 0, -1, 4)
    cfg2, sky2 = small_case("c1", 4)
    eng2 = Engine(cfg2, sky2)
    with pytest.raises(DangGpuError, match="unreachable"):
        eng2.sample_index_mh(0, 0, -2, 4)
    with pytest.raises(DangGpuError, match="CG group"):
        eng.cg_solve(ig=5)
    lib = _lib.load()
    # unknown component type
    rc = lib.dang_gpu_set_component(eng.h, 0, 12, b"what", 30e9, 1, 1, None, None)
    assert rc == 1 and b"unrecognized" in lib.dang_gpu_last_error(eng.h)
    # bad geometry at creation
    h = _lib.vp()
    assert lib.dang_gpu_create(0, 4, 191, 3, 5, 2, 0, 191, C.byref(h)) == 1
    assert lib.dang_gpu_create(0, 4, 192, 3, 5, 2, 10, 5, C.byref(h)) == 1
    assert lib.dang_gpu_create(99, 4, 192, 3, 5, 2, 0, 192, C.byref(h)) == 1
    # operators before the maps are uploaded
    assert lib.dang_gpu_create(0, 4, 192, 3, 5, 2, 0, 192, C.byref(h)) == 0
    planes = (C.c_double * 3)()
    n = C.c_int64()
    assert lib.dang_gpu_chisq(h, 2, 3, planes, C.byref(n)) == 5
    assert b"upload_maps" in lib.dang_gpu_last_error(h)
    lib.dang_gpu_destroy(h)


# ------------------------------------------------------------------ round-2 additions (VERDICT r1 "missing" 4, "weak" 12)
def test_step_size_tuner_marginal_likelihood():
    """tune_spectral_parameter_length with lnl_type 'marginal' (src/dang_sample_mod.f90:650-651, 676-677): the
    streaming tuner runs the same blocks and lands on the same step as the oracle."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c2", 8, perturb=False)
    rng = np.random.default_rng(17)
    for c in cfg.comps:  # non-zero amplitudes: the marginal likelihood divides by sum(TN * model)
        sky.amplitude[c.label][1:3] = sky.truth[c.label][1:3] * (1.0 + 0.05 * rng.standard_normal((2, cfg.npix)))
    spec = cfg.comps[1].indices[0]
    spec.lnl_type, spec.tune = "marginal", True
    nsample, max_blocks = 10, 6
    for step0 in (0.3, 0.002):
        spec.step = step0
        ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
        z, u = rng.standard_normal(nsample * max_blocks), rng.random(nsample * max_blocks)
        nb_o, step_o = ora.tune_step(1, 0, -1, nsample, 1, z, u, max_blocks)
        nb_g, step_g = eng.tune_index(1, 0, -1, nsample, "sample", z, u, max_blocks=max_blocks)
        assert nb_g == nb_o and nb_o >= 1 and step_g == step_o, (step0, nb_g, nb_o, step_g, step_o)


def test_step_size_tuner_starts_a_per_pixel_index_at_the_map_mean():
    """The per-pixel call site (src/dang_sample_mod.f90:341-347) starts the tuner at sum(indices) / sum(mask)."""
    from dang_b200.engine import DangGpuError, Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c1", 8)
    spec = cfg.comps[0].indices[0]
    spec.tune, spec.step = True, 0.4
    nsample, max_blocks = 12, 8
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    rng = np.random.default_rng(23)
    z, u = rng.standard_normal(nsample * max_blocks), rng.random(nsample * max_blocks)
    nb_o, step_o = ora.tune_step(0, 0, -1, nsample, 1, z, u, max_blocks, perpixel_start=True)
    nb_g, step_g = eng.tune_index(0, 0, -1, nsample, "sample", z, u, max_blocks=max_blocks)
    assert nb_g == nb_o and step_g == step_o and step_g != 0.4, (nb_g, nb_o, step_g, step_o)
    # a two-index component cannot be tuned per pixel (the reference calls the tuner with T = 0)
    cfg2, sky2 = small_case("c4", 4)
    cfg2.comps[1].indices[0].region = "per-pixel"
    with pytest.raises(DangGpuError, match="never terminates"):
        Engine(cfg2, sky2).tune_index(1, 0, -1, 4, "sample", z, u, max_blocks=2)


def test_gibbs_loop_tunes_an_untuned_index_once():
    """Engine.sample_spectral_parameters mirrors sample_index_mh: `.not. c%tuned` -> tune first, then draw; once."""
    from dang_b200.engine import Engine
    cfg, sky = small_case("c2", 8, perturb=False)
    spec = cfg.comps[1].indices[0]
    spec.tune, spec.step = True, 0.5
    eng = Engine(cfg, sky)
    eng.sample_cg_groups(seed=1)
    eng.sample_spectral_parameters(seed=2)
    step1 = eng.lib.dang_gpu_get_step_size
    import ctypes as C
    v = C.c_double()
    eng._ck(step1(eng.h, 1, 0, C.byref(v)))
    assert v.value < 0.5 and eng._tuned[1] == [True, True]
    s_after = v.value
    eng.sample_spectral_parameters(seed=3)
    eng._ck(step1(eng.h, 1, 0, C.byref(v)))
    assert v.value == s_after


def test_perpixel_jeffreys_prior():
    """eval_jeffreys_prior (src/dang_lnl_mod.f90:242-304, label 'synch' only) in the per-pixel chains."""
    cfg, sky = small_case("c1", 8)
    cfg.comps[0].indices[0].prior = "jeffreys"
    ora, eng, (acc_o, dec_o, lnl_o), (acc_g, dec_g, lnl_g) = run_perpixel(cfg, sky, 0, 0, 10)
    assert np.array_equal(dec_g, dec_o) and acc_g == acc_o
    ev = dec_o < 2
    assert 0 < (dec_o == 1).sum() < ev.sum()
    assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL
    assert rel_err(eng.indices(0), ora.indices(0)) < 1e-14


def test_reupload_after_cg_swap():
    """swap_cg_maps (src/dang.f90:92-97, dang_data_mod.f90:179-227) replaces sig / rms between iterations:
    dang_gpu_upload_maps again, and the next solve behaves exactly like a fresh handle on the new maps that starts
    from the same amplitudes (self%x survives the swap, Q10); its chi-square matches the oracle on the new maps."""
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c2", 8, perturb=False)
    sky_b = clone_sky(sky)
    rng = np.random.default_rng(29)
    sky_b.sig = sky.sig + 0.5 * sky.rms * rng.standard_normal(sky.sig.shape)
    sky_b.rms = sky.rms * (1.0 + 0.2 * rng.random(sky.rms.shape))
    eng = Engine(cfg, sky)
    eng.sample_cg_groups(eta=rng.standard_normal(2 * cfg.npix))
    eng.upload_maps(sky_b)                       # the swap
    eng2 = Engine(cfg, sky_b)                    # a fresh handle on the swapped maps, same start
    for ic in range(len(cfg.comps)):
        eng2.set_amplitude(ic, eng.amplitude(ic))
    eta2 = rng.standard_normal(2 * cfg.npix)
    it_a, _ = eng.cg_solve(0, 0, "sample", eta=eta2)
    it_b, _ = eng2.cg_solve(0, 0, "sample", eta=eta2)
    assert it_a == it_b
    for ic in range(len(cfg.comps)):
        assert np.array_equal(eng.amplitude(ic), eng2.amplitude(ic))
    ora = Oracle(cfg, sky_b)
    for ic in range(len(cfg.comps)):
        ora.amplitude(ic)[:] = eng.amplitude(ic)
    ora.update_sky_model()
    chisq_o, _ = ora.compute_chisq()
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o


def test_bandpass_quadrature_on_a_jagged_table():
    """The default 8-node Gauss rule against a deliberately jagged bandpass (random tau, unequal spacing): the
    exactness argument does not care about the shape of tau, only about the smoothness of the SED across the band."""
    from dang_b200.config import Band
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = small_case("c3", 4)
    rng = np.random.default_rng(31)
    for j, b in enumerate(cfg.bands):
        nu = np.sort(b.nu_ghz * (1.0 + 0.12 * (2.0 * rng.random(97) - 1.0)))
        tau = rng.random(97) ** 3 + 0.01 * (rng.random(97) < 0.3)
        cfg.bands[j] = Band(nu_ghz=b.nu_ghz, label=b.label, bp_nu_ghz=nu, bp_tau=tau)
    from dang_b200.synth import make_sky
    sky2 = make_sky(cfg)
    sky2.amplitude, sky2.indices = sky.amplitude, sky.indices
    ora, eng = Oracle(cfg, sky2), Engine(cfg, sky2)
    ora.update_sky_model()
    chisq_o, planes_o = ora.compute_chisq()
    planes_g, _ = eng.chisq_planes()
    assert rel_err(planes_g, planes_o) < TOL
    sky_g, _, _ = eng.update_sky_model()
    assert rel_err(sky_g, ora.sky_model()) < 1e-12


@pytest.mark.parametrize("kind", ["ring", "rms", "mask"])
@pytest.mark.parametrize("nside_in,nside_out", [(32, 8), (8, 32), (16, 16), (64, 1)])
def test_udgrade_operators_match_the_oracle(kind, nside_in, nside_out):
    """SURVEY 8f-2: udgrade_ring (HEALPix udgrade_nr) / udgrade_rms / udgrade_mask (src/dang_util_mod.f90:341-376)
    as device operators, bit-equal to the oracle's restatement (same NESTED summation order), bad pixels included."""
    from dang_b200.engine import Engine
    from oracle.binding import udgrade
    cfg, sky = small_case("c1", 4)
    eng = Engine(cfg, sky)
    rng = np.random.default_rng(41)
    n = 12 * nside_in * nside_in
    data = rng.standard_normal((3, n)) if kind == "ring" else np.abs(rng.standard_normal((3, n))) + 0.1
    if kind == "mask":
        data = (rng.random((3, n)) < 0.6).astype(float)
    if kind == "ring":
        data[1, rng.random(n) < 0.3] = -1.6375e30   # HPX bad pixels are skipped by the average
        data[2, :] = -1.6375e30
    out_o = udgrade(kind, data, nside_in, nside_out, 0.5)
    out_g = eng.udgrade(kind, data, nside_in, nside_out, 0.5)
    assert np.array_equal(out_g, out_o)
