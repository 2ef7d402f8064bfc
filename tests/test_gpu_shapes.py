"""Every band-count, component-count and single-plane specialisation of the kernels against the oracle.

The library picks template instances by band count (per-pixel Metropolis: NB = 8 / 12 / 20 / 32 bands per thread, or
2 / 3 / 5 / 8 bands per lane), by component count (CG C = 1..4, chi-square NC = 1..4, 8, statistics 2 / 4 / generic)
and by the number of polarisation planes S of a draw or solve.  The parity tests elsewhere run the four BASELINE
configurations only; here a synthetic run is built for any band list (log-spaced 20..857 GHz, up to DG_MAX_BANDS = 32)
and any component list (up to DG_MAX_COMPS = 8), and every instance, batch tail (B mod 4), size threshold and S = 1
branch is compared with the CPU oracle on injected deviates.

The parameter lists below are module-level constants.  test_dispatch_reaches_every_instance (no GPU) reads the
dispatch lines of the sources and fails when an instance is added that no case reaches."""
import math
import os
import re

import numpy as np
import pytest

from conftest import TOL, rel_err
from helpers import deviates

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dang_b200", "csrc")

# every NB instance (8 / 12 / 20 / 32), every bands-per-lane rounding (2 / 3 / 5 / 8), both sides of the uni / generic
# K1 switch (B 20 / 21) and every tail of the band batches of four (B mod 4 = 0..3)
BANDS = (1, 2, 3, 4, 6, 9, 12, 13, 16, 17, 20, 21, 27, 32)
# the bands of BANDS by the instance they are meant to reach (the CPU guard checks this against the sources)
BAND_GROUPS = ((1, 2, 3, 4, 6), (9, 12), (13, 16, 17, 20), (21, 27, 32))
# the diffuse components in the order a case takes them (labels of repeats get a suffix)
COMPS = ("synch", "dust", "ff", "cmb", "ame", "synch", "dust", "ff")
# (component, index) of each SED mode of the per-pixel kernels, with components COMPS[:2]
SED = {"powerlaw": (0, 0), "mbb_beta": (1, 0), "mbb_T": (1, 1)}


# ------------------------------------------------------------------ builder
def _component(kind):
    from dang_b200.config import Component, IndexSpec
    if kind == "synch":
        return Component("synch", "power-law", 30.0, indices=[
            IndexSpec("BETA", -3.0, prior="gaussian", gauss=(-3.1, 0.1), uni=(-4.0, -2.0), step=0.05)])
    if kind == "dust":
        return Component("dust", "mbb", 353.0, indices=[
            IndexSpec("BETA", 1.5, prior="gaussian", gauss=(1.55, 0.1), uni=(1.0, 2.2), step=0.05),
            IndexSpec("T", 19.0, prior="gaussian", gauss=(19.6, 1.0), uni=(10.0, 35.0), step=0.5)])
    if kind == "ff":
        return Component("ff", "freefree", 40.0, indices=[
            IndexSpec("T_e", 7000.0, prior="uniform", uni=(4000.0, 11000.0), step=300.0)])
    if kind == "cmb":
        return Component("cmb", "cmb", 100.0, indices=[])
    if kind == "ame":
        return Component("ame", "lognormal", 22.0, indices=[IndexSpec("NU_P", 21.0), IndexSpec("W_AME", 0.55)])
    raise ValueError(kind)


def shape_case(nbands, comps=COMPS[:2], nside=16, poltype="Q+U", varying=None, seed=20261020, out_of_group=()):
    """A run over `nbands` delta bands log-spaced over 20..857 GHz (noise from synth.band_sigma) with the diffuse
    components `comps` (kinds of COMPS), all in CG group 1 except the labels in `out_of_group`.  The sky is
    synth.make_sky's, perturbed as helpers.small_case does; components without a simulated sky get random amplitudes.
    `varying`: labels whose index maps vary per pixel (None: all), the others stay uniform."""
    from dang_b200.config import Band, CGGroup, RunConfig
    from dang_b200.synth import TRUE_THETA, make_sky
    nus = np.exp(np.linspace(np.log(20.0), np.log(857.0), nbands))
    clist = []
    for n, kind in enumerate(comps):
        c = _component(kind)
        if kind in comps[:n]:
            c.label = f"{kind}{n}"
        for s in c.indices:
            s.poltype = poltype
        c.cg_group = 2 if c.label in out_of_group else 1
        clist.append(c)
    groups = [CGGroup(sample=True, max_iter=200, converge=1e-12, poltype=poltype)]
    if out_of_group:
        groups.append(CGGroup(sample=False, max_iter=200, converge=1e-12, poltype=poltype))
    cfg = RunConfig(f"shape_b{nbands}_c{len(comps)}", nside, [Band(float(nu)) for nu in nus], clist, groups, nsample=12)
    sky = make_sky(cfg, seed=seed, noise_seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    for c in cfg.comps:
        if c.label in TRUE_THETA:
            sky.amplitude[c.label][1:3] = sky.truth[c.label][1:3] * (1.0 + 0.05 * rng.standard_normal((2, cfg.npix)))
        else:
            sky.amplitude[c.label][1:3] = rng.normal(0.0, 5.0, size=(2, cfg.npix))
        if varying is None or c.label in varying:
            for k, s in enumerate(c.indices):
                sky.indices[c.label][k][:] = (s.init + 0.02 * rng.standard_normal(cfg.npix))[None, :]
    return cfg, sky


def _planes(map_n):
    return (1, 2) if map_n == -1 else (map_n - 1,)


# ------------------------------------------------------------------ (a) per-pixel draws
PP_FAMILIES = {"pixel": dict(fast=3, serial=0), "lane": dict(fast=1, serial=0), "fp64": dict(fast=0, serial=0),
               "serial": dict(fast=1, serial=1)}


def _pp_record_cases():
    cases, used = [], [0] * len(BAND_GROUPS)
    for family in PP_FAMILIES:
        for sed in SED:
            for g, group in enumerate(BAND_GROUPS):
                for map_n in (-1, 2 + used[g] // 2 % 2):   # S = 2, and S = 1 on Q or U
                    cases.append((family, sed, group[used[g] % len(group)], map_n))
                    used[g] += 1
    return cases


PP_RECORD = _pp_record_cases()
# production mode (no recording): the screened forms against the fp64 kernel, one padded band count per instance
PP_PROD_FAMILIES = {"pixel": 3, "lane": 1, "split": 2}
PP_PROD = [(family, sed, B) for family in PP_PROD_FAMILIES for sed in SED for B in (6, 9, 17, 27)]


def _perpixel_record(family, sed, B, map_n, nside=16, nsample=12, pix_range=None):
    from dang_b200.engine import OPT_PERPIXEL_FAST, OPT_PERPIXEL_SERIAL, OPT_RECORD, Engine
    from oracle.binding import Oracle
    ic, nind = SED[sed]
    cfg, sky = shape_case(B, nside=nside)
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region = True, "per-pixel"
    lo, hi = pix_range or (0, cfg.npix)
    if pix_range:
        sky.mask[:lo] = 0.0
        sky.mask[hi:] = 0.0
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky, pix_range=pix_range)
    eng.set_option(OPT_RECORD, 1)
    eng.set_option(OPT_PERPIXEL_SERIAL, PP_FAMILIES[family]["serial"])
    eng.set_option(OPT_PERPIXEL_FAST, PP_FAMILIES[family]["fast"])
    z, u = deviates(cfg, nsample, seed=1000 * B + nside + map_n)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, map_n, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(ic, nind, map_n, nsample, "sample", z, u)
    dec_g, lnl_g = eng.decisions(nsample, fullsky=False)
    dec_g, lnl_g = dec_g.reshape(nsample, -1)[:, lo:hi], lnl_g.reshape(nsample, -1)[:, lo:hi]
    dec_o, lnl_o = dec_o.reshape(nsample, -1)[:, lo:hi], lnl_o.reshape(nsample, -1)[:, lo:hi]
    assert np.array_equal(dec_g, dec_o), f"{(dec_g != dec_o).sum()} decisions differ"
    assert acc_g == acc_o
    ev = dec_o < 2
    assert ev.any() and 0 < acc_o
    assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL
    idx_g, idx_o = eng.indices(ic)[:, :, lo:hi], ora.indices(ic)[:, :, lo:hi]
    assert rel_err(idx_g, idx_o) < 1e-14
    masked = sky.mask[lo:hi] == 0
    idx0 = sky.indices[cfg.comps[ic].label][:, :, lo:hi]
    for l in range(idx_g.shape[0]):
        for k in range(3):
            if l == nind and k in _planes(map_n):
                assert np.all(idx_g[l, k, masked] == 0.0)
            else:  # planes and indices the draw does not own are untouched
                assert np.array_equal(idx_g[l, k], idx0[l, k]), (l, k)
    if family in ("pixel", "lane"):  # record mode checks every screened difference against its error bound
        assert eng.perpixel_stats()[1] == 0
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize("family,sed,B,map_n", PP_RECORD)
def test_perpixel_record_mode(family, sed, B, map_n):
    _perpixel_record(family, sed, B, map_n)


@pytest.mark.gpu
@pytest.mark.parametrize("family,sed,B", PP_PROD)
def test_perpixel_production_matches_fp64(family, sed, B):
    """Long chains with three times the configured steps at nside 64: the screened forms leave the fp64 kernel's maps
    and counts, and the fp64 fallback of every (instance, SED mode) is exercised (padded instance, S = 2 and 1) but
    stays the exception: a screened state gone non-finite (e.g. a padding band's K_j) falls back on every proposal."""
    from dang_b200.engine import OPT_PERPIXEL_FAST, Engine
    ic, nind = SED[sed]
    cfg, sky = shape_case(B, nside=64)
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region = True, "per-pixel"
    spec.step *= 3.0
    nsample = 40
    a, b = Engine(cfg, sky), Engine(cfg, sky)
    a.set_option(OPT_PERPIXEL_FAST, PP_PROD_FAMILIES[family])
    b.set_option(OPT_PERPIXEL_FAST, 0)
    fallbacks, proposals = 0.0, 0
    for map_n in (-1, 2, 3):
        proposals += nsample * int((sky.mask != 0).sum())
        z, u = deviates(cfg, nsample, seed=B + map_n)
        acc_a = a.sample_index_mh(ic, nind, map_n, nsample, "sample", z, u)
        fallbacks += a.perpixel_stats()[0]
        acc_b = b.sample_index_mh(ic, nind, map_n, nsample, "sample", z, u)
        assert acc_a == acc_b and acc_a > 0, map_n
        assert np.array_equal(a.indices(ic), b.indices(ic)), map_n
    print(f"fallbacks {family} {sed} B={B}: {fallbacks:.0f} of {proposals}")
    # (the pixel form's single bound per pixel gives up on ~20 % of these long-step power-law proposals, whose
    # ln(nu / nu_ref) spans 20..857 GHz; a non-finite state falls back on nearly all of them)
    assert 0 < fallbacks < 0.5 * proposals, (fallbacks, proposals)


# ------------------------------------------------------------------ (b) full-sky draws
FS_FAMILIES = ("ring", "uni", "stream")


def _fs_cases():
    cases = []
    for f, family in enumerate(FS_FAMILIES):
        for i, B in enumerate(BANDS):
            n = i + f
            cases.append((family, B, (-1, 2, 3)[n % 3], (24, 200)[n % 2], (2, 3, 4, 5)[n % 4], tuple(SED)[n % 3]))
    return cases


FS_CASES = _fs_cases()


def _fullsky(family, B, map_n, nsample, ncomp, sed, nside=16):
    from dang_b200.engine import OPT_FULLSKY_STREAM, OPT_STREAM_RING, Engine
    from oracle.binding import Oracle
    ic, nind = SED[sed]
    cfg, sky = shape_case(B, COMPS[:ncomp], nside=nside, varying=())
    spec = cfg.comps[ic].indices[nind]
    spec.sample, spec.region, spec.step = True, "fullsky", (0.002, 0.02)[nind]
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eng.set_option(OPT_STREAM_RING, int(family != "uni"))
    eng.set_option(OPT_FULLSKY_STREAM, int(family == "stream"))
    rng = np.random.default_rng(100 * B + nsample)
    z, u = rng.standard_normal(nsample), rng.random(nsample)
    acc_o, dec_o, lnl_o = ora.sample_index_mh(ic, nind, map_n, nsample, 1, z, u, want_trace=True)
    acc_g = eng.sample_index_mh(ic, nind, map_n, nsample, "sample", z, u)
    dec_g, lnl_g = eng.decisions(nsample, fullsky=True)
    dec_o, lnl_o = dec_o[:nsample], lnl_o[:nsample]
    assert np.array_equal(dec_g, dec_o), (dec_g, dec_o)
    assert acc_g == acc_o
    ev = dec_o < 2
    assert ev.any()
    assert rel_err(lnl_g[ev], lnl_o[ev]) < TOL
    assert rel_err(eng.indices(ic), ora.indices(ic)) < 1e-14
    for k in _planes(map_n):
        assert eng.index_fullsky(ic, nind, k + 1) == ora.indices(ic)[nind, k, 0]
    ora.update_sky_model()
    chisq_o, _ = ora.compute_chisq()
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o


@pytest.mark.gpu
@pytest.mark.parametrize("family,B,map_n,nsample,ncomp,sed", FS_CASES)
def test_fullsky_draw(family, B, map_n, nsample, ncomp, sed):
    _fullsky(family, B, map_n, nsample, ncomp, sed)


# ------------------------------------------------------------------ (c) CG
CG_FORMS = ("persistent", "recompute8", "streaming", "two_pass")
# (C, form, K1 path, group poltype, B).  K1: 'ring' all uniform; 'uni1' / 'uni2' one / two components with varying
# indices (staged in shared memory while 2 * B * 2 * 256 * 8 B <= 160 KiB, i.e. B <= 20); 'generic' two varying
# components at B >= 21; 'generic_og' a varying component outside the group.  The persistent solve exists for C <= 2.
CG_CASES = [(C, form, "ring", "Q+U", B) for C, B in ((1, 4), (2, 6), (3, 9), (4, 13))
            for form in CG_FORMS if form != "persistent" or C <= 2] + [
    (1, "persistent", "uni1", "Q+U", 9), (1, "recompute8", "uni1", "U", 3), (2, "persistent", "uni1", "Q", 13),
    (2, "persistent", "uni2", "Q+U", 20), (2, "recompute8", "uni2", "U", 16), (2, "persistent", "generic", "Q+U", 21),
    (2, "two_pass", "generic", "Q", 32), (1, "streaming", "generic_og", "Q+U", 27), (3, "recompute8", "uni2", "Q", 12),
    (3, "two_pass", "generic", "U", 21), (4, "recompute8", "uni2", "Q+U", 17), (4, "streaming", "generic", "Q", 27),
    (4, "persistent", "ring", "U", 8)]


def _cg(C, form, k1, poltype, B, nside=16, pix_range=None):
    from dang_b200.engine import OPT_CG_CHECKPOINT, OPT_CG_PERSISTENT, OPT_CG_TWO_PASS, Engine
    from oracle.binding import Oracle
    comps = COMPS[:C] + (("dust",) if k1 == "generic_og" else ())
    varying = {"ring": (), "uni1": ("synch",), "uni2": ("synch", "dust"), "generic": ("synch", "dust"),
               "generic_og": ("dust",)}[k1]
    cfg, sky = shape_case(B, comps, nside=nside, poltype=poltype, varying=varying,
                          out_of_group=("dust",) if k1 == "generic_og" else ())
    lo, hi = pix_range or (0, cfg.npix)
    if pix_range:
        sky.mask[:lo] = 0.0
        sky.mask[hi:] = 0.0
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky, pix_range=pix_range)
    eng.set_option(OPT_CG_PERSISTENT, int(form == "persistent"))
    eng.set_option(OPT_CG_CHECKPOINT, 0 if form == "streaming" else 8)
    eng.set_option(OPT_CG_TWO_PASS, int(form == "two_pass"))
    S = 2 if poltype == "Q+U" else 1
    rng = np.random.default_rng(B + 10 * C)
    for _ in range(2):  # the second solve starts from the first one's x
        eta = rng.standard_normal(S * cfg.npix)
        it_o, _, trace_o = ora.cg_search_trace(ml_mode=1, eta=eta)
        it_g, _ = eng.cg_solve(0, 0, "sample", eta=eta)
        trace_g = eng.cg_trace()
        assert it_g == it_o, (it_g, it_o)
        assert np.allclose(trace_g, trace_o, rtol=1e-7, atol=0)
        for ic in range(len(cfg.comps)):
            assert rel_err(eng.amplitude(ic)[:, lo:hi], ora.amplitude(ic)[:, lo:hi]) < TOL, ic
    if not pix_range:
        assert rel_err(eng.cg_x(), ora.cg_x()) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("C,form,k1,poltype,B", CG_CASES)
def test_cg_solve(C, form, k1, poltype, B):
    _cg(C, form, k1, poltype, B)


@pytest.mark.gpu
def test_cg_template_group_with_32_fitted_pairs():
    """A template fitted to all 32 bands next to diffuse synchrotron: the border tail at its limit of 32 (component,
    band) pairs.  The bordered system is ill-conditioned (tests/test_gpu_parity.py::test_template_cg_operator_matches_oracle:
    the trajectory of ANY two implementations parts after a few iterations), so parity is asserted on the operator --
    the first residual norms -- and on the converged solution, as for the other template tests."""
    from dang_b200.config import Component
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = shape_case(32, ("synch",), varying=())
    cfg.comps.append(Component(label="tmpl", type="template", nu_ref_ghz=353.0, cg_group=1, corr=[True] * 32))
    cfg.cg_groups[0].converge, cfg.cg_groups[0].max_iter = 1e-20, 300
    rng = np.random.default_rng(32)
    T = np.ones((3, cfg.npix))
    T[1:3] = np.abs(rng.normal(0.0, 1.0, size=(2, cfg.npix))) + 0.05
    T[1:3] /= T[1:3].max(axis=1, keepdims=True)
    for j, b in enumerate(cfg.bands):
        sky.sig[j, 1:3] += 40.0 * (b.nu_ghz / 353.0) ** 1.6 * T[1:3]
    sky.template = {"tmpl": T}
    sky.template_amplitudes = {"tmpl": np.zeros((3, 32))}
    sky.amplitude["tmpl"] = np.zeros((3, cfg.npix))
    sky.indices["tmpl"] = np.zeros((0, 3, cfg.npix))
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky)
    eta = rng.standard_normal(2 * cfg.npix)
    it_o, delta_o, tr_o = ora.cg_search_trace(0, 0, 1, eta)
    it_g, delta_g = eng.cg_solve(0, 0, "sample", eta)
    tr_g = eng.cg_trace()
    assert np.max(np.abs(tr_g[:5] - tr_o[:5]) / tr_o[:5]) < 1e-12
    assert delta_g <= 1e-20 and delta_o <= 1e-20
    assert rel_err(eng.template_amplitudes(1), ora.template_amplitudes(1)) < 1e-8
    assert rel_err(eng.amplitude(0), ora.amplitude(0)) < 1e-8


# ------------------------------------------------------------------ (d) chi-square and sky model
CHISQ_CASES = [(ncomp, varying, BANDS[(2 * ncomp + varying) % len(BANDS)]) for ncomp in range(1, 9) for varying in (0, 1)]


def _chisq(ncomp, varying, B, nside=16, pix_range=None):
    from dang_b200.engine import Engine
    from oracle.binding import Oracle
    cfg, sky = shape_case(B, COMPS[:ncomp], nside=nside, varying=None if varying else ())
    lo, hi = pix_range or (0, cfg.npix)
    if pix_range:
        sky.mask[:lo] = 0.0
        sky.mask[hi:] = 0.0
    ora, eng = Oracle(cfg, sky), Engine(cfg, sky, pix_range=pix_range)
    ora.update_sky_model()
    chisq_o, planes_o = ora.compute_chisq()
    planes_g, n = eng.chisq_planes()
    assert n == int((sky.mask != 0).sum())
    assert rel_err(planes_g, planes_o) < TOL
    assert abs(eng.compute_chisq() - chisq_o) <= TOL * chisq_o
    sky_g, res_g, chi_g = eng.update_sky_model()
    assert rel_err(sky_g[..., lo:hi], ora.sky_model()[..., lo:hi]) < TOL
    assert rel_err(res_g[..., lo:hi], ora.res_map()[..., lo:hi]) < TOL
    assert rel_err(chi_g[..., lo:hi], ora.chi_map()[..., lo:hi]) < TOL
    assert np.all(chi_g[:, sky.mask == 0] == 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("ncomp,varying,B", CHISQ_CASES)
def test_chisq_and_sky_model(ncomp, varying, B):
    _chisq(ncomp, varying, B)


# ------------------------------------------------------------------ (e) sizes and limits
@pytest.mark.gpu
@pytest.mark.parametrize("nside", [1, 2])
def test_tiny_maps(nside):
    """P < 64: one partly filled 64-pixel plane (12 and 48 pixels).

    The C = 3 solve runs at nside 2 only.  At nside 1 a C = 3 solve on one plane has 24 unknowns (8 unmasked pixels,
    condition number 465 with 13 bands, 1.7e3 with 6) and CG ends only by exhausting that 24-dimensional Krylov space:
    its last residual norm drops by 1e3 to the rounding floor, where summation order decides it (measured on a B200:
    2.8e-14 in the oracle against 8.3e-14 on the GPU at 13 bands; at 6 bands 27 against 28 iterations).  The C = 2 solve
    (32 unknowns, condition number 2.6) converges in 13 iterations, well before its Krylov space runs out."""
    _perpixel_record("pixel", "mbb_T", 12, -1, nside=nside)
    _perpixel_record("fp64", "powerlaw", 3, 2, nside=nside)
    _perpixel_record("lane", "mbb_beta", 27, 3, nside=nside)
    _fullsky("ring", 9, -1, 24, 3, "mbb_beta", nside=nside)
    _fullsky("uni", 21, 3, 200, 5, "powerlaw", nside=nside)
    _cg(2, "persistent", "uni2", "Q+U", 9, nside=nside)
    if nside == 2:
        _cg(3, "recompute8", "ring", "Q", 6, nside=nside)
    _chisq(3, 0, 13, nside=nside)
    _chisq(6, 1, 4, nside=nside)


ODD_RANGE = (101, 600)  # 499 pixels of nside 8: odd P, not a ring boundary


@pytest.mark.gpu
def test_odd_pixel_range_handle():
    """A handle over an arbitrary odd range [lo, hi) (the ABI takes one): every pixel outside it is masked, so the
    oracle's global sums are the handle's."""
    _chisq(4, 1, 9, nside=8, pix_range=ODD_RANGE)
    _cg(2, "persistent", "uni2", "Q+U", 9, nside=8, pix_range=ODD_RANGE)
    _cg(3, "streaming", "ring", "U", 12, nside=8, pix_range=ODD_RANGE)
    _perpixel_record("pixel", "powerlaw", 17, -1, nside=8, pix_range=ODD_RANGE)
    _perpixel_record("fp64", "mbb_T", 6, 2, nside=8, pix_range=ODD_RANGE)


@pytest.mark.gpu
def test_limits_are_loud():
    from dang_b200.config import Component
    from dang_b200.engine import DangGpuError, Engine
    cfg, sky = shape_case(33, nside=1)
    with pytest.raises(DangGpuError, match="nbands = 33"):
        Engine(cfg, sky)
    cfg, sky = shape_case(4, COMPS + ("cmb",), nside=1)
    with pytest.raises(DangGpuError, match="ncomp = 9"):
        Engine(cfg, sky)
    cfg, sky = shape_case(8, COMPS[:5], nside=2)
    with pytest.raises(DangGpuError, match="5 diffuse components"):
        Engine(cfg, sky).cg_solve(0, 0, "sample", eta=np.zeros(2 * cfg.npix))
    # 32 + 1 fitted (template, band) pairs in one group: one more than the border tail holds
    cfg, sky = shape_case(32, ("synch",), nside=2, varying=())
    for label, corr in (("t1", [True] * 32), ("t2", [j == 0 for j in range(32)])):
        cfg.comps.append(Component(label=label, type="template", nu_ref_ghz=353.0, cg_group=1, corr=corr))
        sky.template = dict(sky.template or {}, **{label: np.ones((3, cfg.npix))})
        sky.template_amplitudes = dict(sky.template_amplitudes or {}, **{label: np.zeros((3, 32))})
        sky.amplitude[label] = np.zeros((3, cfg.npix))
        sky.indices[label] = np.zeros((0, 3, cfg.npix))
    with pytest.raises(DangGpuError, match="33 fitted"):
        Engine(cfg, sky).cg_solve(0, 0, "sample", eta=np.zeros(2 * cfg.npix))


# ------------------------------------------------------------------ dispatch coverage (CPU)
def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _ladder(text, cond, call):
    """Instance chosen for a value by an if / else-if / else ladder `if (<cond> N) <call>(M) ... else <call>(K)`:
    returns (pick(value), all instances)."""
    steps = [(int(n), int(m)) for n, m in re.findall(cond + r"\s*(\d+)\)\s*" + call + r"\(?(\d+)", text)]
    last = re.findall(r"else\s+" + call + r"\(?(\d+)", text)
    assert steps and len(last) == 1, (cond, call)
    last = int(last[0])
    return (lambda v: next((m for n, m in steps if v <= n), last)), {m for _, m in steps} | {last}


def test_dispatch_reaches_every_instance():
    lanes = int(re.search(r"#define DG_MH_LANES (\d+)", _read("kernels_mh.cuh")).group(1))
    bpl = lambda B: math.ceil(B / lanes)  # noqa: E731
    # per-pixel kernels: the one-thread-per-pixel NB ladder, the bands-per-lane ladders of the lane, split and fp64 forms
    pix, pix_all = _ladder(_read("host_mh_ppx.cu"), r"h->nbands <=", "LAUNCH_PIX_MODE")
    ppf = _read("host_mh_ppf.cu")
    lane, lane_all = _ladder(ppf, r"bpl <=", "LAUNCH_PPF_MODE")
    split, split_all = _ladder(ppf, r"bpl <=", "LAUNCH_SPLIT_MODE")
    pp = _read("host_mh_pp.cu")
    fp64, fp64_all = _ladder(pp, r"bpl <=", "launch_perpixel_fp64_")
    # the shared-memory roundings `bpl <= N ? N : ...` agree with the launch ladders
    for text in (pp, ppf):
        for chain in re.findall(r"bpl <= \d+ \? \d+ :[^;]*;", text):
            steps = [(int(n), int(m)) for n, m in re.findall(r"bpl <= (\d+) \? (\d+)", chain)]
            last = int(re.search(r":\s*(\d+);", chain).group(1))
            for B in range(1, 33):
                assert next((m for n, m in steps if bpl(B) <= n), last) == lane(bpl(B)) == fp64(bpl(B)), chain
    # (the strict serial kernel has no band instance: its cases follow the pixel form's)
    inst = {"pixel": (lambda B: pix(B), pix_all), "lane": (lambda B: lane(bpl(B)), lane_all),
            "fp64": (lambda B: fp64(bpl(B)), fp64_all), "split": (lambda B: split(bpl(B)), split_all),
            "serial": (lambda B: pix(B), pix_all)}
    hit = {(f, inst[f][0](B), sed, len(_planes(m))) for f, sed, B, m in PP_RECORD}
    for f in PP_FAMILIES:
        for nb in inst[f][1]:
            for sed in SED:
                for S in (1, 2):
                    assert (f, nb, sed, S) in hit, ("record mode", f, nb, sed, S)
    prod = {(f, inst[f][0](B), sed) for f, sed, B in PP_PROD}
    for f in PP_PROD_FAMILIES:
        for nb in inst[f][1]:
            for sed in SED:
                assert (f, nb, sed) in prod, ("production mode", f, nb, sed)
    # BAND_GROUPS: each group is one NB instance; together they are BANDS
    assert sorted(B for g in BAND_GROUPS for B in g) == sorted(BANDS)
    for g in BAND_GROUPS:
        assert len({pix(B) for B in g}) == 1
    assert {B for _, _, B, _ in PP_RECORD} == set(BANDS) and {B % 4 for B in BANDS} == {0, 1, 2, 3}
    # full-sky statistics: the ring / uni kernels for ncomp <= 2 and <= 4, the generic kernel above, S = 1 and 2
    fs = _read("host_mh_fs.cu")
    uni_max = int(re.search(r"bool uni = h->ncomp <= (\d+);", fs).group(1))
    small = int(re.search(r"if \(h->ncomp <= (\d+)\) launch\(mh_suffstat_ring_kernel", fs).group(1))
    stat = lambda n: small if n <= small else uni_max if n <= uni_max else "generic"  # noqa: E731
    fs_hit = {(f, stat(nc), len(_planes(m))) for f, B, m, ns, nc, _ in FS_CASES}
    for f in ("ring", "uni"):
        for k in (small, uni_max, "generic"):
            for S in (1, 2):
                assert (f, k, S) in fs_hit, ("full-sky statistics", f, k, S)
    assert {ns for *_, ns, _, _ in FS_CASES} == {24, 200} and max(B for _, B, *_ in FS_CASES) == 32
    # CG: every C of the switch in every form that exists for it
    cg = _read("host_cg.cu")
    max_cg = int(re.search(r"#define DG_MAX_CG (\d+)", _read("common.cuh")).group(1))
    cases = {int(a): int(b) for a, b in re.findall(r"case (\d+): cg_solve_impl<(\d+)>", cg)}
    default = int(re.search(r"default: cg_solve_impl<(\d+)>", cg).group(1))
    pers_max = int(re.search(r"const bool persistent = .*C <= (\d+);", cg).group(1))
    cg_inst = lambda C: cases.get(C, default)  # noqa: E731
    cg_hit = {(cg_inst(C), form) for C, form, *_ in CG_CASES}
    for C in range(1, max_cg + 1):
        for form in CG_FORMS:
            if form != "persistent" or C <= pers_max:
                assert (cg_inst(C), form) in cg_hit, ("CG", C, form)
    assert {k1 for _, _, k1, _, _ in CG_CASES} == {"ring", "uni1", "uni2", "generic", "generic_og"}
    assert {p for *_, p, _ in CG_CASES} == {"Q+U", "Q", "U"}
    assert all(B >= 21 for _, _, k1, _, B in CG_CASES if k1 == "generic")
    # chi-square: every chisq_uni_kernel<NC> (planes, uniform indices) and chisq_kernel<NC> (maps)
    data = _read("host_data.cu")
    uni_nc = int(re.search(r"bool uni = .*h->ncomp <= (\d+);", data).group(1))
    pick_uni, uni_all = _ladder(data.replace("h->ncomp == ", "h->ncomp <= "), r"h->ncomp <=", "LAUNCH_CHISQ_UNI")
    gen = {int(a): int(b) for a, b in re.findall(r"ncomp (?:==|<=) (\d+)\) launch_chisq<(\d+)>", data)}
    gen_else = re.search(r"else launch_chisq<(\w+)>", data).group(1)
    gen_all = set(gen.values()) | {gen_else}
    assert {pick_uni(n) for n, v, _ in CHISQ_CASES if not v and n <= uni_nc} == uni_all
    assert {gen.get(n, gen_else) for n, _, _ in CHISQ_CASES} == gen_all
    assert {n for n, _, _ in CHISQ_CASES} == set(range(1, 9))


# ------------------------------------------------------------------ (f) two GPUs
@pytest.mark.gpu
def test_two_gpus_32_bands_fullsky_and_single_plane():
    """tests/multi_gpu_check.py, case 'b32': a full-sky Q+U draw and a single-plane draw at 32 bands, whose statistics
    rows (3 x 4 x 8 x 2 = 192 values per rank) are the largest the exchange carries -- over NVLink mailboxes and NCCL."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, DANG_MGC_CASE="b32", DANG_MGC_NSIDE="32")
    for mailbox in ("1", "0"):
        env["DANG_GPU_MAILBOX"] = mailbox
        p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29537",
                            os.path.join(ROOT, "tests", "multi_gpu_check.py")],
                           env=env, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        assert p.stdout.count("multi-GPU parity ok") == 2
