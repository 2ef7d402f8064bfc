"""Bandpass-integrated SEDs on the device against the extended-precision reference of test_bandpass_seds.py.

SED probe: one component per handle with amplitude 1 on every plane, so the sky model dang_gpu_get_sky_model returns
is the device's SED per (band, pixel).  Each pixel of an nside-16 map holds its own index value (pair) on a grid over
the parameter box (the sed_theta path), or every pixel holds one corner of the box (sed_table_kernel / sed_uniform).
Three band forms: delta bands, the full table (DANG_OPT_BP_QUADRATURE = 0) and the default (a Gauss rule wherever the
library verified one).

Bars.  1e-14 relative where the formula is well conditioned.  Where the reference's own fp64 operation order loses
digits, the bar is 1e-14 + 8 eps cond, with the condition number of that order at the band's worst sample:
  exp(x) - 1 at small x (mbb's Planck factors at x = h nu / kT, 'cmb' (twice), T_cmb / hi_fit): 1 / x;
  exp(x) at large x (the same factors in the Wien tail): x;
  lognormal exp(-t^2 / 2), t = ln(nu / nu_p) / w: the exponent carries t^2 eps, so t^2 + |t|.
A verified rule may differ from the table by up to 1e-14 (the library's acceptance threshold), which the default
form's bar adds.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import TOL, rel_err
from test_bandpass_seds import BOXES, H, KB, NU_REF, TYPES, expected_samples, ref_sed, synth_c3, tophat

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
CENTRES = sorted(set(np.round(np.geomspace(20.0, 1000.0, 16), 1)) | {30.0, 353.0, 545.0, 857.0})
FORMS = ("delta", "table", "quad")


def bands_for(shape):
    from dang_b200.config import Band
    out = []
    for c in CENTRES:
        if shape == "delta":
            out.append(Band(c))
            continue
        nu_c, nu, tau = {"hw0.25": lambda v: tophat(v, 0.25), "c3": synth_c3}[shape](c * 1e9)
        out.append(Band(nu_ghz=c, label=f"{c:g}", bp_nu_ghz=nu / 1e9, bp_tau=tau))
    return out


def band_table(b):
    """(nu_c, nu0, tau0) as the library receives them (init_bandpass)."""
    from dang_b200.engine import init_bandpass
    return init_bandpass(b)


def cond(kind, nu, th):
    """condition number of the reference's fp64 operation order at the band's samples (see the module docstring)."""
    nu = np.atleast_1d(np.asarray(nu, dtype=np.float64))[None, :]
    th = [np.atleast_1d(np.asarray(t, dtype=np.float64))[:, None] for t in th]
    if kind == "mbb":
        z = H / (KB * th[1])
        x = np.concatenate([z * nu, z * NU_REF[kind] + 0 * nu], axis=1)
        return np.max(1.0 / x + x, axis=1)
    if kind in ("cmb", "T_cmb", "hi_fit"):
        y = H * nu / (KB * th[0])
        return np.max(2.0 / y + y, axis=1)
    if kind == "lognormal":
        t = np.log(nu / (th[0] * 1e9)) / th[1]
        return np.max(t * t + np.abs(t), axis=1)
    return np.zeros(th[0].shape[0])


def probe(kind, shape, form, th, nside=16, t_cmb_values=(None,)):
    """Device SED of one component of `kind` per (band, pixel) for index maps th (one (npix,) array per index)."""
    from dang_b200.config import CGGroup, Component, IndexSpec, RunConfig
    from dang_b200.engine import OPT_BP_QUADRATURE, Engine
    from dang_b200.synth import Sky
    bands = bands_for("delta" if form == "delta" else shape)
    nb, npix = len(bands), 12 * nside * nside
    comp = Component("p", kind, NU_REF[kind] / 1e9, cg_group=1, amp_sample=False,
                     indices=[IndexSpec(f"i{l}", float(t[0])) for l, t in enumerate(th)],
                     corr=[True] * nb if kind == "hi_fit" else None)
    cfg = RunConfig("probe", nside, bands, [comp], [CGGroup()], tqu="TQU")
    ones = np.ones((3, npix))
    sky = Sky(sig=np.zeros((nb, 3, npix)), rms=np.ones((nb, 3, npix)), mask=np.ones(npix), gain=np.ones(nb),
              offset=np.zeros(nb), amplitude={"p": ones}, indices={"p": np.stack([np.tile(t, (3, 1)) for t in th])
                                                                   if th else np.zeros((0, 3, npix))}, truth={})
    if kind == "hi_fit":
        sky.template, sky.template_amplitudes = {"p": ones}, {"p": np.ones((3, nb))}
    eng = Engine(cfg, sky)
    eng.set_option(OPT_BP_QUADRATURE, 0 if form == "table" else 8)
    out, samples = [], []
    for t in t_cmb_values:
        if t is not None:
            eng.set_t_cmb(t)
        out.append(eng.update_sky_model()[0])
        if form == "quad":  # which bands a rule served, and with how many nodes
            samples.append(assert_band_samples(eng, cfg, sky, 2.7255 if t is None else t))
    return bands, out, samples


def check(kind, form, bands, sky_g, th, label):
    """worst err / bar over bands and pixels; asserts every plane equals plane 0 and err <= bar."""
    worst, worst_err = 0.0, 0.0
    for j, b in enumerate(bands):
        nu_c, nu, tau = band_table(b)
        assert np.array_equal(sky_g[j, 1], sky_g[j, 0]) and np.array_equal(sky_g[j, 2], sky_g[j, 0])
        ref = ref_sed(kind, nu_c, nu, tau, th)
        ok = np.abs(ref) > 1e-290  # below the double range the device's sums underflow, as the reference's do
        err = np.zeros(ref.shape)
        err[ok] = np.abs(sky_g[j, 0][ok] / ref[ok] - 1).astype(np.float64)
        samples = nu if len(nu) else np.array([nu_c])
        bar = 1e-14 + 8 * EPS * cond(kind, samples[samples > 0], th) + (1e-14 if form == "quad" else 0.0)
        i = int(np.argmax(err / bar))
        worst, worst_err = max(worst, err[i] / bar[i]), max(worst_err, float(err.max()))
        assert err[i] <= bar[i], (label, b.nu_ghz, [t[i] for t in th], err[i], bar[i])
    print(f"{label}: worst rel. error {worst_err:.1e}, worst error / bar {worst:.2f}")


def pixel_grid(kind, npix):
    """index value (pair) per pixel on a grid over the box, edges included"""
    box = BOXES[kind]
    if len(box) == 1:
        return [np.linspace(box[0][0], box[0][1], npix)]
    n = int(np.sqrt(npix))
    a, b = np.meshgrid(np.linspace(*box[0], n), np.linspace(*box[1], n), indexing="ij")
    a, b = a.ravel(), b.ravel()
    pad = npix - a.size
    return [np.concatenate([a, np.full(pad, box[0][1])]), np.concatenate([b, np.full(pad, box[1][1])])]


@pytest.mark.parametrize("shape,form", [("delta", "delta"), ("hw0.25", "table"), ("hw0.25", "quad"), ("c3", "table"),
                                        ("c3", "quad")])
@pytest.mark.parametrize("kind", [k for k in TYPES if k != "cmb"])
def test_sed_probe_per_pixel_indices(kind, shape, form):
    """sed_theta: a different index value (pair) at every pixel."""
    th = pixel_grid(kind, 12 * 16 * 16)
    bands, (sky_g,), samples = probe(kind, shape, form, th)
    if samples:
        print(f"{kind} {shape}: samples per band {samples[0]}")
    check(kind, form, bands, sky_g, th, f"{kind} {shape} {form} per-pixel")


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("kind", TYPES)
def test_sed_probe_constant_indices(kind, form):
    """sed_table_kernel / sed_uniform: every pixel holds one corner of the box ('cmb': T_CMB over its box, which also
    re-verifies the rules at every new T_CMB).  In the default form the bands at which 8 nodes miss the table by more
    than 1e-14 ('cmb' at 857 GHz: 12 nodes on the c3 shape, 16 on the top-hat) are served by larger rules, so the
    device's sums over 12 ... 32 nodes are compared with the reference too."""
    shapes = ("hw0.25", "c3") if form != "delta" else ("hw0.25",)
    escalated = 0
    for shape in shapes:
        if kind == "cmb":
            ts = (2.6, 2.7255, 2.8)
            bands, skies, samples = probe(kind, shape, form, [], nside=2, t_cmb_values=ts)
            for t, sky_g in zip(ts, skies):
                check(kind, form, bands, sky_g, [np.full(48, t)], f"cmb {shape} {form} T_CMB {t}")
            escalated += sum(8 < n <= 32 for ns in samples for n in ns)
            continue
        for corner in np.array(np.meshgrid(*BOXES[kind], indexing="ij")).reshape(len(BOXES[kind]), -1).T:
            th = [np.full(48, v) for v in corner]
            bands, (sky_g,), samples = probe(kind, shape, form, th, nside=2)
            check(kind, form, bands, sky_g, th, f"{kind} {shape} {form} {tuple(corner)}")
            escalated += sum(8 < n <= 32 for ns in samples for n in ns)
    if form == "quad" and kind in ("cmb", "lognormal", "T_cmb"):
        assert escalated > 0


def band_samples(eng):
    n = C.c_int()
    out = []
    for j in range(eng.nbands):
        eng._ck(eng.lib.dang_gpu_band_samples(eng.h, j, C.byref(n)))
        out.append(n.value)
    return out


def expected_band_samples(cfg, sky, t_cmb=2.7255):
    """What each band of a handle built from (cfg, sky) should be served by, restated from the verification policy
    (dang_gpu_band_samples): each index is checked on 7 points per dimension over the range of its uploaded maps,
    widened to the uniform prior when the index is sampled; 'cmb' at the current T_CMB.  None: more than 32 nodes."""
    points = []
    for c in cfg.comps:
        if c.type in ("template", "monopole"):
            continue
        boxes = [(t_cmb, t_cmb)] if c.type == "cmb" else []
        for l, s in enumerate(c.indices):
            m = sky.indices[c.label][l]
            lo, hi = float(m.min()), float(m.max())
            if s.sample:
                lo, hi = min(lo, s.uni[0]), max(hi, s.uni[1])
            boxes.append((lo, hi))
        axes = [np.linspace(lo, hi, 7) if hi > lo else np.array([lo]) for lo, hi in boxes]
        th = tuple(a.ravel() for a in np.meshgrid(*axes, indexing="ij"))
        points.append((c.type, th, c.nu_ref_ghz * 1e9 if c.nu_ref_ghz < 1e7 else c.nu_ref_ghz))
    out = []
    for b in cfg.bands:
        nu_c, nu, tau = band_table(b)
        out.append(0 if len(nu) == 0 else expected_samples(nu_c, nu, tau, points))
    return out


def assert_band_samples(eng, cfg, sky, t_cmb=2.7255):
    """the device's band forms are the ones the restated policy predicts (more than 32 nodes: a larger rule or the
    table, which this restatement does not distinguish)"""
    got, want = band_samples(eng), expected_band_samples(cfg, sky, t_cmb)
    for g, w in zip(got, want):
        assert g == w if w is not None else g > 32, (got, want)
    return got


def test_c3_bands_keep_the_eight_node_rule():
    """Every c3 band is served by an 8-node rule (the 16x saving of DESIGN 4.2 holds for the flagship config)."""
    from dang_b200.engine import OPT_BP_QUADRATURE, Engine
    from helpers import small_case
    cfg, sky = small_case("c3", 8)
    eng = Engine(cfg, sky)
    assert band_samples(eng) == [8] * 12
    eng.set_option(OPT_BP_QUADRATURE, 0)
    assert band_samples(eng) == [128] * 12


def test_rules_are_reverified_when_the_parameters_move():
    """A lognormal at nu_p = 30 GHz on a 30 GHz top-hat of half-width 0.25: w = 1 is served by 8 nodes; index maps
    with w = 0.1 leave the verified box and the band gets 16 nodes; the 857 GHz band ('cmb' needs 16 nodes there)
    needs more than 32 once w = 0.1 puts the lognormal 34 widths into its tail."""
    from dang_b200.config import Band, CGGroup, Component, IndexSpec, RunConfig
    from dang_b200.engine import Engine
    from dang_b200.synth import Sky
    nside, npix = 2, 48
    nu_c, nu, tau = tophat(30e9, 0.25)
    _, nu8, tau8 = tophat(857e9, 0.25)
    bands = [Band(30.0, "30", nu / 1e9, tau), Band(857.0, "857", nu8 / 1e9, tau8), Band(100.0)]
    comps = [Component("ame", "lognormal", 22.0, indices=[IndexSpec("NU_P", 30.0), IndexSpec("W", 1.0)]),
             Component("cmb", "cmb", 100.0)]
    cfg = RunConfig("rv", nside, bands, comps, [CGGroup()], tqu="TQU")
    idx = np.stack([np.full((3, npix), 30.0), np.full((3, npix), 1.0)])
    sky = Sky(sig=np.zeros((3, 3, npix)), rms=np.ones((3, 3, npix)), mask=np.ones(npix), gain=np.ones(3),
              offset=np.zeros(3), amplitude={"ame": np.ones((3, npix)), "cmb": np.ones((3, npix))},
              indices={"ame": idx, "cmb": np.zeros((0, 3, npix))}, truth={})
    eng = Engine(cfg, sky)
    assert band_samples(eng)[0] == 8 and band_samples(eng)[2] == 0
    n0 = assert_band_samples(eng, cfg, sky)
    idx[1] = 0.1
    eng.set_indices(0, idx)
    assert band_samples(eng)[0] == 16
    n1 = assert_band_samples(eng, cfg, sky)
    assert n1[1] >= n0[1] > 8, (n0, n1)
    sky_g = eng.update_sky_model()[0]
    ref = ref_sed("lognormal", nu_c, nu, tau, ([30.0], [0.1]))[0] + ref_sed("cmb", nu_c, nu, tau, ([2.7255],))[0]
    assert abs(sky_g[0, 0, 0] / ref - 1) <= 3e-14


# ------------------------------------------------------------------ downstream parity on bands that reach the gap
def gap_case(nside=8, seed=77):
    """c3's bands plus tabulated top-hats of half-width 0.25 at 30, 353, 545 and 857 GHz; synchrotron, dust,
    free-free (per-pixel T_e), a narrow lognormal at nu_p = 30 GHz (w = 0.1) and CMB, each bright enough that a
    1e-10 change of its SED in any band moves the chi-square.  The data are the oracle's sky model plus noise."""
    from dang_b200.config import Band, CGGroup, Component, IndexSpec
    from dang_b200.synth import make_config, make_sky
    from oracle.binding import Oracle
    cfg = make_config("c3", nside=nside)
    for c in (30.0, 353.0, 545.0, 857.0):
        _, nu, tau = tophat(c * 1e9, 0.25)
        cfg.bands.append(Band(nu_ghz=c, label=f"{c:g}w", bp_nu_ghz=nu / 1e9, bp_tau=tau))
    cfg.comps[1].indices[0].region = "fullsky"
    cfg.comps += [
        Component("ff", "freefree", 40.0, cg_group=2, indices=[
            IndexSpec("T_e", 7000.0, sample=True, region="per-pixel", prior="uniform", uni=(4000.0, 11000.0), step=300.0)]),
        Component("ame", "lognormal", 22.0, cg_group=2, indices=[IndexSpec("NU_P", 30.0), IndexSpec("W_AME", 0.1)]),
        Component("cmb", "cmb", 100.0, cg_group=2, indices=[]),
    ]
    cfg.cg_groups.append(CGGroup(sample=True, max_iter=100, converge=1e-12, poltype="Q+U"))
    sky = make_sky(cfg, seed=seed, noise_seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    scale = {"synch": 10.0, "dust": 50.0, "ff": 20.0, "ame": 40.0, "cmb": 3e4}
    for c in cfg.comps:
        sky.amplitude[c.label][1:3] = rng.normal(0.0, scale[c.label], size=(2, cfg.npix))
    sky.indices["ff"][0][:] = 7000.0 + 800.0 * rng.standard_normal(cfg.npix)[None, :]
    ora = Oracle(cfg, sky)
    ora.update_sky_model()
    sky.sig = ora.sky_model().copy() + sky.rms * rng.standard_normal(sky.rms.shape)
    for c in cfg.comps:   # start the chain 2 % away from the amplitudes that made the data
        sky.amplitude[c.label][1:3] *= 1.0 + 0.02 * rng.standard_normal((2, cfg.npix))
    return cfg, sky


def run_gap(cfg, sky, eng, ora):
    """chi-square, sky model, both CG groups, a per-pixel T_e draw and a full-sky dust-beta draw."""
    from dang_b200.engine import OPT_RECORD
    eng.set_option(OPT_RECORD, 1)
    out = {"planes": eng.chisq_planes()[0], "sky": eng.update_sky_model()[0]}
    rng = np.random.default_rng(5)
    for ig in (0, 1):
        eta = rng.standard_normal(2 * cfg.npix)
        out[f"it{ig}"] = eng.cg_solve(ig, 0, "sample", eta=eta)[0]
        if ora is not None:
            out[f"it{ig}_o"] = ora.cg_search_trace(ig=ig, ml_mode=1, eta=eta)[0]
    out["amp"] = [eng.amplitude(ic).copy() for ic in range(len(cfg.comps))]
    nsample = 8
    z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
    out["acc_pp"] = eng.sample_index_mh(2, 0, -1, nsample, "sample", z, u)
    out["dec_pp"], out["lnl_pp"] = eng.decisions(nsample, fullsky=False)
    if ora is not None:
        out["acc_pp_o"], out["dec_pp_o"], out["lnl_pp_o"] = ora.sample_index_mh(2, 0, -1, nsample, 1, z, u, want_trace=True)
    zf, uf = rng.standard_normal(16), rng.random(16)
    out["acc_fs"] = eng.sample_index_mh(1, 0, -1, 16, "sample", zf, uf)
    out["dec_fs"], out["lnl_fs"] = eng.decisions(16, fullsky=True)
    if ora is not None:
        out["acc_fs_o"], out["dec_fs_o"], out["lnl_fs_o"] = ora.sample_index_mh(1, 0, -1, 16, 1, zf, uf, want_trace=True)
    out["idx"] = [eng.indices(ic).copy() for ic in (1, 2)]
    return out


def test_gap_config_matches_the_oracle():
    """On bands where 8 nodes miss the table ('cmb' at 545 / 857 GHz and the narrow lognormal at 30 GHz, half-width
    0.25; here 13 bands get rules of 12 to 28 nodes and three keep more than 32 samples) the device still computes what
    the reference computes: chi-square, sky model band by band, the CG amplitudes
    of both groups, the decisions of a per-pixel T_e draw and of a full-sky draw.  The default form and the full table
    agree to 1e-12 with identical decisions."""
    from dang_b200.engine import OPT_BP_QUADRATURE, Engine
    from oracle.binding import Oracle
    cfg, sky = gap_case()
    ora = Oracle(cfg, sky)
    ora.update_sky_model()
    _, planes_o = ora.compute_chisq()
    sky_o = ora.sky_model().copy()
    res = {}
    for nq in (8, 0):
        eng = Engine(cfg, sky)
        eng.set_option(OPT_BP_QUADRATURE, nq)
        r = res[nq] = run_gap(cfg, sky, eng, ora if nq == 8 else None)
        if nq == 8:  # the draws stay in the verified box: the forms are still the ones verified at upload
            samples = assert_band_samples(eng, cfg, sky)
            print(f"samples per band {samples}")
            assert sum(8 < n <= 32 for n in samples) >= 10, samples
        else:
            assert band_samples(eng) == [128] * cfg.nbands
        assert rel_err(r["planes"], planes_o) < TOL, (nq, rel_err(r["planes"], planes_o))
        for j in range(cfg.nbands):
            assert rel_err(r["sky"][j], sky_o[j]) < TOL, (nq, cfg.bands[j].label, rel_err(r["sky"][j], sky_o[j]))
    r = res[8]
    assert r["it0"] == r["it0_o"] and r["it1"] == r["it1_o"]
    for ic in range(len(cfg.comps)):
        assert rel_err(r["amp"][ic], ora.amplitude(ic)) < TOL, (cfg.comps[ic].label, rel_err(r["amp"][ic], ora.amplitude(ic)))
    assert np.array_equal(r["dec_pp"], r["dec_pp_o"]) and r["acc_pp"] == r["acc_pp_o"]
    ev = r["dec_pp_o"] < 2
    assert rel_err(r["lnl_pp"][ev], r["lnl_pp_o"][ev]) < TOL
    assert np.array_equal(r["dec_fs"], r["dec_fs_o"]) and r["acc_fs"] == r["acc_fs_o"]
    ev = r["dec_fs_o"] < 2
    assert rel_err(r["lnl_fs"][ev], r["lnl_fs_o"][ev]) < TOL
    assert rel_err(r["idx"][0], ora.indices(1)) < 1e-14 and rel_err(r["idx"][1], ora.indices(2)) < 1e-14
    # the rule and the table
    a, b = res[8], res[0]
    assert rel_err(a["planes"], b["planes"]) < 1e-12 and rel_err(a["sky"], b["sky"]) < 1e-12
    assert a["it0"] == b["it0"] and a["it1"] == b["it1"]
    for ic in range(len(cfg.comps)):
        assert rel_err(a["amp"][ic], b["amp"][ic]) < 1e-12
    for k in ("dec_pp", "dec_fs"):
        assert np.array_equal(a[k], b[k])
