"""Posterior mean / standard-deviation maps and the Gelman-Rubin R-hat accumulated on the device
(dang_gpu_posterior_*, DESIGN.md section 9).  The update rule is defined operation by operation, so the device's
accumulators are compared bit for bit with a numpy restatement over the states the existing getters download."""
import numpy as np
import pytest

from conftest import ROOT
from helpers import intensity_case, small_case, template_case

POST_ALL = 1 | 2 | 4 | 8 | 16


def welford(samples):
    """The library's update rule, every operation a separately rounded IEEE float64 operation (numpy does not
    contract):  d = x - mean;  mean += d / n;  M2 += d * (x - mean);  std = sqrt(M2 / (n - 1)), NaN for n < 2."""
    mean = np.zeros_like(samples[0])
    m2 = np.zeros_like(samples[0])
    for i, x in enumerate(samples, 1):
        d = x - mean
        mean = mean + d / float(i)
        m2 = m2 + d * (x - mean)
    n = len(samples)
    with np.errstate(invalid="ignore", divide="ignore"):
        std = np.sqrt(m2 / float(n - 1)) if n > 1 else np.full_like(mean, np.nan)
    return mean, m2, std


def rhat_restated(means, m2s, n):
    """dang_gpu_posterior_rhat: sums over the chains in order, separately rounded; NaN where W = 0."""
    m = len(means)
    W = np.zeros_like(means[0])
    mu = np.zeros_like(means[0])
    for c in range(m):
        W = W + m2s[c] / float(n - 1)
        mu = mu + means[c]
    W = W / float(m)
    mu = mu / float(m)
    B = np.zeros_like(means[0])
    for c in range(m):
        d = means[c] - mu
        B = B + d * d
    B = B / float(m - 1)
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.sqrt(((float(n - 1) / float(n)) * W + B) / W)
    r[W == 0.0] = np.nan
    return r


def rhat_textbook(chains):
    """chains[c][i]: sample i of chain c.  R = sqrt(((n-1)/n W + B/n) / W) from np.var(ddof=1) / np.mean."""
    x = np.asarray(chains)
    n = x.shape[1]
    W = np.mean(np.var(x, axis=1, ddof=1), axis=0)
    Bn = np.var(np.mean(x, axis=1), axis=0, ddof=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.sqrt(((n - 1) / n * W + Bn) / W)


# ------------------------------------------------------------------ CPU: the restatements themselves
def test_restated_update_rule_matches_numpy_moments():
    """At 1e-13 relative wherever the variance is well conditioned (|mean| / std of a few): two samples that almost
    coincide lose digits in either formula, so n starts at 3."""
    rng = np.random.default_rng(3)
    for n in (3, 7, 50):
        x = rng.normal(1.0, 1.0, size=(n, 4, 100)) * np.exp(rng.normal(0.0, 3.0, size=(1, 4, 100)))
        mean, _, std = welford(list(x))
        np.testing.assert_allclose(mean, np.mean(x, axis=0), rtol=1e-13, atol=0)
        np.testing.assert_allclose(std, np.std(x, axis=0, ddof=1), rtol=1e-13, atol=0)
    mean, _, std = welford([np.arange(3.0)])
    assert np.array_equal(mean, np.arange(3.0)) and np.all(np.isnan(std))


def test_restated_rhat_matches_the_textbook_formula():
    rng = np.random.default_rng(4)
    for m, n in ((2, 2), (4, 7), (16, 30)):
        x = rng.normal(0.0, 1.0, size=(m, n, 200)) + rng.normal(0.0, 0.5, size=(m, 1, 200))
        means, m2s = zip(*[welford(list(x[c]))[:2] for c in range(m)])
        np.testing.assert_allclose(rhat_restated(means, m2s, n), rhat_textbook(x), rtol=1e-13, atol=0)
    x = np.ones((3, 5, 4))  # W = 0: NaN
    means, m2s = zip(*[welford(list(x[c]))[:2] for c in range(3)])
    assert np.all(np.isnan(rhat_restated(means, m2s, 5)))


# ------------------------------------------------------------------ GPU helpers
def _kinds_of(cfg):
    """(kind, ic, nind) of everything a POST_ALL accumulation holds for this configuration."""
    from dang_b200.engine import POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, POST_RESIDUAL, POST_TEMPLATE_AMPLITUDES
    out = [(POST_CHI_MAP, 0, 0), (POST_RESIDUAL, 0, 0)]
    for ic, c in enumerate(cfg.comps):
        if c.type in ("template", "monopole", "hi_fit"):
            out.append((POST_TEMPLATE_AMPLITUDES, ic, 0))
        elif c.type != "T_cmb":
            out.append((POST_AMPLITUDE, ic, 0))
        for j in range(len(c.indices)):
            out.append((POST_INDICES, ic, j))
    return out


def _state(eng, kinds):
    """Every accumulated quantity, downloaded with the existing getters."""
    from dang_b200.engine import POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, POST_RESIDUAL
    _, res, chi = eng.update_sky_model()
    out = {}
    for kind, ic, j in kinds:
        if kind == POST_AMPLITUDE:
            out[kind, ic, j] = eng.amplitude(ic)
        elif kind == POST_INDICES:
            out[kind, ic, j] = eng.indices(ic)[j]
        elif kind == POST_CHI_MAP:
            out[kind, ic, j] = chi
        elif kind == POST_RESIDUAL:
            out[kind, ic, j] = res
        else:
            out[kind, ic, j] = eng.template_amplitudes(ic)
    return out


def _chain(cfg, sky, n_it=7, seed=5, accumulate=True, record=True, options_from_3=(), async_downloads=False,
           pix_range=None, share=None):
    from dang_b200.engine import Engine
    eng = Engine(cfg, sky, pix_range=pix_range, share_maps_with=share)
    kinds = _kinds_of(cfg)
    if accumulate:
        eng.posterior_begin(POST_ALL)
    states, prev = [], None
    # host buffers of the asynchronous downloads: they must outlive the copies
    amp_bufs = {ic: np.zeros((cfg.nmaps, cfg.npix)) for ic, c in enumerate(cfg.comps)
                if c.type not in ("template", "monopole", "hi_fit", "T_cmb")}
    idx_bufs = {ic: np.zeros((len(c.indices), cfg.nmaps, cfg.npix)) for ic, c in enumerate(cfg.comps) if c.indices}
    for it in range(1, n_it + 1):
        if it == 3:
            for opt, val in options_from_3:
                eng.set_option(opt, val)
        eng.gibbs_iteration(it, seed=seed)
        deferred = dict(options_from_3).get(18, 0)
        ticket = eng.iteration_mark() if deferred and it >= 3 else None
        if accumulate:
            eng.posterior_accumulate()
        if async_downloads:   # interleaved with the accumulations, read back one iteration late
            for ic, b in amp_bufs.items():
                eng.amplitude_async(ic, b, 1, cfg.nmaps)
            for ic, b in idx_bufs.items():
                for j in range(b.shape[0]):
                    eng.indices_async(ic, j, b, 1, cfg.nmaps)
            if prev is not None:
                eng.iteration_scalars(prev)
            prev = ticket
        if record:
            states.append(_state(eng, kinds))
    if prev is not None:
        eng.iteration_scalars(prev)
    eng.download_wait()
    if async_downloads:   # the last requests hold the final state
        for ic, b in amp_bufs.items():
            assert np.array_equal(b, eng.amplitude(ic)), ic
        for ic, b in idx_bufs.items():
            assert np.array_equal(b, eng.indices(ic)), ic
    return eng, states, kinds


def _check_against_restatement(eng, states, kinds, sl=slice(None)):
    for key in kinds:
        mean, std, n = eng.posterior(*key)
        assert n == len(states)
        want_mean, _, want_std = welford([s[key][..., sl] for s in states])
        np.testing.assert_array_equal(mean[..., sl], want_mean, err_msg=str(key))
        np.testing.assert_array_equal(std[..., sl], want_std, err_msg=str(key))


# ------------------------------------------------------------------ 1. bit-identity with the restatement
@pytest.mark.gpu
@pytest.mark.parametrize("name,nside", [("c1", 8), ("c2", 16)])
def test_accumulators_equal_the_restated_update(name, nside):
    """c1 draws beta_s per pixel, c2 beta_d full sky; 7 Gibbs iterations with device deviates, every kind."""
    cfg, sky = small_case(name, nside, perturb=False)
    eng, states, kinds = _chain(cfg, sky)
    _check_against_restatement(eng, states, kinds)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["c3", "template", "intensity_hi"])
def test_accumulators_equal_the_restated_update_other_components(case):
    """Tabulated bands (c3); a template component's amplitudes; monopole and hi_fit (Stokes I)."""
    if case == "c3":
        cfg, sky = small_case("c3", 8, perturb=False)
    elif case == "template":
        cfg, sky, _ = template_case()
    else:
        cfg, sky, _, _ = intensity_case(with_hi=True)
    eng, states, kinds = _chain(cfg, sky, n_it=5)
    assert any(k[0] == 16 for k in kinds) == (case != "c3")
    _check_against_restatement(eng, states, kinds)


# ------------------------------------------------------------------ 2. no behaviour change
@pytest.mark.gpu
@pytest.mark.parametrize("name,nside", [("c1", 8), ("c2", 16)])
def test_accumulating_leaves_the_chain_unchanged(name, nside):
    cfg, sky = small_case(name, nside, perturb=False)
    a, _, _ = _chain(cfg, sky, n_it=6, accumulate=True, record=False)
    b, _, _ = _chain(cfg, sky, n_it=6, accumulate=False, record=False)
    for ic in range(len(cfg.comps)):
        assert np.array_equal(a.amplitude(ic), b.amplitude(ic)), ic
        assert np.array_equal(a.indices(ic), b.indices(ic)), ic
    assert np.array_equal(a.cg_trace(), b.cg_trace())
    if name == "c2":   # the full-sky chain's decisions (per-pixel ones are recorded only in record mode; c1's index
        # maps above hold every per-pixel outcome)
        da, la = a.decisions(cfg.nsample, True)
        db, lb = b.decisions(cfg.nsample, True)
        assert np.array_equal(da, db) and np.array_equal(la, lb, equal_nan=True)
    assert a.compute_chisq() == b.compute_chisq()


# ------------------------------------------------------------------ 3. ordering against deferred work
@pytest.mark.gpu
def test_accumulators_are_ordered_with_deferred_scalars_and_downloads():
    """DEFER_SCALARS and DEFER_D2H on from iteration 3 (as bench.py runs c2), asynchronous amplitude and index
    downloads requested between the accumulations: the accumulators equal the synchronous chain's, bit for bit."""
    from dang_b200.engine import OPT_DEFER_D2H, OPT_DEFER_SCALARS
    cfg, sky = small_case("c2", 16, perturb=False)
    ref, states, kinds = _chain(cfg, sky)
    eng, _, _ = _chain(cfg, sky, record=False, async_downloads=True,
                       options_from_3=((OPT_DEFER_SCALARS, 1), (OPT_DEFER_D2H, 1)))
    for key in kinds:
        m0, s0, n0 = ref.posterior(*key)
        m1, s1, n1 = eng.posterior(*key)
        assert n0 == n1 == 7
        np.testing.assert_array_equal(m1, m0, err_msg=str(key))
        np.testing.assert_array_equal(s1, s0, err_msg=str(key))


# ------------------------------------------------------------------ 4. a pixel slice
@pytest.mark.gpu
def test_odd_pixel_range_writes_only_its_pixels():
    cfg, sky = small_case("c1", 8, perturb=False)
    lo, hi = 37, cfg.npix - 101
    eng, states, kinds = _chain(cfg, sky, n_it=4, pix_range=(lo, hi))
    _check_against_restatement(eng, states, kinds, sl=slice(lo, hi))
    for key in kinds:
        if key[0] == 16:
            continue
        mean, std, _ = eng.posterior(*key)
        assert not mean[..., :lo].any() and not mean[..., hi:].any(), key
        assert not std[..., :lo].any() and not std[..., hi:].any(), key


# ------------------------------------------------------------------ 5. R-hat
@pytest.mark.gpu
def test_rhat_of_chains_sharing_maps():
    """Four c2 chains on one set of maps (dang_gpu_share_maps), different seeds: R-hat equals the restatement bit for
    bit, and the textbook formula to 1e-13 relative times the element's condition number max|x| / sqrt(W) (at least
    1).  Both fp64 variances lose digits in proportion to it: amplitudes that move little against their size
    (condition ~10^3) differ by up to 5e-13 on a B200 run."""
    from dang_b200.engine import posterior_rhat
    cfg, sky = small_case("c2", 16, perturb=False)
    owner = None
    engs, runs = [], []
    for c in range(4):
        eng, states, kinds = _chain(cfg, sky, n_it=6, seed=100 + 17 * c, share=owner)
        owner = owner or eng
        engs.append(eng)
        runs.append(states)
    n = len(runs[0])
    for key in kinds:
        r = posterior_rhat(engs, *key)
        samples = [[s[key] for s in run] for run in runs]
        means, m2s = zip(*[welford(x)[:2] for x in samples])
        want = rhat_restated(means, m2s, n)
        np.testing.assert_array_equal(r, want, err_msg=str(key))
        tb = rhat_textbook(samples)
        ok = np.isfinite(want)
        x = np.asarray(samples)
        with np.errstate(invalid="ignore", divide="ignore"):
            cond = np.max(np.abs(x), axis=(0, 1)) / np.sqrt(np.mean(np.var(x, axis=1, ddof=1), axis=0))
        bar = 1e-13 * np.maximum(1.0, cond[ok]) * np.abs(tb[ok])
        assert np.all(np.abs(r[ok] - tb[ok]) <= bar), (key, np.max(np.abs(r[ok] - tb[ok]) / bar))
    # masked pixels of the chi-square map have W = 0
    assert np.all(np.isnan(posterior_rhat(engs, 4)[:, sky.mask == 0]))


RHAT_NSIDE, RHAT_DRAWS = 64, 20


def _stationary_chains(shift):
    """m = 4 chains on the stationarity set-up of test_gpu_device_rng (every pixel has the same exact posterior of
    beta_s, Q and U drawn together), each started at independent exact draws.  `shift`: the last chain's data are
    multiplied by (nu / nu_ref)^shift, which moves its posterior by `shift` in beta (about 3 posterior widths)."""
    from dang_b200.engine import POST_INDICES, Engine, posterior_rhat
    from test_gpu_device_rng import _cdf, _flat_sky
    cfg, sky, ic, nind, loglike, logprior, spec = _flat_sky("powerlaw", 2, False, RHAT_NSIDE)
    grid = np.linspace(spec.uni[0], spec.uni[1], 2 ** 18 + 1)
    cdf = _cdf(grid, loglike(grid) + logprior(grid, spec.gauss[0]))
    engs = []
    for c in range(4):
        s = sky
        if shift and c == 3:
            import copy
            s = copy.deepcopy(sky)
            nu_ref = cfg.comps[ic].nu_ref_ghz
            for j, b in enumerate(cfg.bands):
                s.sig[j] = s.sig[j] * (b.nu_ghz / nu_ref) ** shift
        eng = Engine(cfg, s)
        idx = s.indices[cfg.comps[ic].label].copy()
        start = np.interp(np.random.default_rng(500 + c).random(cfg.npix), cdf, grid)
        idx[nind, 1] = idx[nind, 2] = start
        eng.set_indices(ic, idx)
        eng.posterior_begin(POST_INDICES)
        engs.append(eng)
    for i in range(RHAT_DRAWS):
        for c, eng in enumerate(engs):
            eng.sample_index_mh(ic, nind, -1, 50, "sample", seed=9000 + 131 * c + i)
            eng.posterior_accumulate()
    return posterior_rhat(engs, POST_INDICES, ic, nind)[1]


@pytest.mark.gpu
def test_rhat_is_near_one_for_chains_of_one_posterior_and_large_when_one_differs():
    """Per-pixel R-hat over the 49152 pixels.  Recorded on a B200 (nside 64, 4 chains x 20 draws of 50 proposals,
    fixed seeds): one posterior, median 0.9997 and 99.9th percentile 1.157; one chain's posterior moved by ~3 widths,
    0.1th percentile 1.226 and median 1.580.  Thresholds: the first set stays within 0.01 of 1 at the median and
    below 1.2 at the 99.9th percentile; the second stays above 1.2 at the 0.1th percentile and above 1.4 at the
    median -- 1.2 separates every pixel of one from every pixel of the other but the extreme 0.1 %."""
    same = _stationary_chains(0.0)
    moved = _stationary_chains(0.3)
    q_same = np.quantile(same, [0.5, 0.999])
    q_moved = np.quantile(moved, [0.001, 0.5])
    print(f"R-hat same posterior: median {q_same[0]:.4f}, 99.9% {q_same[1]:.4f}; "
          f"moved: 0.1% {q_moved[0]:.4f}, median {q_moved[1]:.4f}")
    assert np.all(np.isfinite(same)) and np.all(np.isfinite(moved))
    assert abs(q_same[0] - 1.0) < 0.01 and q_same[1] < 1.2
    assert q_moved[0] > 1.2 and q_moved[1] > 1.4


# ------------------------------------------------------------------ 6. errors and restarts
@pytest.mark.gpu
def test_errors_nan_stddev_and_restart():
    from dang_b200.engine import (POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, POST_TEMPLATE_AMPLITUDES, Engine,
                                  posterior_rhat, DangGpuError)
    EINVAL, ESTATE = 1, 5
    cfg, sky, _ = template_case()
    eng = Engine(cfg, sky)
    lib, h = eng.lib, eng.h
    mean, std, n = np.zeros((3, cfg.npix)), np.zeros((3, cfg.npix)), np.zeros(1, dtype=np.int64)
    from dang_b200._lib import c_dp, c_i64p

    def get(kind, ic=0, nind=0):
        return lib.dang_gpu_posterior_get(h, kind, ic, nind, mean.ctypes.data_as(c_dp), std.ctypes.data_as(c_dp),
                                          n.ctypes.data_as(c_i64p))
    assert lib.dang_gpu_posterior_accumulate(h) == ESTATE
    assert get(POST_AMPLITUDE) == ESTATE
    assert lib.dang_gpu_posterior_end(h) == ESTATE
    for what in (0, 32, -1):
        assert lib.dang_gpu_posterior_begin(h, what, 2, 3) == EINVAL
    assert lib.dang_gpu_posterior_begin(h, POST_CHI_MAP, 3, 2) == EINVAL
    assert lib.dang_gpu_posterior_begin(h, POST_CHI_MAP, 0, 3) == EINVAL
    eng.posterior_begin(POST_AMPLITUDE | POST_INDICES)
    assert get(POST_CHI_MAP) == ESTATE and get(POST_TEMPLATE_AMPLITUDES, 1) == ESTATE
    for kind in (0, 3, 32):
        assert get(kind) == EINVAL
    assert get(POST_AMPLITUDE, 2) == EINVAL and get(POST_AMPLITUDE, -1) == EINVAL
    assert get(POST_AMPLITUDE, 1) == EINVAL          # the template component has no map amplitude
    assert get(POST_INDICES, 0, 1) == EINVAL and get(POST_INDICES, 1, 0) == EINVAL
    eng.gibbs_iteration(1, seed=3)
    eng.posterior_accumulate()
    m, s, k = eng.posterior(POST_AMPLITUDE, 0)
    assert k == 1 and np.array_equal(m, eng.amplitude(0)) and np.all(np.isnan(s))
    with pytest.raises(DangGpuError):   # n < 2
        posterior_rhat([eng, eng], POST_AMPLITUDE, 0)
    eng.gibbs_iteration(2, seed=3)
    eng.posterior_accumulate()
    assert eng.posterior(POST_AMPLITUDE, 0)[2] == 2
    other = Engine(cfg, sky)
    other.posterior_begin(POST_INDICES)
    for _ in range(2):
        other.posterior_accumulate()
    with pytest.raises(DangGpuError):   # kind not begun on one handle
        posterior_rhat([eng, other], POST_AMPLITUDE, 0)
    other.posterior_begin(POST_AMPLITUDE)
    other.posterior_accumulate()
    with pytest.raises(DangGpuError):   # different n
        posterior_rhat([eng, other], POST_AMPLITUDE, 0)
    with pytest.raises(DangGpuError):   # one chain
        posterior_rhat([eng], POST_AMPLITUDE, 0)
    # _begin again starts from zero
    eng.posterior_begin(POST_AMPLITUDE)
    eng.gibbs_iteration(3, seed=3)
    eng.posterior_accumulate()
    m, s, k = eng.posterior(POST_AMPLITUDE, 0)
    assert k == 1 and np.array_equal(m, eng.amplitude(0)) and np.all(np.isnan(s))
    eng.posterior_end()
    assert lib.dang_gpu_posterior_end(h) == ESTATE


# ------------------------------------------------------------------ 8. two GPUs
@pytest.mark.gpu
def test_two_gpus_accumulate_their_own_pixels():
    """tests/multi_gpu_posterior_check.py on two ring-partitioned ranks, over the NVLink mailboxes and over NCCL:
    nothing crosses ranks; each rank's accumulators are the restatement over its own slice."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, DANG_MGC_NSIDE="16")
    for mailbox in ("1", "0"):
        env["DANG_GPU_MAILBOX"] = mailbox
        p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                            "--master-addr", "127.0.0.1", "--master-port", "29547",
                            os.path.join(ROOT, "tests", "multi_gpu_posterior_check.py")],
                           env=env, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        assert p.stdout.count("multi-GPU posterior ok") == 2
