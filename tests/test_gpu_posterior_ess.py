"""Batch-means effective sample size and Monte Carlo standard error of the posterior mean, accumulated on the device
(dang_gpu_posterior_begin_batched / dang_gpu_posterior_ess, DESIGN.md section 9).  The batch rule and the read-out
are defined operation by operation, so the device is compared bit for bit with a numpy restatement over the states
the existing getters download; the restatement is checked against the textbook estimator and, for AR(1) chains,
against the estimator's closed-form expectation."""
import numpy as np
import pytest

from helpers import intensity_case, small_case, template_case
from test_gpu_posterior import _chain, _kinds_of, welford

EINVAL, ESTATE = 1, 5


def batch_moments(samples, b):
    """The batch rule, every operation a separately rounded float64 operation: sample i (1-based) at position
    j = ((i-1) mod b) + 1 of its batch: bsum = x if j == 1 else bsum + x; when j == b, k = i / b and y = bsum / b
    go through Welford's update into (bmean, bM2).  Returns (mean, M2, bmean, bM2)."""
    mean, m2, _ = welford(samples)
    bsum = np.zeros_like(samples[0])
    bmean = np.zeros_like(samples[0])
    bm2 = np.zeros_like(samples[0])
    for i, x in enumerate(samples, 1):
        j = (i - 1) % b + 1
        bsum = x.copy() if j == 1 else bsum + x
        if j == b:
            y = bsum / float(b)
            d = y - bmean
            bmean = bmean + d / float(i // b)
            bm2 = bm2 + d * (y - bmean)
    return mean, m2, bmean, bm2


def ess_restated(moments, n, b):
    """dang_gpu_posterior_ess over the chains' (mean, M2, bmean, bM2), summed in order, separately rounded:
    s2 = (A + n D) / (m n - 1), sig2 = b (Ab + K Db) / (m K - 1), ess = (m n) s2 / sig2, mcse = sqrt(sig2 / (m n)),
    NaN where sig2 = 0."""
    m, K = len(moments), n // b
    mu, A, mub, Ab = (np.zeros_like(moments[0][0]) for _ in range(4))
    for mean, m2, bmean, bm2 in moments:
        mu, A, mub, Ab = mu + mean, A + m2, mub + bmean, Ab + bm2
    mu, mub = mu / float(m), mub / float(m)
    D, Db = np.zeros_like(mu), np.zeros_like(mu)
    for mean, _, bmean, _ in moments:
        d, db = mean - mu, bmean - mub
        D, Db = D + d * d, Db + db * db
    s2 = (A + float(n) * D) / float(m * n - 1)
    sig2 = (float(b) * (Ab + float(K) * Db)) / float(m * K - 1)
    with np.errstate(invalid="ignore", divide="ignore"):
        ess = (float(m * n) * s2) / sig2
        mcse = np.sqrt(sig2 / float(m * n))
    ess[sig2 == 0.0] = np.nan
    mcse[sig2 == 0.0] = np.nan
    return ess, mcse


def ess_textbook(x, b):
    """x[c][i]: sample i of chain c.  s2: the variance (ddof=1) of all m n samples; sig2: b times the variance
    (ddof=1) of all m K means of the first K b samples of each chain, taken in rows of b."""
    x = np.asarray(x)
    m, n, K = x.shape[0], x.shape[1], x.shape[1] // b
    s2 = np.var(x.reshape((m * n,) + x.shape[2:]), axis=0, ddof=1)
    y = x[:, :K * b].reshape((m, K, b) + x.shape[2:]).mean(axis=2)
    sig2 = b * np.var(y.reshape((m * K,) + x.shape[2:]), axis=0, ddof=1)
    return m * n * s2 / sig2, np.sqrt(sig2 / (m * n))


def ar1(rng, rho, n, shape):
    """n steps of x_t = rho x_{t-1} + sqrt(1 - rho^2) e_t started in stationarity (unit variance)."""
    x = rng.standard_normal(shape)
    out = np.empty((n,) + shape)
    c = np.sqrt(1.0 - rho * rho)
    for t in range(n):
        out[t] = x
        x = rho * x + c * rng.standard_normal(shape)
    return out


def var_of_mean(rho, L):
    """v_L = (L + 2 sum_{k<L} (L - k) rho^k) / L^2: the variance of the mean of L consecutive AR(1) samples."""
    k = np.arange(1, L)
    return (L + 2.0 * np.sum((L - k) * rho ** k)) / (L * L)


def expected_sig2(rho, b, K):
    """E[sig2] of one chain of K b samples: b K / (K - 1) (v_b - v_{Kb})."""
    return b * K / (K - 1) * (var_of_mean(rho, b) - var_of_mean(rho, K * b))


# ------------------------------------------------------------------ CPU: the restatement itself
@pytest.mark.parametrize("m", [1, 4])
@pytest.mark.parametrize("n,b", [(60, 6), (67, 6), (50, 1), (9, 4)])
def test_restated_batch_means_match_the_textbook_estimator(m, n, b):
    """n a multiple of b and not (the partial batch is left out of sig2 but not s2), one chain and four."""
    rng = np.random.default_rng(10 * m + n + b)
    x = rng.normal(0.0, 1.0, size=(m, n, 300)) + rng.normal(0.0, 0.3, size=(m, 1, 300)) + 2.0
    moments = [batch_moments(list(x[c]), b) for c in range(m)]
    ess, mcse = ess_restated(moments, n, b)
    ess_t, mcse_t = ess_textbook(x, b)
    np.testing.assert_allclose(ess, ess_t, rtol=1e-13, atol=0)
    np.testing.assert_allclose(mcse, mcse_t, rtol=1e-13, atol=0)
    if b == 1:   # batches of one sample: the batch moments are the moments
        for mean, m2, bmean, bm2 in moments:
            assert np.array_equal(mean, bmean) and np.array_equal(m2, bm2)


@pytest.mark.parametrize("rho", [0.0, 0.5, 0.9])
def test_restated_estimator_has_the_ar1_closed_form_expectation(rho):
    """Averaged over 20000 seeded chains of K b = 40 x 25 samples, n sig2 = n MCSE^2 of one chain matches
    b K / (K - 1) (v_b - v_{Kb}) within 5 standard errors of the average (from the chains' spread)."""
    b, K, chains = 25, 40, 20000
    x = ar1(np.random.default_rng(int(rho * 10) + 77), rho, K * b, (chains,))
    moments = batch_moments(list(x), b)
    _, mcse = ess_restated([moments], K * b, b)
    sig2 = mcse * mcse * (K * b)
    want = expected_sig2(rho, b, K)
    se = np.std(sig2) / np.sqrt(chains)
    assert abs(np.mean(sig2) - want) < 5 * se, (rho, np.mean(sig2), want, se)


# ------------------------------------------------------------------ GPU helpers
def _begin_batched(monkeypatch, b):
    """Make test_gpu_posterior's chain driver begin every handle with batch length b (0: without batches)."""
    from dang_b200.engine import Engine
    begin = getattr(Engine.posterior_begin, "unbatched", Engine.posterior_begin)

    def batched(self, what, *args, **kw):
        return begin(self, what, *args, batch_len=b, **kw)
    batched.unbatched = begin
    monkeypatch.setattr(Engine, "posterior_begin", batched)


def _case(case):
    if case in ("c1", "c2"):
        return small_case(case, 8 if case == "c1" else 16, perturb=False)
    if case == "c3":
        return small_case("c3", 8, perturb=False)
    if case == "template":
        return template_case()[:2]
    return intensity_case(with_hi=True)[:2]


def _ensemble(cfg, sky, m, n_it, **kw):
    """m chains on one set of maps (dang_gpu_share_maps), different seeds, each with its recorded states."""
    owner, engs, runs = None, [], []
    for c in range(m):
        eng, states, kinds = _chain(cfg, sky, n_it=n_it, seed=100 + 17 * c, share=owner, **kw)
        owner = owner or eng
        engs.append(eng)
        runs.append(states)
    return engs, runs, kinds


def _check_ess(engs, runs, kinds, b, sl=slice(None)):
    from dang_b200.engine import posterior_ess
    n = len(runs[0])
    for key in kinds:
        moments = [batch_moments([s[key][..., sl] for s in run], b) for run in runs]
        for chains in (slice(0, 1), slice(None)):
            ess, mcse = posterior_ess(engs[chains], *key)
            want_ess, want_mcse = ess_restated(moments[chains], n, b)
            np.testing.assert_array_equal(ess[..., sl], want_ess, err_msg=str((key, len(engs[chains]))))
            np.testing.assert_array_equal(mcse[..., sl], want_mcse, err_msg=str((key, len(engs[chains]))))


# ------------------------------------------------------------------ 3. bit-identity with the restatement
@pytest.mark.gpu
@pytest.mark.parametrize("b,n", [(1, 5), (3, 7), (4, 8)])
@pytest.mark.parametrize("case", ["c1", "c2", "c3", "template", "intensity_hi"])
def test_ess_and_mcse_equal_the_restatement(monkeypatch, case, b, n):
    """Every kind, of one chain and pooled over four sharing one set of maps: b = 1, a partial last batch (b = 3,
    n = 7) and two batches (b = n / 2).  c1 per-pixel beta_s, c2 full-sky beta_d, c3 tabulated bands, template
    amplitudes, monopole and hi_fit."""
    cfg, sky = _case(case)
    _begin_batched(monkeypatch, b)
    engs, runs, kinds = _ensemble(cfg, sky, 4, n)
    _check_ess(engs, runs, kinds, b)


# ------------------------------------------------------------------ 4. existing behaviour unchanged
@pytest.mark.gpu
@pytest.mark.parametrize("name,nside", [("c1", 8), ("c2", 16)])
def test_batched_accumulation_changes_neither_the_moments_nor_the_chain(monkeypatch, name, nside):
    """A batched handle's mean / std equal an unbatched handle's bit for bit, and a chain that accumulates batched
    ends where a chain that does not accumulate ends."""
    cfg, sky = small_case(name, nside, perturb=False)
    _begin_batched(monkeypatch, 3)
    a, _, kinds = _chain(cfg, sky, n_it=7, record=False)
    _begin_batched(monkeypatch, 0)
    u, _, _ = _chain(cfg, sky, n_it=7, record=False)
    z, _, _ = _chain(cfg, sky, n_it=7, accumulate=False, record=False)
    for key in kinds:
        ma, sa, na = a.posterior(*key)
        mu, su, nu = u.posterior(*key)
        assert na == nu == 7
        np.testing.assert_array_equal(ma, mu, err_msg=str(key))
        np.testing.assert_array_equal(sa, su, err_msg=str(key))
    for ic in range(len(cfg.comps)):
        assert np.array_equal(a.amplitude(ic), z.amplitude(ic)), ic
        assert np.array_equal(a.indices(ic), z.indices(ic)), ic
    assert np.array_equal(a.cg_trace(), z.cg_trace())
    if name == "c2":
        da, la = a.decisions(cfg.nsample, True)
        dz, lz = z.decisions(cfg.nsample, True)
        assert np.array_equal(da, dz) and np.array_equal(la, lz, equal_nan=True)
    assert a.compute_chisq() == z.compute_chisq()


@pytest.mark.gpu
def test_batched_accumulators_are_ordered_with_deferred_scalars_and_downloads(monkeypatch):
    """DEFER_SCALARS and DEFER_D2H from iteration 3, asynchronous downloads between the accumulations: the ESS and
    MCSE equal the restatement over the synchronous chain's states, and the moments equal that chain's."""
    from dang_b200.engine import OPT_DEFER_D2H, OPT_DEFER_SCALARS
    cfg, sky = small_case("c2", 16, perturb=False)
    _begin_batched(monkeypatch, 3)
    ref, states, kinds = _chain(cfg, sky)
    eng, _, _ = _chain(cfg, sky, record=False, async_downloads=True,
                       options_from_3=((OPT_DEFER_SCALARS, 1), (OPT_DEFER_D2H, 1)))
    _check_ess([eng], [states], kinds, 3)
    for key in kinds:
        m0, s0, _ = ref.posterior(*key)
        m1, s1, _ = eng.posterior(*key)
        np.testing.assert_array_equal(m1, m0, err_msg=str(key))
        np.testing.assert_array_equal(s1, s0, err_msg=str(key))


@pytest.mark.gpu
def test_batched_odd_pixel_range_writes_only_its_pixels(monkeypatch):
    from dang_b200.engine import posterior_ess
    cfg, sky = small_case("c1", 8, perturb=False)
    lo, hi = 37, cfg.npix - 101
    _begin_batched(monkeypatch, 2)
    eng, states, kinds = _chain(cfg, sky, n_it=5, pix_range=(lo, hi))
    _check_ess([eng], [states], kinds, 2, sl=slice(lo, hi))
    for key in kinds:
        if key[0] == 16:
            continue
        ess, mcse = posterior_ess([eng], *key)
        assert not ess[..., :lo].any() and not ess[..., hi:].any(), key
        assert not mcse[..., :lo].any() and not mcse[..., hi:].any(), key


# ------------------------------------------------------------------ 5. b = 1
@pytest.mark.gpu
def test_batches_of_one_sample_give_ess_n_and_mcse_std_over_sqrt_n(monkeypatch):
    """With b = 1 every sample closes its batch: y = x / 1 and k = n, so {bmean, bM2} follow {mean, M2} exactly and
    sig2 = s2.  ESS = n and MCSE = std / sqrt(n) to 4 ulp wherever std > 0; NaN where it is 0 (masked chi-square
    pixels)."""
    from dang_b200.engine import posterior_ess
    cfg, sky = small_case("c2", 16, perturb=False)
    _begin_batched(monkeypatch, 1)
    n = 6
    engs, runs, kinds = _ensemble(cfg, sky, 4, n)
    _check_ess(engs, runs, kinds, 1)
    for key in kinds:
        _, std, k = engs[0].posterior(*key)
        assert k == n
        ess, mcse = posterior_ess(engs[:1], *key)
        ok = std > 0
        assert np.all(np.isnan(ess[~ok])) and np.all(np.isnan(mcse[~ok])), key
        assert np.all(np.abs(ess[ok] - n) <= 4 * np.spacing(float(n))), key
        want = std[ok] / np.sqrt(n)
        assert np.all(np.abs(mcse[ok] - want) <= 4 * np.spacing(want)), key


# ------------------------------------------------------------------ 6. statistical meaning
STAT_NSIDE, STAT_N, STAT_B = 32, 4000, 100
STAT_RHO = (0.0, 0.5, 0.9)      # planes I, Q, U
AMP_OFFSET = (10.0, -5.0, 3.0)  # distinct offsets per plane; the estimators do not see them
IDX_SCALE = 0.01                # index maps move by 0.01 x around their start


@pytest.mark.gpu
def test_ess_and_mcse_of_ar1_chains():
    """Per-plane AR(1) series fed through set_amplitude / set_indices on four handles at nside 32 (n = 4000,
    b = 100, K = 40), each pixel its own chain:
    - one chain's n MCSE^2, averaged over the pixels, matches b K / (K - 1) (v_b - v_{Kb}) within 5 standard errors
      of that average, for rho = 0, 0.5, 0.9 on I, Q, U of the amplitude and of the index map;
    - four i.i.d. chains (rho = 0): m n / ESS averages to 1 within 5 standard errors (for Gaussian i.i.d. samples
      sig2 / s2 has mean exactly 1);
    - the index map's I plane of the fourth chain is offset by one standard deviation: the pooled ESS falls more
      than 10x below the aligned case (about 16x from the formula at these sizes)."""
    from dang_b200.engine import POST_AMPLITUDE, POST_INDICES, Engine, posterior_ess
    cfg, sky = small_case("c2", STAT_NSIDE, perturb=False)
    m, P = 4, cfg.npix
    owner, engs, start = None, [], None
    for c in range(m):
        eng = Engine(cfg, sky, share_maps_with=owner)
        owner = owner or eng
        start = eng.indices(0) if start is None else start
        eng.posterior_begin(POST_AMPLITUDE | POST_INDICES, batch_len=STAT_B)
        engs.append(eng)
    rng = np.random.default_rng(2026)
    rho = np.asarray(STAT_RHO)[:, None]
    # unit-variance AR(1) per plane and pixel, started in stationarity: [chain][amp, idx][plane][pixel]
    x = rng.standard_normal((m, 2, 3, P))
    offs = np.asarray(AMP_OFFSET)[:, None]
    for _ in range(STAT_N):
        for c, eng in enumerate(engs):
            eng.set_amplitude(0, offs + x[c, 0])
            idx = start.copy()
            idx[0] = start[0] + IDX_SCALE * x[c, 1]
            if c == m - 1:
                idx[0, 0] += IDX_SCALE   # one standard deviation
            eng.set_indices(0, idx)
            eng.posterior_accumulate()
        x = rho * x + np.sqrt(1.0 - rho * rho) * rng.standard_normal(x.shape)
    K = STAT_N // STAT_B
    report = []
    for kind, scale in ((POST_AMPLITUDE, 1.0), (POST_INDICES, IDX_SCALE)):
        _, mcse = posterior_ess(engs[:1], kind, 0, 0)
        for k, rho in enumerate(STAT_RHO):
            v = mcse[k] ** 2 * STAT_N / scale ** 2
            want, se = expected_sig2(rho, STAT_B, K), np.std(v) / np.sqrt(P)
            report.append(f"kind {kind} rho {rho}: {np.mean(v):.4f} vs {want:.4f} (se {se:.4f})")
            assert abs(np.mean(v) - want) < 5 * se, report[-1]
    ess_aligned, _ = posterior_ess(engs, POST_AMPLITUDE, 0, 0)
    r = m * STAT_N / ess_aligned[0]
    report.append(f"m n / ESS, aligned: {np.mean(r):.4f} (se {np.std(r) / np.sqrt(P):.4f})")
    assert abs(np.mean(r) - 1.0) < 5 * np.std(r) / np.sqrt(P), report[-1]
    ess_offset, _ = posterior_ess(engs, POST_INDICES, 0, 0)
    drop = np.median(ess_aligned[0]) / np.median(ess_offset[0])
    report.append(f"median ESS aligned {np.median(ess_aligned[0]):.0f}, one chain offset "
                  f"{np.median(ess_offset[0]):.0f}: {drop:.1f}x")
    print("\n".join(report))
    assert drop > 10.0, report[-1]


# ------------------------------------------------------------------ 7. errors
@pytest.mark.gpu
def test_ess_errors():
    from dang_b200._lib import c_dp, vp
    from dang_b200.engine import POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, Engine
    cfg, sky = small_case("c1", 8, perturb=False)
    a = Engine(cfg, sky)
    lib = a.lib
    buf = np.zeros((2, cfg.nmaps, cfg.npix))

    def ess(engs, kind=POST_AMPLITUDE, m=None, out=(True, True)):
        hs = (vp * len(engs))(*[e.h for e in engs])
        e = buf[0].ctypes.data_as(c_dp) if out[0] else None
        s = buf[1].ctypes.data_as(c_dp) if out[1] else None
        return lib.dang_gpu_posterior_ess(hs, len(engs) if m is None else m, kind, 0, 0, e, s)

    assert ess([a]) == ESTATE                                   # not begun
    for b in (0, -1):
        assert lib.dang_gpu_posterior_begin_batched(a.h, POST_AMPLITUDE, 2, 3, b) == EINVAL
    a.posterior_begin(POST_AMPLITUDE)
    assert ess([a]) == ESTATE                                   # begun without batches
    a.posterior_begin(POST_AMPLITUDE | POST_INDICES, batch_len=2)
    for _ in range(3):
        a.posterior_accumulate()
    assert ess([a]) == EINVAL                                   # K = 1
    a.posterior_accumulate()
    assert ess([a]) == 0                                        # K = 2
    assert ess([a], out=(True, False)) == 0 and ess([a], out=(False, True)) == 0
    assert ess([a], out=(False, False)) == EINVAL
    assert ess([a], kind=POST_CHI_MAP) == EINVAL                # kind not begun
    assert ess([a], m=0) == EINVAL
    many = [a] * 257
    assert ess(many) == EINVAL and ess(many[:256]) == 0

    b = Engine(cfg, sky, share_maps_with=a)
    b.posterior_begin(POST_AMPLITUDE, batch_len=2)
    for _ in range(5):
        b.posterior_accumulate()
    assert ess([a, b]) == EINVAL                                # different n
    b.posterior_begin(POST_AMPLITUDE, batch_len=1)
    for _ in range(4):
        b.posterior_accumulate()
    assert ess([a, b]) == EINVAL                                # different batch length
    b.posterior_begin(POST_AMPLITUDE, batch_len=2)
    for _ in range(4):
        b.posterior_accumulate()
    assert ess([a, b]) == 0
    b.posterior_begin(POST_AMPLITUDE)
    assert ess([a, b]) == ESTATE                                # one handle without batches
    b.posterior_end()
    assert ess([a, b]) == ESTATE                                # one handle not begun
    c = Engine(cfg, sky, pix_range=(0, cfg.npix // 2))
    c.posterior_begin(POST_AMPLITUDE, batch_len=2)
    for _ in range(4):
        c.posterior_accumulate()
    assert ess([a, c]) == EINVAL                                # different pixel range
    assert "pixel range" in lib.dang_gpu_last_error(a.h).decode()
