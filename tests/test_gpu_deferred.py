"""Deferred scalars (DANG_OPT_DEFER_SCALARS, include/dang_gpu.h): the calls of one Gibbs iteration enqueue their kernels
without waiting for the numbers of the terminal line (write_stats_to_term, src/dang.f90:100-104);
dang_gpu_iteration_mark / dang_gpu_iteration_scalars hand them back one iteration late.  Everything -- iteration
counts, residuals, chi-squares, acceptance ratios, index values, the maps -- must be bit-identical to the default
mode, which the other parity tests tie to the oracle."""
import numpy as np
import pytest

from helpers import small_case

pytestmark = pytest.mark.gpu


def _run(cfg, sky, n_iter, deferred, lag):
    from dang_b200.engine import OPT_DEFER_SCALARS, Engine
    eng = Engine(cfg, sky)
    rows = []
    if not deferred:
        for it in range(1, n_iter + 1):
            r1, r2 = eng.gibbs_iteration(it, seed=11)
            rows.append((r1[0][0], r1[0][1], r1[1], None if r2 is None else r2[0][0], None if r2 is None else r2[1]))
    else:
        # iteration 1 (no spectral-parameter block, tuner not yet run) and 2 (the tuner runs) in the default mode
        for it in range(1, 3):
            r1, r2 = eng.gibbs_iteration(it, seed=11)
            rows.append((r1[0][0], r1[0][1], r1[1], None if r2 is None else r2[0][0], None if r2 is None else r2[1]))
        eng.set_option(OPT_DEFER_SCALARS, 1)
        tickets = []
        for it in range(3, n_iter + 1):
            r1, r2 = eng.gibbs_iteration(it, seed=11)
            assert r1[0][0] == -1 and np.isnan(r1[0][1]) and np.isnan(r1[1])      # nothing came back yet
            assert np.isnan(r2[0][0]) and np.isnan(r2[1])
            tickets.append(eng.iteration_mark())
            if len(tickets) > lag:
                s = eng.iteration_scalars(tickets[-1 - lag])
                rows.append((s["n_iter"], s["delta"], s["chisq_amplitudes"], s["accept"], s["chisq_index"], s["index_value"]))
        for t in tickets[len(tickets) - lag:]:
            s = eng.iteration_scalars(t)
            rows.append((s["n_iter"], s["delta"], s["chisq_amplitudes"], s["accept"], s["chisq_index"], s["index_value"]))
        eng.set_option(OPT_DEFER_SCALARS, 0)
    amps = [eng.amplitude(ic).copy() for ic in range(len(cfg.comps))]
    idx = [eng.indices(ic).copy() for ic in range(len(cfg.comps))]
    return rows, amps, idx, eng


@pytest.mark.parametrize("lag", [0, 1, 3])
def test_deferred_scalars_are_bit_identical(lag):
    cfg, sky = small_case("c2", nside=32)
    n_iter = 9
    rows_s, amps_s, idx_s, eng_s = _run(cfg, sky, n_iter, False, 0)
    rows_d, amps_d, idx_d, eng_d = _run(cfg, sky, n_iter, True, lag)
    assert len(rows_s) == len(rows_d) == n_iter
    for it, (a, b) in enumerate(zip(rows_s, rows_d), start=1):
        assert a[:5] == b[:5], (it, a, b)
    assert rows_d[-1][5] == idx_d[1][0][1][0] or rows_d[-1][5] == idx_d[0][0][1][0]   # the value the chain left in the map
    for x, y in zip(amps_s, amps_d):
        assert np.array_equal(x, y)
    for x, y in zip(idx_s, idx_d):
        assert np.array_equal(x, y)
    # back in the default mode both engines continue identically (host bookkeeping caught up)
    r_s, r_d = eng_s.gibbs_iteration(n_iter + 1, seed=11), eng_d.gibbs_iteration(n_iter + 1, seed=11)
    assert r_s[0][0] == r_d[0][0] and r_s[0][1] == r_d[0][1] and r_s[1][1] == r_d[1][1]
    assert eng_d.index_fullsky(*_sampled(cfg), 2) == eng_s.index_fullsky(*_sampled(cfg), 2)


def _sampled(cfg):
    for ic, c in enumerate(cfg.comps):
        for j, s in enumerate(c.indices):
            if s.sample:
                return ic, j
    raise AssertionError("no sampled index")


def test_deferred_mode_is_loud_about_misuse():
    from dang_b200.engine import OPT_DEFER_SCALARS, DangGpuError, Engine
    cfg, sky = small_case("c2", nside=16)
    eng = Engine(cfg, sky)
    eng.gibbs_iteration(1, seed=3)
    eng.gibbs_iteration(2, seed=3)
    eng.set_option(OPT_DEFER_SCALARS, 1)
    eng.gibbs_iteration(3, seed=3)
    with pytest.raises(DangGpuError, match="pending"):
        eng.set_option(OPT_DEFER_SCALARS, 0)          # results would be lost
    t = [eng.iteration_mark()]
    for it in range(4, 7):
        eng.gibbs_iteration(it, seed=3)
        t.append(eng.iteration_mark())
    eng.gibbs_iteration(7, seed=3)
    with pytest.raises(DangGpuError, match="has not been read"):
        eng.iteration_mark()                          # four unread tickets: the fifth would overwrite the first
    with pytest.raises(DangGpuError, match="never issued"):
        eng.iteration_scalars(99)
    s = [eng.iteration_scalars(x) for x in t]
    assert all(x["n_iter"] > 1 for x in s)
    t5 = eng.iteration_mark()
    with pytest.raises(DangGpuError, match="overwritten"):
        eng.iteration_scalars(t[0])
    assert eng.iteration_scalars(t5)["n_iter"] > 1
    # a mark holds one full-sky outcome: a second full-sky draw before it (index poltype 'Q,U', or two full-sky
    # indices in one iteration) would overwrite the first draw's acceptance, value and chi-square
    eng.sample_index_mh(1, 0, 2, 8, seed=4)
    with pytest.raises(DangGpuError, match="iteration_mark"):
        eng.sample_index_mh(1, 0, 3, 8, seed=4)
    with pytest.raises(DangGpuError, match="iteration_mark"):
        eng.tune_index(1, 0, 3, 8, seed=4, max_blocks=2)
    t6 = eng.iteration_mark()
    eng.sample_index_mh(1, 0, 3, 8, seed=4)
    t7 = eng.iteration_mark()
    s6, s7 = eng.iteration_scalars(t6), eng.iteration_scalars(t7)
    assert s6["index_value"] == eng.index_fullsky(1, 0, 2) and s7["index_value"] == eng.index_fullsky(1, 0, 3)
    assert s6["accept"] >= 0.0 and s7["accept"] >= 0.0  # (NaN: nothing was snapshot)
