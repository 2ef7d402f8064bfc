"""Multi-rank parity check, one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29511 tests/multi_gpu_check.py

Every rank owns a contiguous HEALPix ring range; the CG dot products, full-sky lnL statistics and
chi-square sums cross ranks through NCCL all-gathers inside libdang_gpu.so.  Each rank checks its
own pixel slice against the CPU oracle run on the full sky with the same injected deviates.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist

    from dang_b200.engine import Engine, setup_torch_comm
    from dang_b200.healpix import ring_partition
    from helpers import small_case
    from oracle.binding import Oracle

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    worst = 0.0
    ns = int(os.environ.get("DANG_MGC_NSIDE", "16"))
    if os.environ.get("DANG_MGC_CASE") == "b32":
        check_32_bands(rank, world, local, ns)
        dist.destroy_process_group()
        return
    if os.environ.get("DANG_MGC_CASE") == "rng":
        check_device_deviates(rank, world, local, ns)
        dist.destroy_process_group()
        return
    from dang_b200.engine import OPT_CG_CHECKPOINT
    # (config, nside, CG form): the default checkpointed-recompute form, the streaming form (checkpoint 0) and a
    # solve with i_max >= DG_CG_HIST (1024), which also takes the streaming form -- all exchange the CG sums
    # inside the pass kernel when the NVLink mailboxes are on, and must follow the single-rank oracle
    for name, nside, form in (("c1", ns, "recompute"), ("c2", ns, "recompute"), ("c2", 16, "streaming"), ("c1", 16, "imax2000")):
        cfg, sky = small_case(name, nside, perturb=(name == "c1"))
        if form == "imax2000":
            cfg.cg_groups[0].max_iter = 2000
        bounds = ring_partition(cfg.nside, world, weights=(sky.mask != 0).astype(np.float64))
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
        if form == "streaming":
            eng.set_option(OPT_CG_CHECKPOINT, 0)
        setup_torch_comm(eng, mailboxes=os.environ.get("DANG_GPU_MAILBOX", "1") != "0")
        ora = Oracle(cfg, sky)
        rng = np.random.default_rng(77)
        nsample = 8
        for it in (1, 2, 3):
            eta = rng.standard_normal(2 * cfg.npix)
            its_o, _ = ora.sample_cg_group(0, 1, eta)
            r = eng.sample_cg_groups(eta=eta)
            assert r[0][0] == its_o[0], (rank, name, form, r[0], its_o)
            # every rank took the same decisions from the same sums: identical final residual everywhere
            dl = torch.tensor([r[0][1]], dtype=torch.float64, device="cuda")
            dall = [torch.zeros_like(dl) for _ in range(world)]
            dist.all_gather(dall, dl)
            assert all(float(t.item()) == r[0][1] for t in dall), (rank, name, form, [float(t.item()) for t in dall])
            chisq_o, _ = ora.compute_chisq()
            assert abs(r[1] - chisq_o) <= 1e-10 * chisq_o, (rank, r[1], chisq_o)
            if it > 1:
                z, u = rng.standard_normal(nsample * cfg.npix), rng.random(nsample * cfg.npix)
                ora.sample_spectral_parameters(nsample, 1, z, u)
                acc, chisq_g = eng.sample_spectral_parameters(nsample=nsample, z=z, u=u)
                chisq_o, _ = ora.compute_chisq()
                assert abs(chisq_g - chisq_o) <= 1e-10 * chisq_o, (rank, chisq_g, chisq_o)
            for ic in range(len(cfg.comps)):
                a, b = eng.amplitude(ic)[:, lo:hi], ora.amplitude(ic)[:, lo:hi]
                e = np.max(np.abs(a - b)) / np.max(np.abs(ora.amplitude(ic)))
                worst = max(worst, e)
                assert e < 1e-10, (rank, name, it, ic, e)
                ia, ib = eng.indices(ic)[:, :, lo:hi], ora.indices(ic)[:, :, lo:hi]
                assert np.max(np.abs(ia - ib)) < 1e-12, (rank, name, it, ic)
        eng.comm_check()
        eng.close()
        dist.barrier()
    # a CG group with a template component: border-row sums cross ranks like the CG dot products
    from helpers import template_case
    cfg, sky, _ = template_case(16)
    cfg.cg_groups[0].converge, cfg.cg_groups[0].max_iter = 1e-20, 300
    bounds = ring_partition(cfg.nside, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
    setup_torch_comm(eng, mailboxes=os.environ.get("DANG_GPU_MAILBOX", "1") != "0")
    ora = Oracle(cfg, sky)
    rng = np.random.default_rng(78)
    for it in (1, 2):
        eta = rng.standard_normal(2 * cfg.npix)
        ora.sample_cg_group(0, 1, eta)
        r = eng.sample_cg_groups(eta=eta)
        chisq_o, _ = ora.compute_chisq()
        assert abs(r[1] - chisq_o) <= 1e-8 * chisq_o, (rank, r[1], chisq_o)
        ta_g, ta_o = eng.template_amplitudes(1), ora.template_amplitudes(1)
        assert np.max(np.abs(ta_g - ta_o)) <= 1e-8 * np.max(np.abs(ta_o)), (rank, ta_g, ta_o)
        a, b = eng.amplitude(0)[:, lo:hi], ora.amplitude(0)[:, lo:hi]
        assert np.max(np.abs(a - b)) <= 1e-8 * np.max(np.abs(ora.amplitude(0))), (rank, "template group amplitudes")
    eng.comm_check()
    eng.close()
    dist.barrier()
    # deferred scalars (DANG_OPT_DEFER_SCALARS) on several ranks: same numbers as the default mode, one iteration late
    if os.environ.get("DANG_GPU_MAILBOX", "1") != "0":   # (the persistent solve needs the mailboxes)
        from dang_b200.engine import OPT_DEFER_SCALARS
        cfg, sky = small_case("c2", ns, perturb=False)
        bounds = ring_partition(cfg.nside, world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        rows = {}
        for mode in ("default", "deferred"):
            eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
            setup_torch_comm(eng, mailboxes=True)
            out, prev = [], None
            for it in range(1, 8):
                if mode == "deferred" and it == 3:
                    eng.set_option(OPT_DEFER_SCALARS, 1)
                r1, r2 = eng.gibbs_iteration(it, seed=5)
                if mode == "deferred" and it >= 3:
                    assert r1[0][0] == -1
                    t = eng.iteration_mark()
                    if prev is not None:
                        q = eng.iteration_scalars(prev)
                        out.append((q["n_iter"], q["delta"], q["chisq_amplitudes"], q["accept"], q["chisq_index"]))
                    prev = t
                else:
                    out.append((r1[0][0], r1[0][1], r1[1], r2[0][0] if r2 else None, r2[1] if r2 else None))
            if prev is not None:
                q = eng.iteration_scalars(prev)
                out.append((q["n_iter"], q["delta"], q["chisq_amplitudes"], q["accept"], q["chisq_index"]))
                eng.set_option(OPT_DEFER_SCALARS, 0)
            rows[mode] = (out, [eng.amplitude(ic)[:, lo:hi].copy() for ic in range(len(cfg.comps))],
                          [eng.indices(ic)[:, :, lo:hi].copy() for ic in range(len(cfg.comps))])
            eng.comm_check()
            eng.close()
            dist.barrier()
        assert rows["default"][0] == rows["deferred"][0], (rank, rows["default"][0], rows["deferred"][0])
        for a, b in zip(rows["default"][1] + rows["default"][2], rows["deferred"][1] + rows["deferred"][2]):
            assert np.array_equal(a, b), (rank, "deferred-scalars maps differ")
    print(f"rank {rank}/{world}: multi-GPU parity ok (pixels [{lo},{hi}), worst amplitude error {worst:.2e})", flush=True)
    dist.destroy_process_group()


def check_32_bands(rank, world, local, nside):
    """DANG_MGC_CASE=b32: full-sky draws at 32 bands (S = 2, then S = 1 on Q), whose statistics rows of
    3 x 4 x 8 chunks x S values per rank are the largest the scalar exchange carries."""
    import torch.distributed as dist

    from dang_b200.engine import Engine, setup_torch_comm
    from dang_b200.healpix import ring_partition
    from oracle.binding import Oracle
    from test_gpu_shapes import shape_case
    cfg, sky = shape_case(32, nside=nside, varying=())
    spec = cfg.comps[1].indices[0]
    spec.sample, spec.region, spec.step = True, "fullsky", 0.002
    bounds = ring_partition(cfg.nside, world, weights=(sky.mask != 0).astype(np.float64))
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
    setup_torch_comm(eng, mailboxes=os.environ.get("DANG_GPU_MAILBOX", "1") != "0")
    ora = Oracle(cfg, sky)
    rng = np.random.default_rng(79)
    for map_n, nsample in ((-1, 24), (2, 200)):
        z, u = rng.standard_normal(nsample), rng.random(nsample)
        acc_o, dec_o, lnl_o = ora.sample_index_mh(1, 0, map_n, nsample, 1, z, u, want_trace=True)
        acc_g = eng.sample_index_mh(1, 0, map_n, nsample, "sample", z, u)
        dec_g, lnl_g = eng.decisions(nsample, fullsky=True)
        assert np.array_equal(dec_g, dec_o[:nsample]) and acc_g == acc_o, (rank, map_n, dec_g, dec_o[:nsample])
        ev = dec_o[:nsample] < 2
        assert np.max(np.abs(lnl_g[ev] - lnl_o[:nsample][ev])) <= 1e-10 * np.max(np.abs(lnl_o[:nsample][ev])), (rank, map_n)
        ia, ib = eng.indices(1)[:, :, lo:hi], ora.indices(1)[:, :, lo:hi]
        assert np.max(np.abs(ia - ib)) <= 1e-14 * np.max(np.abs(ib)), (rank, map_n)
        ora.update_sky_model()
        chisq_o, _ = ora.compute_chisq()
        assert abs(eng.compute_chisq() - chisq_o) <= 1e-10 * chisq_o, (rank, map_n)
    eng.comm_check()
    eng.close()
    dist.barrier()
    print(f"rank {rank}/{world}: multi-GPU parity ok (32 bands, pixels [{lo},{hi}))", flush=True)


def check_device_deviates(rank, world, local, nside):
    """DANG_MGC_CASE=rng: Gibbs iterations with the device's own deviates, as bench.py runs them -- c2 (full-sky beta_d,
    tuned once) and c1 (per-pixel beta_s).  Every rank draws its pixels' eta and z / u at global slots, so its slice
    must follow the single-process oracle fed the Philox arrays (tests/test_gpu_device_rng.py)."""
    import torch.distributed as dist

    from dang_b200.engine import Engine, setup_torch_comm
    from dang_b200.healpix import ring_partition
    from helpers import small_case
    from oracle.binding import Oracle
    from test_gpu_device_rng import oracle_gibbs_iteration
    seed = 9
    for name, ns in (("c2", nside), ("c1", 16)):
        cfg, sky = small_case(name, ns, perturb=False)
        if name == "c2":
            cfg.comps[1].indices[0].tune = True
        bounds = ring_partition(cfg.nside, world, weights=(sky.mask != 0).astype(np.float64))
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
        setup_torch_comm(eng, mailboxes=os.environ.get("DANG_GPU_MAILBOX", "1") != "0")
        ora = Oracle(cfg, sky)
        tuned = [[not s.tune for s in c.indices] for c in cfg.comps]
        for it in range(1, 5):
            n_o, chi_cg_o, acc_o, chi_mh_o, _ = oracle_gibbs_iteration(ora, cfg, it, seed, tuned)
            r1, r2 = eng.gibbs_iteration(it, seed=seed)
            assert r1[0][0] == n_o[0], (rank, name, it, r1[0][0], n_o)
            assert abs(r1[1] - chi_cg_o) <= 1e-10 * chi_cg_o, (rank, name, it, r1[1], chi_cg_o)
            if it > 1:
                assert r2[0] == acc_o, (rank, name, it, r2[0], acc_o)
                assert abs(r2[1] - chi_mh_o) <= 1e-10 * chi_mh_o, (rank, name, it, r2[1], chi_mh_o)
            for ic in range(len(cfg.comps)):
                a, b = eng.amplitude(ic)[:, lo:hi], ora.amplitude(ic)[:, lo:hi]
                assert np.max(np.abs(a - b)) <= 1e-10 * np.max(np.abs(ora.amplitude(ic))), (rank, name, it, ic)
                ia, ib = eng.indices(ic)[:, :, lo:hi], ora.indices(ic)[:, :, lo:hi]
                assert np.max(np.abs(ia - ib)) <= 1e-14 * np.max(np.abs(ib)), (rank, name, it, ic)
        eng.comm_check()
        eng.close()
        dist.barrier()
    print(f"rank {rank}/{world}: multi-GPU parity ok (device deviates, pixels [{lo},{hi}))", flush=True)


if __name__ == "__main__":
    main()
