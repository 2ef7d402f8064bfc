#!/usr/bin/env python
"""bench.py -- Gibbs iterations/sec of dang's hot path (BASELINE.json metric) on B200.

A "step" is one full Gibbs iteration of the reference's loop body for iter > 1
(src/dang.f90:101-111 restricted to the hot path): sample_cg_groups (rhs + CG + unpack +
chi-square) followed by sample_spectral_parameters (Metropolis + chi-square).

  python bench.py --gpus N --steps K --warmup W          our arm (one process per GPU)
  python bench.py --impl reference ...                   the CPU oracle on the host cores
  python bench.py ... --dump-outputs DIR                 also write the last timed step's outputs to DIR/*.npy

The workload is BASELINE.json configs[1] ("c2": nside=512, 8 delta bands, Q+U, synch+dust, CG
amplitudes + full-sky beta_d, NUMSAMPLE=20) on synthetic maps (dang_b200/synth.py).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Gibbs iterations/sec (nside=512, Q+U, synch+dust)"
UNIT = "it/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json, written by profiles/summarize.py)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(kernel)


def ncu_pipe(kernel: str, config: str):
    """Pipe utilisation of `kernel` on `config` from the committed ncu capture (profiles/ncu_pipes.json): the bound
    of the per-pixel Metropolis kernels is an execution pipe, not HBM (SURVEY.md section 8d), and pipe-busy
    percentages cannot be measured outside a profiler."""
    p = os.path.join(ROOT, "profiles", "ncu_pipes.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(f"{kernel}@{config}")


def roofline_block(top, stats, config, peak, peak_src, capture_share=None):
    """The `roofline` object of the JSON line for the dominant kernel `top` of `stats` (dang_gpu_kernel_stats).
    `capture_share`: this rank's share of the workload the committed ncu capture was taken on (c2 at nside 512 on one
    GPU): the captured DRAM bytes per launch scale with it; None when the run is another workload (no traffic figure)."""
    s = stats[top]
    ach = s["bytes"] / (s["ms"] * 1e-3) / 1e9
    tot = sum(v["ms"] for v in stats.values())
    traffic = ncu_traffic(top) if capture_share is not None else None
    if traffic is not None:
        traffic = round(traffic * capture_share)
    roof = {"bound": "hbm", "kernel": top, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
            "frac": round(ach / peak, 4), "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": round(s["bytes"] / max(s["launches"], 1)),
            "avg_launch_us": round(1e3 * s["ms"] / max(s["launches"], 1), 2),
            "share_of_kernel_time": round(s["ms"] / tot, 3),
            "per_kernel": {k: {"launches": v["launches"], "ms": round(v["ms"], 3),
                               "GBps": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if (v["ms"] > 0 and v["bytes"] > 0) else None}
                           for k, v in stats.items() if v["launches"]}}
    pipe = ncu_pipe(top, config)
    if pipe:  # not an HBM-bound kernel: report the pipe that bounds it, keep the (small) HBM figures beside it
        roof["hbm"] = {"achieved": roof["achieved"], "peak": peak, "unit": "GB/s", "frac": roof["frac"]}
        roof.update({"bound": pipe["bound"], "achieved": pipe["busy_pct"], "peak": 100.0,
                     "unit": f"% of the {pipe['bound']} pipe's issue slots busy", "frac": round(pipe["busy_pct"] / 100.0, 4),
                     "peak_source": f"ncu capture {pipe['capture']} (a pipe-busy fraction cannot be measured live; launch time above is live)",
                     "issue_active_pct": pipe.get("issue_active_pct")})
    return roof


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  The region is short (20 steps x 1.5 ms), so
    an `nvidia-smi -lms` child process never gets a sample in (its start-up alone is longer); this is an NVML
    polling thread (pynvml) started before the region and stopped right after it, ~1 ms per sample.  Falls
    back to one nvidia-smi query if NVML is not importable."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, cuda_index: int):
        import threading
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._stop = threading.Event()
        self._t = None
        self.src = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:  # NVML ignores CUDA_VISIBLE_DEVICES: address the device by UUID
                uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
                hdl = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                hdl = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(hdl, pynvml.NVML_CLOCK_SM))
            self.src = "nvml"

            def loop():
                while not self._stop.is_set():
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(hdl, pynvml.NVML_CLOCK_SM)))
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(hdl)
                        for bit, name in self.REASONS.items():
                            if r & bit:
                                self.reasons.add(name)
                        self.power.append(pynvml.nvmlDeviceGetPowerUsage(hdl) / 1e3)
                    except Exception:
                        break
                    time.sleep(0.003)
            self._t = threading.Thread(target=loop, daemon=True)
            self._t.start()
        except Exception:
            self._t = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0, "source": self.src}
        if self._t is not None:
            self._stop.set()
            self._t.join(timeout=2)
        if not self.samples:  # last resort: one query (after the region; says so)
            try:
                r = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0].split(", ")
                out.update(sm_mhz=float(r[0]), sm_max_mhz=float(r[1]), samples=1, source="nvidia-smi after the region")
            except Exception:
                pass
            return out
        out["sm_mhz"] = float(np.median(self.samples))
        out["sm_mhz_min"] = float(np.min(self.samples))
        out["power_w_max"] = round(float(np.max(self.power)), 1) if self.power else None
        out["reasons"] = sorted(self.reasons)
        out["samples"] = len(self.samples)
        return out


# ------------------------------------------------------------------ pinned host buffers
def pinned_array(lib, shape):
    n = int(np.prod(shape))
    ptr = C.c_void_p()
    rc = lib.dang_gpu_host_alloc(C.byref(ptr), n * 8)
    if rc != 0:
        raise RuntimeError("dang_gpu_host_alloc failed")
    buf = (C.c_double * n).from_address(ptr.value)
    return np.frombuffer(buf, dtype=np.float64).reshape(shape)


# ------------------------------------------------------------------ outputs of the timed path
DUMP_BUDGET_BYTES = 60_000_000
DUMP_SEED = 20260107


def dump_outputs(out_dir, eng, cfg, n_cg, chisq):
    """What the last timed Gibbs iteration left a caller: every component's amplitude maps [nmaps][npix] and index
    maps [nind][nmaps][npix], the CG iteration count and the chi-square, as float64 .npy files.  When the maps exceed
    the budget (60 MB in all), the same seeded, sorted sample of pixels is taken from every map (`pixels.npy` lists
    it), so two builds run with the same arguments can be compared file by file."""
    rows = sum(cfg.nmaps * (1 + len(c.indices)) for c in cfg.comps)
    m = min(cfg.npix, DUMP_BUDGET_BYTES // (8 * (rows + 1)))
    pix = np.arange(cfg.npix) if m == cfg.npix else np.sort(
        np.random.default_rng(DUMP_SEED).choice(cfg.npix, size=m, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"pixels": pix.astype(np.float64), "n_cg": np.array([n_cg], dtype=np.float64),
              "chisq": np.array([chisq], dtype=np.float64)}
    for ic, c in enumerate(cfg.comps):
        arrays[f"amplitude_{c.label}"] = np.ascontiguousarray(eng.amplitude(ic)[:, pix])
        if c.indices:
            arrays[f"indices_{c.label}"] = np.ascontiguousarray(eng.indices(ic)[:, :, pix])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------ our arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    from dang_b200.engine import OPT_DEFER_SCALARS, OPT_PROFILE, Engine, setup_torch_comm
    from dang_b200.healpix import ring_partition
    from dang_b200.synth import make_config, make_sky, make_sky_slice
    from dang_b200.healpix import pix2z_ring

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or world == 1, (world, args.gpus)
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs: run a single process (each rank holds only its own pixels)")

    cfg = make_config(args.config, nside=args.nside)
    # big configs (nside >= 1024): every rank builds only its own pixel slice of the synthetic sky
    big = cfg.nside >= 1024
    if big:
        z_all = pix2z_ring(cfg.nside, np.arange(cfg.npix))
        mask_all = np.where(np.abs(z_all) < np.sin(np.deg2rad(5.0)), 0.0, 1.0)
        del z_all
    else:
        sky = make_sky(cfg)
        mask_all = sky.mask
    # streaming kernels cost the same for masked and unmasked pixels; per-pixel Metropolis chains run
    # only on unmasked ones: balance total pixels, or unmasked pixels when a per-pixel index is sampled
    per_pixel = any(s.sample and s.region != "fullsky" for c in cfg.comps for s in c.indices)
    bounds = ring_partition(cfg.nside, world, weights=(mask_all != 0).astype(np.float64) if per_pixel else None)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    if big:
        del mask_all
        sky = make_sky_slice(cfg, lo, hi)
    mask_slice = sky.mask[lo:hi]
    eng = Engine(cfg, sky, device=local, pix_range=(lo, hi))
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(int(k), float(v))
    mailboxes = os.environ.get("DANG_GPU_MAILBOX", "1") != "0"
    if world > 1:
        setup_torch_comm(eng, mailboxes=mailboxes)

    def barrier():
        eng.sync()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    info = {}
    # Deferred scalars (DANG_OPT_DEFER_SCALARS, include/dang_gpu.h): the numbers of the reference's terminal line
    # (CG iterations, chi-square, acceptance) reach the host one Gibbs iteration late instead of stalling the device
    # three times per iteration.  Covers the one-solve + full-sky-draw shape of c1 / c2; every number still arrives
    # (and is counted below), the kernels and their results are bit-identical (tests/test_gpu_deferred.py).
    fullsky_only = all(s.region == "fullsky" for c in cfg.comps for s in c.indices if s.sample)
    one_solve = len(cfg.cg_groups) == 1 and "," not in cfg.cg_groups[0].poltype
    defer = bool(args.defer_scalars) and fullsky_only and one_solve and (world == 1 or mailboxes)
    pending = []
    n_cg = []

    def take(q):
        n_cg.append(q["n_iter"])
        info["chisq"] = q["chisq_index"]
        info["index_value"] = q["index_value"]

    def step(it, seed=0):
        r1, r2 = eng.gibbs_iteration(it, seed=seed)
        if r1[0][0] == -1:  # deferred: mark this iteration, pick up the one before it
            pending.append(eng.iteration_mark())
            if len(pending) > 1:
                take(eng.iteration_scalars(pending.pop(0)))
        else:
            n_cg.append(r1[0][0])
            info["chisq"] = r2[1] if r2 else r1[-1]

    def drain():
        while pending:
            take(eng.iteration_scalars(pending.pop(0)))

    # --- device-resident timing: `value`
    step(2)  # (the step-size tuner runs here, once)
    if defer:
        eng.set_option(OPT_DEFER_SCALARS, 1)
    for w in range(1, args.warmup):
        step(2 + w)
    drain()
    # the NVML sampler is set up BEFORE the barrier: its start-up (tens of ms on rank 0 only) inside the timed region
    # would leave the other ranks' kernels spinning in their first scalar exchange, and max-over-ranks would report it
    sampler = ClockSampler(local) if (rank == 0 and os.environ.get("DANG_BENCH_NO_CLOCKS") != "1") else None
    barrier()
    eng.launch_count(reset=True)
    eng.event_record(0)
    t_value0 = time.perf_counter()
    n_cg.clear()
    for k in range(args.steps):
        step(2 + args.warmup + k)
    drain()
    assert len(n_cg) == args.steps and np.isfinite(info["chisq"]), (len(n_cg), info)
    eng.event_record(1)
    eng.sync()
    wall_value_ms = (time.perf_counter() - t_value0) * 1e3
    barrier()
    ms = max_over_ranks(eng.event_elapsed_ms(0, 1))
    launches = eng.launch_count()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:  # before the legs below move the chain on
        dump_outputs(args.dump_outputs, eng, cfg, n_cg[-1], info["chisq"])

    # --- per-kernel timing for the roofline: same steps with CUDA events around every launch
    eng.kernel_stats(reset=True)
    eng.set_option(OPT_PROFILE, 1)
    ncg_value = list(n_cg)
    for k in range(max(1, min(args.steps, 5))):
        step(2 + args.warmup + args.steps + k)
    drain()
    n_cg = ncg_value
    stats = eng.kernel_stats(reset=True)
    eng.set_option(OPT_PROFILE, 0)
    k5_fallbacks = eng.perpixel_stats()[0] if per_pixel else None

    # --- end to end through the C ABI with host buffers: deviates in, maps out, every step
    npix = cfg.npix
    # three different sets of deviates, cycled: with ONE set every other solve would start from the previous
    # solution of the same right-hand side and converge at once
    eta_hs = [pinned_array(eng.lib, (2 * npix,)) for _ in range(3)]
    eta_h = eta_hs[0]
    # one (z, u) pair per sample_index_mh call: nsample slots for a full-sky index,
    # nsample*npix for a per-pixel one
    calls = [s for c in cfg.comps for s in c.indices if s.sample for _ in s.poltype.split(",")]
    # injected per-pixel Metropolis deviates are nsample*npix doubles per call (16 GB per step at nside 2048):
    # big configs draw them on the device in the end-to-end leg too and say so
    host_zu = not (big and per_pixel)
    if host_zu:
        z_h = [pinned_array(eng.lib, (cfg.nsample * (1 if s.region == "fullsky" else npix),)) for s in calls]
        u_h = [pinned_array(eng.lib, (cfg.nsample * (1 if s.region == "fullsky" else npix),)) for s in calls]
    else:
        z_h = u_h = None
    amp_h = [pinned_array(eng.lib, (cfg.nmaps, npix)) for _ in cfg.comps]
    idx_h = [pinned_array(eng.lib, (len(c.indices), cfg.nmaps, npix)) for c in cfg.comps]
    rng = np.random.default_rng(20260103 + rank * 0)
    for e in eta_hs:
        e[:] = rng.standard_normal(2 * npix)
    for zz, uu in zip(z_h or [], u_h or []):
        zz[:] = rng.standard_normal(zz.size)
        uu[:] = rng.random(uu.size)
    P = hi - lo
    h2d = 8 * (2 * P + (sum(2 * cfg.nsample * (1 if s.region == "fullsky" else P) for s in calls) if host_zu else 0))

    # Every step: this step's deviates host -> device (eta staged on a copy stream while the
    # previous step computes; z/u inside the sampler call), this step's results device -> host
    # (the Q/U planes the step changed: component amplitudes and the sampled index maps, started
    # right after they are final so the copy overlaps the rest of the step and the next solve;
    # chi-square scalars come back synchronously).  All results have landed when the clock stops.
    sampled = [(ic, j) for ic, c in enumerate(cfg.comps) for j, s in enumerate(c.indices) if s.sample]
    single_solve = len(cfg.cg_groups) == 1 and "," not in cfg.cg_groups[0].poltype
    fs_val = {}

    e2e_ncg = []

    def e2e_step(it):
        if single_solve:
            eng.stage_eta(eta_hs[(it + 1) % 3])     # next step's deviates: upload overlaps this step's solve
            r1 = eng.sample_cg_groups(eta=None)     # consumes the deviates staged one step earlier
        else:
            r1 = eng.sample_cg_groups(eta=eta_hs[it % 3])
        if r1[0][0] != -1:
            e2e_ncg.append(r1[0][0])
        for ic in range(len(cfg.comps)):
            eng.amplitude_async(ic, amp_h[ic])
        eng.sample_spectral_parameters(z=z_h, u=u_h, seed=7 + 2 * it)
        if r1[0][0] == -1:  # deferred scalars: iterations, chi-square and the full-sky index value arrive one step late
            pending.append(eng.iteration_mark())
            if len(pending) > 1:
                q = eng.iteration_scalars(pending.pop(0))
                e2e_ncg.append(q["n_iter"])
                fs_val["deferred"] = q["index_value"]
            return
        for ic, j in sampled:
            if cfg.comps[ic].indices[j].region == "fullsky":
                # the whole plane holds the chain's final sample (dang_sample_mod.f90:329,483): 8 bytes per
                # plane come back; the host-side assignment c%indices(:,k,nind) = value is the reference's own
                fs_val[(ic, j)] = (eng.index_fullsky(ic, j, 2), eng.index_fullsky(ic, j, 3))
            else:
                eng.indices_async(ic, j, idx_h[ic])

    if single_solve:
        eng.stage_eta(eta_hs[0])
    def e2e_drain():
        while pending:
            q = eng.iteration_scalars(pending.pop(0))
            e2e_ncg.append(q["n_iter"])
            fs_val["deferred"] = q["index_value"]

    for w in range(3):
        e2e_step(w)
    eng.download_wait()
    e2e_drain()
    e2e_ncg.clear()
    barrier()
    eng.event_record(2)
    t0 = time.perf_counter()
    ke = max(1, min(args.steps, 50))
    for k in range(ke):
        e2e_step(3 + k)
    eng.download_wait()
    e2e_drain()
    assert len(e2e_ncg) == ke, (len(e2e_ncg), ke)
    eng.event_record(3)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_dev_ms = eng.event_elapsed_ms(2, 3)
    e2e_ms = max_over_ranks(max(e2e_dev_ms, wall_ms))
    n_pp = sum(1 for ic, j in sampled if cfg.comps[ic].indices[j].region != "fullsky")
    nplanes_out = 2 * len(cfg.comps) + 2 * n_pp
    d2h = 8 * P * nplanes_out + 8 * 8 + 16 * (len(sampled) - n_pp)

    # --- the same loop with fewer bytes on the host link (reported beside `e2e`, which stays the worst case:
    #     injected deviates in AND all changed maps out on every iteration, i.e. OUTPUT_ITER = 1)
    variants = {}
    if fullsky_only and one_solve and not args.no_variants:
        def run_variant(kind):
            def vstep(it):
                if kind == "device_rng":      # the shim's production path: deviates drawn on the device, maps out
                    r1 = eng.sample_cg_groups(eta=None, seed=1000 + it)
                    for ic in range(len(cfg.comps)):
                        eng.amplitude_async(ic, amp_h[ic])
                    eng.sample_spectral_parameters(seed=7 + 2 * it)
                else:                          # maps stay on the device between output iterations (OUTPUT_ITER > 1)
                    eng.stage_eta(eta_hs[(it + 1) % 3])
                    r1 = eng.sample_cg_groups(eta=None)
                    eng.sample_spectral_parameters(z=z_h, u=u_h, seed=7 + 2 * it)
                if r1[0][0] == -1:
                    pending.append(eng.iteration_mark())
                    if len(pending) > 1:
                        eng.iteration_scalars(pending.pop(0))
                else:
                    for ic, j in sampled:
                        eng.index_fullsky(ic, j, 2)

            def vdrain():
                while pending:
                    eng.iteration_scalars(pending.pop(0))
                eng.download_wait()

            if kind == "scalars_only":
                eng.stage_eta(eta_hs[0])
            for w in range(3):
                vstep(w)
            vdrain()
            barrier()
            eng.event_record(4)
            tv = time.perf_counter()
            for k in range(ke):
                vstep(3 + k)
            vdrain()
            eng.event_record(5)
            barrier()
            wall = (time.perf_counter() - tv) * 1e3
            vms = max_over_ranks(max(eng.event_elapsed_ms(4, 5), wall))
            if kind == "scalars_only":     # leave no staged deviates behind
                eng.sample_cg_groups(eta=None)
                vdrain()
            return round(1e3 * ke / vms, 3)

        variants["device_rng_maps_out"] = {"value": run_variant("device_rng"), "unit": UNIT, "h2d_bytes_per_step": 0,
                                           "d2h_bytes_per_step": d2h}
        variants["deviates_in_scalars_out"] = {"value": run_variant("scalars_only"), "unit": UNIT, "h2d_bytes_per_step": h2d,
                                               "d2h_bytes_per_step": 8 * 8 + 16 * len(sampled)}

    eng.comm_check()  # a timed-out scalar exchange would have poisoned the sums: fail instead of printing
    if rank == 0:
        peak, peak_src = peaks()
        ms_per_step = ms / args.steps
        top = max((k for k in stats if stats[k]["ms"] > 0), key=lambda k: stats[k]["ms"], default=None)
        # the ncu capture behind `traffic` is c2 at nside 512 on one GPU; a rank of an N-GPU run moves its share of it
        share = (P / cfg.npix) if (cfg.name == "c2" and cfg.nside == 512) else None
        roof = roofline_block(top, stats, cfg.name, peak, peak_src, capture_share=share) if top else None
        line = {
            "metric": METRIC if (cfg.name == "c2" and cfg.nside == 512) else f"Gibbs iterations/sec (nside={cfg.nside}, Q+U, synch+dust)",
            "value": round(1e3 / ms_per_step, 3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
            "ms_per_step_wall_rank0": round(wall_value_ms / args.steps, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(cfg),
                       "npix": cfg.npix,
                       "n_cg_iterations": {"min": int(min(n_cg)), "max": int(max(n_cg)), "mean": round(float(np.mean(n_cg)), 2)},
                       "parallelism": f"ring-range pixel shards x{world}" + ("" if world == 1 else (", scalar exchange over NVLink mailboxes" if mailboxes else ", scalar exchange by NCCL all-gather")),
                       "l2": f"working set per GPU (sig+rms {16e-9 * cfg.nbands * 2 * P:.2f} GB + CG state) >> 126 MB L2, no flush needed",
                       "rng": "device Philox4x32-10",
                       "scalars": ("deferred: CG iterations / chi-square / acceptance of step k read by the host during step k+1 "
                                   "(DANG_OPT_DEFER_SCALARS); all read before the clock stops") if defer else "every call returns its own scalars (three host waits per step)",
                       **({"k5_fp64_fallbacks_per_proposal": round(k5_fallbacks / (cfg.nsample * float((mask_slice != 0).sum()) * world), 6)}
                          if k5_fallbacks is not None else {})},
            "pixel_band_updates_per_s": round(2 * cfg.npix * cfg.nbands * 1e3 / ms_per_step, 1),
            "gpu_launches": launches,
            "clocks": clocks,
            "e2e": {"value": round(1e3 * ke / e2e_ms, 3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": ke,
                    "n_cg_iterations": {"min": int(min(e2e_ncg)), "max": int(max(e2e_ncg)), "mean": round(float(np.mean(e2e_ncg)), 2)},
                    "ms_per_step_device_rank0": round(e2e_dev_ms / ke, 4), "ms_per_step_wall_rank0": round(wall_ms / ke, 4),
                    "what": "per step: injected deviates (eta, z, u) pinned host -> device; changed Q/U planes of every amplitude map and of the per-pixel-sampled index maps, the value of every full-sky-sampled index (one double per plane) + chi-square device -> pinned host; copies overlap compute on dedicated streams"
                            + ("" if host_zu else "; per-pixel Metropolis deviates drawn on the device (16 GB per step otherwise)"),
                    **({"variants": variants,
                        "variants_what": "same loop, fewer bytes on the host link: `device_rng_maps_out` = the Fortran shim's production path (device Philox, all changed maps out every iteration); `deviates_in_scalars_out` = injected deviates in, only the terminal-line scalars out (maps stay on the device between OUTPUT_ITER iterations, src/dang.f90:119-121)"}
                       if variants else {})},
            "roofline": roof,
        }
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args, sky=None if big else sky)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ CPU arm (oracle, all host cores)
def host_threads() -> int:
    """Cores this process may run on.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, so the
    thread count is set explicitly (ora_set_num_threads) instead of inherited from the environment."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_gibbs_time(nside, nsteps: int, config: str, budget_s: float = 1e9, sky=None):
    """Seconds per Gibbs iteration of the OpenMP oracle on the SAME config and map size as the GPU arm
    (reference cost structure: three-sweep compute_Ax with SED re-evaluation, full-map data copies,
    per-proposal sweeps).  One untimed cold iteration (iter == 1: no spectral draw, cold-start CG), then at most
    `nsteps` timed iterations, stopping early once `budget_s` seconds of timed work are spent."""
    from dang_b200.synth import make_config, make_sky
    from oracle.binding import Oracle, load
    cfg = make_config(config, nside=nside)
    if sky is None:
        sky = make_sky(cfg)
    threads = host_threads()
    load(omp=True).ora_set_num_threads(threads)
    ora = Oracle(cfg, sky, omp=True)
    rng = np.random.default_rng(3)
    calls = [s for c in cfg.comps for s in c.indices if s.sample for _ in s.poltype.split(",")]
    # a full-sky chain reads nsample deviates; a per-pixel one nsample * npix (slot-indexed)
    nz = cfg.nsample if (len(calls) == 1 and calls[0].region == "fullsky") else cfg.nsample * cfg.npix * max(1, len(calls))
    times, n_cg = [], []
    for it in range(nsteps + 1):
        eta = rng.standard_normal(2 * cfg.npix)
        z, u = rng.standard_normal(nz), rng.random(nz)
        t0 = time.perf_counter()
        its, _ = ora.sample_cg_group(0, 1, eta)
        ora.compute_chisq()
        if it > 0:
            ora.sample_spectral_parameters(cfg.nsample, 1, z, u)
            ora.compute_chisq()
        dt = time.perf_counter() - t0
        if it > 0:
            times.append(dt)
            n_cg.append(its[0])
            if sum(times) > budget_s:
                break
    return cfg, float(np.mean(times)), n_cg, ora.lib.ora_num_threads()


def cpu_baseline(args, sky=None):
    """rank 0, N = 1 only: a bounded sample (one timed Gibbs iteration after the cold one, 10-30 s of CPU work)
    of the same workload at the same size."""
    cfg, sec, n_cg, threads = cpu_gibbs_time(args.nside, 1, args.config, sky=sky)
    return {"value": round(1.0 / sec, 5), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"1 timed Gibbs iteration (after the cold first one) of the OpenMP oracle -- the CPU restatement of "
                      f"the reference -- on the same config at the same size (nside={cfg.nside}): {sec:.2f} s, n_cg={n_cg[0]}"}


def run_reference(args):
    """The reference arm: the reference's own CPU implementation of the path (its C restatement: the Fortran cannot
    be built, DESIGN.md section 2) on all host cores, on THIS config at THIS size.  Steps are whole Gibbs
    iterations; the run stops after --steps of them or ~150 s of timed work, whichever comes first, and reports
    the steps actually timed.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, sec, n_cg, threads = cpu_gibbs_time(args.nside, max(1, args.steps), args.config, budget_s=150.0)
    v = round(1.0 / sec, 5)
    sample = (f"{len(n_cg)} Gibbs iterations of the OpenMP oracle (CPU restatement of the reference; no Fortran compiler "
              f"exists here or on the GPU box) on {threads} threads, config {cfg.name} at nside={cfg.nside}, same workload as the GPU arm")
    line = {"impl": "reference", "metric": METRIC if (cfg.name == "c2" and cfg.nside == 512) else f"Gibbs iterations/sec (nside={cfg.nside}, Q+U, synch+dust)",
            "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(n_cg), "warmup": 1, "ms_per_step": round(sec * 1e3, 2),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(cfg), "npix": cfg.npix,
                       "n_cg_iterations": {"min": int(min(n_cg)), "max": int(max(n_cg)), "mean": round(float(np.mean(n_cg)), 2)},
                       "steps_requested": args.steps},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_name(cfg) -> str:
    return (f"{cfg.name}: nside={cfg.nside}, {cfg.nbands} bands, Q+U, synch+dust, CG amplitudes + "
            + " + ".join(f"{s.region} {c.label} {s.label}" for c in cfg.comps for s in c.indices if s.sample)
            + f", NUMSAMPLE={cfg.nsample}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--nside", type=int, default=None, help="override the map size (tests only)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the reduced-traffic e2e variants")
    ap.add_argument("--defer-scalars", type=int, default=1, help="1: DANG_OPT_DEFER_SCALARS on the one-solve + full-sky configs")
    ap.add_argument("--opt", action="append", default=[], help="library option id=value (experiments), e.g. --opt 8=16")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's maps and scalars to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
