"""Cost of the device-side posterior summaries (dang_gpu_posterior_accumulate) on full-size runs:
    python scripts/posterior_cost.py [--steps 20] [--reps 5]

For c2 and c4 (20 bands, per-pixel beta_d and T_d) at nside 512, Gibbs iterations (device deviates, device-resident
state) are timed with CUDA events in three arms that share one set of maps and alternate rep by rep: no accumulation,
AMPLITUDE | INDICES after every iteration, and every kind after every iteration.  The accumulate call alone is
timed between dang_gpu_event_record slots; its bytes are computed from the shapes and set against the project's
measured 6.39 TB/s device copy peak.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_PEAK = 6.39e12  # B/s, measured device-to-device copy rate of a B200 (README)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def pass_bytes(cfg, what):
    """Compulsory HBM bytes of one accumulation: 40 B per accumulated element of the streaming pass (8 read from the
    state, 16 read and 16 written of {mean, M2}); the residual / chi-square pass reads sig, rms, the amplitudes and
    indices once and moves 32 B of accumulators per residual and chi-square element."""
    from dang_b200.engine import POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, POST_RESIDUAL
    P, S, B = cfg.npix, cfg.nmaps, cfg.nbands
    planes = 0
    for c in cfg.comps:
        if what & POST_AMPLITUDE and c.type not in ("template", "monopole", "hi_fit", "T_cmb"):
            planes += S
        if what & POST_INDICES:
            planes += S * len(c.indices)
    stream = 40.0 * planes * P
    k6 = 0.0
    if what & (POST_CHI_MAP | POST_RESIDUAL):
        k6 = 8.0 * P * S * (2 * B + sum(1 + len(c.indices) for c in cfg.comps)) + P
        k6 += 32.0 * P * S * ((B if what & POST_RESIDUAL else 0) + (1 if what & POST_CHI_MAP else 0))
    return stream, k6


def run(name, nside, steps, reps):
    from dang_b200.engine import POST_AMPLITUDE, POST_INDICES, Engine
    from dang_b200.synth import make_config, make_sky
    cfg = make_config(name, nside=nside)
    sky = make_sky(cfg)
    arms = {"none": 0, "amp_idx": POST_AMPLITUDE | POST_INDICES, "all": 31}
    engs = {}
    for arm, what in arms.items():
        engs[arm] = Engine(cfg, sky, share_maps_with=engs.get("none"))
        if what:
            engs[arm].posterior_begin(what)
    it = {arm: 1 for arm in arms}

    def steps_of(arm, k):
        eng, what = engs[arm], arms[arm]
        for _ in range(k):
            eng.gibbs_iteration(it[arm], seed=11)
            it[arm] += 1
            if what:
                eng.posterior_accumulate()

    for arm in arms:  # warm-up: tuner, first solves, every kernel shape
        steps_of(arm, 3)
        engs[arm].sync()
    ms = {arm: [] for arm in arms}
    for _ in range(reps):
        for arm in arms:
            eng = engs[arm]
            eng.sync()
            eng.event_record(0)
            steps_of(arm, steps)
            eng.event_record(1)
            eng.sync()
            ms[arm].append(eng.event_elapsed_ms(0, 1) / steps)
    out = {"config": name, "nside": nside, "steps": steps, "reps": reps,
           "ms_per_iteration": {a: [round(v, 4) for v in ms[a]] for a in arms}}
    base = float(np.median(ms["none"]))
    for arm, what in arms.items():
        if not what:
            continue
        eng = engs[arm]
        acc_ms = []
        for _ in range(20):
            eng.sync()
            eng.event_record(2)
            eng.posterior_accumulate()
            eng.event_record(3)
            eng.sync()
            acc_ms.append(eng.event_elapsed_ms(2, 3))
        t = float(np.median(acc_ms)) * 1e-3
        stream, k6 = pass_bytes(cfg, what)
        out[arm] = {"iteration_overhead": round(float(np.median(ms[arm])) / base - 1.0, 4),
                    "accumulate_ms": round(t * 1e3, 4), "bytes": stream + k6,
                    "fraction_of_copy_peak": round((stream + k6) / t / COPY_PEAK, 3)}
    for eng in engs.values():
        eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nside", type=int, default=512)
    args = ap.parse_args()
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    for name in ("c2", "c4"):
        print(json.dumps(run(name, args.nside, args.steps, args.reps)), flush=True)


if __name__ == "__main__":
    main()
