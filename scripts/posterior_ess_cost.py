"""Cost of the batch-means accumulators behind dang_gpu_posterior_ess on full-size runs:
    python scripts/posterior_ess_cost.py [--steps 32] [--reps 5] [--batch 32]

For c2 and c4 at nside 512, Gibbs iterations (device deviates, device-resident state) are timed with CUDA events in
four arms that share one set of maps and alternate rep by rep: no accumulation, AMPLITUDE | INDICES unbatched,
AMPLITUDE | INDICES with batch means (b = --batch), and every kind with batch means.  The accumulate call alone is
timed over one whole batch (b consecutive calls, so every phase is in it) between dang_gpu_event_record slots; its
bytes are computed from the shapes and set against the project's measured device copy peak (posterior_cost.py).
The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from posterior_cost import COPY_PEAK, gpu_info  # noqa: E402


def per_element_bytes(b):
    """Mean bytes per element of one accumulation, over the b phases of a batch.  Streaming pass: 40 unbatched;
    batched, open 48 (bsum written, not read), middle 56, close 80 (bsum read, {bmean, bM2} read and written), b = 1
    72.  K6 sink: 32 of {mean, M2}, plus 8 / 16 / 40 (b = 1: 32) for the batch arrays."""
    if b == 0:
        return 40.0, 32.0
    if b == 1:
        return 72.0, 64.0
    return (48.0 + 56.0 * (b - 2) + 80.0) / b, 32.0 + (8.0 + 16.0 * (b - 2) + 40.0) / b


def pass_bytes(cfg, what, b):
    """Compulsory HBM bytes of one accumulation, averaged over a batch: the streaming pass's elements times
    per_element_bytes; the residual / chi-square pass reads sig, rms, the amplitudes and indices once and moves the
    accumulators of every residual and chi-square element."""
    from dang_b200.engine import POST_AMPLITUDE, POST_CHI_MAP, POST_INDICES, POST_RESIDUAL
    P, S, B = cfg.npix, cfg.nmaps, cfg.nbands
    planes = 0
    for c in cfg.comps:
        if what & POST_AMPLITUDE and c.type not in ("template", "monopole", "hi_fit", "T_cmb"):
            planes += S
        if what & POST_INDICES:
            planes += S * len(c.indices)
    e_stream, e_k6 = per_element_bytes(b)
    stream = e_stream * planes * P
    k6 = 0.0
    if what & (POST_CHI_MAP | POST_RESIDUAL):
        k6 = 8.0 * P * S * (2 * B + sum(1 + len(c.indices) for c in cfg.comps)) + P
        k6 += e_k6 * P * S * ((B if what & POST_RESIDUAL else 0) + (1 if what & POST_CHI_MAP else 0))
    return stream, k6


def run(name, nside, steps, reps, batch):
    from dang_b200.engine import POST_AMPLITUDE, POST_INDICES, Engine
    from dang_b200.synth import make_config, make_sky
    cfg = make_config(name, nside=nside)
    sky = make_sky(cfg)
    ai = POST_AMPLITUDE | POST_INDICES
    arms = {"none": (0, 0), "amp_idx": (ai, 0), f"amp_idx_b{batch}": (ai, batch), f"all_b{batch}": (31, batch)}
    engs = {}
    for arm, (what, b) in arms.items():
        engs[arm] = Engine(cfg, sky, share_maps_with=engs.get("none"))
        if what:
            engs[arm].posterior_begin(what, batch_len=b)
    it = {arm: 1 for arm in arms}

    def steps_of(arm, k):
        eng, (what, _) = engs[arm], arms[arm]
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
    out = {"config": name, "nside": nside, "steps": steps, "reps": reps, "batch": batch,
           "ms_per_iteration": {a: [round(v, 4) for v in ms[a]] for a in arms}}
    base = float(np.median(ms["none"]))
    for arm, (what, b) in arms.items():
        if not what:
            continue
        eng = engs[arm]
        calls = max(b, 1)  # one whole batch: every phase once
        acc_ms = []
        for _ in range(max(1, 64 // calls)):
            eng.sync()
            eng.event_record(2)
            for _ in range(calls):
                eng.posterior_accumulate()
            eng.event_record(3)
            eng.sync()
            acc_ms.append(eng.event_elapsed_ms(2, 3) / calls)
        t = float(np.median(acc_ms)) * 1e-3
        stream, k6 = pass_bytes(cfg, what, b)
        out[arm] = {"iteration_overhead": round(float(np.median(ms[arm])) / base - 1.0, 4),
                    "accumulate_ms": round(t * 1e3, 4), "bytes": stream + k6,
                    "fraction_of_copy_peak": round((stream + k6) / t / COPY_PEAK, 3)}
    for eng in engs.values():
        eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--nside", type=int, default=512)
    args = ap.parse_args()
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    for name in ("c2", "c4"):
        print(json.dumps(run(name, args.nside, args.steps, args.reps, args.batch)), flush=True)


if __name__ == "__main__":
    main()
