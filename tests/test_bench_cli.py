"""bench.py's CPU legs (no GPU): the reference arm prints one JSON line with the contract's keys, on rank 0 only
under a multi-rank launch, and the product arm fails loudly without a device instead of falling back to the CPU.
--dump-outputs is checked on a stub engine here and end to end on the GPU (marked `gpu`)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                          timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--nside", "16", "--steps", "2", "--warmup", "1", "--gpus", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "it/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["value"] > 0 and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "c2: nside=16" in d["config"]["workload"] and d["config"]["n_cg_iterations"]["min"] >= 2


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--nside", "16", "--steps", "1", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = _run(["--nside", "16", "--steps", "1", "--warmup", "1", "--no-cpu"])
    assert r.returncode != 0
    assert "dang_gpu" in (r.stderr + r.stdout) or "CUDA" in (r.stderr + r.stdout)


def test_steps_and_dump_outputs_arguments_are_checked():
    r = _run(["--impl", "reference", "--nside", "16", "--steps", "0"])
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run(["--impl", "reference", "--nside", "16", "--steps", "1", "--dump-outputs", "unused"])
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


class _StubEngine:
    """amplitude / indices as Engine returns them, filled with values that encode (array, row, pixel)."""

    def __init__(self, cfg):
        import numpy as np
        self.cfg, self.pix = cfg, np.arange(cfg.npix, dtype=np.float64)

    def amplitude(self, ic):
        import numpy as np
        return np.stack([1e7 * ic + 1e6 * k + self.pix for k in range(self.cfg.nmaps)])

    def indices(self, ic):
        import numpy as np
        nind = len(self.cfg.comps[ic].indices)
        return np.stack([self.amplitude(ic) + 1e5 * (j + 1) for j in range(nind)])


def test_dump_outputs_writes_a_fixed_sample_within_the_budget(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from dang_b200.synth import make_config
    for nside, sampled in ((16, False), (512, True)):      # the bench workload at a small size and at its own size
        cfg = make_config("c2", nside=nside)
        dumps = []
        for k in range(2):
            d = tmp_path / f"n{nside}_{k}"
            bench.dump_outputs(str(d), _StubEngine(cfg), cfg, 17, 1.25)
            dumps.append({p.stem: np.load(p) for p in d.iterdir()})
            assert sum(p.stat().st_size for p in d.iterdir()) <= 64_000_000
        a, b = dumps
        assert sorted(a) == ["amplitude_dust", "amplitude_synch", "chisq", "indices_dust", "indices_synch", "n_cg", "pixels"]
        assert all(v.dtype == np.float64 for v in a.values())
        assert all(np.array_equal(a[n], b[n]) for n in a)    # same arguments, same files
        assert a["n_cg"].tolist() == [17.0] and a["chisq"].tolist() == [1.25]
        pix = a["pixels"].astype(np.int64)
        assert np.all(np.diff(pix) > 0) and (len(pix) < cfg.npix) == sampled
        assert a["amplitude_dust"].shape == (cfg.nmaps, len(pix)) and a["indices_dust"].shape == (2, cfg.nmaps, len(pix))
        assert np.array_equal(a["amplitude_dust"][2], 1e7 + 2e6 + pix)
        assert np.array_equal(a["indices_synch"][0, 1], 1e6 + 1e5 + pix)


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_on_the_gpu(tmp_path):
    """Same arguments, same outputs (also with the scalars read every step); one timed step more moves the chain on."""
    import numpy as np

    def dump(name, *extra, steps=3):
        d = tmp_path / name
        r = _run(["--nside", "16", "--steps", str(steps), "--warmup", "2", "--no-cpu", "--no-variants",
                  "--dump-outputs", str(d), *extra], env={"DANG_BENCH_NO_CLOCKS": "1"})
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([x for x in r.stdout.splitlines() if x.startswith("{")][-1])["steps"] == steps
        return {p.stem: np.load(p) for p in d.iterdir()}

    a, b, sync, more = dump("a"), dump("b"), dump("sync", "--defer-scalars", "0"), dump("more", steps=4)
    assert sorted(a) == sorted(more) and len(a["pixels"]) == 3072 and 1 < a["n_cg"][0] < 100
    for n in a:
        assert np.array_equal(a[n], b[n]) and np.array_equal(a[n], sync[n]), n
        assert np.all(np.isfinite(a[n])), n
    assert not np.array_equal(a["amplitude_dust"], more["amplitude_dust"])


def test_roofline_block_reports_the_bounding_pipe(monkeypatch):
    """HBM-bound kernels report bytes / time against the measured copy peak; a kernel listed in
    profiles/ncu_pipes.json (per-pixel Metropolis: an execution pipe bounds it) reports that pipe, with the
    HBM figures kept beside it."""
    sys.path.insert(0, ROOT)
    import bench
    stats = {"cg_pass_kernel": {"launches": 2, "ms": 2.0, "bytes": 10.0e9},
             "mh_perpixel_kernel": {"launches": 2, "ms": 20.0, "bytes": 4.0e9},
             "scalar kernels": {"launches": 4, "ms": 0.1, "bytes": 0.0}}
    monkeypatch.setattr(bench, "ncu_pipe", lambda k, c: None)
    monkeypatch.setattr(bench, "ncu_traffic", lambda k: 4_000_000_000 if k == "cg_pass_kernel" else None)
    r = bench.roofline_block("cg_pass_kernel", stats, "c2", 6388.0, "measured", capture_share=1.0)
    assert r["bound"] == "hbm" and r["achieved"] == 5000.0 and abs(r["frac"] - 5000.0 / 6388.0) < 1e-4
    assert r["traffic"] == 4_000_000_000
    assert bench.roofline_block("cg_pass_kernel", stats, "c2", 6388.0, "measured", capture_share=0.125)["traffic"] == 500_000_000
    assert bench.roofline_block("cg_pass_kernel", stats, "c2", 6388.0, "measured")["traffic"] is None   # another workload
    assert r["per_kernel"]["scalar kernels"]["GBps"] is None and r["avg_launch_us"] == 1000.0
    monkeypatch.setattr(bench, "ncu_pipe", lambda k, c: {"bound": "fp64", "busy_pct": 41.5, "issue_active_pct": 60.0,
                                                         "capture": "profiles/x.csv"} if (k, c) == ("mh_perpixel_kernel", "c3") else None)
    r = bench.roofline_block("mh_perpixel_kernel", stats, "c3", 6388.0, "measured")
    assert r["bound"] == "fp64" and r["achieved"] == 41.5 and r["peak"] == 100.0 and r["frac"] == 0.415
    assert r["hbm"]["achieved"] == 200.0 and r["avg_launch_us"] == 10000.0
    r = bench.roofline_block("mh_perpixel_kernel", stats, "c4", 6388.0, "measured")
    assert r["bound"] == "hbm"
