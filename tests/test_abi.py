"""CPU-side checks of the drop-in boundary: the shared library builds, loads and exports every
symbol include/dang_gpu.h declares; without a GPU the product path fails loudly."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT, has_gpu


def header_symbols():
    text = open(os.path.join(ROOT, "include", "dang_gpu.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dang_gpu_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from dang_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    lib = C.CDLL(_lib.LIB_PATH)
    syms = header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(lib, s), f"libdang_gpu.so does not export {s}"
    # the ctypes signature table covers exactly the header
    assert sorted(_lib.SIGNATURES) == syms


def test_library_is_sm100a_and_has_no_oracle_dependency():
    from dang_b200 import _lib
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"  # build.sh's default toolkit, off PATH
    out = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    ldd = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in ldd


def test_product_sources_never_reference_the_oracle():
    pkg = os.path.join(ROOT, "dang_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "dang_oracle" not in src, f


@pytest.mark.skipif(has_gpu(), reason="only meaningful without a GPU")
def test_fails_loudly_without_a_gpu():
    from dang_b200.engine import DangGpuError, Engine
    from helpers import small_case
    cfg, sky = small_case(nside=4)
    with pytest.raises(DangGpuError) as ei:
        Engine(cfg, sky)
    assert "no CPU fallback" in str(ei.value) or "CUDA" in str(ei.value)


def test_bandpass_gauss_quadrature_reproduces_the_table_sums():
    """Host-only: the 8-point Gauss rule the library hands to the device instead of a 128-sample bandpass
    (DANG_OPT_BP_QUADRATURE) reproduces the bandpass-integrated power-law and modified-blackbody SEDs of
    evaluate_powerlaw / evaluate_mbb (src/dang_component_mod.f90:909-914, 949-955) to rounding, for every c3 band
    and the extremes of the priors; short, wide or negative-weight tables are refused (the table is kept)."""
    import ctypes as C

    import numpy as np

    from dang_b200 import _lib
    from dang_b200.synth import H_PLANCK, K_B, make_config
    lib = _lib.load()
    dp = lambda a: a.ctypes.data_as(_lib.c_dp)
    cfg = make_config("c3", nside=4)
    worst = 0.0
    for band in cfg.bands:
        nu = np.ascontiguousarray(band.bp_nu_ghz, dtype=np.float64) * 1e9
        tau = np.ascontiguousarray(band.bp_tau, dtype=np.float64)
        tau = tau / tau.sum()
        nq, wq = np.zeros(8), np.zeros(8)
        assert lib.dang_gpu_bandpass_quadrature(band.nu_ghz * 1e9, len(nu), dp(nu), dp(tau), 8, dp(nq), dp(wq)) == 0
        assert abs(wq.sum() - 1.0) < 1e-13 and np.all(wq > 0) and nu.min() < nq.min() and nq.max() < nu.max()
        for beta, T, nu_ref in [(-3.1, None, 30e9), (-2.0, None, 30e9), (-4.0, None, 30e9), (1.55, 19.6, 353e9),
                                (2.2, 10.0, 353e9), (1.0, 35.0, 353e9)]:
            if T is None:
                g = lambda v: (v / nu_ref) ** beta
            else:
                z = H_PLANCK / (K_B * T)
                g = lambda v: (np.exp(z * nu_ref) - 1.0) / (np.exp(z * v) - 1.0) * (v / nu_ref) ** (beta + 1.0)
            full, quad = np.sum(tau * g(nu)), np.sum(wq * g(nq))
            worst = max(worst, abs(full - quad) / abs(full))
    assert worst < 5e-15, worst
    # refused: too few samples for the rule, a negative weight, a band wider than +-0.25 in ln(nu)
    nu = np.linspace(90e9, 110e9, 12)
    tau = np.full(12, 1.0 / 12)
    out = np.zeros(8)
    assert lib.dang_gpu_bandpass_quadrature(100e9, 12, dp(nu), dp(tau), 8, dp(out), dp(out.copy())) == 3
    nu = np.linspace(90e9, 110e9, 64)
    tau = np.full(64, 1.0 / 64)
    tau[5] = -1e-3
    assert lib.dang_gpu_bandpass_quadrature(100e9, 64, dp(nu), dp(tau), 8, dp(out), dp(out.copy())) == 3
    nu = np.linspace(50e9, 150e9, 64)
    tau = np.full(64, 1.0 / 64)
    assert lib.dang_gpu_bandpass_quadrature(100e9, 64, dp(nu), dp(tau), 8, dp(out), dp(out.copy())) == 3


def test_fortran_shim_binds_the_declared_abi():
    """fortran/dang_gpu_mod.f90 cannot be compiled in this image (no Fortran compiler), so at least keep it
    consistent with the header: every name it binds is declared in include/dang_gpu.h, and everything a host
    needs (all but the test / bench instrumentation) is bound."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "dang_gpu.h")).read()
    shim = open(os.path.join(root, "fortran", "dang_gpu_mod.f90")).read()
    declared = set(re.findall(r"\b(dang_gpu_[a-z_0-9]+)\s*\(", header))
    bound = set(re.findall(r"name='(dang_gpu_[a-z_0-9]+)'", shim))
    assert bound <= declared, bound - declared
    instrumentation = {"dang_gpu_cg_trace", "dang_gpu_get_cg_x", "dang_gpu_get_decisions", "dang_gpu_event_record",
                       "dang_gpu_event_elapsed_ms", "dang_gpu_launch_count", "dang_gpu_kernel_stats",
                       "dang_gpu_kernel_name", "dang_gpu_perpixel_stats", "dang_gpu_share_maps",
                       "dang_gpu_bandpass_quadrature", "dang_gpu_timeline", "dang_gpu_comm_probe"}
    assert declared - bound <= instrumentation, (declared - bound) - instrumentation


def test_python_constants_match_the_header_enums():
    """dang_b200/engine.py and config.py mirror the header's enums by value: keep them in step."""
    import os
    import re

    from dang_b200 import config, engine
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "dang_gpu.h")).read()
    enums = {k: int(v) for k, v in re.findall(r"\b(DANG_[A-Z0-9_]+)\s*=\s*(\d+)", header)}
    for name, value in vars(engine).items():
        if name.startswith("OPT_"):
            key = "DANG_" + name
            alias = {"DANG_OPT_RECORD": "DANG_OPT_RECORD_DECISIONS"}
            assert enums[alias.get(key, key)] == value, name
    assert engine.KERNEL_COUNT == enums["DANG_K_COUNT"]
    assert config.COMP_TYPES == {"power-law": enums["DANG_COMP_POWERLAW"], "mbb": enums["DANG_COMP_MBB"],
                                 "freefree": enums["DANG_COMP_FREEFREE"], "lognormal": enums["DANG_COMP_LOGNORMAL"],
                                 "cmb": enums["DANG_COMP_CMB"], "template": enums["DANG_COMP_TEMPLATE"],
                                 "T_cmb": enums["DANG_COMP_T_CMB"], "monopole": enums["DANG_COMP_MONOPOLE"],
                                 "hi_fit": enums["DANG_COMP_HI_FIT"]}
    assert config.LNL_TYPES == {"chisq": enums["DANG_LNL_CHISQ"], "marginal": enums["DANG_LNL_MARGINAL"],
                                "prior": enums["DANG_LNL_PRIOR"]}
    assert config.PRIOR_TYPES == {"uniform": enums["DANG_PRIOR_UNIFORM"], "gaussian": enums["DANG_PRIOR_GAUSSIAN"],
                                  "jeffreys": enums["DANG_PRIOR_JEFFREYS"]}
    assert config.ML_MODES == {"optimize": enums["DANG_ML_OPTIMIZE"], "sample": enums["DANG_ML_SAMPLE"]}
    assert config.INDEX_MODES == {"fullsky": enums["DANG_INDEX_FULLSKY"], "per-pixel": enums["DANG_INDEX_PERPIXEL"]}
