"""Host-side mirror of the reference's Gibbs-loop operators over the C ABI.

`Engine` plays the role of the Fortran host (`dang.f90` + the thin shim in
fortran/dang_gpu_mod.f90): it keeps the run description (RunConfig) as the source of truth,
pushes bands / maps / components / CG groups through include/dang_gpu.h exactly as the shim
does, and exposes the reference's own operator names:

    sample_cg_groups            src/dang_cg_mod.f90:142-177
    sample_spectral_parameters  src/dang_sample_mod.f90:21-86
    sample_index_mh             src/dang_sample_mod.f90:88-485
    update_sky_model            src/dang_data_mod.f90:339-396
    compute_chisq               src/dang_data_mod.f90:494-526

All computation happens in libdang_gpu.so on the GPU; nothing here falls back to numpy.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from .config import (COMP_TYPES, INDEX_MODES, LNL_TYPES, ML_MODES, PRIOR_TYPES, RunConfig,
                     flag_to_map_n, return_poltype_flag)

OPT_FIX_SAMPLE_VECTOR, OPT_CG_TWO_PASS, OPT_FULLSKY_STREAM, OPT_PROFILE, OPT_CG_CHUNK, OPT_RECORD = 1, 2, 3, 4, 5, 6
OPT_PERPIXEL_SERIAL = 7
OPT_CG_CHECKPOINT = 8
OPT_TMA = 9
OPT_STAT_CACHE = 10
OPT_L2_PERSIST_MB = 11
OPT_PERPIXEL_FAST = 12
OPT_PERPIXEL_BP_SERIES = 13
OPT_BP_QUADRATURE = 14
OPT_CG_PERSISTENT = 15
OPT_STREAM_RING = 16
OPT_DEFER_D2H = 17
OPT_DEFER_SCALARS = 18
KERNEL_COUNT = 12
# kinds of dang_gpu_posterior_* (a bit set at posterior_begin, one bit per posterior / posterior_rhat call)
POST_AMPLITUDE, POST_INDICES, POST_CHI_MAP, POST_RESIDUAL, POST_TEMPLATE_AMPLITUDES = 1, 2, 4, 8, 16


class DangGpuError(RuntimeError):
    pass


def _dp(a: Optional[np.ndarray]):
    if a is None:
        return None
    if a.dtype != np.float64 or not a.flags["C_CONTIGUOUS"]:
        raise ValueError("expected a C-contiguous float64 array")
    return a.ctypes.data_as(_lib.c_dp)


def init_bandpass(band) -> Tuple[float, np.ndarray, np.ndarray]:
    """Host part of init_bp_mod / read_bandpass / normalize_bandpass
    (src/dang_bp_mod.f90:19-81,138): nu_c GHz -> Hz if < 1e9, nu0 GHz -> Hz, tau0 / sum(tau0)."""
    nu_c = band.nu_ghz
    if nu_c < 1e9:
        nu_c = nu_c * 1e9
    if band.is_delta:
        return nu_c, np.zeros(0), np.zeros(0)
    nu0 = np.ascontiguousarray(band.bp_nu_ghz, dtype=np.float64) * 1.0e9
    tau = np.ascontiguousarray(band.bp_tau, dtype=np.float64)
    total = 0.0
    for t in tau:  # Fortran sum(): sequential
        total = total + t
    return nu_c, nu0, tau / total


class Engine:
    def __init__(self, cfg: RunConfig, sky, device: int = 0,
                 pix_range: Optional[Tuple[int, int]] = None, share_maps_with: Optional["Engine"] = None):
        self.lib = _lib.load()
        self.cfg = cfg
        self.npix, self.nmaps, self.nbands = cfg.npix, cfg.nmaps, cfg.nbands
        self.lo, self.hi = pix_range if pix_range is not None else (0, cfg.npix)
        self.h = _lib.vp()
        rc = self.lib.dang_gpu_create(device, cfg.nside, cfg.npix, cfg.nmaps, cfg.nbands,
                                      len(cfg.comps), self.lo, self.hi, C.byref(self.h))
        if rc != 0:
            msg = self.lib.dang_gpu_last_error(None).decode()
            self.h = None
            raise DangGpuError(f"dang_gpu_create failed (rc={rc}): {msg}")
        self.nranks, self.rank = 1, 0
        # c%tuned(j) = .not. fg_spec_tune (src/dang_component_mod.f90:177): untuned indices are tuned by the first
        # sample_index_mh that meets them, and the tuner then marks ALL of the component's indices tuned (:711)
        self._tuned = [[not s.tune for s in c.indices] for c in cfg.comps]
        self._n_unmasked = 0
        # init_bp_mod
        for j, b in enumerate(cfg.bands):
            nu_c, nu0, tau0 = init_bandpass(b)
            self._ck(self.lib.dang_gpu_set_band(self.h, j, nu_c, len(nu0), _dp(nu0) if len(nu0) else None,
                                                _dp(tau0) if len(tau0) else None))
        # initialize_data_module (an ensemble member borrows the owner's device maps instead)
        self._owner = share_maps_with
        if share_maps_with is None:
            self.upload_maps(sky)
        else:
            self._ck(self.lib.dang_gpu_share_maps(self.h, share_maps_with.h))
        # initialize_components
        for ic, c in enumerate(cfg.comps):
            nu_ref = c.nu_ref_ghz * 1e9 if c.nu_ref_ghz < 1e7 else c.nu_ref_ghz  # dang_param_mod.f90:571-573
            if c.type in ("template", "monopole", "hi_fit"):
                # c%template ('template': already divided by temp_norm; 'monopole': the constructor's own map),
                # c%template_amplitudes(nbands,nmaps), c%corr, c%nfit; hi_fit also carries its T_d index map
                idx = np.ascontiguousarray(sky.indices[c.label], dtype=np.float64) if c.type == "hi_fit" else None
                self._ck(self.lib.dang_gpu_set_component(self.h, ic, COMP_TYPES[c.type], c.label.encode(), nu_ref,
                                                         c.cg_group, int(c.amp_sample), None, _dp(idx)))
                corr = (C.c_int * cfg.nbands)(*[int(bool(v)) for v in c.corr])
                tmap = None if c.type == "monopole" else np.ascontiguousarray(sky.template[c.label], dtype=np.float64)
                tamp = np.ascontiguousarray(sky.template_amplitudes[c.label], dtype=np.float64)
                self._ck(self.lib.dang_gpu_set_template(self.h, ic, _dp(tmap), _dp(tamp), corr, int(sum(map(bool, c.corr)))))
                if c.type != "hi_fit":
                    continue
                self._set_indices_spec(ic, c)
                continue
            amp = np.ascontiguousarray(sky.amplitude[c.label], dtype=np.float64)
            idx = np.ascontiguousarray(sky.indices[c.label], dtype=np.float64)
            self._ck(self.lib.dang_gpu_set_component(self.h, ic, COMP_TYPES[c.type], c.label.encode(), nu_ref,
                                                     c.cg_group, int(c.amp_sample), _dp(amp), _dp(idx)))
            self._set_indices_spec(ic, c)
        # initialize_cg_groups
        for ig, g in enumerate(cfg.cg_groups):
            flags = return_poltype_flag(g.poltype)
            fl = (C.c_int * len(flags))(*flags)
            self._ck(self.lib.dang_gpu_set_cg_group(self.h, ig + 1, g.max_iter, g.converge, fl, len(flags)))

    def _set_indices_spec(self, ic: int, c):
        for k, s in enumerate(c.indices):
            flags = return_poltype_flag(s.poltype)
            fl = (C.c_int * max(len(flags), 1))(*flags)
            g = np.asarray(s.gauss, dtype=np.float64)
            u = np.asarray(s.uni, dtype=np.float64)
            self._ck(self.lib.dang_gpu_set_index(self.h, ic, k, int(s.sample), INDEX_MODES[s.region],
                                                 LNL_TYPES[s.lnl_type], PRIOR_TYPES[s.prior], _dp(g), _dp(u),
                                                 s.step, s.samp_nside or self.cfg.nside, fl, len(flags)))

    # ------------------------------------------------------------------ plumbing
    def _ck(self, rc: int):
        if rc != 0:
            raise DangGpuError(f"libdang_gpu rc={rc}: {self.lib.dang_gpu_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.dang_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, opt: int, value: float):
        self._ck(self.lib.dang_gpu_set_option(self.h, opt, float(value)))

    def comm_init(self, nranks: int, rank: int, uid: bytes):
        self._ck(self.lib.dang_gpu_comm_init(self.h, nranks, rank, uid))
        self.nranks, self.rank = nranks, rank

    def comm_ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self.lib.dang_gpu_comm_ipc_handle(self.h, buf))
        return buf.raw

    def comm_open_peers(self, handles: bytes):
        """handles: the nranks 64-byte IPC handles, rank-major; enables the NVLink mailbox path."""
        self._ck(self.lib.dang_gpu_comm_open_peers(self.h, handles))

    def comm_check(self):
        self._ck(self.lib.dang_gpu_comm_check(self.h))

    def upload_maps(self, sky):
        """ddata%sig_map / rms_map / masks / gain / offset -> device (also after swap_cg_maps)."""
        self._ck(self.lib.dang_gpu_upload_maps(self.h, _dp(sky.sig), _dp(sky.rms), _dp(sky.mask),
                                               _dp(np.ascontiguousarray(sky.gain, dtype=np.float64)),
                                               _dp(np.ascontiguousarray(sky.offset, dtype=np.float64))))

    # ------------------------------------------------------------------ state access
    def amplitude(self, ic: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        out = np.zeros((self.nmaps, self.npix)) if out is None else out
        self._ck(self.lib.dang_gpu_get_amplitude(self.h, ic, _dp(out)))
        return out

    def indices(self, ic: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        nind = len(self.cfg.comps[ic].indices)
        out = np.zeros((nind, self.nmaps, self.npix)) if out is None else out
        self._ck(self.lib.dang_gpu_get_indices(self.h, ic, _dp(out)))
        return out

    # asynchronous staging (copies overlap later calls; host arrays should be pinned)
    def amplitude_async(self, ic: int, out: np.ndarray, k_lo: int = 2, k_hi: int = 3):
        self._ck(self.lib.dang_gpu_get_amplitude_async(self.h, ic, k_lo, k_hi, _dp(out)))

    def indices_async(self, ic: int, nind: int, out: np.ndarray, k_lo: int = 2, k_hi: int = 3):
        self._ck(self.lib.dang_gpu_get_indices_async(self.h, ic, nind, k_lo, k_hi, _dp(out)))

    def download_wait(self):
        self._ck(self.lib.dang_gpu_download_wait(self.h))

    def stage_eta(self, eta: np.ndarray, nplanes: int = 2):
        """Upload the next cg_solve's normals in the background; call that solve with eta=None."""
        self._ck(self.lib.dang_gpu_stage_eta(self.h, _dp(eta), nplanes))

    def template_amplitudes(self, ic: int) -> np.ndarray:
        """c%template_amplitudes as [plane][band] (Fortran (nbands, nmaps))."""
        out = np.zeros((self.nmaps, self.nbands))
        self._ck(self.lib.dang_gpu_get_template_amplitudes(self.h, ic, _dp(out)))
        return out

    def index_fullsky(self, ic: int, nind: int, map_n: int) -> float:
        """The value the whole plane holds after a full-sky draw (8 bytes instead of a map download)."""
        v = C.c_double()
        self._ck(self.lib.dang_gpu_get_index_fullsky(self.h, ic, nind, map_n, C.byref(v)))
        return v.value

    def set_t_cmb(self, t_cmb: float):
        """The module-global T_CMB (src/dang_util_mod.f90:15), which a 'T_cmb' component overwrites after its draw."""
        self._ck(self.lib.dang_gpu_set_t_cmb(self.h, float(t_cmb)))

    def _bcast_t_cmb(self, ic: int) -> float:
        # a full-sky draw leaves the same value on every rank; a rank that does not own pixel 0 reads its own first pixel
        return float(self.indices(ic)[0, 0, self.lo])

    def set_amplitude(self, ic: int, amp: np.ndarray):
        self._ck(self.lib.dang_gpu_set_amplitude(self.h, ic, _dp(np.ascontiguousarray(amp, dtype=np.float64))))

    def set_indices(self, ic: int, idx: np.ndarray):
        self._ck(self.lib.dang_gpu_set_indices(self.h, ic, _dp(np.ascontiguousarray(idx, dtype=np.float64))))

    def cg_x(self, ig: int = 0, flag_n: int = 0) -> np.ndarray:
        g = self.cfg.cg_groups[ig]
        S = 2 if return_poltype_flag(g.poltype)[flag_n] & 8 else 1
        ncg = sum(1 for c in self.cfg.comps if c.cg_group == ig + 1 and c.amp_sample)
        out = np.zeros((ncg * S, self.npix))
        self._ck(self.lib.dang_gpu_get_cg_x(self.h, ig + 1, flag_n, _dp(out)))
        return out.reshape(-1)

    # ------------------------------------------------------------------ operators
    def cg_solve(self, ig: int = 0, flag_n: int = 0, ml_mode: str = "sample",
                 eta: Optional[np.ndarray] = None, seed: int = 0) -> Tuple[int, float]:
        """compute_rhs + cg_search + unpack_amplitudes for one (group, flag)."""
        n_iter = C.c_int()
        delta = C.c_double()
        e = None if eta is None else np.ascontiguousarray(eta, dtype=np.float64)
        self._ck(self.lib.dang_gpu_cg_solve(self.h, ig + 1, flag_n, ML_MODES[ml_mode], _dp(e), seed,
                                            C.byref(n_iter), C.byref(delta)))
        return n_iter.value, delta.value

    def cg_trace(self) -> np.ndarray:
        buf = np.zeros(256)
        n = C.c_int()
        self._ck(self.lib.dang_gpu_cg_trace(self.h, _dp(buf), 256, C.byref(n)))
        return buf[: n.value].copy()

    def sample_cg_groups(self, ml_mode: Optional[str] = None, eta: Optional[np.ndarray] = None,
                         seed: int = 0, stats: bool = True):
        """sample_cg_groups: per sampled group, per flag: rhs -> CG -> unpack; then the chi-square
        print of write_stats_to_term.  `eta` holds the normals of all solves back to back."""
        ml_mode = ml_mode or self.cfg.ml_mode
        out = []
        off = 0
        for ig, g in enumerate(self.cfg.cg_groups):
            if not g.sample:
                continue
            flags = return_poltype_flag(g.poltype)
            for f, flag in enumerate(flags):
                m = (2 if flag & 8 else 1) * self.npix
                e = None if eta is None else eta[off: off + m]
                off += m
                out.append(self.cg_solve(ig, f, ml_mode, e, seed + 1000003 * (ig * 3 + f)))
            if stats:
                out.append(self.compute_chisq())
        return out

    def sample_index_mh(self, ic: int, nind: int, map_n: int, nsample: Optional[int] = None,
                        ml_mode: Optional[str] = None, z: Optional[np.ndarray] = None,
                        u: Optional[np.ndarray] = None, seed: int = 0) -> float:
        nsample = self.cfg.nsample if nsample is None else nsample
        ml_mode = ml_mode or self.cfg.ml_mode
        acc = C.c_double()
        zz = None if z is None else np.ascontiguousarray(z, dtype=np.float64)
        uu = None if u is None else np.ascontiguousarray(u, dtype=np.float64)
        self._ck(self.lib.dang_gpu_sample_index(self.h, ic, nind, map_n, nsample, ML_MODES[ml_mode],
                                                _dp(zz), _dp(uu), seed, C.byref(acc)))
        return acc.value

    def perpixel_stats(self) -> Tuple[float, float]:
        """(fp64 fallbacks, bound violations) of the last per-pixel draw's fp32 screening."""
        f, v = C.c_double(), C.c_double()
        self._ck(self.lib.dang_gpu_perpixel_stats(self.h, C.byref(f), C.byref(v)))
        return f.value, v.value

    def tune_index(self, ic: int, nind: int, map_n: int, nsample: Optional[int] = None,
                   ml_mode: Optional[str] = None, z: Optional[np.ndarray] = None,
                   u: Optional[np.ndarray] = None, seed: int = 0, max_blocks: int = 20) -> Tuple[int, float]:
        """tune_spectral_parameter_length (src/dang_sample_mod.f90:623-717): returns
        (blocks run, tuned step size); the step is stored in the component for later draws."""
        nsample = self.cfg.nsample if nsample is None else nsample
        ml_mode = ml_mode or self.cfg.ml_mode
        zz = None if z is None else np.ascontiguousarray(z, dtype=np.float64)
        uu = None if u is None else np.ascontiguousarray(u, dtype=np.float64)
        nb, step = C.c_int(), C.c_double()
        self._ck(self.lib.dang_gpu_tune_index(self.h, ic, nind, map_n, nsample, ML_MODES[ml_mode], _dp(zz),
                                              _dp(uu), seed, max_blocks, C.byref(nb), C.byref(step)))
        return nb.value, step.value

    def sample_spectral_parameters(self, nsample: Optional[int] = None, ml_mode: Optional[str] = None,
                                   z: Optional[np.ndarray] = None, u: Optional[np.ndarray] = None,
                                   seed: int = 0, stats: bool = True):
        """sample_spectral_parameters: components -> indices -> pol flags, in reference order.
        Deviate arrays are consumed call by call with stride nsample*npix (as the oracle does);
        alternatively `z` / `u` may be lists holding one array per sample_index_mh call."""
        nsample = self.cfg.nsample if nsample is None else nsample
        stride = nsample * self.npix
        per_call = isinstance(z, (list, tuple))
        ncall, sampled, acc = 0, False, []
        for ic, c in enumerate(self.cfg.comps):
            if not c.indices or not any(s.sample for s in c.indices):
                continue
            sampled = True
            for j, s in enumerate(c.indices):
                if not s.sample:
                    continue
                for flag in return_poltype_flag(s.poltype):
                    if per_call:
                        zz, uu = z[ncall], (None if u is None else u[ncall])
                    else:
                        zz = None if z is None else z[stride * ncall: stride * (ncall + 1)]
                        uu = None if u is None else u[stride * ncall: stride * (ncall + 1)]
                    if not self._tuned[ic][j] and s.lnl_type != "prior":
                        # sample_index_mh: `if (.not. c%tuned(nind))` -> tune_spectral_parameter_length first
                        # (src/dang_sample_mod.f90:270-273 full sky, :341-347 per pixel); device deviates
                        self.tune_index(ic, j, flag_to_map_n(flag), nsample, ml_mode, seed=seed + 104729 * (ncall + 1),
                                        max_blocks=1000)
                        self._tuned[ic] = [True] * len(c.indices)
                    acc.append(self.sample_index_mh(ic, j, flag_to_map_n(flag), nsample, ml_mode, zz, uu,
                                                    seed + 7919 * ncall))
                    ncall += 1
            if c.type == "T_cmb":  # :76-78: T_CMB = c%indices(0,1,1)
                self.set_t_cmb(float(self.indices(ic)[0, 0, self.lo]) if self.rank == 0 else self._bcast_t_cmb(ic))
        chisq = self.compute_chisq() if (sampled and stats) else None
        return acc, chisq

    def decisions(self, nsample: int, fullsky: bool):
        n = nsample if fullsky else nsample * self.npix
        dec = np.full(n, 255, dtype=np.uint8)
        lnl = np.full(n, np.nan)
        self._ck(self.lib.dang_gpu_get_decisions(self.h, dec.ctypes.data_as(C.POINTER(C.c_ubyte)), _dp(lnl)))
        return dec, lnl

    def chisq_planes(self) -> Tuple[np.ndarray, int]:
        planes = np.zeros(self.nmaps)
        n = C.c_int64()
        lo, hi = self.cfg.pol_type
        self._ck(self.lib.dang_gpu_chisq(self.h, lo, hi, _dp(planes), C.byref(n)))
        self._n_unmasked = n.value
        return planes, n.value

    def compute_chisq(self) -> float:
        """compute_chisq: sum(chi_map)/nump with nump = nmaps * #unmasked (SURVEY Q9 convention)."""
        planes, n = self.chisq_planes()
        total = 0.0
        for k in range(self.nmaps):
            total = total + planes[k]
        return total / float(self.nmaps * n)

    def update_sky_model(self):
        """update_sky_model (+ chi_map): downloads sky_model, res_map, chi_map for this handle's pixels."""
        sky = np.zeros((self.nbands, self.nmaps, self.npix))
        res = np.zeros((self.nbands, self.nmaps, self.npix))
        chi = np.zeros((self.nmaps, self.npix))
        lo, hi = self.cfg.pol_type
        self._ck(self.lib.dang_gpu_get_sky_model(self.h, lo, hi, _dp(sky), _dp(res), _dp(chi)))
        return sky, res, chi

    def fit_band_gain(self, map_n: int, band: int, ml_mode: Optional[str] = None, z: Optional[float] = None,
                      seed: int = 0) -> float:
        """fit_band_gain (src/dang_sample_mod.f90:570-621); the new gain stays in the handle."""
        ml_mode = ml_mode or self.cfg.ml_mode
        g = C.c_double()
        zz = None if z is None else C.byref(C.c_double(z))
        self._ck(self.lib.dang_gpu_fit_band_gain(self.h, map_n, band, ML_MODES[ml_mode], zz, seed, C.byref(g)))
        return g.value

    def udgrade(self, kind: str, data: np.ndarray, nside_in: int, nside_out: int, threshold: float = 0.5) -> np.ndarray:
        """udgrade_ring / udgrade_rms / udgrade_mask (HEALPix udgrade_nr; src/dang_util_mod.f90:341-376) on full-sky
        RING maps [nmaps][npix] -- the resolution changes of sample_index_mh's low-resolution branch."""
        data = np.ascontiguousarray(data, dtype=np.float64)
        out = np.zeros((data.shape[0], 12 * nside_out * nside_out))
        self._ck(self.lib.dang_gpu_udgrade(self.h, {"ring": 0, "rms": 1, "mask": 2}[kind], _dp(data), nside_in, _dp(out),
                                           nside_out, data.shape[0], float(threshold)))
        return out

    def index_mean(self, ic: int, nind: int, map_n: int) -> float:
        m = C.c_double()
        self._ck(self.lib.dang_gpu_index_mean(self.h, ic, nind, map_n, C.byref(m)))
        return m.value

    def gibbs_iteration(self, it: int, eta=None, z=None, u=None, seed: int = 0):
        """Loop body of src/dang.f90:87-126 restricted to the hot path: sample_cg_groups, then
        (iter > 1) sample_spectral_parameters.  Returns the chi-square after each block."""
        r1 = self.sample_cg_groups(eta=eta, seed=seed + 2 * it)
        r2 = None
        if it > 1:
            r2 = self.sample_spectral_parameters(z=z, u=u, seed=seed + 2 * it + 1)
        return r1, r2

    # ------------------------------------------------------------------ deferred scalars (OPT_DEFER_SCALARS)
    def iteration_mark(self) -> int:
        """Snapshot the results the deferred calls since the last mark left on the device; returns a ticket."""
        t = C.c_int64()
        self._ck(self.lib.dang_gpu_iteration_mark(self.h, C.byref(t)))
        return t.value

    def iteration_scalars(self, ticket: int) -> dict:
        """The terminal line of src/dang.f90:100-104 for the iteration a ticket closed: waits for that snapshot only."""
        n_iter, delta, acc, val = C.c_int(), C.c_double(), C.c_double(), C.c_double()
        chi_a, chi_i = np.zeros(self.cfg.nmaps), np.zeros(self.cfg.nmaps)
        self._ck(self.lib.dang_gpu_iteration_scalars(self.h, ticket, C.byref(n_iter), C.byref(delta), _dp(chi_a), C.byref(acc),
                                                     C.byref(val), _dp(chi_i)))
        def total(planes):  # compute_chisq's normalisation
            t = 0.0
            for k in range(self.nmaps):
                t = t + planes[k]
            return t / float(self.nmaps * self._n_unmasked) if self._n_unmasked else float("nan")

        return dict(n_iter=n_iter.value, delta=delta.value, chisq_after_amplitudes=chi_a, accept=acc.value,
                    index_value=val.value, chisq_after_index=chi_i, chisq_amplitudes=total(chi_a), chisq_index=total(chi_i))

    # ------------------------------------------------------------------ posterior summaries (not in the reference)
    def posterior_begin(self, what: int, pol_lo: Optional[int] = None, pol_hi: Optional[int] = None,
                        batch_len: int = 0):
        """Zero running moments of the POST_* kinds in `what`; CHI_MAP / RESIDUAL are those of update_sky_model over
        pol_lo..pol_hi (default cfg.pol_type).  The caller decides burn-in and thinning by when it accumulates.
        batch_len > 0 also keeps batch means of batch_len consecutive samples, for posterior_ess; 0: none."""
        lo, hi = self.cfg.pol_type
        lo, hi = lo if pol_lo is None else pol_lo, hi if pol_hi is None else pol_hi
        if batch_len:
            self._ck(self.lib.dang_gpu_posterior_begin_batched(self.h, int(what), lo, hi, int(batch_len)))
        else:
            self._ck(self.lib.dang_gpu_posterior_begin(self.h, int(what), lo, hi))

    def posterior_accumulate(self):
        """Add the current state as one sample (stream ordered, no host wait)."""
        self._ck(self.lib.dang_gpu_posterior_accumulate(self.h))

    def _posterior_shape(self, kind: int):
        if kind == POST_RESIDUAL:
            return (self.nbands, self.nmaps, self.npix)
        if kind == POST_TEMPLATE_AMPLITUDES:
            return (self.nmaps, self.nbands)
        return (self.nmaps, self.npix)

    def posterior(self, kind: int, ic: int = 0, nind: int = 0) -> Tuple[np.ndarray, np.ndarray, int]:
        """(mean, std, n) in the shapes of amplitude / indices(ic)[nind] / update_sky_model / template_amplitudes;
        std is NaN while n < 2.  Only this handle's pixels are written (the rest stay 0)."""
        mean, std = np.zeros(self._posterior_shape(kind)), np.zeros(self._posterior_shape(kind))
        n = C.c_int64()
        self._ck(self.lib.dang_gpu_posterior_get(self.h, int(kind), ic, nind, _dp(mean), _dp(std), C.byref(n)))
        return mean, std, n.value

    def posterior_end(self):
        self._ck(self.lib.dang_gpu_posterior_end(self.h))

    # ------------------------------------------------------------------ instrumentation
    def sync(self):
        self._ck(self.lib.dang_gpu_sync(self.h))

    def event_record(self, slot: int):
        self._ck(self.lib.dang_gpu_event_record(self.h, slot))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        self._ck(self.lib.dang_gpu_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def launch_count(self, reset: bool = False) -> int:
        n = C.c_int64()
        self._ck(self.lib.dang_gpu_launch_count(self.h, C.byref(n), int(reset)))
        return n.value

    def kernel_stats(self, reset: bool = False):
        out = {}
        for k in range(KERNEL_COUNT):
            n, ms, by = C.c_int64(), C.c_double(), C.c_double()
            self._ck(self.lib.dang_gpu_kernel_stats(self.h, k, C.byref(n), C.byref(ms), C.byref(by), int(reset)))
            out[self.lib.dang_gpu_kernel_name(k).decode()] = dict(launches=n.value, ms=ms.value, bytes=by.value)
        return out


def posterior_rhat(engines: Sequence[Engine], kind: int, ic: int = 0, nind: int = 0) -> np.ndarray:
    """Gelman-Rubin R-hat per element across chains (one Engine each, same device and pixel range, same samples
    accumulated), in the shape of Engine.posterior."""
    lib = _lib.load()
    hs = (_lib.vp * len(engines))(*[e.h for e in engines])
    out = np.zeros(engines[0]._posterior_shape(kind))
    rc = lib.dang_gpu_posterior_rhat(hs, len(engines), int(kind), ic, nind, _dp(out))
    if rc != 0:
        raise DangGpuError(f"dang_gpu_posterior_rhat rc={rc}: {lib.dang_gpu_last_error(engines[0].h).decode()}")
    return out


def posterior_ess(engines: Sequence[Engine], kind: int, ic: int = 0, nind: int = 0) -> Tuple[np.ndarray, np.ndarray]:
    """(ess, mcse): batch-means effective sample size and Monte Carlo standard error of the posterior mean per
    element, of one chain or pooled over several (one Engine each, begun with the same batch_len, same device and
    pixel range, same samples accumulated), in the shape of Engine.posterior."""
    lib = _lib.load()
    hs = (_lib.vp * len(engines))(*[e.h for e in engines])
    ess, mcse = np.zeros(engines[0]._posterior_shape(kind)), np.zeros(engines[0]._posterior_shape(kind))
    rc = lib.dang_gpu_posterior_ess(hs, len(engines), int(kind), ic, nind, _dp(ess), _dp(mcse))
    if rc != 0:
        raise DangGpuError(f"dang_gpu_posterior_ess rc={rc}: {lib.dang_gpu_last_error(engines[0].h).decode()}")
    return ess, mcse


def setup_torch_comm(eng: "Engine", mailboxes: bool = True):
    """Wire an Engine into an initialised torch.distributed NCCL process group (one process per
    GPU): broadcast the NCCL unique id, then (optionally) all-gather the CUDA-IPC mailbox handles
    for the NVLink scalar-exchange path.  torch.distributed is plumbing only."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(), dist.get_rank()
    if world == 1:
        return
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.frombuffer(bytearray(comm_unique_id()), dtype=torch.uint8).cuda()
    dist.broadcast(uid, 0)
    eng.comm_init(world, rank, uid.cpu().numpy().tobytes())
    if mailboxes:
        mine = torch.frombuffer(bytearray(eng.comm_ipc_handle()), dtype=torch.uint8).cuda()
        allh = [torch.zeros(64, dtype=torch.uint8, device="cuda") for _ in range(world)]
        dist.all_gather(allh, mine)
        eng.comm_open_peers(b"".join(t.cpu().numpy().tobytes() for t in allh))
        dist.barrier()


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = _lib.load().dang_gpu_comm_unique_id(buf)
    if rc != 0:
        raise DangGpuError(f"dang_gpu_comm_unique_id rc={rc}: {_lib.load().dang_gpu_last_error(None).decode()}")
    return buf.raw
