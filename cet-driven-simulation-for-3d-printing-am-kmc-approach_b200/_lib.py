"""ctypes binding of libcetkmc.so (include/cetkmc.h) — the only way the host side reaches
the GPU.  There is no CPU fallback: if the library or a CUDA device is missing every compute
call raises.

`Context` owns one lattice (or one slab of it) resident in HBM.  The drop-in modules
(`thermal_solver`, `kmc_event_rates`, `kmc_simulation`) are thin layers over it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcetkmc.so")

EV_NAMES = (b"dep", b"diff", b"nuc", b"att")      # cetkmc.h CET_EV_* order


class RateParams(C.Structure):                      # cet_rate_params
    _fields_ = [("nu", C.c_double), ("nu_dep", C.c_double),
                ("E_b", C.c_double * 3), ("E_diff", C.c_double * 3),
                ("kT", C.c_double), ("T_melt", C.c_double), ("i0", C.c_double),
                ("delta_T_c", C.c_double), ("k_nuc", C.c_double), ("beta_imp_nuc", C.c_double),
                ("max_imp_fraction", C.c_double), ("rate_threshold", C.c_double),
                ("anisotropy", C.c_double), ("impurity_re", C.c_double), ("impurity_c", C.c_double),
                ("states_w", C.c_int32), ("states_re", C.c_int32), ("states_c", C.c_int32),
                ("defect_id", C.c_int32)]


class ThermalParams(C.Structure):                   # cet_thermal_params
    _fields_ = [("dt_alpha", C.c_double), ("inv_dx2", C.c_double), ("lo", C.c_double),
                ("hi", C.c_double), ("nan_value", C.c_double),
                ("nan_to_num", C.c_int32), ("pad_", C.c_int32)]


class ThermalFullParams(C.Structure):               # cet_thermal_full_params
    _fields_ = [("dt", C.c_double), ("alpha", C.c_double), ("inv_dx2", C.c_double),
                ("rho_cp", C.c_double), ("latent_over_cp", C.c_double), ("lo", C.c_double),
                ("hi", C.c_double)]


class KmcResult(C.Structure):                       # cet_kmc_result
    _fields_ = [("steps_done", C.c_int64), ("py_used", C.c_int64), ("np_used", C.c_int64),
                ("sp_used", C.c_int64), ("nucleation_count", C.c_int64),
                ("fallback_last", C.c_int64), ("total_time", C.c_double),
                ("last_total_rate", C.c_double), ("terminated", C.c_int32), ("starved", C.c_int32)]


class SweepParams(C.Structure):                     # cet_sweep_params
    _fields_ = [("seed", C.c_uint64), ("events_per_sweep", C.c_double), ("p_max", C.c_double),
                ("defect_fraction", C.c_double), ("thermal_every", C.c_int32), ("pad_", C.c_int32)]


class SweepResult(C.Structure):                     # cet_sweep_result
    _fields_ = [("sweeps_done", C.c_int64), ("events_fired", C.c_int64),
                ("events_applied", C.c_int64), ("nucleation_count", C.c_int64),
                ("sweep_index", C.c_int64), ("time", C.c_double), ("last_total_rate", C.c_double),
                ("last_max_rate", C.c_double), ("last_tau", C.c_double),
                ("terminated", C.c_int32), ("overflow", C.c_int32), ("sites_refreshed", C.c_int64)]


class InitDesc(C.Structure):                        # cet_init_desc
    _fields_ = [("n_nuclei", C.c_int64), ("site", C.c_void_p), ("byte", C.c_void_p), ("theta", C.c_void_p),
                ("phi", C.c_void_p), ("T_row", C.c_void_p)]


class MetricsParams(C.Structure):                   # cet_metrics_params
    _fields_ = [("theta_threshold", C.c_double), ("ar_threshold", C.c_double), ("pct_pos", C.c_int64 * 4),
                ("refresh", C.c_int32), ("carbon_id", C.c_int32), ("epoch", C.c_uint32), ("pad_", C.c_int32),
                ("seed", C.c_uint64), ("prob_base", C.c_double), ("e_mig", C.c_double), ("kT", C.c_double),
                ("T_default", C.c_double)]


class MetricsResult(C.Structure):                   # cet_metrics_result
    _fields_ = [("counts", C.c_int64 * 16), ("n_carbon", C.c_int64), ("n_defects", C.c_int64),
                ("n_grains", C.c_int64), ("size_sum", C.c_int64), ("n_equiaxed", C.c_int64),
                ("pct_index", C.c_int64 * 4), ("ar_sum", C.c_double)]


_lib = None
_lock = threading.Lock()

_VP, _I64, _I32, _F64 = C.c_void_p, C.c_int64, C.c_int32, C.c_double

# name -> argtypes; every function returns int except cet_last_error / cet_abi_version
SIGNATURES = {
    "cet_device_count": [C.POINTER(C.c_int)],
    "cet_device_name": [C.c_int, C.c_char_p, C.c_int],
    "cet_create": [C.POINTER(_VP), C.c_int, _I64, _I64, _I64, _I32],
    "cet_create_slab": [C.POINTER(_VP), C.c_int, _I64, _I64, _I64, _I64, _I32],
    "cet_create_shape": [C.POINTER(_VP), C.c_int, _I64, _I64, _I64],
    "cet_destroy": [_VP],
    "cet_sync": [_VP],
    "cet_set_rate_params": [_VP, C.POINTER(RateParams)],
    "cet_upload": [_VP, _VP, _VP, _VP, _VP, _VP],
    "cet_download": [_VP, _VP, _VP, _VP, _VP, _VP],
    "cet_upload_prev_state": [_VP, _VP],
    "cet_snapshot_state": [_VP],
    "cet_upload_packed": [_VP, _VP],
    "cet_download_packed": [_VP, _VP],
    "cet_device_ptr": [_VP, C.c_int, C.POINTER(_VP), C.POINTER(_I64)],
    "cet_counts": [_VP, C.POINTER(_I64 * 16)],
    "cet_thermal_cet": [_VP, C.POINTER(ThermalParams)],
    "cet_thermal_full": [_VP, C.POINTER(ThermalFullParams), _VP],
    "cet_thermal_full_group": [C.POINTER(_VP), _I32, C.POINTER(ThermalFullParams), C.POINTER(_VP), _I32],
    "cet_thermal_fill_gradient": [_VP, _F64, _F64],
    "cet_rates_build": [_VP],
    "cet_rates_total": [_VP, C.POINTER(_F64), C.POINTER(_I64)],
    "cet_rates_download": [_VP, _VP, _VP],
    "cet_events_count": [_VP, C.POINTER(_I64), C.POINTER(_I64)],
    "cet_events_export": [_VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP, C.POINTER(_I64)],
    "cet_kmc_run": [_VP, _I64, _I64, _F64, C.POINTER(ThermalParams), _I32, _VP, _I64, _VP, _I64,
                    _VP, _I64, _F64, C.POINTER(KmcResult), _VP, _VP, _VP, _VP, _VP, _VP],
    "cet_sweep_reset": [_VP],
    "cet_sweep_get_state": [_VP, C.POINTER(_I64), C.POINTER(_F64), C.POINTER(_F64)],
    "cet_sweep_set_state": [_VP, _I64, _F64, _F64],
    "cet_sweep_run": [_VP, _I64, C.POINTER(SweepParams), C.POINTER(ThermalParams),
                      C.POINTER(SweepResult)],
    "cet_sweep_run_group": [C.POINTER(_VP), _I32, _I64, C.POINTER(SweepParams), C.POINTER(ThermalParams),
                            C.POINTER(SweepResult)],
    "cet_comm_unique_id": [_VP],
    "cet_comm_init": [_VP, _VP, C.c_int, C.c_int],
    "cet_comm_destroy": [_VP],
    "cet_halo_exchange": [_VP, C.c_int],
    "cet_allreduce_f64": [_VP, _VP, C.c_int, C.c_int],
    "cet_defects_refresh": [_VP, _VP, _I64, C.c_uint64, C.c_uint32, _F64, _F64, _F64, _F64, _I32, _I32, _I32,
                            C.POINTER(_I64), C.POINTER(_I64)],
    "cet_grains_label": [_VP, _F64, C.POINTER(_I64)],
    "cet_grains_label_ex": [_VP, _F64, C.c_int, C.POINTER(_I64)],
    "cet_grains_stats": [_VP, _I64, _VP, _VP, _VP, _VP],
    "cet_grains_download_labels": [_VP, _VP],
    "cet_grains_download_planes": [_VP, _I64, _I64, _VP],
    "cet_init_group": [C.POINTER(_VP), _I32, C.POINTER(InitDesc), _I32],
    "cet_counts_group": [C.POINTER(_VP), _I32, C.POINTER(_I64)],
    "cet_metrics_group": [C.POINTER(_VP), _I32, C.POINTER(MetricsParams), C.POINTER(_VP), C.POINTER(_I64),
                          C.POINTER(MetricsResult)],
    "cet_grain_profile_group": [C.POINTER(_VP), _I32, _I32, _F64, C.POINTER(_I64)],
    "cet_debug_nst_mismatches": [_VP, C.POINTER(_I64)],
    "cet_debug_flags": [_VP, C.c_int],
    "cet_profile_enable": [_VP, C.c_int],
    "cet_profile_read": [_VP, C.c_int, C.POINTER(_F64), C.POINTER(_I64), C.c_int],
    "cet_timer_begin": [_VP],
    "cet_timer_end_ms": [_VP, C.POINTER(C.c_float)],
}


def build(force: bool = False) -> str:
    """Compile libcetkmc.so in-tree with nvcc for sm_100a (see Makefile)."""
    args = ["make", "-C", _HERE, "-j8"]
    if force:
        args.append("-B")
    subprocess.run(args, check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build the CUDA library first (python -c 'import "
                "__graft_entry__ as g; g.build()' or `make` in the package directory). "
                "There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.cet_last_error.restype = C.c_char_p
        L.cet_last_error.argtypes = []
        L.cet_abi_version.restype = C.c_int
        L.cet_abi_version.argtypes = []
        for name, argtypes in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        _lib = L
        return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().cet_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libcetkmc {what} failed (code {rc}): {msg}")


def device_count() -> int:
    n = C.c_int(0)
    check(lib().cet_device_count(C.byref(n)), "cet_device_count")
    return n.value


def require_gpu():
    if device_count() < 1:
        raise RuntimeError("no CUDA device visible: the cetkmc B200 path has no CPU fallback")


def _arr(a, dtype):
    """C-contiguous array of exactly `dtype` (copy only when needed); None passes through."""
    if a is None:
        return None
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One lattice (or one slab of planes [i_begin, i_end) with `halo` ghost planes per side)
    resident on one GPU."""

    def __init__(self, L=None, shape=None, device=0, i_begin=0, i_end=None, halo=0, n0=None):
        """L: edge length (cubic lattice, the reference's case).  n0: number of planes along axis 0
        when it differs from L (stacked slabs for multi-GPU weak scaling).  shape: thermal-only
        context of arbitrary (n0, n1, n2)."""
        self._h = C.c_void_p(None)
        l = lib()
        if shape is not None and (L is None):
            n0, n1, n2 = (int(x) for x in shape)
            if n0 == n1 == n2:
                check(l.cet_create(C.byref(self._h), device, n0, 0, n0, 0), "cet_create")
            else:
                check(l.cet_create_shape(C.byref(self._h), device, n0, n1, n2), "cet_create_shape")
            self.shape = (n0, n1, n2)
            self.i_begin, self.i_end, self.halo = 0, n0, 0
        else:
            L = int(L)
            n0 = L if n0 is None else int(n0)
            i_end = n0 if i_end is None else int(i_end)
            check(l.cet_create_slab(C.byref(self._h), device, n0, L, int(i_begin), i_end, int(halo)),
                  "cet_create_slab")
            self.shape = (n0, L, L)
            self.i_begin, self.i_end, self.halo = int(i_begin), i_end, int(halo)
        self.device = device
        self.n0 = self.shape[0]
        self.rank, self.world = 0, 1
        self.owned_shape = (self.i_end - self.i_begin, self.shape[1], self.shape[2])

    # -- life cycle -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().cet_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def sync(self):
        check(lib().cet_sync(self._h), "cet_sync")

    # -- fields -----------------------------------------------------------------------------
    def _chk(self, a, name):
        if a is not None and tuple(a.shape) != self.owned_shape:
            raise ValueError(f"{name}: shape {a.shape} != {self.owned_shape}")

    def upload(self, state=None, theta=None, phi=None, T=None, defects=None):
        st, df = _arr(state, np.int64), _arr(defects, np.int64)
        th, ph, t = _arr(theta, np.float64), _arr(phi, np.float64), _arr(T, np.float64)
        for a, n in ((st, "state"), (th, "theta"), (ph, "phi"), (t, "T"), (df, "defects")):
            self._chk(a, n)
        check(lib().cet_upload(self._h, _ptr(st), _ptr(th), _ptr(ph), _ptr(t), _ptr(df)), "cet_upload")

    def download(self, state=False, atom_type=False, theta=False, phi=False, T=False, out=None):
        """Returns a dict of freshly allocated arrays (or fills the arrays given in `out`)."""
        out = dict(out or {})
        want = dict(state=(state, np.int64), atom_type=(atom_type, np.int64),
                    theta=(theta, np.float64), phi=(phi, np.float64), T=(T, np.float64))
        bufs = {}
        for name, (flag, dt) in want.items():
            if name in out:
                a = out[name]
                if a.dtype != dt or not a.flags.c_contiguous or tuple(a.shape) != self.owned_shape:
                    raise ValueError(f"{name}: need C-contiguous {dt} array of shape {self.owned_shape}")
                bufs[name] = a
            elif flag:
                bufs[name] = np.empty(self.owned_shape, dtype=dt)
        check(lib().cet_download(self._h, _ptr(bufs.get("state")), _ptr(bufs.get("atom_type")),
                                 _ptr(bufs.get("theta")), _ptr(bufs.get("phi")), _ptr(bufs.get("T"))),
              "cet_download")
        return bufs

    def upload_prev_state(self, prev_state):
        ps = _arr(prev_state, np.int64)
        self._chk(ps, "prev_state")
        check(lib().cet_upload_prev_state(self._h, _ptr(ps)), "cet_upload_prev_state")

    def snapshot_state(self):
        check(lib().cet_snapshot_state(self._h), "cet_snapshot_state")

    def upload_packed(self, packed):
        p = _arr(packed, np.uint8)
        self._chk(p, "packed")
        check(lib().cet_upload_packed(self._h, _ptr(p)), "cet_upload_packed")

    def download_packed(self, out=None):
        """Packed state (state | defects << 4); `out`: a C-contiguous uint8 array of the owned shape
        to fill (e.g. page-locked memory) instead of a fresh pageable one."""
        if out is None:
            p = np.empty(self.owned_shape, np.uint8)
        else:
            p = out
            if p.dtype != np.uint8 or not p.flags.c_contiguous or tuple(p.shape) != self.owned_shape:
                raise ValueError(f"packed: need C-contiguous uint8 array of shape {self.owned_shape}")
        check(lib().cet_download_packed(self._h, _ptr(p)), "cet_download_packed")
        return p

    def device_ptr(self, which: int):
        p, nb = C.c_void_p(None), C.c_int64(0)
        check(lib().cet_device_ptr(self._h, which, C.byref(p), C.byref(nb)), "cet_device_ptr")
        return p.value, nb.value

    def counts(self):
        c = (C.c_int64 * 16)()
        check(lib().cet_counts(self._h, C.byref(c)), "cet_counts")
        return np.array(list(c), dtype=np.int64)

    # -- thermal ----------------------------------------------------------------------------
    def thermal_cet(self, tp: ThermalParams):
        check(lib().cet_thermal_cet(self._h, C.byref(tp)), "cet_thermal_cet")

    def thermal_full(self, p: ThermalFullParams, q_top):
        q = _arr(q_top, np.float64)
        check(lib().cet_thermal_full(self._h, C.byref(p), _ptr(q)), "cet_thermal_full")

    def fill_gradient(self, t0, g):
        check(lib().cet_thermal_fill_gradient(self._h, float(t0), float(g)), "cet_thermal_fill_gradient")

    # -- rates ------------------------------------------------------------------------------
    def set_rate_params(self, rp: RateParams):
        check(lib().cet_set_rate_params(self._h, C.byref(rp)), "cet_set_rate_params")

    def rates_build(self):
        check(lib().cet_rates_build(self._h), "cet_rates_build")

    def rates_total(self):
        t, n = C.c_double(0.0), C.c_int64(0)
        check(lib().cet_rates_total(self._h, C.byref(t), C.byref(n)), "cet_rates_total")
        return t.value, n.value

    def rates_download(self, dep=True):
        sr = np.empty(self.owned_shape, np.float64)
        dr = np.empty(self.shape[1:], np.float64) if dep else None
        check(lib().cet_rates_download(self._h, _ptr(sr), _ptr(dr)), "cet_rates_download")
        return sr, dr

    def events_count(self):
        n, nd = C.c_int64(0), C.c_int64(0)
        check(lib().cet_events_count(self._h, C.byref(n), C.byref(nd)), "cet_events_count")
        return n.value, nd.value

    def events_export(self, species_draws=None):
        """SoA event list in the reference's order (kmc_event_rates.py:162-176)."""
        n, nd = self.events_count()
        sd = _arr(species_draws, np.float64)
        ty = np.empty(n, np.uint8); po = np.empty(n, np.int64); ra = np.empty(n, np.float64)
        ta = np.empty(n, np.int64); at = np.empty(n, np.int32)
        nw = C.c_int64(0)
        check(lib().cet_events_export(self._h, _ptr(sd), 0 if sd is None else sd.size, n,
                                      _ptr(ty), _ptr(po), _ptr(ra), _ptr(ta), _ptr(at), C.byref(nw)),
              "cet_events_export")
        if nw.value != n:
            raise RuntimeError("event count changed between count and export")
        return dict(type=ty, pos=po, rate=ra, target=ta, atom=at, n_dep=nd)

    # -- exact BKL --------------------------------------------------------------------------
    def kmc_run(self, step0, n_steps, defect_fraction, tp, thermal_every, py_draws, np_draws,
                sp_draws=None, total_time0=0.0, log=False):
        py, npd, sp = _arr(py_draws, np.float64), _arr(np_draws, np.float64), _arr(sp_draws, np.float64)
        res = KmcResult()
        lg = {}
        if log:
            lg = dict(type=np.zeros(n_steps, np.uint8), pos=np.zeros(n_steps, np.int64),
                      target=np.zeros(n_steps, np.int64), atom=np.zeros(n_steps, np.int32),
                      rate=np.zeros(n_steps, np.float64), total=np.zeros(n_steps, np.float64))
        check(lib().cet_kmc_run(self._h, int(step0), int(n_steps), float(defect_fraction),
                                None if tp is None else C.byref(tp), int(thermal_every),
                                _ptr(py), py.size, _ptr(npd), npd.size,
                                _ptr(sp), 0 if sp is None else sp.size, float(total_time0),
                                C.byref(res), _ptr(lg.get("type")), _ptr(lg.get("pos")),
                                _ptr(lg.get("target")), _ptr(lg.get("atom")), _ptr(lg.get("rate")),
                                _ptr(lg.get("total"))), "cet_kmc_run")
        out = {f: getattr(res, f) for f, _ in KmcResult._fields_}
        for k, v in lg.items():
            out["log_" + k] = v[:res.steps_done]
        return out

    # -- sublattice sweeps --------------------------------------------------------------------
    def sweep_run(self, n_sweeps, sp: SweepParams, tp: ThermalParams = None):
        res = SweepResult()
        check(lib().cet_sweep_run(self._h, int(n_sweeps), C.byref(sp),
                                  None if tp is None else C.byref(tp), C.byref(res)), "cet_sweep_run")
        return {f: getattr(res, f) for f, _ in SweepResult._fields_ if f != "pad_"}

    # -- slabs over several GPUs ----------------------------------------------------------------
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        check(lib().cet_comm_init(self._h, buf, rank, world), "cet_comm_init")
        self.rank, self.world = int(rank), int(world)

    def halo_exchange(self, fields=7):
        check(lib().cet_halo_exchange(self._h, int(fields)), "cet_halo_exchange")

    def allreduce(self, values, op=0):
        v = np.ascontiguousarray(values, dtype=np.float64).copy()
        check(lib().cet_allreduce_f64(self._h, _ptr(v), v.size, op), "cet_allreduce_f64")
        return v

    # -- defects (defects.py on the resident lattice) ------------------------------------------------
    def defects_refresh(self, draws=None, seed=0, epoch=0, prob_base=0.12, e_mig=0.3, kT=8.617333262e-5,
                        T_default=2800.0, carbon_id=3, defect_id=4, apply_to_state=False):
        """defects.track_defects / introduce_defects (defects.py:4-31) in place: the defect mask of
        the resident lattice is redrawn.  draws: the reference's draw stream (one per carbon site, C
        order), or None for the device's Philox stream keyed by (seed, epoch, site).
        Returns (n_carbon, n_defects)."""
        d = None if draws is None else np.ascontiguousarray(draws, dtype=np.float64)
        nc, nd = C.c_int64(0), C.c_int64(0)
        check(lib().cet_defects_refresh(self._h, _ptr(d), 0 if d is None else d.size, int(seed), int(epoch),
                                        float(prob_base), float(e_mig), float(kT), float(T_default), int(carbon_id),
                                        int(defect_id), 1 if apply_to_state else 0, C.byref(nc), C.byref(nd)),
              "cet_defects_refresh")
        return nc.value, nd.value

    # -- grains (utils.get_clusters on the resident lattice) ------------------------------------
    def grains(self, theta_threshold=0.5, labels=False, theta_only=False):
        """Grains of the resident lattice in the reference's cluster order (raster order of each
        grain's first voxel, utils.py:28-84).  Returns a dict: n, root (C-order site index of the
        first voxel), size (voxels), box_lo / box_hi (n, 3); with labels=True also `labels`, the
        reference's `visited` volume (grain number 1.. per occupied site, 0 for empty).
        theta_only: the |theta1 - theta2| criterion of utils.py:49-50 instead of the misorientation."""
        n = C.c_int64(0)
        check(lib().cet_grains_label_ex(self._h, float(theta_threshold), 1 if theta_only else 0, C.byref(n)),
              "cet_grains_label_ex")
        n = n.value
        root, size = np.empty(n, np.int32), np.empty(n, np.int32)
        lo, hi = np.empty((n, 3), np.int32), np.empty((n, 3), np.int32)
        if n:
            check(lib().cet_grains_stats(self._h, n, _ptr(root), _ptr(size), _ptr(lo), _ptr(hi)), "cet_grains_stats")
        order = np.argsort(root, kind="stable")
        out = dict(n=n, root=root[order], size=size[order], box_lo=lo[order], box_hi=hi[order])
        if labels:
            lab = np.empty(self.owned_shape, np.int32)
            check(lib().cet_grains_download_labels(self._h, _ptr(lab)), "cet_grains_download_labels")
            vis = np.zeros(self.owned_shape, np.int32)
            occ = lab >= 0
            vis[occ] = np.searchsorted(out["root"], lab[occ]).astype(np.int32) + 1
            out["labels"] = vis
        return out

    def grains_local(self, theta_threshold=0.5):
        """Slab-local labelling (owned planes + 2 ghost planes per cut face; the ghost planes must be
        current): dict of root (GLOBAL site index of each local component's first voxel), size (owned
        voxels), box_lo / box_hi (global coordinates), unsorted.  metrics.grains_distributed joins the
        components of all slabs."""
        n = C.c_int64(0)
        check(lib().cet_grains_label_ex(self._h, float(theta_threshold), 0, C.byref(n)), "cet_grains_label_ex")
        n = n.value
        root, size = np.empty(n, np.int32), np.empty(n, np.int32)
        lo, hi = np.empty((n, 3), np.int32), np.empty((n, 3), np.int32)
        if n:
            check(lib().cet_grains_stats(self._h, n, _ptr(root), _ptr(size), _ptr(lo), _ptr(hi)), "cet_grains_stats")
        return dict(root=root.astype(np.int64), size=size.astype(np.int64), box_lo=lo, box_hi=hi)

    def grain_label_planes(self, i_lo, i_hi):
        """Labels (global root index, -1 = empty) of global planes [i_lo, i_hi) of the last labelling."""
        n1, n2 = self.owned_shape[1], self.owned_shape[2]
        out = np.empty((int(i_hi - i_lo), n1, n2), np.int32)
        check(lib().cet_grains_download_planes(self._h, int(i_lo), int(i_hi), _ptr(out)), "cet_grains_download_planes")
        return out

    def nst_mismatches(self):
        n = C.c_int64(0)
        check(lib().cet_debug_nst_mismatches(self._h, C.byref(n)), "cet_debug_nst_mismatches")
        return n.value

    def debug_flags(self, flags):
        """Refresh-kernel selection of sweep_run (tests / profiling); bit values in cetkmc.h (cet_debug_flags)."""
        check(lib().cet_debug_flags(self._h, int(flags)), "cet_debug_flags")

    def sweep_state(self):
        """(sweep_index, tau, time) of the sweep clock — see sweep_set_state."""
        i, tau, t = C.c_int64(0), C.c_double(0.0), C.c_double(0.0)
        check(lib().cet_sweep_get_state(self._h, C.byref(i), C.byref(tau), C.byref(t)), "cet_sweep_get_state")
        return i.value, tau.value, t.value

    def sweep_set_state(self, sweep_index, tau, time):
        """Restore the sweep clock of a checkpoint: the resumed run continues bit for bit."""
        check(lib().cet_sweep_set_state(self._h, int(sweep_index), float(tau), float(time)), "cet_sweep_set_state")

    def sweep_reset(self):
        check(lib().cet_sweep_reset(self._h), "cet_sweep_reset")

    # -- timing -----------------------------------------------------------------------------
    PROF_KINDS = dict(decide=0, apply=1, thermal=2, rates=3, halo=4, step=5, pick=6, refresh=7, allreduce=8, boundary=9)

    def profile_enable(self, on=True):
        check(lib().cet_profile_enable(self._h, 1 if on else 0), "cet_profile_enable")

    def profile_read(self, kind, reset=True):
        """(total ms, launches) of a kernel kind since the last reset."""
        ms, n = C.c_double(0.0), C.c_int64(0)
        check(lib().cet_profile_read(self._h, self.PROF_KINDS[kind], C.byref(ms), C.byref(n), 1 if reset else 0),
              "cet_profile_read")
        return ms.value, n.value

    def timer_begin(self):
        check(lib().cet_timer_begin(self._h), "cet_timer_begin")

    def timer_end_ms(self) -> float:
        ms = C.c_float(0.0)
        check(lib().cet_timer_end_ms(self._h, C.byref(ms)), "cet_timer_end_ms")
        return ms.value


GROUP_MAX = 64                                      # cet_sweep_run_group's limit on n_ctx


def sweep_run_group(ctxs, n_sweeps, sps, tps=None):
    """Advance the lattices of `ctxs` (whole-lattice Contexts of one L on one device) by n_sweeps sweeps each,
    with one launch per kernel for the whole group.  sps: one SweepParams per context; tps: one
    ThermalParams per context, or None when no context has a thermal step.  Every context ends exactly as
    its own ctx.sweep_run(n_sweeps, sps[q], tps[q]) would leave it.  Returns one result dict per context,
    with the keys of Context.sweep_run."""
    ctxs, sps = list(ctxs), list(sps)
    n = len(ctxs)
    if len(sps) != n:
        raise ValueError(f"sweep_run_group: {len(sps)} sweep params for {n} contexts")
    if tps is not None:
        tps = list(tps)
        if len(tps) != n:
            raise ValueError(f"sweep_run_group: {len(tps)} thermal params for {n} contexts")
    if any(not isinstance(c, Context) for c in ctxs):
        raise TypeError("sweep_run_group: ctxs must be Context objects")
    handles = (C.c_void_p * n)(*[c._h.value for c in ctxs])
    sp_arr = (SweepParams * n)(*sps)
    tp_arr = None if tps is None else (ThermalParams * n)(*tps)
    res = (SweepResult * n)()
    check(lib().cet_sweep_run_group(handles, n, int(n_sweeps), sp_arr, tp_arr, res), "cet_sweep_run_group")
    return [{f: getattr(r, f) for f, _ in SweepResult._fields_ if f != "pad_"} for r in res]


def thermal_full_group(ctxs, params, q_tops, snapshot=True):
    """update_temperature on a group of whole-lattice Contexts of one L on one device, one stencil launch for the
    group: context q takes params[q] (ThermalFullParams) and the source plane q_tops[q] (an (L, L) C-contiguous
    float64 array, thermal_solver.laser_source_top).  Every context ends exactly as its own
    ctx.thermal_full(params[q], q_tops[q]) followed, with snapshot=True, by ctx.snapshot_state() would leave it."""
    ctxs, params, q_tops = list(ctxs), list(params), list(q_tops)
    n = len(ctxs)
    if len(params) != n:
        raise ValueError(f"thermal_full_group: {len(params)} params for {n} contexts")
    if len(q_tops) != n:
        raise ValueError(f"thermal_full_group: {len(q_tops)} source planes for {n} contexts")
    if any(not isinstance(p, ThermalFullParams) for p in params):
        raise TypeError("thermal_full_group: params must be ThermalFullParams")
    handles = _group_handles("thermal_full_group", ctxs)
    for q, (c, a) in enumerate(zip(ctxs, q_tops)):
        if not isinstance(a, np.ndarray) or a.dtype != np.float64 or not a.flags.c_contiguous:
            raise TypeError(f"thermal_full_group: q_tops[{q}] must be a C-contiguous float64 array")
        if tuple(a.shape) != tuple(c.shape[1:]):
            raise ValueError(f"thermal_full_group: q_tops[{q}] has shape {a.shape}, the lattice needs {tuple(c.shape[1:])}")
    tfp = (ThermalFullParams * n)(*params)
    q_ptr = (C.c_void_p * n)(*[a.ctypes.data for a in q_tops])
    check(lib().cet_thermal_full_group(handles, n, tfp, q_ptr, 1 if snapshot else 0), "cet_thermal_full_group")


def _group_handles(fn, ctxs):
    if any(not isinstance(c, Context) for c in ctxs):
        raise TypeError(f"{fn}: ctxs must be Context objects")
    return (C.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])


def init_group(ctxs, nuclei, snapshot=False):
    """The initial lattices of a group of whole-lattice Contexts of one L on one device, built on the device with one
    copy and two launches.  nuclei[q] = (site, byte, theta, phi, T_row) as _host.initial_nuclei returns them: int64,
    uint8, float64 and float64 arrays of one length and a float64 array of L.  Context q ends exactly as
    ctxs[q].upload() of the dense arrays would leave it (followed, with snapshot=True, by ctxs[q].snapshot_state())."""
    ctxs, nuclei = list(ctxs), list(nuclei)
    n = len(ctxs)
    if len(nuclei) != n:
        raise ValueError(f"init_group: {len(nuclei)} nucleus sets for {n} contexts")
    handles = _group_handles("init_group", ctxs)
    dtypes = (np.int64, np.uint8, np.float64, np.float64, np.float64)
    for q, (c, nu) in enumerate(zip(ctxs, nuclei)):
        if len(nu) != 5:
            raise ValueError(f"init_group: nuclei[{q}] must be (site, byte, theta, phi, T_row)")
        for a, dt in zip(nu, dtypes):
            if not isinstance(a, np.ndarray) or a.dtype != dt or a.ndim != 1 or not a.flags.c_contiguous:
                raise TypeError(f"init_group: nuclei[{q}] needs 1-D C-contiguous arrays of "
                                "int64, uint8, float64, float64, float64")
        if len({len(a) for a in nu[:4]}) != 1:
            raise ValueError(f"init_group: nuclei[{q}]: site, byte, theta and phi differ in length")
        if len(nu[4]) != c.shape[2]:
            raise ValueError(f"init_group: nuclei[{q}]: T_row has {len(nu[4])} values, the lattice needs {c.shape[2]}")
    desc = (InitDesc * n)(*[InitDesc(len(nu[0]), *[a.ctypes.data for a in nu]) for nu in nuclei])
    check(lib().cet_init_group(handles, n, desc, 1 if snapshot else 0), "cet_init_group")


def counts_group(ctxs):
    """Context.counts() of every context of `ctxs` (whole-lattice Contexts of one L on one device) with one launch
    and one synchronisation: an (n, 16) int64 array."""
    ctxs = list(ctxs)
    handles = _group_handles("counts_group", ctxs)
    out = np.zeros((len(ctxs), 16), np.int64)
    check(lib().cet_counts_group(handles, len(ctxs), out.ctypes.data_as(C.POINTER(C.c_int64))), "cet_counts_group")
    return out


def metrics_group(ctxs, params, draws=None):
    """The metrics cadence of a group of whole-lattice Contexts of one L on one device, each kernel one launch for
    the group: per context the optional defect-mask refresh (params[q].refresh; draws[q] the NumPy stream's draws,
    or None for the Philox stream), the state histogram, the grain labelling (Context.grains() reports it
    afterwards) and the reductions of a metrics row.  params: one MetricsParams per context; draws: None or a list
    with one entry per context.  Returns one dict per context with the fields of MetricsResult (counts and
    pct_index as int64 arrays)."""
    ctxs, params = list(ctxs), list(params)
    n = len(ctxs)
    if len(params) != n:
        raise ValueError(f"metrics_group: {len(params)} params for {n} contexts")
    if any(not isinstance(p, MetricsParams) for p in params):
        raise TypeError("metrics_group: params must be MetricsParams")
    if draws is not None:
        draws = list(draws)
        if len(draws) != n:
            raise ValueError(f"metrics_group: {len(draws)} draw arrays for {n} contexts")
        draws = [None if d is None else np.ascontiguousarray(d, dtype=np.float64) for d in draws]
    handles = _group_handles("metrics_group", ctxs)
    mp = (MetricsParams * n)(*params)
    res = (MetricsResult * n)()
    d_ptr = n_draws = None
    if draws is not None:
        d_ptr = (C.c_void_p * n)(*[None if d is None else d.ctypes.data for d in draws])
        n_draws = (C.c_int64 * n)(*[0 if d is None else d.size for d in draws])
    check(lib().cet_metrics_group(handles, n, mp, d_ptr, n_draws, res), "cet_metrics_group")
    out = []
    for r in res:
        d = {f: getattr(r, f) for f, _ in MetricsResult._fields_}
        d["counts"] = np.array(list(r.counts), np.int64)
        d["pct_index"] = np.array(list(r.pct_index), np.int64)
        out.append(d)
    return out


PROFILE_COLUMNS = ("Solid", "EquiaxedSolid", "GrainsSpanning", "EquiaxedGrainsSpanning")    # cet_grain_profile_group's f


def grain_profile_group(ctxs, axis, ar_threshold):
    """Per-plane grain profile of the last grain labelling (Context.grains(), metrics_group) of every context of `ctxs`
    (whole-lattice Contexts of one L on one device), along `axis` (0, 1 or 2), with five launches and one copy for the
    group.  Returns an (n, 4, L) int64 array: for context q and plane z, [q, 0, z] occupied sites, [q, 1, z] of those
    the sites of grains with aspect ratio < ar_threshold, [q, 2, z] grains whose bounding box along `axis` contains z,
    [q, 3, z] of those the grains with aspect ratio < ar_threshold (PROFILE_COLUMNS).  The call does not relabel and
    changes nothing the next metrics row or sweep reads."""
    ctxs = list(ctxs)
    if isinstance(axis, bool) or not isinstance(axis, (int, np.integer)) or int(axis) not in (0, 1, 2):
        raise ValueError(f"grain_profile_group: axis must be 0, 1 or 2, got {axis!r}")
    thr = float(ar_threshold)
    if not np.isfinite(thr):
        raise ValueError(f"grain_profile_group: ar_threshold must be finite, got {ar_threshold!r}")
    handles = _group_handles("grain_profile_group", ctxs)
    L = ctxs[0].shape[2] if ctxs else 0
    out = np.zeros((len(ctxs), 4, L), np.int64)
    check(lib().cet_grain_profile_group(handles, len(ctxs), int(axis), thr, out.ctypes.data_as(C.POINTER(C.c_int64))),
          "cet_grain_profile_group")
    return out


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    check(lib().cet_comm_unique_id(buf), "cet_comm_unique_id")
    return buf.raw
