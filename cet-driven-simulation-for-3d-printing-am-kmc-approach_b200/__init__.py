"""cetkmc — B200-native KMC / thermal hot path for the CET additive-manufacturing simulator.

Drop-in modules (same public names, signatures and array layouts as the reference):
    cetkmc.kmc_event_rates   get_event_rates, compute_row_events, get_bcc_neighbors, compute_misorientation
    cetkmc.kmc_simulation    run_kmc (+ run_kmc_sublattice for the large-lattice path)
    cetkmc.thermal_solver    update_temperature_cet, update_temperature, build_temperature_field
All compute goes through libcetkmc.so (include/cetkmc.h) via ctypes; there is no CPU fallback.
Import the package as `import cetkmc` (alias module at the repository root).
"""
__version__ = "0.1.0"

from . import _lib  # noqa: F401  (ctypes binding; the shared library is loaded on first use)
from ._lib import Context, build, counts_group, device_count, grain_profile_group, init_group, metrics_group, sweep_run_group, thermal_full_group  # noqa: F401
