"""Host-side set-up used by `run_kmc` when the user's own modules (`lattice_init`, `defects`) are
not importable: the initial lattice and the initial defect mask.  They are out of the hot path
(SURVEY §2 rows 5-6): O(L^3) NumPy work that runs once per run, before anything is uploaded.

Each function reproduces the observable behaviour of the reference function it names (same
global-RNG draws in the same order, same return types) so that a run driven through either
implementation yields the same trajectory and the same metrics.csv.  Observables (grain
clustering, metrics rows) have no host implementation in the product: csrc/grains.cu + metrics.py.
"""
from __future__ import annotations

import numpy as np

from ._config import constants as K

# kmc_event_rates.py:29-36 — neighbour offsets, reference order
NEIGHBOR_OFFSETS = np.array(
    [(1, 1, 0), (1, -1, 0), (-1, 1, 0), (-1, -1, 0), (0, 1, 1), (0, 1, -1), (0, -1, 1), (0, -1, -1),
     (2, 0, 0), (-2, 0, 0), (0, 2, 0), (0, -2, 0), (0, 0, 2), (0, 0, -2)], dtype=np.int64)


def initialize_lattice(lattice_size=None, n_seeds=None, T_sub=None, T_melt=None, random_seed=42,
                       impurity_c=0.0, verbose=False):
    """lattice_init.py:10-59 — seeds NumPy's global stream and consumes it identically."""
    L = K.LATTICE_SIZE if lattice_size is None else lattice_size
    n_seeds = K.N_SEEDS if n_seeds is None else n_seeds
    T_sub = K.T_SUB if T_sub is None else T_sub
    T_melt = K.T_MELT if T_melt is None else T_melt
    np.random.seed(random_seed)
    state = np.zeros((L, L, L), dtype=int)
    atom_type = np.zeros((L, L, L), dtype=int)
    theta = np.zeros((L, L, L))
    phi = np.zeros((L, L, L))
    grad = (T_melt - T_sub) / L
    T = np.ascontiguousarray(np.broadcast_to(T_sub + grad * np.arange(L), (L, L, L)))
    for flat in np.random.choice(L * L, n_seeds, replace=False):
        x, y = int(flat) // L, int(flat) % L
        r = np.random.random()
        if r < K.IMPURITY_RE:
            atom = 2
        elif r < K.IMPURITY_RE + impurity_c:
            atom = 3
        else:
            atom = 1
        state[x, y, 0] = atom
        atom_type[x, y, 0] = atom
        theta[x, y, 0] = np.random.uniform(0, np.pi)
        phi[x, y, 0] = np.random.uniform(0, 2 * np.pi)
    return state, theta, phi, T, atom_type


def initial_nuclei(L, n_seeds, T_sub, random_seed, impurity_c, T_melt=None):
    """initialize_lattice(L, n_seeds, T_sub, T_melt, random_seed, impurity_c) followed by
    introduce_defects(state, atom_type, T, apply_to_state=False) in sparse form, consuming NumPy's global stream
    exactly as that pair does.  The initial lattice is empty but for the nuclei on the k = 0 plane, and T depends
    on k only.  Returns (site, byte, theta, phi, T_row):
        site   int64 (n,)  C-order flat site index of each nucleus, in draw order
        byte   uint8 (n,)  atom | defect << 4
        theta, phi  float64 (n,)
        T_row  float64 (L,)  the temperature along k that the dense T repeats over (i, j)."""
    T_melt = K.T_MELT if T_melt is None else T_melt
    np.random.seed(random_seed)
    grad = (T_melt - T_sub) / L
    T_row = T_sub + grad * np.arange(L)
    flat = np.random.choice(L * L, n_seeds, replace=False)
    n = len(flat)
    atom = np.empty(n, np.uint8)
    theta, phi = np.empty(n), np.empty(n)
    for q in range(n):
        r = np.random.random()
        atom[q] = 2 if r < K.IMPURITY_RE else (3 if r < K.IMPURITY_RE + impurity_c else 1)
        theta[q] = np.random.uniform(0, np.pi)
        phi[q] = np.random.uniform(0, 2 * np.pi)
    site = np.asarray(flat, dtype=np.int64) * L
    defect = np.zeros(n, np.uint8)
    carbon = np.flatnonzero(atom == 3)
    if len(carbon):
        # introduce_defects draws one number per carbon site in C order, and every carbon site has T = T_row[0]
        carbon = carbon[np.argsort(site[carbon])]
        tv = np.full(len(carbon), T_row[0])
        with np.errstate(divide="ignore", invalid="ignore"):
            tv = np.where(tv > 0, tv, K.T_SUB)
            prob = K.DEFECT_PROB_BASE * np.exp(-0.3 / (K.K_T * tv))
        prob = np.clip(prob, 0.0, 1.0)
        defect[carbon] = np.random.random(len(carbon)) < prob
    return site, atom | (defect << 4), theta, phi, T_row


def introduce_defects(state, atom_type, T=None, apply_to_state=False, voxel_size=5e-6):
    """defects.py:4-31 — Bernoulli defect mask on carbon sites (one global-stream draw each)."""
    L = state.shape[0]
    mask = np.zeros((L, L, L), dtype=int)
    carbon = (atom_type == 3)
    n_c = int(carbon.sum())
    if n_c:
        if T is not None:
            tv = T[carbon]
            with np.errstate(divide="ignore", invalid="ignore"):
                tv = np.where(tv > 0, tv, K.T_SUB)
                prob = K.DEFECT_PROB_BASE * np.exp(-0.3 / (K.K_T * tv))
        else:
            prob = np.full(n_c, K.DEFECT_PROB_BASE)
        prob = np.clip(prob, 0.0, 1.0)
        mask[carbon] = (np.random.random(n_c) < prob).astype(int)
    if apply_to_state:
        state[mask == 1] = 4
    volume = mask.size * (voxel_size ** 3)
    density = np.sum(mask) / volume if volume > 0 else 0.0
    return mask, density
