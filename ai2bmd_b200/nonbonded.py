"""Host side of the non-bonded terms -- mirrors of ``MMNonBondedCalculator`` (``src/Calculators/nonbonded.py:9-63``)
and ``PMENonBondedCalculator`` (``src/Calculators/pme.py:113-214``), the two choices of ``--fragment-longrange-calc``.

The reference obtains per-atom charges / sigmas / epsilons from OpenMM's amber14 force field
(``src/AIMD/protein.py:153-175``); OpenMM is not part of this image, so the parameters are inputs here, in the
reference's units (e, nm, kJ/mol).  The pair list (all ordered pairs minus atoms sharing a dipeptide,
``protein.py:133-151`` + ``distancefrag.py:355-363``) is never materialised: the device kernel walks all sources
per destination atom and consults a per-atom exclusion table (CSR) built by :func:`exclusion_table`.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

from .engine import Engine


def dipeptide_atom_sets(frags, recipe, pm) -> list:
    """Protein-atom indices of every dipeptide fragment (``prot.all_dipeptide_index`` at ``distancefrag.py:325-327``):
    the real atoms of the fragments whose sign in the bonded combination is +1."""
    sets = []
    for g in range(len(frags)):
        if pm.frag_sign[g] > 0:
            real = np.asarray(recipe.real[int(frags.start[g]):int(frags.end[g])])
            sets.append(np.unique(real[real >= 0]))
    return sets


def exclusion_table(n_atoms: int, groups: Sequence[np.ndarray]) -> Tuple[np.ndarray, np.ndarray]:
    """CSR table (rowptr [n+1], col) of excluded partners: j is listed under i iff i != j share a group
    (``distancefrag.py:355-361``: every combination inside a dipeptide, both orders).  Rows are ascending."""
    partners = [set() for _ in range(n_atoms)]
    for g in groups:
        g = [int(a) for a in g]
        for a in g:
            partners[a].update(g)
    rowptr = np.zeros(n_atoms + 1, dtype=np.int32)
    cols = []
    for i, s in enumerate(partners):
        s.discard(i)
        cols.extend(sorted(s))
        rowptr[i + 1] = len(cols)
    return rowptr, np.asarray(cols, dtype=np.int32)


class MMNonBondedCalculator:
    """``set_parameters`` once, then ``calc(positions) -> (energy [eV], forces [n,3] eV/A)`` per step."""

    def __init__(self, engine: Engine):
        import torch
        self.torch = torch
        self.engine = engine
        self.n = 0

    def set_parameters(self, charges, sigmas_nm, epsilons_kj, excl_rowptr, excl_col, atom_lo: int = 0, atom_hi: int = -1):
        torch = self.torch
        self.engine.set_nonbonded(charges, sigmas_nm, epsilons_kj, excl_rowptr, excl_col, atom_lo, atom_hi)
        self.n = len(charges)
        dev = torch.device("cuda", self.engine.device)
        self.pos = torch.empty((self.n, 3), dtype=torch.float32, device=dev)
        self.ef = torch.empty(3 * self.n + 1, dtype=torch.float32, device=dev)

    def __call__(self, positions) -> Tuple[float, np.ndarray]:
        torch = self.torch
        p = np.ascontiguousarray(positions, dtype=np.float32)        # nonbonded.py:39 casts to fp32
        if p.shape != (self.n, 3):
            raise ValueError(f"positions must be [{self.n}, 3]")
        stream = torch.cuda.current_stream(self.pos.device)
        self.pos.copy_(torch.from_numpy(p), non_blocking=True)
        self.ef.zero_()
        self.engine.nonbonded_device(self.pos.data_ptr(), self.ef.data_ptr(), stream.cuda_stream)
        ef = self.ef.cpu().numpy()
        return float(ef[-1]), ef[:-1].reshape(-1, 3).copy()


class PMENonBondedCalculator:
    """Mirror of the reference's ``PMENonBondedCalculator`` (``src/Calculators/pme.py:113-214``) on the device:
    ``set_parameters`` once, then ``calc(positions) -> (energy [eV], forces [n,3] eV/A)`` per step."""

    def __init__(self, engine: Engine, beta: float = 0.3, cutoff: float = 9.0, grid_spacing: float = 1.0):
        import torch
        self.torch = torch
        self.engine = engine
        self.beta, self.cutoff, self.grid_spacing = float(beta), float(cutoff), float(grid_spacing)
        self.n = 0

    def grid(self, cell) -> Tuple[int, int, int]:
        """Mesh points per axis, ``int(cell_len / grid_spacing)`` (pme.py:146-149)."""
        return tuple(int(c / self.grid_spacing) for c in cell)

    def set_parameters(self, charges, sigmas_nm, epsilons_kj, excl_rowptr, excl_col, cell, atom_lo: int = 0,
                       atom_hi: int = -1):
        """``cell``: the orthorhombic cell lengths (A), e.g. :func:`ai2bmd_b200.pdbfrag.read_cell` of the input PDB."""
        torch = self.torch
        cell = tuple(float(c) for c in cell)
        self.engine.set_pme(charges, sigmas_nm, epsilons_kj, excl_rowptr, excl_col, cell, self.grid(cell), self.beta,
                            self.cutoff, atom_lo, atom_hi)
        self.n = len(charges)
        dev = torch.device("cuda", self.engine.device)
        self.pos = torch.empty((self.n, 3), dtype=torch.float32, device=dev)
        self.ef = torch.empty(3 * self.n + 1, dtype=torch.float32, device=dev)

    def __call__(self, positions) -> Tuple[float, np.ndarray]:
        torch = self.torch
        p = np.ascontiguousarray(positions, dtype=np.float32)        # pme.py:162 casts to fp32
        if p.shape != (self.n, 3):
            raise ValueError(f"positions must be [{self.n}, 3]")
        stream = torch.cuda.current_stream(self.pos.device)
        self.pos.copy_(torch.from_numpy(p), non_blocking=True)
        self.ef.zero_()
        self.engine.pme_device(self.pos.data_ptr(), self.ef.data_ptr(), stream.cuda_stream)
        ef = self.ef.cpu().numpy()
        return float(ef[-1]), ef[:-1].reshape(-1, 3).copy()


def synthetic_parameters(numbers, seed: int = 0):
    """Amber-like per-atom parameters for benchmarks and tests when no force field is available: charges in
    [-0.8, 0.6] e shifted to a neutral total, sigma / epsilon by element in amber14's typical ranges."""
    rng = np.random.default_rng(seed)
    numbers = np.asarray(numbers)
    sig = {1: 0.11, 6: 0.34, 7: 0.325, 8: 0.296, 16: 0.356}
    eps = {1: 0.066, 6: 0.36, 7: 0.71, 8: 0.88, 16: 1.05}
    q = rng.uniform(-0.8, 0.6, size=len(numbers))
    q -= q.mean()
    sigma = np.array([sig[int(z)] for z in numbers]) * rng.uniform(0.9, 1.1, size=len(numbers))
    epsilon = np.array([eps[int(z)] for z in numbers]) * rng.uniform(0.8, 1.2, size=len(numbers))
    return q.astype(np.float32), sigma.astype(np.float32), epsilon.astype(np.float32)
