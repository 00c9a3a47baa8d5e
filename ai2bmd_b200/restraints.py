"""Hookean restraints: the pre-equilibration and the hydrogen-bond constraints of the reference's MD driver.

The reference's MD driver (``src/AIMD/simulator.py`` of microsoft/AI2BMD) adds ASE ``Hookean`` constraints to the protein twice:

* pre-equilibration (``:139-166``): five stages of ``--preeq-steps`` steps (2000 by default), every protein atom tied to
  where it stood at the start of the stage with k = 10, 5, 1, 0.5, 0.1 kcal/mol/A^2 (times ``kcalmol2ev``; the log line
  says "eV/A^2"), the previous constraint list restored after each stage;
* ``--constraints`` (``:168-180``): every hydrogen gets a flat-bottom spring to its covalent partner,
  ``Hookean(a1=h, a2=partner, k=15 eV/A^2, rt=r_cov(H) + r_cov(partner) + 0.2)`` with the pairs of
  ``PDBAnalyzer.find_bonded_atoms("H")`` (``src/utils/utils.py:169-221``).

ASE is not installed here, so :func:`hookean` restates ASE 3.22 ``ase/constraints.py`` ``Hookean`` (point and two-atom
types; recalled, not pinned) in fp64 numpy.  It is the checker of the device term (``csrc/k_restraint.cuh``,
``vb_set_restraints``).  ASE adds ``adjust_forces`` to whatever the calculator returns and
``adjust_potential_energy`` to the energy, and ``Langevin.step`` asks for the forces afresh every step, so a changed
restraint set acts from the next half-kick on: :func:`set_restraints` refreshes the forces of either integrator.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

KCAL_MOL = 4184.0 / (6.022140857e23 * 1.6021766208e-19)     # kcal/mol in eV, ASE's CODATA-2014 units
PREEQ_STAGES = (10.0, 5.0, 1.0, 0.5, 0.1)                    # kcal/mol/A^2, simulator.py:142
COVALENT_RADII = {"H": 0.31, "C": 0.76, "N": 0.71, "O": 0.66, "P": 1.07, "S": 1.05}   # utils.py:172-179
HBOND_K = 15.0                                              # eV/A^2, utils.py:217


def _arr(a, dtype, shape):
    return np.ascontiguousarray(np.asarray(a, dtype=dtype).reshape(shape))


@dataclass
class RestraintSet:
    """Point restraints (atom, anchor, k, rt) and pair restraints (i, j, k, rt); k in eV/A^2, lengths in A.
    ``[atom_lo, atom_hi)`` are the destination atoms whose forces are computed (``atom_hi < 0``: all); a restraint's
    energy is counted where its first atom is computed."""
    point_atom: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    point_anchor: np.ndarray = field(default_factory=lambda: np.zeros((0, 3)))
    point_k: np.ndarray = field(default_factory=lambda: np.zeros(0))
    point_rt: np.ndarray = field(default_factory=lambda: np.zeros(0))
    pair_ij: np.ndarray = field(default_factory=lambda: np.zeros((0, 2), np.int32))
    pair_k: np.ndarray = field(default_factory=lambda: np.zeros(0))
    pair_rt: np.ndarray = field(default_factory=lambda: np.zeros(0))
    atom_lo: int = 0
    atom_hi: int = -1

    def __post_init__(self):
        self.point_atom = _arr(self.point_atom, np.int32, -1)
        self.point_anchor = _arr(self.point_anchor, np.float64, (-1, 3)).copy()     # a fixed copy: it does not follow the atom
        self.point_k, self.point_rt = _arr(self.point_k, np.float64, -1), _arr(self.point_rt, np.float64, -1)
        self.pair_ij = _arr(self.pair_ij, np.int32, (-1, 2))
        self.pair_k, self.pair_rt = _arr(self.pair_k, np.float64, -1), _arr(self.pair_rt, np.float64, -1)
        if not (len(self.point_atom) == len(self.point_anchor) == len(self.point_k) == len(self.point_rt)
                and len(self.pair_ij) == len(self.pair_k) == len(self.pair_rt)):
            raise ValueError("restraint arrays have inconsistent lengths")

    @property
    def n_point(self) -> int:
        return len(self.point_atom)

    @property
    def n_pair(self) -> int:
        return len(self.pair_ij)

    @property
    def empty(self) -> bool:
        return self.n_point == 0 and self.n_pair == 0

    def __add__(self, other: "RestraintSet") -> "RestraintSet":
        """Both sets' restraints (this one's first), with this set's slice."""
        return RestraintSet(np.concatenate([self.point_atom, other.point_atom]),
                            np.concatenate([self.point_anchor, other.point_anchor]),
                            np.concatenate([self.point_k, other.point_k]), np.concatenate([self.point_rt, other.point_rt]),
                            np.concatenate([self.pair_ij, other.pair_ij]), np.concatenate([self.pair_k, other.pair_k]),
                            np.concatenate([self.pair_rt, other.pair_rt]), self.atom_lo, self.atom_hi)

    def sliced(self, atom_lo: int, atom_hi: int) -> "RestraintSet":
        return RestraintSet(self.point_atom, self.point_anchor, self.point_k, self.point_rt, self.pair_ij, self.pair_k,
                            self.pair_rt, int(atom_lo), int(atom_hi))

    def install(self, engine) -> None:
        """Make this set the engine's restraint term (an empty set removes it)."""
        engine.set_restraints(self.point_atom, self.point_anchor, self.point_k, self.point_rt, self.pair_ij, self.pair_k,
                              self.pair_rt, self.atom_lo, self.atom_hi)


def hookean(x, rs: RestraintSet):
    """(E [eV], F [n,3] eV/A) of the restraints at positions x [n,3], fp64: ASE 3.22 ``Hookean`` without minimum image.
    point: d = p0 - x_a; pair: d = x_j - x_i; r = |d|; if r > rt: F_a / F_i += k (r - rt) d/r (F_j -= the same) and
    E += k (r - rt)^2 / 2.  Only atoms in the slice receive forces; energies are counted at the first atom."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    lo, hi = rs.atom_lo, (n if rs.atom_hi < 0 else rs.atom_hi)
    F = np.zeros_like(x)
    E = 0.0

    def term(d, k, rt):
        r = np.sqrt((d * d).sum(1))
        on = r > rt
        s = np.where(on, k * (r - rt), 0.0)
        return s[:, None] * d / np.where(on, r, 1.0)[:, None], np.where(on, 0.5 * s * (r - rt), 0.0)

    if rs.n_point:
        a = rs.point_atom
        f, e = term(rs.point_anchor - x[a], rs.point_k, rs.point_rt)
        own = (a >= lo) & (a < hi)
        np.add.at(F, a[own], f[own])
        E += float(e[own].sum())
    if rs.n_pair:
        i, j = rs.pair_ij[:, 0], rs.pair_ij[:, 1]
        f, e = term(x[j] - x[i], rs.pair_k, rs.pair_rt)
        own_i, own_j = (i >= lo) & (i < hi), (j >= lo) & (j < hi)
        np.add.at(F, i[own_i], f[own_i])
        np.add.at(F, j[own_j], -f[own_j])
        E += float(e[own_i].sum())
    return E, F


def hydrogen_bond_restraints(names, positions) -> RestraintSet:
    """The ``--constraints`` springs: ``PDBAnalyzer.find_bonded_atoms("H")`` restated (utils.py:201-221).  Every atom whose
    name starts with "H" is paired with every other atom within r_cov(H) + r_cov(partner) + 0.2 A, the partner's radius
    looked up by the first letter of its name (0 for letters not in the table); pairs in the reference's order (hydrogens
    by index, partners by index), k = 15 eV/A^2, rt = that bound.  ``names`` / ``positions`` must come from the same
    file as the protein state (atom orders differ between the example PDBs).  Raises ``ValueError`` where the reference
    asserts: when the number of pairs differs from the number of hydrogens."""
    names = [str(s).strip() for s in names]
    pos = np.asarray(positions, dtype=np.float64)
    r_h = COVALENT_RADII["H"]
    bound = np.array([(r_h + COVALENT_RADII.get(s[0], 0)) + 0.2 for s in names])
    hyd = [i for i, s in enumerate(names) if s.startswith("H")]
    pairs, rt = [], []
    for h in hyd:
        dist = np.linalg.norm(pos[h] - pos, axis=1)
        for p in np.flatnonzero(dist <= bound):
            if p != h:
                pairs.append((h, int(p)))
                rt.append(bound[p])
    if len(pairs) != len(hyd):
        raise ValueError(f"hydrogen constraints: {len(pairs)} hydrogen covalent bonds for {len(hyd)} hydrogens")
    return RestraintSet(pair_ij=np.asarray(pairs, dtype=np.int32).reshape(-1, 2), pair_k=np.full(len(pairs), HBOND_K),
                        pair_rt=np.asarray(rt))


def position_restraints(x, k_kcal: float) -> RestraintSet:
    """Every atom tied to its position in x (a copy) with k = k_kcal kcal/mol/A^2, rt = 0 (simulator.py:148-155)."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    return RestraintSet(np.arange(n, dtype=np.int32), x.copy(), np.full(n, k_kcal * KCAL_MOL), np.zeros(n))


class Restrained:
    """``force_fn`` wrapper for the host :class:`ai2bmd_b200.md.Langevin`: the wrapped (E, F) plus :func:`hookean` on
    ``self.restraints``, a mutable set the caller may replace between steps (then call :func:`set_restraints`)."""

    def __init__(self, force_fn, restraints: RestraintSet = None):
        self.force_fn = force_fn
        self.restraints = restraints if restraints is not None else RestraintSet()

    def __call__(self, x):
        e, f = self.force_fn(x)
        if self.restraints.empty:
            return e, f
        er, fr = hookean(x, self.restraints)
        return e + er, f + fr


def _is_device(md) -> bool:
    return hasattr(md, "engine")


def _wrapper(md) -> Restrained:
    if not isinstance(md.force_fn, Restrained):
        raise TypeError("the host integrator needs its force_fn wrapped in restraints.Restrained")
    return md.force_fn


def get_restraints(md) -> RestraintSet:
    """The restraint set in force on a DeviceLangevin or on a host Langevin with a :class:`Restrained` force_fn."""
    return md.restraints if _is_device(md) else _wrapper(md).restraints


def set_restraints(md, rs: RestraintSet) -> None:
    """Replace the restraint set of either integrator and recompute its forces at the current positions, so the next
    half-kick already uses the new set (ASE's Langevin.step applies the current constraints to every force request)."""
    if _is_device(md):
        md.set_restraints(rs)
        return
    _wrapper(md).restraints = rs
    md.energy, md.f = md.force_fn(md.x)


def positions(md) -> np.ndarray:
    return md.state()[0] if _is_device(md) else md.x.copy()


def pre_equilibrate(md, steps_per_stage: int, stages=PREEQ_STAGES) -> None:
    """The reference's pre-equilibration (simulator.py:139-166) on either integrator: for every stage k, tie every atom
    to where it stands now with k kcal/mol/A^2 on top of the current set, run ``steps_per_stage`` steps, restore the
    previous set.  Forces are refreshed at every change of the set."""
    prev = get_restraints(md)
    for k in stages:
        set_restraints(md, prev + position_restraints(positions(md), k))
        md.run(steps_per_stage)
        set_restraints(md, prev)
