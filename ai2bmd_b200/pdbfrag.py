"""Capped-protein PDB -> packed dipeptide / ACE-NME fragments (+ whole-protein force map).

A compact restatement of the reference's one-off fragmentation tables, far enough to produce real
``FragmentData`` geometry for the four example proteins:

* residue windows: ``/root/reference/src/Fragmentation/basefrag.py:44-167`` (``get_fragments_index``)
* cap-hydrogen choice and first-approximation placement on the acceptor->removed-atom ray at the sum
  of covalent radii: ``src/Fragmentation/distancefrag.py:365-504`` and ``:34-54``
* ACE-NME k shares its 12 positions with dipeptides k+1 (leading cap group) and k (trailing cap group):
  ``distancefrag.py:286-307``
* interleaved packing dipeptide 0, ACE-NME 0, dipeptide 1, ...: ``distancefrag.py:250-284``
* signed force map (+ dipeptide atoms, - ACE-NME atoms, added hydrogens dropped):
  ``distancefrag.py:335-353``, ``src/Calculators/combiner.py:38-39``

* CYX-CYX pairs: the two dipeptides of a disulfide bridge are evaluated as ONE graph; the second one (by residue number)
  stays in the batch as an empty fragment: ``distancefrag.py:185-238``, pairing rule ``get_cystine_bonds`` ``:804-844``

Atom order inside a fragment is this module's own (leading cap group, residue, trailing cap group, added hydrogens after
the real atoms of their group); the reference reorders every dipeptide into AMBER order through ``seq_dict.pkl``
(``distancefrag.py:506-737``).  ViSNet is permutation-equivariant, so energies and forces do not depend on it as long as no
atom has more than 32 candidates inside the cutoff (the first-32-by-index rule is order dependent: ``neighbour_cap_margin``
reports the margin, and the AMBER order of a dipeptide is available through ``ai2bmd_b200.caph.table_layout``).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Tuple

import numpy as np

from .fragment_data import FragmentData

_Z = {"H": 1, "C": 6, "N": 7, "O": 8, "S": 16}
_RCOV = {"C": 0.76, "N": 0.71, "H": 0.31}   # distancefrag.py:383-388


@dataclass
class CappedProtein:
    names: List[str]        # atom names (CA, HA, ...)
    resnames: List[str]
    resnums: np.ndarray     # 1-based, contiguous
    elements: List[str]
    positions: np.ndarray   # [n,3] float64 Angstrom

    def __len__(self):
        return len(self.names)


def read_pdb(path: str) -> CappedProtein:
    names, resn, resi, elem, xyz = [], [], [], [], []
    with open(path) as fh:
        for line in fh:
            if not line.startswith(("ATOM", "HETATM")):
                continue
            names.append(line[12:16].strip())
            resn.append(line[17:20].strip())
            resi.append(int(line[22:26]))
            xyz.append((float(line[30:38]), float(line[38:46]), float(line[46:54])))
            e = line[76:78].strip() if len(line) >= 78 else ""
            elem.append(e if e else names[-1][0])
    resi = np.asarray(resi)
    resi = resi - resi.min() + 1
    return CappedProtein(names, resn, resi, elem, np.asarray(xyz, dtype=np.float64))


def read_cell(path: str) -> Tuple[float, float, float]:
    """Cell lengths a, b, c (A) of the PDB's ``CRYST1`` record -- the cell the reference's PME term uses
    (``pme.py:146``, an orthorhombic ``XAligned`` lattice).  Raises ``ValueError`` when the record is missing or an
    angle is not 90 degrees."""
    with open(path) as fh:
        for line in fh:
            if line.startswith("CRYST1"):
                a, b, c = float(line[6:15]), float(line[15:24]), float(line[24:33])
                angles = (float(line[33:40]), float(line[40:47]), float(line[47:54]))
                if any(abs(x - 90.0) > 1e-6 for x in angles):
                    raise ValueError(f"{path}: CRYST1 angles {angles} are not all 90 degrees (PME needs an orthorhombic cell)")
                return a, b, c
    raise ValueError(f"{path}: no CRYST1 record (PME needs the cell)")


@dataclass
class ProteinMap:
    """Whole-protein reduction map: F_prot[dst_atom] += sign * F_frag[src_atom]; E = sum sign_g * E_g."""
    n_protein: int
    src_atom: np.ndarray    # int32 [M] index into the packed fragment atoms
    dst_atom: np.ndarray    # int32 [M] index into the protein
    sign: np.ndarray        # float32 [M]
    frag_sign: np.ndarray   # float32 [G] (+1 dipeptide, -1 ACE-NME)


@dataclass
class FragmentRecipe:
    """How every packed fragment atom follows the protein coordinates (``distancefrag.py:34-54``): real atoms
    copy ``P[real]``; an added cap hydrogen sits at ``P[acc] + unit(P[rem] - P[acc]) * blen``."""
    real: np.ndarray        # int32 [N] protein index, -1 for an added hydrogen
    acc: np.ndarray         # int32 [N] acceptor protein index (added hydrogens only, else 0)
    rem: np.ndarray         # int32 [N] removed-atom protein index (added hydrogens only, else 0)
    blen: np.ndarray        # float32 [N] bond length

    def positions(self, prot_pos: np.ndarray) -> np.ndarray:
        p = np.asarray(prot_pos, dtype=np.float64)
        out = p[np.maximum(self.real, 0)]
        cap = self.real < 0
        if cap.any():
            d = p[self.rem[cap]] - p[self.acc[cap]]
            d /= np.linalg.norm(d, axis=1, keepdims=True)
            out[cap] = p[self.acc[cap]] + d * self.blen[cap, None]
        return out.astype(np.float32)


class _Cap:
    """Marker for an added hydrogen: (acceptor, removed atom, bond length)."""
    def __init__(self, acc, rem, blen):
        self.acc, self.rem, self.blen = acc, rem, blen


def _cap_h(pos, acceptor, removed, acc_elem):
    return _Cap(acceptor, removed, _RCOV[acc_elem] + _RCOV["H"])


def cystine_pairs(prot: CappedProtein, centres) -> dict:
    """``{dipeptide i: dipeptide j}`` for the dipeptides (indices into ``centres``, the centre residue numbers) whose centre
    residue is CYX, paired by the shortest SG-SG distance exactly as ``DistanceFragment.get_cystine_bonds`` does
    (``distancefrag.py:804-844``): walk the CYX dipeptides in order, take each one's nearest SG partner unless either of the
    two is already paired."""
    cyx, sg = [], []
    for k, c in enumerate(centres):
        members = [i for i in range(len(prot)) if prot.resnums[i] == c]
        if prot.resnames[members[0]] != "CYX":
            continue
        s_atoms = [i for i in members if prot.names[i] == "SG"]
        if len(s_atoms) != 1:
            raise ValueError(f"CYX residue {c} has {len(s_atoms)} SG atoms")
        cyx.append(k)
        sg.append(s_atoms[0])
    if len(cyx) % 2:
        raise ValueError("odd number of CYX residues")
    if not cyx:
        return {}
    P = np.asarray(prot.positions, dtype=np.float64)[sg]
    dist = np.linalg.norm(P[None, :] - P[:, None], axis=-1)
    np.fill_diagonal(dist, np.inf)
    pairs = {}
    for i, j in enumerate(np.argmin(dist, axis=-1)):
        if i in pairs or int(j) in pairs:
            continue
        pairs[i] = int(j)
    return {cyx[i]: cyx[j] for i, j in pairs.items()}


def neighbour_cap_margin(frags: FragmentData, cutoff: float = 5.0, cap: int = 32) -> int:
    """``cap`` minus the largest number of atoms (itself included) any atom has strictly inside the cutoff within its own
    fragment.  Non-negative: no neighbour list is truncated, so the atom order inside the fragments cannot change the
    result; negative: the first-32-by-index rule drops neighbours and the reference's AMBER order matters."""
    worst = 0
    for g in range(len(frags)):
        p = np.asarray(frags.pos[int(frags.start[g]):int(frags.end[g])], dtype=np.float32)
        if len(p) == 0:
            continue
        d2 = ((p[:, None, :] - p[None, :, :]) ** 2).sum(-1)
        worst = max(worst, int((d2 < np.float32(cutoff) ** 2).sum(1).max()))
    return cap - worst


def fragment_protein(prot: CappedProtein, with_recipe: bool = False):
    R = int(prot.resnums.max())
    assert len(set(prot.resnums.tolist())) == R, "residue numbers are not continuous"
    nd, na = R - 2, R - 3
    if nd < 2:
        raise NotImplementedError("3 or fewer residues (incl. caps): run un-fragmented (--mode visnet)")
    by_res = {r: [i for i in range(len(prot)) if prot.resnums[i] == r] for r in range(1, R + 1)}

    def pick(r, pred):
        return [i for i in by_res[r] if pred(prot.names[i])]

    def atom(r, name):
        hit = [i for i in by_res[r] if prot.names[i] == name]
        return hit[0] if hit else None

    is_ca = lambda n: n == "CA" or n.startswith("HA")
    P = prot.positions

    # leading (ACE-like) and trailing (NME-like) cap groups per junction
    def lead_group(r):
        """Atoms dipeptide (centre r+1) takes from residue r: [(protein index | None, element, xyz)]."""
        if prot.resnames[by_res[r][0]] == "ACE":
            return [(i, prot.elements[i], P[i]) for i in by_res[r]]
        out = [(i, prot.elements[i], P[i]) for i in pick(r, lambda n: is_ca(n) or n in ("C", "O"))]
        ca = atom(r, "CA")
        out.append((None, "H", _cap_h(P, ca, atom(r, "N"), "C")))
        if prot.resnames[by_res[r][0]] != "GLY":
            out.append((None, "H", _cap_h(P, ca, atom(r, "CB"), "C")))
        return out

    def trail_group(r):
        """Atoms dipeptide (centre r-1) takes from residue r."""
        if prot.resnames[by_res[r][0]] == "NME":
            return [(i, prot.elements[i], P[i]) for i in by_res[r]]
        out = [(i, prot.elements[i], P[i]) for i in pick(r, lambda n: is_ca(n) or n in ("N", "H"))]
        ca = atom(r, "CA")
        out.append((None, "H", _cap_h(P, ca, atom(r, "C"), "C")))
        rn = prot.resnames[by_res[r][0]]
        if rn != "GLY":
            out.append((None, "H", _cap_h(P, ca, atom(r, "CB"), "C")))
        if rn == "PRO":
            out.append((None, "H", _cap_h(P, atom(r, "N"), atom(r, "CD"), "N")))
        return out

    frags = []  # (sign, [(prot_idx|None, elem, xyz)])
    for k in range(nd):
        centre = k + 2
        atoms = lead_group(centre - 1) + [(i, prot.elements[i], P[i]) for i in by_res[centre]] + \
            trail_group(centre + 1)
        frags.append((+1.0, atoms))
        if k < na:
            # ACE-NME k: leading group of dipeptide k+1 (from residue k+2) + trailing group of dipeptide k (k+3)
            frags.append((-1.0, lead_group(centre) + trail_group(centre + 1)))

    # disulfide bridges: the pair is one graph, the partner's slot stays as an empty fragment (distancefrag.py:185-238)
    for i, j in cystine_pairs(prot, [k + 2 for k in range(nd)]).items():
        frags[2 * i] = (frags[2 * i][0], frags[2 * i][1] + frags[2 * j][1])
        frags[2 * j] = (frags[2 * j][0], [])

    z, batch, start, end = [], [], [], []
    src, dst, sgn, fsgn = [], [], [], []
    r_real, r_acc, r_rem, r_len = [], [], [], []
    off = 0
    for g, (s, atoms) in enumerate(frags):
        start.append(off)
        for (pi, el, xyz) in atoms:
            z.append(_Z[el])
            batch.append(g)
            if pi is not None:
                src.append(off)
                dst.append(pi)
                sgn.append(s)
                r_real.append(pi); r_acc.append(0); r_rem.append(0); r_len.append(0.0)
            else:
                r_real.append(-1); r_acc.append(xyz.acc); r_rem.append(xyz.rem); r_len.append(xyz.blen)
            off += 1
        end.append(off)
        fsgn.append(s)
    recipe = FragmentRecipe(np.asarray(r_real, dtype=np.int32), np.asarray(r_acc, dtype=np.int32),
                            np.asarray(r_rem, dtype=np.int32), np.asarray(r_len, dtype=np.float32))
    pos = recipe.positions(P)
    fd = FragmentData(np.asarray(z, dtype=np.int64), np.asarray(pos, dtype=np.float32),
                      np.asarray(start, dtype=np.int64), np.asarray(end, dtype=np.int64),
                      np.asarray(batch, dtype=np.int64))
    pm = ProteinMap(len(prot), np.asarray(src, dtype=np.int32), np.asarray(dst, dtype=np.int32),
                    np.asarray(sgn, dtype=np.float32), np.asarray(fsgn, dtype=np.float32))
    return (fd, pm, recipe) if with_recipe else (fd, pm)


def single_graph(z, pos) -> FragmentData:
    """Un-fragmented mode (``visnet_calculator.py:142-148``): the whole input is one graph."""
    n = len(z)
    return FragmentData(np.asarray(z, dtype=np.int64), np.asarray(pos, dtype=np.float32),
                        np.array([0], dtype=np.int64), np.array([n], dtype=np.int64),
                        np.zeros((n,), dtype=np.int64))
