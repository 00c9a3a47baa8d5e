#!/usr/bin/env python
"""Generate ``reference_pme.npz``.  Runs ONLY where the reference source tree is available.

    python tests/golden/make_pme_golden.py

Energy, forces and terms of the reference's OWN ``src/Calculators/pme.py``: the module functions (``setup``,
``set_lattice_vectors``, ``compute_E_rec``, ``electro_dir`` / ``_slf`` / ``_adj`` / ``_neutral``) and the
``PMENonBondedCalculator`` class body, extracted with ``ast`` because the module imports helpmelib / torch_geometric /
torch_scatter / ase / AIMD.  Stand-ins:

* ``helpmelib.PMEInstanceF`` -- its reciprocal energy is ``oracle.pme_ref.spme_erec`` (helpme is not vendored);
* ``torch_geometric.nn.radius_graph`` -- brute force over all pairs, fp32 ``d^2 < r^2``, ``loop=False``, no neighbour cap;
* ``torch_scatter.scatter_add`` -- ``index_add_``;
* the six ``ase.units`` constants of ``oracle/nonbonded_ref.py`` (CODATA 2014, recalled);
* a ``Protein`` stub with the attributes the class touches; ``exclude_index`` holds the ordered dipeptide pairs of
  ``distancefrag.py:355-363`` sorted (the reference lists a Python set).

Pinned: everything in ``pme.py`` except helpme's arithmetic and ``radius_graph``.  Inputs: ``synthetic_parameters`` (seed
1, as ``reference_nonbonded.npz``) on Chignolin with the ``chig.pdb`` cell, the same coordinates with the
``chig-preeq-nowat.pdb`` cell, and ABD (746 atoms) in a synthetic 60 A cube.  Writes only ``reference_pme.npz``.
"""
import ast
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)
REF = "/root/reference"

from ai2bmd_b200.fixtures import load_fragments, load_protein          # noqa: E402
from ai2bmd_b200.nonbonded import dipeptide_atom_sets, synthetic_parameters   # noqa: E402
from ai2bmd_b200.pdbfrag import read_cell                              # noqa: E402
from oracle import nonbonded_ref as NB, pme_ref as PR                  # noqa: E402

CASES = (("chig", "chig", f"{REF}/examples/chig.pdb"),
         ("chig_preeq", "chig", f"{REF}/examples/chig_preprocessed/chig-preeq-nowat.pdb"),
         ("abd", "abd", (60.0, 60.0, 60.0)))


class _PMEInstanceF:
    """helpmelib.PMEInstanceF: setup / set_lattice_vectors / compute_E_rec for rPower 1, orthorhombic XAligned cells."""
    class LatticeType:
        XAligned = "XAligned"

    def setup(self, rPower, kappa, splineOrder, dimA, dimB, dimC, scaleFactor, numThreads):
        assert rPower == 1 and splineOrder == 4 and scaleFactor == 1
        self.kappa, self.dims = kappa, (dimA, dimB, dimC)

    def set_lattice_vectors(self, a, b, c, alpha, beta, gamma, latticeType):
        assert (alpha, beta, gamma) == (90, 90, 90) and latticeType == "XAligned"
        self.cell = (a, b, c)

    def compute_E_rec(self, parameterAngMom, parameters, coordinates):
        assert parameterAngMom == 0
        return PR.spme_erec(np.asarray(coordinates), np.asarray(parameters).reshape(-1), self.cell, self.dims, self.kappa)


def _radius_graph(x, r, max_num_neighbors=32, loop=False):
    assert loop is False and max_num_neighbors >= len(x)
    src, dst = PR.radius_pairs(x.numpy(), r)
    return torch.stack([src, dst])


def load_reference_pme():
    helpmelib = types.SimpleNamespace(PMEInstanceF=_PMEInstanceF, MatrixF=lambda a: np.asarray(a, dtype=np.float32))
    ns = {"np": np, "torch": torch, "helpmelib": helpmelib, "radius_graph": _radius_graph,
          "erf": torch.special.erf, "erfc": torch.special.erfc,
          "scatter_add": lambda src, index, dim=0, dim_size=None: torch.zeros((dim_size,) + src.shape[1:], dtype=src.dtype).index_add_(dim, index, src),
          "C": NB.C, "_eps0": NB._eps0, "kJ": NB.kJ, "mol": NB.mol, "nm": NB.nm, "pi": NB.pi, "Protein": object}
    tree = ast.parse(open(f"{REF}/src/Calculators/pme.py").read())
    body = [n for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef))]
    exec(compile(ast.Module(body=body, type_ignores=[]), "ref_pme", "exec"), ns)
    return ns


def main():
    ns = load_reference_pme()
    out = {}
    for key, prot_name, cell_src in CASES:
        fd, pm = load_fragments(prot_name)
        prot_pos, prot_z, recipe = load_protein(prot_name)
        cell = read_cell(cell_src) if isinstance(cell_src, str) else cell_src
        q, sg, ep = synthetic_parameters(prot_z, seed=1)
        groups = dipeptide_atom_sets(fd, recipe, pm)
        ex = PR.exclude_index(groups)

        class FakeProtein:                   # the attributes PMENonBondedCalculator touches
            def __init__(self):
                self.positions = np.asarray(prot_pos, dtype=np.float64)
                self.sigmas, self.epsilons, self.charges = sg, ep, q
                self.exclude_index = ex
                self.cell = np.diag(np.asarray(cell, dtype=np.float64))

            def get_positions(self):
                return self.positions

            def __len__(self):
                return len(self.positions)

        prot = FakeProtein()
        calc = ns["PMENonBondedCalculator"](device="cpu")
        calc.set_parameters(prot)
        energy, force = calc(prot)
        pos = torch.tensor(prot.get_positions(), dtype=torch.float)
        src, dst = _radius_graph(pos, calc.cutoff, max_num_neighbors=len(pos), loop=False)
        ch = calc.charges
        terms = dict(E_rec=ns["compute_E_rec"](calc.pme, ns["helpmelib"].MatrixF, 0, calc.charges_cpu, pos),
                     E_dir=float(ns["electro_dir"](pos, ch, (src, dst), calc.beta)),
                     E_adj=float(ns["electro_adj"](pos, ch, prot.exclude_index, calc.beta)),
                     E_ex=float(ns["electro_dir"](pos, ch, (calc.src_ex, calc.dst_ex), calc.beta)),
                     slf=float(calc.coulomb_slf), neutral=float(calc.coulomb_neutral))
        out.update({f"{key}_{k}": v for k, v in dict(
            positions=prot.positions, charges=q, sigmas=sg, epsilons=ep, cell=np.asarray(cell, np.float64),
            grid=np.array(calc.pme.dims, np.int32), src_ex=ex[0].numpy(), dst_ex=ex[1].numpy(),
            energy=np.float64(energy), forces=force, **{f"term_{k}": np.float64(v) for k, v in terms.items()}).items()})
        print(f"pme reference ({key}): {len(q)} atoms, cell {cell}, grid {calc.pme.dims}, {src.numel()} pairs < "
              f"{calc.cutoff} A, {ex.shape[1]} excluded, E = {energy:.6f} eV, max|F| = {np.abs(force).max():.4f} eV/A")
    np.savez_compressed(os.path.join(HERE, "reference_pme.npz"), **out)


if __name__ == "__main__":
    main()
