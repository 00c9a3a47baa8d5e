#!/usr/bin/env python
"""Generate ``reference_hbond_restraints.json``.  Runs ONLY where the reference source tree is available.

    python tests/golden/make_hbond_golden.py

The hydrogen / partner pairs of the reference's OWN ``PDBAnalyzer.find_bonded_atoms("H")`` (``src/utils/utils.py:169-221``,
the ``--constraints`` springs of ``src/AIMD/simulator.py:168-180``) on chig / chig-preeq-nowat / trpcage / ww / abd, with
the atom names and coordinates the analyzer parsed.  Checker of ``ai2bmd_b200.restraints.hydrogen_bond_restraints``
(``tests/test_restraints.py``).  Kept apart from ``make_golden.py`` so that writing this fixture touches no other one.
"""
import importlib.util
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"

PDBS = (("chig", "chig.pdb"), ("chig-preeq-nowat", "chig_preprocessed/chig-preeq-nowat.pdb"),
        ("trpcage", "trpcage.pdb"), ("ww", "ww.pdb"), ("abd", "abd.pdb"))


def load_reference_utils():
    """The reference's ``utils/utils.py``.  It imports ase / AIMD.arguments by name only (MDObserver uses them,
    PDBAnalyzer does not): stand-in modules are installed for the import and removed after."""
    stubs = {"ase": dict(Atoms=object), "ase.io": {}, "ase.io.trajectory": dict(TrajectoryWriter=object), "ase.md": {},
             "ase.md.md": dict(MolecularDynamics=object), "AIMD": {}, "AIMD.arguments": {}}
    saved = {k: sys.modules.get(k) for k in stubs}
    try:
        for k, attrs in stubs.items():
            sys.modules[k] = types.ModuleType(k)
            for a, v in attrs.items():
                setattr(sys.modules[k], a, v)
        sys.modules["AIMD"].arguments = sys.modules["AIMD.arguments"]
        spec = importlib.util.spec_from_file_location("ref_utils", f"{REF}/src/utils/utils.py")
        um = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(um)
    finally:
        for k, m in saved.items():
            if m is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = m
    return um


def main():
    um = load_reference_utils()
    out = {}
    for name, rel in PDBS:
        an = um.PDBAnalyzer(f"{REF}/examples/{rel}")
        pairs = an.find_bonded_atoms("H")
        out[name] = {"names": [a[0] for a in an.atoms], "positions": [[float(c) for c in a[1]] for a in an.atoms],
                     "pairs": [[int(i), int(j), float(rt), float(k)] for i, j, rt, k in pairs]}
        print(f"hydrogen-bond restraints ({name}): {len(an.atoms)} atoms, {len(pairs)} pairs, "
              f"rt {sorted({round(p[2], 6) for p in pairs})}")
    with open(os.path.join(HERE, "reference_hbond_restraints.json"), "w") as fh:
        json.dump(out, fh, sort_keys=True)


if __name__ == "__main__":
    main()
