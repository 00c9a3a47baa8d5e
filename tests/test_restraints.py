"""Host side of the Hookean restraints (ai2bmd_b200/restraints.py): the hydrogen-bond pairs against the reference's own
PDBAnalyzer, the fp64 restatement of ASE's Hookean, and the pre-equilibration protocol on the host integrator."""
import json
import os

import numpy as np
import pytest

from ai2bmd_b200 import restraints as R
from ai2bmd_b200.md import Langevin

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_hbond_restraints.json")


@pytest.fixture(scope="module")
def hbond_golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


@pytest.mark.parametrize("name", ["chig", "chig-preeq-nowat", "trpcage", "ww", "abd"])
def test_hydrogen_bond_restraints_equal_reference(hbond_golden, name):
    g = hbond_golden[name]
    rs = R.hydrogen_bond_restraints(g["names"], np.asarray(g["positions"]))
    ref = g["pairs"]
    assert rs.n_point == 0 and rs.n_pair == len(ref)
    assert rs.pair_ij.tolist() == [[i, j] for i, j, _, _ in ref]
    assert rs.pair_rt.tolist() == [rt for _, _, rt, _ in ref]          # bit-exact: same float operations
    assert rs.pair_k.tolist() == [k for _, _, _, k in ref]


@pytest.mark.parametrize("name", ["chig", "trpcage", "ww", "abd"])
def test_hydrogen_bond_input_is_the_protein_state_file(hbond_golden, name):
    """The example proteins of the fixtures list their atoms as the PDBs the reference's analyzer reads, so the pairs
    index the device state directly."""
    from ai2bmd_b200.fixtures import load_capped_protein
    prot = load_capped_protein(name)
    g = hbond_golden[name]
    assert list(prot.names) == g["names"]
    assert np.array_equal(prot.positions, np.asarray(g["positions"]))


def test_hydrogen_bond_restraints_raise_where_reference_asserts():
    names = ["N", "H", "CA", "HA"]
    pos = np.array([[0.0, 0, 0], [1.0, 0, 0], [5.0, 0, 0], [9.0, 0, 0]])      # HA has no partner
    with pytest.raises(ValueError):
        R.hydrogen_bond_restraints(names, pos)
    pos[3] = [5.0, 1.05, 0]
    rs = R.hydrogen_bond_restraints(names, pos)
    assert rs.pair_ij.tolist() == [[1, 0], [3, 2]]


def _mixed_set(n, rng, x):
    """Point and pair restraints with rt drawn so that about half of them are stretched beyond rt."""
    a = rng.integers(0, n, 10)
    anchor = x[a] + rng.normal(0, 0.5, (10, 3))
    dp = np.linalg.norm(anchor - x[a], axis=1)
    ij = np.array([(i, j) for i, j in rng.integers(0, n, (20, 2)) if i != j][:12])
    dq = np.linalg.norm(x[ij[:, 1]] - x[ij[:, 0]], axis=1)
    return R.RestraintSet(a, anchor, rng.uniform(0.5, 15, 10), dp * rng.uniform(0.3, 1.7, 10),
                          ij, rng.uniform(0.5, 15, len(ij)), dq * rng.uniform(0.3, 1.7, len(ij)))


def test_hookean_forces_are_minus_gradient():
    rng = np.random.default_rng(0)
    n = 16
    x = rng.uniform(0, 4, (n, 3))
    rs = _mixed_set(n, rng, x)
    e0, f = R.hookean(x, rs)
    assert e0 > 0 and np.abs(f).max() > 0.1
    h = 1e-6
    g = np.zeros_like(x)
    for a in range(n):
        for c in range(3):
            xp, xm = x.copy(), x.copy()
            xp[a, c] += h
            xm[a, c] -= h
            g[a, c] = (R.hookean(xp, rs)[0] - R.hookean(xm, rs)[0]) / (2 * h)
    assert np.abs(f + g).max() <= 1e-6 * np.abs(f).max() + 1e-8


def test_hookean_flat_bottom_and_zero_distance():
    x = np.array([[0.0, 0, 0], [1.0, 0, 0], [2.0, 0, 0]])
    inside = R.RestraintSet(point_atom=[0], point_anchor=[[0.3, 0, 0]], point_k=[5.0], point_rt=[0.5],
                            pair_ij=[[1, 2]], pair_k=[15.0], pair_rt=[1.2])
    e, f = R.hookean(x, inside)
    assert e == 0.0 and not f.any()
    at_anchor = R.RestraintSet(point_atom=[2], point_anchor=[[2.0, 0, 0]], point_k=[5.0], point_rt=[0.0])
    e, f = R.hookean(x, at_anchor)
    assert e == 0.0 and np.isfinite(f).all() and not f.any()
    stretched = R.RestraintSet(pair_ij=[[0, 2]], pair_k=[4.0], pair_rt=[1.5])
    e, f = R.hookean(x, stretched)
    assert e == pytest.approx(0.5 * 4.0 * 0.25) and f[0].tolist() == pytest.approx([2.0, 0, 0]) and f[2].tolist() == pytest.approx([-2.0, 0, 0])


def test_hookean_pair_forces_sum_to_zero():
    rng = np.random.default_rng(1)
    x = rng.uniform(0, 4, (20, 3))
    rs = _mixed_set(20, rng, x)
    pairs = R.RestraintSet(pair_ij=rs.pair_ij, pair_k=rs.pair_k, pair_rt=rs.pair_rt)
    e, f = R.hookean(x, pairs)
    assert e > 0 and np.abs(f.sum(0)).max() <= 1e-12 * max(1.0, np.abs(f).max())


@pytest.mark.parametrize("m", [0, 1, 7, 19, 20])
def test_hookean_slices_sum_to_whole(m):
    rng = np.random.default_rng(2)
    x = rng.uniform(0, 4, (20, 3))
    rs = _mixed_set(20, rng, x)
    e, f = R.hookean(x, rs)
    e0, f0 = R.hookean(x, rs.sliced(0, m))
    e1, f1 = R.hookean(x, rs.sliced(m, 20))
    assert abs(e0 + e1 - e) <= 1e-12 * e and np.abs(f0 + f1 - f).max() <= 1e-12 * np.abs(f).max()
    assert not f0[m:].any() and not f1[:m].any()


class _Recording(R.Restrained):
    """Restrained force_fn that remembers every set installed and the positions at that moment."""

    def __init__(self, force_fn, md_ref):
        self.log, self._md = [], md_ref
        super().__init__(force_fn)

    @property
    def restraints(self):
        return self._rs

    @restraints.setter
    def restraints(self, rs):
        self._rs = rs
        md = self._md()
        if md is not None:
            self.log.append((rs, md.x.copy(), md.nsteps))


def _host_md(prev=None):
    rng = np.random.default_rng(4)
    n = 12
    x0 = rng.uniform(0, 6, (n, 3))
    c = 0.3

    def well(x):                       # cheap analytic potential: every atom in a harmonic well around x0
        d = x - x0
        return 0.5 * c * float((d * d).sum()), -c * d

    holder = {}
    fn = _Recording(well, lambda: holder.get("md"))
    if prev is not None:
        fn.restraints = prev
    md = Langevin(x0, np.full(n, 6), fn, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.01, seed=0)
    holder["md"] = md
    return md, fn, well


@pytest.mark.parametrize("with_prev", [False, True])
def test_pre_equilibrate_host_protocol(with_prev):
    prev = R.RestraintSet(pair_ij=[[0, 1]], pair_k=[15.0], pair_rt=[1.2]) if with_prev else R.RestraintSet()
    md, fn, well = _host_md(prev)
    steps = 7
    R.pre_equilibrate(md, steps)
    assert md.nsteps == 5 * steps
    assert R.get_restraints(md) is prev
    log = fn.log
    assert len(log) == 10                                              # set, restore per stage
    for s, k in enumerate(R.PREEQ_STAGES):
        rs, x_at, nsteps = log[2 * s]
        assert nsteps == s * steps
        assert rs.n_pair == prev.n_pair and np.array_equal(rs.pair_ij, prev.pair_ij)
        assert rs.n_point == len(md.x) and rs.point_atom.tolist() == list(range(len(md.x)))
        assert np.array_equal(rs.point_k, np.full(len(md.x), k * R.KCAL_MOL)) and not rs.point_rt.any()
        assert np.array_equal(rs.point_anchor, x_at)                   # anchored where the atoms stood at the stage start
        assert log[2 * s + 1][0] is prev and log[2 * s + 1][2] == (s + 1) * steps
    # the forces were refreshed with the restored set
    e, f = well(md.x)
    er, fr = R.hookean(md.x, prev)
    assert md.energy == e + er and np.array_equal(md.f, f + fr)


def test_kcal_mol_is_ase_codata_2014():
    assert R.KCAL_MOL == pytest.approx(0.0433641, rel=1e-6)
    assert R.position_restraints(np.zeros((3, 3)), 10).point_k.tolist() == [10 * R.KCAL_MOL] * 3
