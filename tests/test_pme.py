"""PME non-bonded term on CPU: the SPME oracle against the exact Ewald sum, its invariants, the whole-calculator oracle
against the reference's own pme.py (tests/golden/reference_pme.npz), fixture guards and the host builders."""
import os

import numpy as np
import pytest
import torch

from ai2bmd_b200.pdbfrag import read_cell
from oracle import pme_ref as PR

CHIG_CELL = (25.939, 27.327, 23.669)            # CRYST1 of the reference's examples/chig.pdb
PREEQ_CELL = (55.216, 59.157, 53.428)           # CRYST1 of examples/chig_preprocessed/chig-preeq-nowat.pdb
CASES = ("chig", "chig_preeq", "abd")
# Measured gap between the reference's fp32 output and the fp64 net-per-pair oracle on these fixtures: 4.7e-3 / 4.7e-3 /
# 7.4e-3 eV in energy and 1.9e-2 / 1.9e-2 / 1.2e-2 eV/A in forces.  It is the reference's own fp32 cancellation noise:
# the dipeptide pairs inside the cutoff are added in the sum over P and subtracted in the sum over X, sums of ~1e6
# kJ/mol (the fp64 oracle in either formulation agrees with itself to 1e-10).  Stated tolerance: 2.5x the largest gap.
GOLDEN_E_TOL, GOLDEN_F_TOL = 2e-2, 5e-2


def _random_system(cell, n=175, seed=0):
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0.0, 1.0, (n, 3)) * np.asarray(cell)
    q = rng.uniform(-1.0, 1.0, n)
    return pos, q - q.mean()


@pytest.mark.parametrize("cell", [CHIG_CELL, PREEQ_CELL])
def test_spme_converges_to_ewald(cell):
    """Relative E_rec error of order-4 SPME falls as h^4 with the grid spacing h (measured 2.8e-4 / 1.6e-5 / 8.5e-7 on the
    Chignolin cell and 2.3e-4 / 1.3e-5 / 7.8e-7 on the 55 A cell at 1 / 0.5 / 0.25 A)."""
    pos, q = _random_system(cell)
    ew = PR.ewald_erec(pos, q, cell, 0.3)
    spacings = (1.0, 0.5, 0.25) if cell == CHIG_CELL else (1.0, 0.5)
    bounds = {1.0: 5e-4, 0.5: 3e-5, 0.25: 2e-6}
    err = [abs(PR.spme_erec(pos, q, cell, PR.grid_dims(cell, h), 0.3) - ew) / abs(ew) for h in spacings]
    for h, e in zip(spacings, err):
        assert e <= bounds[h], (h, e)
    for a, b in zip(err, err[1:]):
        assert a / b >= 10.0                      # h^4: 16 per halving


def test_spme_invariants():
    pos, q = _random_system(PREEQ_CELL, seed=1)
    grid = PR.grid_dims(PREEQ_CELL)
    e = PR.spme_erec(pos, q, PREEQ_CELL, grid, 0.3)
    shift = np.array([PREEQ_CELL[0], -2 * PREEQ_CELL[1], 3 * PREEQ_CELL[2]])
    assert abs(PR.spme_erec(pos + shift, q, PREEQ_CELL, grid, 0.3) - e) <= 1e-12 * abs(e)
    perm = np.random.default_rng(2).permutation(len(q))
    assert abs(PR.spme_erec(pos[perm], q[perm], PREEQ_CELL, grid, 0.3) - e) <= 1e-12 * abs(e)
    # the single-particle term behind `neutral` (pme.py:99-110): a lone charge at the origin against the exact sum
    for cell in (CHIG_CELL, PREEQ_CELL):
        g = PR.grid_dims(cell)
        one = PR.spme_erec(np.zeros((1, 3)), [1.5], cell, g, 0.3)
        assert abs(one - PR.ewald_erec(np.zeros((1, 3)), [1.5], cell, 0.3)) <= 1e-3 * abs(one)
        assert PR.neutral_energy([1.0, 0.5], cell, g, 0.3) == -one + 0.3 * 1.5 ** 2 / np.sqrt(np.pi)
        assert abs(PR.neutral_energy([0.5, -0.5], cell, g, 0.3)) == 0.0


def _golden(golden_dir, key):
    g = np.load(os.path.join(golden_dir, "reference_pme.npz"))
    c = {k[len(key) + 1:]: g[k] for k in g.files if k.startswith(key + "_") and not k.startswith(key + "_preeq")}
    c["ex"] = torch.stack([torch.from_numpy(c["src_ex"]), torch.from_numpy(c["dst_ex"])])
    return c


def _oracle(c, dtype):
    return PR.pme(c["positions"], c["charges"], c["sigmas"], c["epsilons"], c["ex"], tuple(c["cell"]), tuple(c["grid"]),
                  dtype=dtype)


@pytest.mark.parametrize("key", CASES)
def test_oracle_equals_the_reference_pme(golden_dir, key):
    """The fp32 oracle restates pme.py's formulation and matches its output to fp32 rounding; the fp64 net-per-pair
    oracle is within the cancellation noise of the reference's fp32 sums (GOLDEN_E_TOL / GOLDEN_F_TOL)."""
    c = _golden(golden_dir, key)
    e32, f32, t32 = _oracle(c, torch.float32)
    assert abs(e32 - float(c["energy"])) <= 1e-4                    # measured <= 1.1e-5 eV (summation order)
    assert np.abs(f32 - c["forces"]).max() <= 1e-6 * np.abs(c["forces"]).max()
    for k in ("E_dir", "E_adj", "E_ex"):
        assert t32[k] == pytest.approx(float(c["term_" + k]), rel=1e-6)
    e64, f64, t64 = _oracle(c, torch.float64)
    assert abs(e64 - float(c["energy"])) <= GOLDEN_E_TOL
    assert np.abs(f64 - c["forces"]).max() <= GOLDEN_F_TOL
    assert t64["E_rec"] == pytest.approx(float(c["term_E_rec"]), rel=1e-6)     # helpme stand-in fed fp32 coordinates
    assert t64["slf"] == pytest.approx(float(c["term_slf"]), rel=1e-6)
    assert abs(t64["neutral"] - float(c["term_neutral"])) <= 1e-12          # neutral charges: both ~0
    assert t64["E_adj"] == pytest.approx(float(c["term_E_adj"]), rel=1e-6)
    net_ref = float(c["term_E_dir"]) - float(c["term_E_ex"])
    assert abs((t64["E_dir"] - t64["E_ex"]) - net_ref) <= 1e-5 * (abs(float(c["term_E_dir"])) + abs(float(c["term_E_ex"])))


def test_fixture_guards(golden_dir):
    """No pair sits within 10 fp32 ulps of d^2 = cutoff^2 (the plain Coulomb force jumps across the cutoff, so the pair
    sets of fp32 and fp64 code must agree), and the excluded pairs beyond the cutoff -- subtracted by the reference
    although never added -- occur."""
    ulp = float(np.spacing(np.float32(81.0)))
    beyond = 0
    for key in CASES:
        c = _golden(golden_dir, key)
        p = c["positions"].astype(np.float32)
        d2 = ((p[:, None, :] - p[None, :, :]) ** 2).sum(-1)
        np.fill_diagonal(d2, 0.0)
        assert np.abs(d2 - np.float32(81.0)).min() >= 10 * ulp, key
        beyond += int((d2[c["dst_ex"], c["src_ex"]] >= 81.0).sum())
    assert beyond > 0


def _pdb(tmp_path, first_line):
    p = tmp_path / "x.pdb"
    p.write_text(first_line + "ATOM      1  N   GLY A   1      -0.001   0.002   0.003  1.00  0.00           N\nEND\n")
    return str(p)


def test_read_cell_and_grid(tmp_path, golden_dir):
    from ai2bmd_b200.nonbonded import PMENonBondedCalculator
    cell = read_cell(_pdb(tmp_path, "CRYST1   25.939   27.327   23.669  90.00  90.00  90.00               1\n"))
    assert cell == CHIG_CELL
    assert PMENonBondedCalculator(None).grid(cell) == (25, 27, 23) == PR.grid_dims(cell)
    assert PMENonBondedCalculator(None).grid(PREEQ_CELL) == (55, 59, 53)
    assert PMENonBondedCalculator(None, grid_spacing=0.5).grid(cell) == (51, 54, 47)
    assert tuple(_golden(golden_dir, "chig")["cell"]) == CHIG_CELL
    assert tuple(_golden(golden_dir, "chig_preeq")["cell"]) == PREEQ_CELL
    with pytest.raises(ValueError, match="no CRYST1"):
        read_cell(_pdb(tmp_path, ""))
    with pytest.raises(ValueError, match="not all 90"):
        read_cell(_pdb(tmp_path, "CRYST1   25.939   27.327   23.669  90.00 109.47  90.00               1\n"))
