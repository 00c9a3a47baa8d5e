"""CPU restatement of the reference's PME non-bonded term -- TEST INFRASTRUCTURE ONLY (checker of
``ai2bmd_b200/csrc/k_pme.cuh``; never imported by the product path).

Follows ``PMENonBondedCalculator`` (``/root/reference/src/Calculators/pme.py:77-214``):

  E = [k (E_rec + E_dir(P) + E_adj(X) + slf + neutral - E_dir(X)) + E_LJ(P) - E_LJ(X)] * kJ/mol
  F = sum_P (F_LJ + F_C) - sum_X (F_LJ + F_C)          on dst, F_C the plain (unscreened) Coulomb force

with P every ordered pair i != j closer than the cutoff (no periodic images, pairs inside a dipeptide included), X every
ordered pair inside a dipeptide (``distancefrag.py:355-363``), every pair sum carrying 1/2.  The reciprocal term gives
no force.

* :func:`spme_erec` -- smooth PME reciprocal energy (Essmann et al., J. Chem. Phys. 103, 8577 (1995)), order-4 cardinal
  B-splines, Euler exponential-spline moduli, fp64 numpy.  helpme (the library the reference calls) is not vendored, so
  its arithmetic is not pinned; this is the standard algorithm restated.
* :func:`ewald_erec` -- the exact Ewald reciprocal sum, the checker of :func:`spme_erec`.
* :func:`pme` -- the whole calculator in fp64 with the net-per-pair formulation the kernel uses (an excluded pair inside
  the cutoff contributes only its erf term, beyond it also minus its LJ / Coulomb / erfc terms), or, with
  ``dtype=torch.float32``, in the reference's own formulation (sums over P and X, subtracted) in fp32.
"""
import numpy as np
import torch

from oracle.nonbonded_ref import C, _eps0, kJ, mol, nm, pi

COULOMB_K = 1 / (4 * pi * _eps0) * 10e6 * mol * C ** (-2)      # pme.py:120


def grid_dims(cell, spacing=1.0):
    """pme.py:146-149: dim = int(cell_len / grid_spacing) per axis."""
    return tuple(int(c / spacing) for c in cell)


def _spline4(u):
    """Order-4 cardinal B-spline weights of fractional grid coordinates u [n]: (base [n] int, w [n,4]); grid point
    base - t gets weight M4(frac(u) + t), t = 0..3."""
    base = np.floor(u)
    w = u - base
    ws = np.stack([w ** 3 / 6, (-3 * w ** 3 + 3 * w ** 2 + 3 * w + 1) / 6, (3 * w ** 3 - 6 * w ** 2 + 4) / 6,
                   (1 - w) ** 3 / 6], axis=1)
    return base.astype(np.int64), ws


def bspline_moduli(K):
    """|b(m)|^2 of the order-4 Euler exponential spline: 1 / |sum_k M4(k+1) exp(2 pi i m k / K)|^2 = 36 / (4 + 2 cos)^2."""
    return 36.0 / (4.0 + 2.0 * np.cos(2 * np.pi * np.arange(K) / K)) ** 2


def _mvec(K, L):
    m = np.arange(K)
    return np.where(m <= K // 2, m, m - K) / L


def spme_erec(pos, q, cell, grid, beta):
    """Smooth PME reciprocal energy (units of e^2 / Angstrom), orthorhombic cell, fp64."""
    pos = np.asarray(pos, np.float64).reshape(-1, 3)
    q = np.asarray(q, np.float64).reshape(-1)
    K = [int(k) for k in grid]
    Q = np.zeros(K)
    idx, wts = [], []
    for a in range(3):
        base, w = _spline4(pos[:, a] * K[a] / cell[a])
        idx.append((base[:, None] - np.arange(4)[None, :]) % K[a])
        wts.append(w)
    for t1 in range(4):
        for t2 in range(4):
            for t3 in range(4):
                np.add.at(Q, (idx[0][:, t1], idx[1][:, t2], idx[2][:, t3]), q * wts[0][:, t1] * wts[1][:, t2] * wts[2][:, t3])
    F = np.fft.fftn(Q)
    m1, m2, m3 = np.meshgrid(*[_mvec(K[a], cell[a]) for a in range(3)], indexing="ij")
    m2s = m1 ** 2 + m2 ** 2 + m3 ** 2
    m2s[0, 0, 0] = 1.0
    B = np.einsum("i,j,k->ijk", *[bspline_moduli(k) for k in K])
    term = np.exp(-np.pi ** 2 * m2s / beta ** 2) / m2s * B * np.abs(F) ** 2
    term[0, 0, 0] = 0.0
    return float(term.sum() / (2 * np.pi * cell[0] * cell[1] * cell[2]))


def ewald_erec(pos, q, cell, beta, tol=1e-17):
    """Exact Ewald reciprocal energy 1/(2 pi V) sum_{m != 0} exp(-pi^2 m^2 / beta^2) / m^2 |S(m)|^2, truncated where
    the Gaussian factor falls below ``tol``."""
    pos = np.asarray(pos, np.float64).reshape(-1, 3)
    q = np.asarray(q, np.float64).reshape(-1)
    nmax = [int(np.ceil(beta * L * np.sqrt(-np.log(tol)) / np.pi)) for L in cell]
    ex = [np.exp(2j * np.pi * np.outer(pos[:, a] / cell[a], np.arange(-nmax[a], nmax[a] + 1))) for a in range(3)]
    n = len(q)
    S = ((q[:, None] * ex[0])[:, :, None] * ex[1][:, None, :]).reshape(n, -1).T @ ex[2]
    S = S.reshape(len(ex[0][0]), len(ex[1][0]), len(ex[2][0]))
    m1, m2, m3 = np.meshgrid(*[np.arange(-nmax[a], nmax[a] + 1) / cell[a] for a in range(3)], indexing="ij")
    m2s = m1 ** 2 + m2 ** 2 + m3 ** 2
    c = tuple(nmax)
    m2s[c] = 1.0
    term = np.exp(-np.pi ** 2 * m2s / beta ** 2) / m2s * np.abs(S) ** 2
    term[c] = 0.0
    return float(term.sum() / (2 * np.pi * cell[0] * cell[1] * cell[2]))


def self_energy(q, beta):
    """electro_slf, pme.py:86-87."""
    return float(-beta / np.sqrt(np.pi) * (np.asarray(q, np.float64) ** 2).sum())


def neutral_energy(q, cell, grid, beta):
    """electro_neutral, pme.py:99-110: minus the reciprocal and self energy of the total charge alone at the origin
    (helpmelib.MatrixF hands the reciprocal part q_tot in fp32)."""
    q_tot = float(np.asarray(q, np.float64).sum())
    return -spme_erec(np.zeros((1, 3)), [float(np.float32(q_tot))], cell, grid, beta) + beta * q_tot ** 2 / np.sqrt(np.pi)


def radius_pairs(pos32, cutoff):
    """All ordered pairs (src, dst), src != dst, with fp32 |pos[dst] - pos[src]|^2 < cutoff^2 (radius_graph, loop=False,
    no neighbour cap); rows sorted by (dst, src)."""
    p = torch.as_tensor(np.asarray(pos32, np.float32))
    d2 = ((p[:, None, :] - p[None, :, :]) ** 2).sum(-1)
    dst, src = torch.nonzero(d2 < np.float32(cutoff) ** 2, as_tuple=True)
    keep = src != dst
    return src[keep], dst[keep]


def exclude_index(groups):
    """Ordered pairs inside a dipeptide (distancefrag.py:355-363) as a [2, X] tensor, sorted."""
    from oracle.nonbonded_ref import exclude_pairs_from_groups
    return torch.tensor(sorted(exclude_pairs_from_groups(groups)), dtype=torch.long).t().reshape(2, -1)


def _lj_coul(vec, d2, sig_s, sig_d, eps_s, eps_d, q_s, q_d, k):
    """Per-pair LJ energy (unhalved), LJ + plain Coulomb force vectors, in the reference's operation order."""
    sigmaij = 0.5 * (sig_s + sig_d) * nm
    epsij = torch.sqrt(eps_s * eps_d)
    c6 = (sigmaij ** 2 / d2) ** 3
    c12 = c6 ** 2
    e_lj = 4 * epsij * (c12 - c6)
    f = (24 * epsij * (2 * c12 - c6) / d2).unsqueeze(-1) * vec
    d = torch.sqrt(d2)
    f = f + (k * q_s * q_d / d / d2).unsqueeze(-1) * vec
    return e_lj, f


def pme(positions, charges, sigmas, epsilons, ex_index, cell, grid, beta=0.3, cutoff=9.0, dtype=torch.float64,
        e_rec=None):
    """(energy [eV], forces [n,3] eV/A, terms) of pme.py:155-214.  ``ex_index`` [2, X] (src, dst) of the excluded pairs.
    terms: E_dir, E_adj, E_ex, E_rec, slf, neutral (e^2/A), E_LJ, E_LJ_ex (kJ/mol), each pair sum halved.  In fp64 E_dir /
    E_LJ are over the non-excluded pairs inside the cutoff and E_ex / E_LJ_ex over the excluded pairs beyond it (the
    net formulation); in fp32 they are the reference's sums over P and X."""
    n = len(charges)
    k = COULOMB_K
    pos = torch.as_tensor(np.asarray(positions, np.float32).astype(np.float64 if dtype == torch.float64 else np.float32))
    q = torch.as_tensor(np.asarray(charges), dtype=dtype)
    sig = torch.as_tensor(np.asarray(sigmas), dtype=dtype)
    eps = torch.as_tensor(np.asarray(epsilons), dtype=dtype)
    src, dst = radius_pairs(positions, cutoff)
    src_ex, dst_ex = ex_index
    if dtype == torch.float64:                        # net formulation: drop the excluded pairs from P
        ex = set(zip(src_ex.tolist(), dst_ex.tolist()))
        keep = torch.tensor([(a, b) not in ex for a, b in zip(src.tolist(), dst.tolist())], dtype=torch.bool)
        src, dst = src[keep], dst[keep]
        vx = pos[dst_ex] - pos[src_ex]
        far = (vx.to(torch.float32) ** 2).sum(-1) >= np.float32(cutoff) ** 2   # the kernel's fp32 cutoff test
        src_far, dst_far = src_ex[far], dst_ex[far]
    else:
        src_far, dst_far = src_ex, dst_ex
    vec = pos[dst] - pos[src]
    d2 = (vec ** 2).sum(-1)
    e_lj, f = _lj_coul(vec, d2, sig[src], sig[dst], eps[src], eps[dst], q[src], q[dst], k)
    vec_x = pos[dst_far] - pos[src_far]
    d2_x = (vec_x ** 2).sum(-1)
    e_lj_x, f_x = _lj_coul(vec_x, d2_x, sig[src_far], sig[dst_far], eps[src_far], eps[dst_far], q[src_far], q[dst_far], k)

    def dir_(s, d, fn):
        dist = torch.norm(pos[d] - pos[s], dim=1)
        return 0.5 * (q[s] * q[d] * fn(beta * dist) / dist).sum()

    t = dict(E_dir=dir_(src, dst, torch.special.erfc), E_adj=-dir_(src_ex, dst_ex, torch.special.erf),
             E_ex=dir_(src_far, dst_far, torch.special.erfc),
             E_rec=torch.tensor(spme_erec(np.asarray(positions, np.float32), charges, cell, grid, beta) if e_rec is None else e_rec,
                                dtype=dtype),
             slf=torch.tensor(self_energy(charges, beta), dtype=dtype),
             neutral=torch.tensor(neutral_energy(charges, cell, grid, beta), dtype=dtype),
             E_LJ=(e_lj / 2).sum(), E_LJ_ex=(e_lj_x / 2).sum())
    e_c = (t["E_rec"] + t["E_dir"] + t["E_adj"] + t["slf"] + t["neutral"] - t["E_ex"]) * k      # in `dtype`, pme.py:195-209
    energy = float(t["E_LJ"] - t["E_LJ_ex"] + e_c) * (kJ / mol)
    force = torch.zeros((n, 3), dtype=dtype).index_add_(0, dst, f) - torch.zeros((n, 3), dtype=dtype).index_add_(0, dst_far, f_x)
    return energy, force.numpy().astype(np.float64) * (kJ / mol), {key: float(v) for key, v in t.items()}
