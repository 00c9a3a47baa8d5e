"""PME non-bonded term on the device (csrc/k_pme.cuh behind vb_set_pme / vb_pme) against the fp64 oracle and the
reference's own output, alone, sharded and inside the device-resident MD step."""
import os
import sys

import numpy as np
import pytest
import torch

from ai2bmd_b200.fixtures import load_fragments, load_protein
from ai2bmd_b200.nonbonded import dipeptide_atom_sets, exclusion_table, synthetic_parameters
from oracle import pme_ref as PR

sys.path.insert(0, os.path.dirname(__file__))
from test_pme import CHIG_CELL, GOLDEN_E_TOL, GOLDEN_F_TOL, _golden   # noqa: E402

pytestmark = pytest.mark.gpu

X_TOL, V_TOL = 2e-5, 2e-4          # as test_md_step_includes_the_nonbonded_term


def _tables(c):
    n = len(c["charges"])
    groups = {}
    for s, d in zip(c["src_ex"], c["dst_ex"]):
        groups.setdefault(int(d), set()).add(int(s))
    rowptr = np.zeros(n + 1, np.int32)
    for i in range(n):
        rowptr[i + 1] = rowptr[i] + len(groups.get(i, ()))
    col = np.concatenate([sorted(groups.get(i, ())) for i in range(n)]).astype(np.int32)
    return rowptr, col


def _calc(real_weights, c, lo=0, hi=-1, charges=None):
    from ai2bmd_b200.engine import Engine
    from ai2bmd_b200.nonbonded import PMENonBondedCalculator
    calc = PMENonBondedCalculator(Engine(real_weights, 0))
    calc.set_parameters(c["charges"] if charges is None else charges, c["sigmas"], c["epsilons"], *_tables(c),
                        tuple(c["cell"]), lo, hi)
    assert calc.grid(tuple(c["cell"])) == tuple(int(k) for k in c["grid"])
    return calc


@pytest.mark.parametrize("key", ["chig", "chig_preeq", "abd"])
def test_pme_matches_oracle_and_reference(real_weights, golden_dir, key):
    """fp32 per-pair kernel vs the fp64 net-per-pair oracle: per-atom sums differ only in fp32 rounding (stated as
    test_nonbonded.py does: |dF| <= 2e-5 max|F| + 1e-6 eV/A, |dE| <= 2e-5 |E| + 1e-4 eV); E_rec and the constants are
    fp64 on both sides (1e-9 relative).  Against the reference's own fp32 output: its cancellation noise
    (tests/test_pme.py GOLDEN_E_TOL / GOLDEN_F_TOL)."""
    c = _golden(golden_dir, key)
    e64, f64, t64 = PR.pme(c["positions"], c["charges"], c["sigmas"], c["epsilons"], c["ex"], tuple(c["cell"]),
                           tuple(c["grid"]))
    calc = _calc(real_weights, c)
    assert calc.engine.get_option("pme_ready") == 1
    e, f = calc(c["positions"])
    t = calc.engine.pme_terms()
    assert np.abs(f - f64).max() <= 2e-5 * np.abs(f64).max() + 1e-6
    assert abs(e - e64) <= 2e-5 * abs(e64) + 1e-4
    for k in ("E_rec", "slf"):
        assert abs(t[k] - t64[k]) <= 1e-9 * abs(t64[k]), k
    assert abs(t["neutral"] - t64["neutral"]) <= 1e-12
    for k in ("E_dir", "E_adj", "E_ex", "E_LJ", "E_LJ_ex"):
        assert abs(t[k] - t64[k]) <= 1e-5 * abs(t64[k]) + 1e-6, k
    assert abs(e - float(c["energy"])) <= GOLDEN_E_TOL
    assert np.abs(f - c["forces"]).max() <= GOLDEN_F_TOL
    # two calls: bit-identical (no atomics, fixed-order sums)
    e2, f2 = calc(c["positions"])
    assert e2 == e and np.array_equal(f2, f)
    assert calc.engine.pme_terms() == t


def test_neutral_term_of_a_charged_system(real_weights, golden_dir):
    """neutral = -E_rec(q_tot at the origin) + beta q_tot^2 / sqrt(pi), computed at set-up by the reciprocal kernels."""
    c = _golden(golden_dir, "chig")
    q = (c["charges"] + np.float32(0.01)).astype(np.float32)
    calc = _calc(real_weights, c, charges=q)
    calc(c["positions"])
    t = calc.engine.pme_terms()
    ref = PR.neutral_energy(q, tuple(c["cell"]), tuple(c["grid"]), 0.3)
    assert abs(ref) > 0.1 and abs(t["neutral"] - ref) <= 1e-9 * abs(ref)
    assert abs(t["E_rec"] - PR.spme_erec(c["positions"].astype(np.float32), q, tuple(c["cell"]), tuple(c["grid"]), 0.3)) \
        <= 1e-9 * abs(t["E_rec"])


def test_slices_sum_to_the_whole(real_weights, golden_dir):
    c = _golden(golden_dir, "abd")
    n = len(c["charges"])
    whole = _calc(real_weights, c)
    e, f = whole(c["positions"])
    t_whole = whole.engine.pme_terms()
    parts_f, parts_e = np.zeros_like(f), 0.0
    for lo, hi in ((0, n // 2), (n // 2, n)):
        part = _calc(real_weights, c, lo, hi)
        es, fs = part(c["positions"])
        t = part.engine.pme_terms()
        assert not fs[:lo].any() and not fs[hi:].any()
        if lo == 0:                                     # E_rec and the constants: counted by the slice at atom 0 only
            assert (t["E_rec"], t["slf"], t["neutral"]) == (t_whole["E_rec"], t_whole["slf"], t_whole["neutral"])
        else:
            assert t["E_rec"] == t["slf"] == t["neutral"] == 0.0
        parts_f += fs
        parts_e += es
    assert np.array_equal(parts_f, f)
    assert abs(parts_e - e) <= 1e-5 * abs(e) + 1e-5


def _chig_pme(seed=3):
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    n = len(prot_z)
    rowptr, col = exclusion_table(n, dipeptide_atom_sets(fd, recipe, pm))
    q, sg, ep = synthetic_parameters(prot_z, seed=seed)
    q *= 0.25                                                   # synthetic charges: keep the toy system gentle
    return fd, pm, prot_pos, prot_z, recipe, (q, sg, ep, rowptr, col)


def test_md_eval_adds_the_pme_term(real_weights):
    """vb_md_eval with PME = the same evaluation without it + vb_pme at the same positions (up to the run-to-run
    spread of the bonded forces, whose adjoint accumulates with atomics)."""
    from ai2bmd_b200.md import DeviceLangevin
    fd, pm, prot_pos, prot_z, recipe, prm = _chig_pme()
    n = len(prot_z)
    dev = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=0.5, friction_per_fs=0.0, seed=4)
    torch.cuda.synchronize()
    ef_bonded = dev.ef.cpu().numpy().copy()
    dev.engine.set_pme(*prm, CHIG_CELL, (25, 27, 23))
    dev._eval()
    torch.cuda.synchronize()
    ef_md = dev.ef.cpu().numpy().copy()
    pos = torch.as_tensor(prot_pos.astype(np.float32), device="cuda:0")
    ef_pme = torch.zeros(3 * n + 1, dtype=torch.float32, device="cuda:0")
    dev.engine.pme_device(pos.data_ptr(), ef_pme.data_ptr(), torch.cuda.current_stream().cuda_stream)
    ef_pme = ef_pme.cpu().numpy()
    f_sum = ef_bonded[:-1] + ef_pme[:-1]
    assert np.abs(ef_md[:-1] - f_sum).max() <= 1e-5 * np.abs(f_sum).max() + 1e-5
    assert abs(float(ef_md[-1]) - float(ef_bonded[-1] + ef_pme[-1])) <= 1e-6 * abs(float(ef_bonded[-1])) + 1e-5


def test_md_step_includes_the_pme_term(real_weights):
    """Device MD with PME follows the host integrator driven by bonded + PMENonBondedCalculator."""
    from ai2bmd_b200.md import BondedForceField, DeviceLangevin, Langevin
    from ai2bmd_b200.nonbonded import PMENonBondedCalculator
    fd, pm, prot_pos, prot_z, recipe, prm = _chig_pme()
    ff = BondedForceField(real_weights, fd, pm, recipe)
    nb = PMENonBondedCalculator(ff.engine)
    nb.set_parameters(*prm, CHIG_CELL)

    def force_fn(x):
        eb, fb = ff(x)
        en, fn = nb(x)
        return eb + en, fb + fn

    host = Langevin(prot_pos, prot_z, force_fn, dt_fs=0.5, friction_per_fs=0.0, seed=4)
    dev = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=0.5, friction_per_fs=0.0, seed=4,
                         velocities=host.v.copy())
    dev.engine.set_pme(*prm, CHIG_CELL, nb.grid(CHIG_CELL))
    dev._eval()                                                 # forces of the start positions now include the term
    assert abs(dev.energy - host.energy) <= 1e-4 * abs(host.energy)
    for _ in range(20):
        host.step()
    dev.run(20)
    x, v, step, hist = dev.state(1)
    assert step == 20 and np.abs(x - host.x).max() <= X_TOL and np.abs(v - host.v).max() <= V_TOL
    assert abs(hist[0] - host.energy) <= 1e-4 * abs(host.energy)


def test_mm_and_pme_replace_each_other(real_weights):
    from ai2bmd_b200.engine import Engine
    _, pm, prot_pos, _, _, prm = _chig_pme()
    n = len(prot_pos)
    eng = Engine(real_weights, 0)
    pos = torch.as_tensor(prot_pos.astype(np.float32), device="cuda:0")
    ef = torch.zeros(3 * n + 1, dtype=torch.float32, device="cuda:0")
    sp = torch.cuda.current_stream().cuda_stream
    assert eng.get_option("pme_ready") == 0
    eng.set_nonbonded(*prm)
    eng.set_pme(*prm, CHIG_CELL, (25, 27, 23))
    assert eng.get_option("pme_ready") == 1
    with pytest.raises(RuntimeError, match=r"\(-3\).*vb_set_nonbonded first"):
        eng.nonbonded_device(pos.data_ptr(), ef.data_ptr(), sp)
    eng.pme_device(pos.data_ptr(), ef.data_ptr(), sp)
    eng.set_nonbonded(*prm)
    assert eng.get_option("pme_ready") == 0
    with pytest.raises(RuntimeError, match=r"\(-3\).*vb_set_pme first"):
        eng.pme_device(pos.data_ptr(), ef.data_ptr(), sp)
    eng.nonbonded_device(pos.data_ptr(), ef.data_ptr(), sp)
    torch.cuda.synchronize()


def test_set_pme_error_paths(real_weights):
    from ai2bmd_b200.engine import Engine
    fd, pm, prot_pos, _, _, (q, sg, ep, rowptr, col) = _chig_pme()
    n = len(q)
    eng = Engine(real_weights, 0)
    pos = torch.as_tensor(prot_pos.astype(np.float32), device="cuda:0")
    ef = torch.zeros(3 * n + 1, dtype=torch.float32, device="cuda:0")
    sp = torch.cuda.current_stream().cuda_stream
    with pytest.raises(RuntimeError, match=r"\(-3\).*vb_set_pme first"):
        eng.pme_device(pos.data_ptr(), ef.data_ptr(), sp)
    good = dict(cell=CHIG_CELL, grid=(25, 27, 23), beta=0.3, cutoff=9.0)
    eng.set_pme(q, sg, ep, rowptr, col, **good)
    nan, inf = float("nan"), float("inf")
    bad_col = col.copy()
    bad_col[1] = bad_col[0]                                         # row 0 not strictly ascending
    cases = [
        ("cell lengths must be finite and positive", dict(cell=(nan, 27.3, 23.7))),
        ("cell lengths must be finite and positive", dict(cell=(25.9, inf, 23.7))),
        ("cell lengths must be finite and positive", dict(cell=(25.9, 27.3, 0.0))),
        ("cell lengths must be finite and positive", dict(cell=(-25.9, 27.3, 23.7))),
        ("grid dimensions must be at least 4", dict(grid=(25, 3, 23))),
        ("grid dimensions must be at least 4", dict(grid=(0, 27, 23))),
        ("beta must be finite and positive", dict(beta=0.0)),
        ("beta must be finite and positive", dict(beta=nan)),
        ("beta must be finite and positive", dict(beta=-0.3)),
        ("cutoff must be finite and positive", dict(cutoff=0.0)),
        ("cutoff must be finite and positive", dict(cutoff=inf)),
        ("bad slice", dict(atom_lo=5, atom_hi=3)),
        ("bad slice", dict(atom_lo=0, atom_hi=n + 1)),
        ("bad slice", dict(atom_lo=-1, atom_hi=n)),
    ]
    for text, kw in cases:
        with pytest.raises(RuntimeError, match=rf"\(-1\).*{text}"):
            eng.set_pme(q, sg, ep, rowptr, col, **{**good, **kw})
        assert eng.get_option("pme_ready") == 1                    # a rejected call leaves the installed term in place
    with pytest.raises(RuntimeError, match=r"\(-1\).*strictly ascending"):
        eng.set_pme(q, sg, ep, rowptr, bad_col, **good)
    rp = rowptr.copy()
    rp[0] = 1
    with pytest.raises(RuntimeError, match=r"\(-1\).*bad exclusion table"):
        eng.set_pme(q, sg, ep, rp, col, **good)
    # n_protein_atoms must equal the protein map's
    eng.set_topology(fd.z, fd.batch, n_graphs=len(fd))
    eng.set_protein_map(pm.n_protein, pm.src_atom, pm.dst_atom, pm.sign, pm.frag_sign)
    r2, c2 = exclusion_table(n - 1, [])
    with pytest.raises(RuntimeError, match=r"\(-1\).*differs from the protein map"):
        eng.set_pme(q[:-1], sg[:-1], ep[:-1], r2, c2, **good)
    assert eng.get_option("pme_ready") == 1
    eng.pme_device(pos.data_ptr(), ef.data_ptr(), sp)
    torch.cuda.synchronize()
    assert np.isfinite(ef.cpu().numpy()).all()


# ---- sharded run (native all-reduce), two or more GPUs ---------------------------------------------------------------
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from ai2bmd_b200.md import DeviceLangevin
    from ai2bmd_b200.parallel import DeviceShard
    from ai2bmd_b200.pdbfrag import FragmentRecipe
    from ai2bmd_b200.weights import load_state_dict
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sd = load_state_dict(os.path.join(ROOT, "tests", "golden", "weights_2ef43f29.npz"))
    fd, pm, prot_pos, prot_z, recipe, prm = _chig_pme()
    sh = DeviceShard(sd, fd, pm, rank, world, rank, native_comm=True)
    lo, hi = sh.plan.atom_lo, sh.plan.atom_hi
    rec = FragmentRecipe(recipe.real[lo:hi], recipe.acc[lo:hi], recipe.rem[lo:hi], recipe.blen[lo:hi])
    md = DeviceLangevin(None, None, pm, rec, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0,
                        device=rank, group=dist.group.WORLD, engine=sh.engine)
    n = pm.n_protein                                            # an even slice of the destination atoms per rank
    sh.engine.set_pme(*prm, CHIG_CELL, (25, 27, 23), atom_lo=rank * n // world, atom_hi=(rank + 1) * n // world)
    md._eval()
    md.run(20)
    x, _, step, _ = md.state()
    xt = torch.as_tensor(x, device=torch.device("cuda", rank))
    gathered = [torch.empty_like(xt) for _ in range(world)]
    dist.all_gather(gathered, xt)
    res = {"x": x, "step": step, "one_graph": md._native_comm,
           "identical_on_all_ranks": all(bool((g == xt).all()) for g in gathered)}
    if rank == 0:
        np.savez(out, **res)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_sharded_pme_equals_single_gpu(tmp_path, real_weights):
    import torch.multiprocessing as mp
    from ai2bmd_b200.md import DeviceLangevin
    from test_multigpu import _free_port
    world = min(torch.cuda.device_count(), 8)
    out = str(tmp_path / "ranks.npz")
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    r = np.load(out)
    assert bool(r["one_graph"]) and int(r["step"]) == 20 and bool(r["identical_on_all_ranks"])
    fd, pm, prot_pos, prot_z, recipe, prm = _chig_pme()
    one = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001,
                         seed=0, device=0)
    one.engine.set_pme(*prm, CHIG_CELL, (25, 27, 23))
    one._eval()
    one.run(20)
    x1, _, _, _ = one.state()
    assert np.abs(r["x"] - x1).max() <= X_TOL
