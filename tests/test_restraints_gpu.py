"""Hookean restraints on the device (csrc/k_restraint.cuh behind vb_set_restraints / vb_restraints) against the fp64 host
restatement (ai2bmd_b200/restraints.py), alone and inside the device-resident MD step."""
import os
import sys

import numpy as np
import pytest
import torch

from ai2bmd_b200 import restraints as R
from ai2bmd_b200.fixtures import load_capped_protein, load_fragments, load_protein

pytestmark = pytest.mark.gpu

# same bounds as tests/test_md_gpu.py: fp32 force rounding amplified by a few tens of steps
X_TOL, V_TOL = 2e-5, 2e-4


def _engine(real_weights, protein_map=True):
    from ai2bmd_b200.engine import Engine
    fd, pm = load_fragments("chig")
    eng = Engine(real_weights, 0)
    eng.set_topology(fd.z, fd.batch, n_graphs=len(fd))
    if protein_map:
        eng.set_protein_map(pm.n_protein, pm.src_atom, pm.dst_atom, pm.sign, pm.frag_sign)
    return eng


def _both_branches_set(x0, rng):
    """Position restraints with random flat bottoms and the hydrogen-bond springs, on positions perturbed so that every
    flat bottom is crossed by some restraints and not by others."""
    prot = load_capped_protein("chig")
    n = len(x0)
    pts = R.position_restraints(x0, 10.0)
    pts.point_rt[:] = rng.uniform(0.0, 0.5, n)
    pts.point_rt[:5] = 0.0
    pts.point_anchor[:5] = x0[:5]                            # r = rt = 0 at the unperturbed atoms 0..4
    return pts + R.hydrogen_bond_restraints(prot.names, prot.positions)


def test_vb_restraints_matches_hookean(real_weights):
    prot_pos, _, _ = load_protein("chig")
    n = len(prot_pos)
    rng = np.random.default_rng(0)
    rs = _both_branches_set(prot_pos, rng)
    x = prot_pos + rng.normal(0.0, 0.15, prot_pos.shape)
    x[:5] = prot_pos[:5]
    r_pt = np.linalg.norm(rs.point_anchor - x[rs.point_atom], axis=1)
    r_pr = np.linalg.norm(x[rs.pair_ij[:, 1]] - x[rs.pair_ij[:, 0]], axis=1)
    for r, rt in ((r_pt, rs.point_rt), (r_pr, rs.pair_rt)):
        assert (r > rt).sum() >= 10 and (r <= rt).sum() >= 5          # both branches of the flat bottom occur
    e_ref, f_ref = R.hookean(x, rs)

    eng = _engine(real_weights)
    assert eng.get_option("restraints_ready") == 0
    rs.install(eng)
    assert eng.get_option("restraints_ready") == 1
    dev = torch.device("cuda", 0)
    xd = torch.as_tensor(x, device=dev)
    sp = torch.cuda.current_stream().cuda_stream

    def run(engine):
        ef = torch.zeros(3 * n + 1, dtype=torch.float32, device=dev)
        engine.restraints_device(xd.data_ptr(), ef.data_ptr(), sp)
        torch.cuda.synchronize()
        return ef.cpu().numpy()

    ef = run(eng)
    f = ef[:-1].reshape(n, 3).astype(np.float64)
    assert np.abs(f - f_ref).max() <= 1e-6 * np.abs(f_ref).max() + 1e-7
    assert abs(float(ef[-1]) - e_ref) <= 2 ** -23 * abs(e_ref)
    assert np.isfinite(f).all()                                      # r = rt = 0 gives no 0/0
    assert np.array_equal(run(eng), ef)                              # no atomics: bit-identical
    # slices [0, m) and [m, n) of the destination atoms sum to the whole term
    m = 77
    rs.sliced(0, m).install(eng)
    e0 = run(eng)
    rs.sliced(m, n).install(eng)
    e1 = run(eng)
    assert not e0[3 * m:-1].any() and not e1[:3 * m].any()
    assert np.array_equal(e0[:-1] + e1[:-1], ef[:-1])
    assert abs(float(e0[-1]) + float(e1[-1]) - e_ref) <= 2 ** -22 * abs(e_ref)
    eng.clear_restraints()
    assert eng.get_option("restraints_ready") == 0
    assert not run(eng).any()                                        # no set: the call adds nothing


def _pair(real_weights, friction=0.01, seed=11):
    """(host Langevin with a Restrained force_fn, DeviceLangevin, start velocities) on Chignolin from the same start, the
    host fed with the device's Philox stream."""
    from ai2bmd_b200.md import BondedForceField, DeviceLangevin, Langevin, philox_normals
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    n_prot = len(prot_z)

    def src(step):
        xi, eta = philox_normals(seed, step, 3 * n_prot)
        return xi.reshape(n_prot, 3), eta.reshape(n_prot, 3)

    ff = BondedForceField(real_weights, fd, pm, recipe)
    host = Langevin(prot_pos, prot_z, R.Restrained(ff), dt_fs=1.0, temperature_K=300.0, friction_per_fs=friction,
                    seed=seed, normal_source=src)
    dev = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0,
                         friction_per_fs=friction, seed=seed, velocities=host.v.copy())
    return host, dev, host.v.copy()


def test_device_md_with_position_restraints_matches_host(real_weights):
    from ai2bmd_b200.md import DeviceLangevin
    host, dev, v0 = _pair(real_weights)
    prot_pos = host.x.copy()
    rng = np.random.default_rng(1)
    rs = R.position_restraints(prot_pos + rng.normal(0.0, 0.05, prot_pos.shape), 10.0)
    e_rs0, _ = R.hookean(prot_pos, rs)
    assert e_rs0 > 0.1                                               # well above the energy tolerance below
    e_free = host.energy
    R.set_restraints(host, rs)
    R.set_restraints(dev, rs)
    assert abs(host.energy - (e_free + e_rs0)) <= 2e-2              # the bonded term is re-evaluated (fp32 sums)
    assert abs(dev.energy - host.energy) <= 2e-2
    n = 25
    host_e = [host.step() for _ in range(n)]
    dev.run(n)
    x, v, step, hist = dev.state(n_hist=n)
    assert step == n
    assert np.abs(x - host.x).max() <= X_TOL and np.abs(v - host.v).max() <= V_TOL
    assert np.abs(hist - np.asarray(host_e)).max() <= 2e-2           # epot_hist includes the restraint energy
    # without the restraints the same start goes elsewhere: the comparison above is not vacuous
    fd, pm = load_fragments("chig")
    _, prot_z, recipe = load_protein("chig")
    free = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0,
                          friction_per_fs=0.01, seed=11, velocities=v0)
    free.run(n)
    xf, _, _, _ = free.state()
    assert np.abs(xf - x).max() >= 1000 * X_TOL


def test_pre_equilibrate_device_matches_host(real_weights):
    host, dev, _ = _pair(real_weights, seed=5)
    steps = 4
    R.pre_equilibrate(host, steps)
    R.pre_equilibrate(dev, steps)
    x, v, step, _ = dev.state()
    assert step == 5 * steps and host.nsteps == 5 * steps
    assert np.abs(x - host.x).max() <= X_TOL and np.abs(v - host.v).max() <= V_TOL
    assert dev.restraints.empty and dev.engine.get_option("restraints_ready") == 0
    for _ in range(6):                                               # production steps after the protocol
        host.step()
    dev.run(6)
    x, v, step, _ = dev.state()
    assert step == 5 * steps + 6
    assert np.abs(x - host.x).max() <= X_TOL and np.abs(v - host.v).max() <= V_TOL


def test_hydrogen_bond_restraints_active_match_host(real_weights):
    host, dev, _ = _pair(real_weights, seed=7)
    prot = load_capped_protein("chig")
    rs = R.hydrogen_bond_restraints(prot.names, prot.positions)
    rs.pair_rt[:] = 0.9                                              # below every X-H bond length: all springs pull
    r = np.linalg.norm(host.x[rs.pair_ij[:, 1]] - host.x[rs.pair_ij[:, 0]], axis=1)
    assert (r > 0.9).all()
    R.set_restraints(host, rs)
    R.set_restraints(dev, rs)
    n = 20
    for _ in range(n):
        host.step()
    dev.run(n)
    x, v, step, _ = dev.state()
    assert step == n
    assert np.abs(x - host.x).max() <= X_TOL and np.abs(v - host.v).max() <= V_TOL


def test_clearing_restraints_equals_never_restrained(real_weights):
    from ai2bmd_b200.md import DeviceLangevin
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    a = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, friction_per_fs=0.01, seed=3)
    a.set_restraints(R.position_restraints(prot_pos + 0.05, 10.0))
    a.run(10)
    a.set_restraints(None)
    assert a.engine.get_option("restraints_ready") == 0
    x, v, step, _ = a.state()
    b = DeviceLangevin(real_weights, fd, pm, recipe, x, prot_z, friction_per_fs=0.01, seed=3, velocities=v)
    b.engine.md_set_state(x, v, step)
    b._eval()
    assert abs(a.energy - b.energy) <= 2e-2
    a.run(15)
    b.run(15)
    xa, va, sa, _ = a.state()
    xb, vb, sb, _ = b.state()
    assert sa == sb == step + 15
    assert np.abs(xa - xb).max() <= X_TOL and np.abs(va - vb).max() <= V_TOL


def _expect_error(eng, status, text, **kw):
    with pytest.raises(RuntimeError) as ei:
        eng.set_restraints(**kw)
    assert f"({status})" in str(ei.value) and text in str(ei.value), str(ei.value)


def test_set_restraints_error_paths(real_weights):
    eng = _engine(real_weights, protein_map=False)
    _expect_error(eng, -3, "vb_set_protein_map first", pair_ij=[[0, 1]], pair_k=[1.0], pair_rt=[1.0])
    eng.close()
    eng = _engine(real_weights)
    n = eng.n_protein
    good = R.RestraintSet(point_atom=[3], point_anchor=[[0.0, 0, 0]], point_k=[1.0], point_rt=[0.0],
                          pair_ij=[[0, 1]], pair_k=[15.0], pair_rt=[1.2])
    good.install(eng)
    pt = dict(point_atom=[3], point_anchor=[[0.0, 0, 0]], point_k=[1.0], point_rt=[0.0])
    pr = dict(pair_ij=[[0, 1]], pair_k=[15.0], pair_rt=[1.2])
    nan, inf = float("nan"), float("inf")
    cases = [
        ("atom index out of range", {**pt, "point_atom": [n]}),
        ("atom index out of range", {**pt, "point_atom": [-1]}),
        ("atom index out of range", {**pr, "pair_ij": [[0, n]]}),
        ("i == j", {**pr, "pair_ij": [[4, 4]]}),
        ("k and rt must be finite and non-negative", {**pt, "point_k": [-1.0]}),
        ("k and rt must be finite and non-negative", {**pt, "point_rt": [inf]}),
        ("k and rt must be finite and non-negative", {**pr, "pair_k": [nan]}),
        ("k and rt must be finite and non-negative", {**pr, "pair_rt": [-0.1]}),
        ("non-finite anchor", {**pt, "point_anchor": [[0.0, nan, 0.0]]}),
        ("bad slice", {**pr, "atom_lo": 5, "atom_hi": 3}),
        ("bad slice", {**pr, "atom_lo": 0, "atom_hi": n + 1}),
        ("bad slice", {**pr, "atom_lo": -1, "atom_hi": n}),
    ]
    for text, kw in cases:
        _expect_error(eng, -1, text, **kw)
        assert eng.get_option("restraints_ready") == 1               # a rejected set leaves the installed one in place
    # the installed set still computes its term
    x = torch.zeros(3 * n, dtype=torch.float64, device="cuda:0")
    x[3:6] = 2.0                                                     # atom 1 at (2, 2, 2): pair (0, 1) stretched
    ef = torch.zeros(3 * n + 1, dtype=torch.float32, device="cuda:0")
    eng.restraints_device(x.data_ptr(), ef.data_ptr(), torch.cuda.current_stream().cuda_stream)
    e_ref, _ = R.hookean(x.cpu().numpy().reshape(n, 3), good)
    assert abs(float(ef[-1].item()) - e_ref) <= 1e-6 * e_ref


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
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    sh = DeviceShard(sd, fd, pm, rank, world, rank, native_comm=True)
    lo, hi = sh.plan.atom_lo, sh.plan.atom_hi
    rec = FragmentRecipe(recipe.real[lo:hi], recipe.acc[lo:hi], recipe.rem[lo:hi], recipe.blen[lo:hi])
    md = DeviceLangevin(None, None, pm, rec, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0,
                        device=rank, group=dist.group.WORLD, engine=sh.engine)
    md.set_restraints(_sharded_set(prot_pos))
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


def _sharded_set(prot_pos):
    prot = load_capped_protein("chig")
    return R.position_restraints(prot_pos + 0.03, 1.0) + R.hydrogen_bond_restraints(prot.names, prot.positions)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_sharded_restraints_equal_single_gpu(tmp_path, real_weights):
    import torch.multiprocessing as mp
    from ai2bmd_b200.md import DeviceLangevin
    sys.path.insert(0, os.path.dirname(__file__))
    from test_multigpu import _free_port
    world = min(torch.cuda.device_count(), 8)
    out = str(tmp_path / "ranks.npz")
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    r = np.load(out)
    assert bool(r["one_graph"]) and int(r["step"]) == 20 and bool(r["identical_on_all_ranks"])
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    one = DeviceLangevin(real_weights, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001,
                         seed=0, device=0)
    one.set_restraints(_sharded_set(prot_pos))
    one.run(20)
    x1, _, _, _ = one.state()
    assert np.abs(r["x"] - x1).max() <= X_TOL
