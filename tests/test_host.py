"""Host-side logic: FragmentData semantics, fixtures, weight packing, C-ABI symbol table, loud failure."""
import ctypes
import json
import os

import numpy as np
import pytest

from ai2bmd_b200 import build as vbuild
from ai2bmd_b200 import engine as vengine
from ai2bmd_b200.calculator import DipeptideBondedCombiner
from ai2bmd_b200.fragment_data import FragmentInfo
from ai2bmd_b200.parallel import combine_local, partition_fragments, shard_protein_map
from ai2bmd_b200.weights import pack_weights

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def lib():
    vbuild.build()            # nvcc cross-compiles without a GPU
    return vengine.load_library()


def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "visnet_b200.h")).read()
    import re
    declared = set(re.findall(r"\b(vb_[a-z_0-9]+)\s*\(", header))
    assert declared == set(vengine.EXPORTED_SYMBOLS)
    for sym in declared:
        assert hasattr(lib, sym), sym


def test_weight_blob_matches_manifest(lib, real_weights):
    manifest = lib.vb_weight_manifest().decode()
    blob = pack_weights(real_weights, manifest)
    total = sum(int(x.split(":")[1]) for x in manifest.strip(";").split(";"))
    assert blob.dtype == np.float32 and blob.size == total
    # spot-check the transposed / native pairs and the fused matrices
    off = {}
    o = 0
    for item in manifest.strip(";").split(";"):
        n, c = item.split(":")
        off[n] = (o, int(c))
        o += int(c)
    get = lambda n, shape: blob[off[n][0]:off[n][0] + off[n][1]].reshape(shape)
    wq = real_weights["representation_model.vis_mp_layers.2.q_proj.weight"]
    assert np.array_equal(get("layer2.WqkvN", (384, 128))[:128], wq)
    assert np.array_equal(get("layer2.WqkvT", (128, 384))[:, :128], wq.T)
    assert np.array_equal(get("layer5.W1N", (384, 128))[256:], np.zeros((128, 128), np.float32))   # no f_proj in the last layer
    assert np.array_equal(get("layer4.WtuN", (256, 128))[128:], real_weights["representation_model.vis_mp_layers.4.w_src_proj.weight"])
    assert get("atomref", (100,))[6] == pytest.approx(-1027.537, abs=1e-2)


def test_engine_fails_loudly_without_gpu(lib, real_weights):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no usable CUDA device|no CPU fallback"):
        vengine.Engine(real_weights)
    from ai2bmd_b200.calculator import ViSNetModel
    with pytest.raises(RuntimeError, match="no CPU path"):
        ViSNetModel(real_weights, device="cpu")


def test_create_rejects_bad_arguments(lib):
    hp = vengine._HParams(256, 9, 8, 32, 32, 5.0)
    h = ctypes.c_void_p()
    blob = np.zeros(16, np.float32)
    assert lib.vb_create(blob.ctypes.data, blob.size, ctypes.byref(hp), 0, ctypes.byref(h)) == -1
    assert b"hyper-parameters" in lib.vb_last_error(None)
    hp = vengine._HParams(128, 6, 8, 32, 32, 5.0)
    assert lib.vb_create(blob.ctypes.data, blob.size, ctypes.byref(hp), 0, ctypes.byref(h)) == -1
    assert b"manifest" in lib.vb_last_error(None)


def test_fragment_data_slicing_and_splits(chig):
    fd, _ = chig
    assert len(fd) == 19 and fd.end[-1] == 391
    sub = fd[2:5]
    assert len(sub) == 3 and sub.start[0] == 0 and sub.batch[0] == 0 and sub.batch[-1] == 2
    assert np.array_equal(sub.pos, fd.pos[fd.start[2]:fd.end[4]])
    one = fd[1]
    assert len(one) == 1 and len(one.z) == 12
    dip, an = fd.scalar_split()
    assert dip.sum() == 10 and an.sum() == 9 and dip[0] and an[1]
    vd, va = fd.vector_split()
    assert vd.sum() + va.sum() == 391 and va.sum() == 9 * 12
    assert vd[:fd.end[0]].all() and va[fd.start[1]:fd.end[1]].all()
    assert FragmentInfo.split(19) == (10, 9)
    with pytest.raises(IndexError):
        fd[3:3]


def test_fixture_shapes_match_survey(golden_dir):
    sizes = {"chig": (19, 391, 175), "trpcage": (39, 737, 281), "ww": (69, 1387, 571), "abd": (93, 1850, 746)}
    for name, (g, n, p) in sizes.items():
        f = np.load(os.path.join(golden_dir, f"fragments_{name}.npz"))
        assert len(f["start"]) == g and len(f["z"]) == n and int(f["n_protein"]) == p
        assert set(np.unique(f["z"])) <= {1, 6, 7, 8, 16}
        assert ((f["end"] - f["start"])[1::2] == 12).all()                     # ACE-NME fragments
        net = np.zeros(p)
        np.add.at(net, f["dst_atom"], f["sign"])
        assert (net == 1).all()                                                 # inclusion-exclusion covers every atom once


def test_combiner_matches_signed_map(chig):
    fd, pm = chig
    rng = np.random.default_rng(0)
    e = rng.normal(size=(len(fd), 1)).astype(np.float32)
    f = rng.normal(size=(len(fd.z), 3)).astype(np.float32)
    dip, an = fd.scalar_split()
    vd, va = fd.vector_split()
    # reference layout: [all dipeptide atoms | all ACE-NME atoms], select = real atoms, origin = protein index
    order = np.concatenate([np.flatnonzero(vd), np.flatnonzero(va)])
    inv = np.empty_like(order)
    inv[order] = np.arange(len(order))
    select, origin = inv[pm.src_atom], pm.dst_atom
    F = DipeptideBondedCombiner.forces_combine(pm.n_protein, f[vd], f[va], select, origin)
    E = DipeptideBondedCombiner.energy_combine(e[dip], e[an])
    ef = combine_local(pm, e, f)
    assert np.allclose(ef[:-1].reshape(-1, 3), F, atol=1e-5)
    assert float(E) == pytest.approx(float(ef[-1]), abs=1e-4)


@pytest.mark.parametrize("n_parts", [1, 2, 3, 4, 8, 32])
def test_partition_is_contiguous_balanced_cover(chig, trpcage, n_parts):
    for fd, pm in (chig, trpcage):
        parts = partition_fragments(fd.start, fd.end, n_parts)
        assert len(parts) == n_parts and parts[0][0] == 0 and parts[-1][1] == len(fd)
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
        atoms = [int(fd.end[hi - 1] - fd.start[lo]) if hi > lo else 0 for lo, hi in parts]
        assert sum(atoms) == int(fd.end[-1])
        if n_parts <= 8:
            assert max(atoms) <= int(fd.end[-1]) / n_parts + 36 + 12          # within one fragment of the ideal share
        # shard maps partition the full map
        total = sum(len(shard_protein_map(pm, fd, lo, hi).src_atom) for lo, hi in parts)
        assert total == len(pm.src_atom)


def test_philox_known_answers_and_normals():
    """Random123 known-answer vectors for Philox4x32-10 pin the host restatement of the device RNG (k_md.cuh)."""
    from ai2bmd_b200.md import philox4x32_10, philox_normals
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = tuple(int(w[0]) for w in philox4x32_10(*ctr, *key))
        assert got == want
    xi, eta = philox_normals(7, 3, 200000)
    for a in (xi, eta):
        assert abs(a.mean()) < 0.01 and abs(a.std() - 1.0) < 0.01 and np.isfinite(a).all()
    assert abs(np.corrcoef(xi, eta)[0, 1]) < 0.01
    xi2, _ = philox_normals(7, 4, 200000)
    assert abs(np.corrcoef(xi, xi2)[0, 1]) < 0.01                 # steps are independent streams
    assert np.array_equal(philox_normals(7, 3, 16)[0], xi[:16])     # component i does not depend on the array length


def test_host_langevin_with_normal_source_and_verlet_limit():
    """The host integrator (checker of the device one): harmonic forces, friction 0 conserves energy; a supplied
    normal source is used step by step."""
    from ai2bmd_b200.md import Langevin, philox_normals
    rng = np.random.default_rng(0)
    x0 = rng.standard_normal((12, 3))
    z = np.array([1, 6, 7, 8] * 3)

    def force_fn(x):
        return 0.5 * float((x * x).sum()), -x

    md = Langevin(x0, z, force_fn, dt_fs=0.5, friction_per_fs=0.0, seed=1)
    e0 = md.energy + md.kinetic_energy()
    md.run(200)
    assert abs(md.energy + md.kinetic_energy() - e0) < 1e-3 * abs(e0) and md.nsteps == 200
    calls = []

    def src(step):
        calls.append(step)
        xi, eta = philox_normals(9, step, 36)
        return xi.reshape(12, 3), eta.reshape(12, 3)

    md2 = Langevin(x0, z, force_fn, friction_per_fs=0.01, seed=1, normal_source=src)
    md2.run(5)
    assert calls == [0, 1, 2, 3, 4] and np.isfinite(md2.x).all()
    assert np.abs((md2.m * md2.v).sum(0)).max() < 1e-12


@pytest.mark.parametrize("name", ["chig", "trpcage", "ww", "abd"])
def test_fragment_compositions_match_the_reference_tables(golden_dir, name):
    """Every dipeptide fragment holds exactly the atoms the reference's own table lists for its central residue
    (``src/utils/reference.py:36-64``), every ACE-NME the 12 atoms of "AN"; fragments alternate dipeptide / ACE-NME
    (``distancefrag.py:250-284``) and dipeptide k is centred on residue k+2 of the capped chain."""
    import json
    from ai2bmd_b200.fixtures import load_fragments
    tables = json.load(open(os.path.join(golden_dir, "fragment_tables.json")))
    zref, seq = tables["z_by_residue"], tables["sequence"][name]
    fd, pm = load_fragments(name)
    assert seq[0] == "ACE" and seq[-1] == "NME"
    n_dip = len(seq) - 2
    assert len(fd) == 2 * n_dip - 1
    for g in range(len(fd)):
        z = sorted(int(v) for v in fd.z[fd.start[g]:fd.end[g]])
        if g % 2 == 0:
            assert pm.frag_sign[g] > 0
            assert z == sorted(zref[seq[g // 2 + 1]]), (g, seq[g // 2 + 1])
        else:
            assert pm.frag_sign[g] < 0 and z == sorted(zref["AN"])


def test_partition_rule_equals_the_reference_function(golden_dir):
    """``partition_fragments`` against blocks computed by the reference's own
    ``DeviceStrategy._set_combined_work_partitions`` (``device_strategy.py:83-127``; generated by make_golden.py)."""
    import json
    from ai2bmd_b200.fixtures import load_fragments
    ref = json.load(open(os.path.join(golden_dir, "reference_partitions.json")))
    assert len(ref) == 16
    for key, blocks in ref.items():
        name, n = key.split(":")
        fd, _ = load_fragments(name)
        mine = partition_fragments(fd.start, fd.end, int(n))
        assert [list(p) for p in mine] == blocks, key


def test_host_mirrors_equal_the_reference_classes(golden_dir, chig):
    """FragmentData slicing / splits, the bonded combiner and the device-epilogue restatement against outputs of the
    reference's OWN classes (``src/AIMD/fragment.py:7-47``, ``src/Calculators/combiner.py:11-41``) generated by
    tests/golden/make_golden.py on the Chignolin fixture."""
    from ai2bmd_b200.calculator import DipeptideBondedCombiner
    g = np.load(os.path.join(golden_dir, "reference_host_logic.npz"))
    fd, pm = chig
    for tag, idx in (("s3_7", slice(3, 7)), ("s0_1", slice(0, 1)), ("i5", 5), ("s10_19", slice(10, 19))):
        sub = fd[idx]
        for field in ("z", "pos", "start", "end", "batch"):
            assert np.array_equal(np.asarray(getattr(sub, field)), g[f"{tag}_{field}"]), (tag, field)
    sd_, sa_ = fd.scalar_split()
    vd_, va_ = fd.vector_split()
    assert np.array_equal(sd_, g["scalar_dip"]) and np.array_equal(sa_, g["scalar_an"])
    assert np.array_equal(vd_, g["vector_dip"]) and np.array_equal(va_, g["vector_an"])
    sub = fd[4:11]
    assert np.array_equal(sub.scalar_split()[0], g["sub_scalar_dip"]) and np.array_equal(sub.vector_split()[1], g["sub_vector_an"])
    e, f = g["comb_e_in"], g["comb_f_in"]
    E = DipeptideBondedCombiner.energy_combine(e[sd_], e[sa_])
    F = DipeptideBondedCombiner.forces_combine(pm.n_protein, f[vd_], f[va_], g["comb_select"], g["comb_origin"])
    assert abs(float(E) - float(g["comb_energy"])) <= 1e-3          # fp32 sums of 19 terms of O(100)
    assert np.abs(F - g["comb_forces"]).max() <= 1e-5
    ef = combine_local(pm, e.reshape(-1), f)                          # what vb_forward_protein computes on the device
    assert np.abs(ef[:-1].reshape(-1, 3) - g["comb_forces"]).max() <= 1e-5 and abs(ef[-1] - float(g["comb_energy"])) <= 1e-3


def test_cap_hydrogen_placement_equals_the_reference_body(golden_dir):
    """``FragmentRecipe.positions`` (host checker of the device placement kernel) against the output of the reference's own
    ``DistanceFragment.get_dipeptide_positions`` body (``distancefrag.py:34-54``; fp32 there, fp64-then-cast here)."""
    from ai2bmd_b200.fixtures import load_protein
    g = np.load(os.path.join(golden_dir, "reference_caph.npz"))
    prot_pos, _, recipe = load_protein("chig")
    mine = recipe.positions(prot_pos)[g["dip_atoms"]]
    assert mine.dtype == np.float32 and np.abs(mine - g["positions"]).max() <= 4e-6      # <= 4 ulp at 10 A
    assert int((recipe.real[g["dip_atoms"]] < 0).sum()) == 35


def test_bench_roofline_arithmetic():
    """bench.py's algorithmic byte / flop counts (SURVEY 8d) -- pure host arithmetic, checked without a GPU."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert b.algorithmic_bytes("edge_fwd0", 10, 100) == 100 * 1044 + 10 * 4096
    assert b.algorithmic_bytes("edge_fwd5", 10, 100) == 100 * 532 + 10 * 4096
    assert b.algorithmic_bytes("edge_bwd3", 10, 100) == 100 * 1572 + 10 * 8192
    stages = [f"edge_bwd{l}" for l in range(6)]
    t = b.tensor_roofline(stages, 1000, 1e-3, 3)
    products = 5 * 5 + 4
    assert abs(t["fp32_equivalent_tflops"] - 2 * 128 * 128 * 1000 * products / 1e-3 / 1e12) < 1e-9
    assert abs(t["achieved"] - 3 * t["fp32_equivalent_tflops"]) < 1e-9 and t["bound"] == "tensor" and 0 < t["frac"] < 1
    assert b.tensor_roofline(stages, 1000, 1e-3, 1) is None           # adjoint stage on SIMT: no tensor roofline
    assert b.tensor_roofline(["node_fwd0"], 1000, 1e-3, 3) is None


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the whole-protein buffer [3*n + 1] as forces [n, 3] and energy [1], float32; forces over
    the size limit as the same seeded sample of rows in every run."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    ef = np.arange(3 * 50 + 1, dtype=np.float32)
    b.dump_outputs(str(tmp_path / "full"), ef, 50)
    f, e = np.load(tmp_path / "full" / "forces.npy"), np.load(tmp_path / "full" / "energy.npy")
    assert f.dtype == np.float32 and np.array_equal(f, ef[:-1].reshape(50, 3))
    assert e.dtype == np.float32 and e.tolist() == [150.0]
    monkeypatch.setattr(b, "DUMP_FORCE_BYTES", 10 * 12)
    b.dump_outputs(str(tmp_path / "s1"), ef, 50)
    b.dump_outputs(str(tmp_path / "s2"), ef, 50)
    s1, s2 = np.load(tmp_path / "s1" / "forces.npy"), np.load(tmp_path / "s2" / "forces.npy")
    assert s1.shape == (10, 3) and np.array_equal(s1, s2)
    rows = s1[:, 0].astype(np.int64) // 3
    assert (np.diff(rows) > 0).all() and np.array_equal(s1, f[rows])


@pytest.mark.parametrize("name", ["chig", "trpcage", "ww", "abd"])
def test_fragment_membership_equals_the_reference_function(golden_dir, name):
    """Which protein atoms belong to every dipeptide / ACE-NME: the fixtures (ai2bmd_b200/pdbfrag.py) against the output
    of the reference's own ``DipeptideFragment.get_fragments_index`` (``basefrag.py:44-167``; make_golden.py).  Atom order
    inside a fragment is this repo's own (the model is permutation-equivariant); the rest of a fragment is added hydrogens."""
    import json
    from ai2bmd_b200.fixtures import load_fragments, load_protein
    ref = json.load(open(os.path.join(golden_dir, "reference_fragment_index.json")))[name]
    fd, pm = load_fragments(name)
    _, _, recipe = load_protein(name)
    assert len(ref["dipeptides"]) + len(ref["acenmes"]) == len(fd)
    for g in range(len(fd)):
        real = recipe.real[fd.start[g]:fd.end[g]]
        want = ref["dipeptides"][g // 2] if g % 2 == 0 else ref["acenmes"][g // 2]
        assert sorted(real[real >= 0].tolist()) == sorted(want), g
        n_added = int((real < 0).sum())
        assert n_added == (fd.end[g] - fd.start[g]) - len(want) and 0 <= n_added <= 5
    # the added hydrogens of every dipeptide: (acceptor, removed atom, bond length) as the reference's own
    # ``get_hydrogen_indices`` chooses them (``distancefrag.py:365-504``)
    for k, caps in enumerate(ref["added_hydrogens"]):
        sl = slice(fd.start[2 * k], fd.end[2 * k])
        m = recipe.real[sl] < 0
        mine = sorted((int(a), int(r), round(float(b), 5)) for a, r, b in zip(recipe.acc[sl][m], recipe.rem[sl][m], recipe.blen[sl][m]))
        assert mine == sorted((a, r, round(b, 5)) for a, r, b in caps), k


def test_host_langevin_keeps_the_centre_of_mass_in_place():
    """ASE 3.22 Langevin.step with fix_com: the centre of mass is put back after the drift and its velocity removed after
    the second half-kick, so 100 steps in a force field with a net force leave it where it started."""
    from ai2bmd_b200.md import Langevin
    rng = np.random.default_rng(0)
    z = np.array([1, 6, 7, 8, 16, 1, 6, 1])
    x0 = rng.normal(size=(8, 3)) * 2.0

    def force_fn(x):
        return 0.0, -0.3 * (x - 1.0) + np.array([0.2, -0.1, 0.05])          # harmonic well + a constant net force

    md = Langevin(x0, z, force_fn, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.01, seed=4)
    com0 = (md.m * x0).sum(0) / md.m.sum()
    assert np.abs((md.m * md.v).sum(0)).max() > 1e-3                       # the Maxwell-Boltzmann draw is not made stationary
    md.run(100)
    assert np.abs((md.m * md.x).sum(0) / md.m.sum() - com0).max() <= 1e-12
    assert np.abs((md.m * md.v).sum(0)).max() <= 1e-12
    assert np.abs(md.x - x0).max() > 1e-2


def test_cystine_pairing_equals_the_reference_function():
    """CYX-CYX dipeptides are paired by the reference's own ``get_cystine_bonds`` (golden) and packed as ONE graph, the
    partner's slot staying in the batch as an empty fragment (distancefrag.py:185-238)."""
    from ai2bmd_b200.fixtures import load_fragments, load_synthetic_cyx
    from ai2bmd_b200.pdbfrag import cystine_pairs, fragment_protein
    prot, gold = load_synthetic_cyx()
    R = int(prot.resnums.max())
    pairs = cystine_pairs(prot, [k + 2 for k in range(R - 2)])
    assert {str(k): v for k, v in pairs.items()} == gold["pairs"]
    fd, pm, rc = fragment_protein(prot, with_recipe=True)
    fd0, pm0 = load_fragments("ww")
    assert len(fd) == len(fd0) and len(fd.z) == len(fd0.z)            # same atoms, regrouped
    sizes, sizes0 = fd.end - fd.start, fd0.end - fd0.start
    assert (sizes[[2 * j for j in pairs.values() if j not in pairs]] == 0).all()
    assert sizes.sum() == sizes0.sum() and (sizes == 0).sum() >= 1 and sizes.max() > sizes0.max()
    # the whole-protein map still addresses every real fragment atom exactly once
    assert len(pm.src_atom) == len(pm0.src_atom) and len(set(pm.src_atom.tolist())) == len(pm.src_atom)
    assert np.array_equal(np.sort(pm.dst_atom), np.sort(pm0.dst_atom))
    assert (np.diff(fd.batch) >= 0).all() and set(np.unique(fd.batch).tolist()) == set(np.flatnonzero(sizes > 0).tolist())


def test_example_fragments_never_exceed_the_neighbour_cap():
    """The engine keeps, like the reference, the FIRST 32 candidates by atom index.  This repository orders the atoms of a
    fragment differently from the reference's AMBER permutation, which is harmless exactly as long as no atom has more
    than 32 atoms (itself included) inside the cutoff -- fail loudly the day a fixture crosses that line."""
    from ai2bmd_b200.fixtures import load_fragments
    from ai2bmd_b200.pdbfrag import neighbour_cap_margin
    for name in ("chig", "trpcage", "ww", "abd"):
        fd, _ = load_fragments(name)
        assert neighbour_cap_margin(fd) >= 0, f"{name}: an atom has more than 32 candidates: atom order now matters"


def test_topology_check_follows_in_place_edits_of_writable_arrays():
    """``dl_potential_loader`` must notice a changed z / batch even when the caller reuses the same array objects (the
    reference re-uploads both every call, visnet_calculator.py:47-52); only read-only arrays may be trusted by identity."""
    from ai2bmd_b200.calculator import ViSNetModel
    from ai2bmd_b200.fragment_data import FragmentData

    class FakeEngine:
        def __init__(self):
            self.topologies = 0

        def set_topology(self, z, batch, n_graphs=None):
            self.topologies += 1

    m = ViSNetModel.__new__(ViSNetModel)
    m.engine, m._topo_key = FakeEngine(), None
    z = np.array([6, 1, 1, 8], dtype=np.int64)
    batch = np.zeros(4, dtype=np.int64)
    fd = FragmentData(z, np.zeros((4, 3), np.float32), np.array([0]), np.array([4]), batch)
    m._ensure_topology(fd); m._ensure_topology(fd)
    assert m.engine.topologies == 1
    z[1] = 7                                             # same object, new content
    m._ensure_topology(fd)
    assert m.engine.topologies == 2
    z.flags.writeable = False; batch.flags.writeable = False
    m._ensure_topology(fd); m._ensure_topology(fd)      # frozen arrays: identity is enough from now on
    assert m.engine.topologies == 2 and m._topo_arrays is not None
