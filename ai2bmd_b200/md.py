"""Minimal MD driver for the bonded (ViSNet fragment) potential -- the loop that drives the hot path.

The reference runs ASE's ``Langevin`` (``/root/reference/src/AIMD/simulator.py:96-137``: dt = 1 fs, 300 K,
friction 0.001 / fs, Maxwell-Boltzmann start) and asks ``FragmentCalculator`` for forces once per step.  ASE is
not available here, so this module restates that integrator (ASE 3.22 ``ase/md/langevin.py``, recalled; SURVEY
App. C) in numpy around :class:`BondedForceField`, which performs per step exactly what
``DLBondedCalculator.__call__`` does (``src/Calculators/bonded.py:102-123``) minus the cap-hydrogen LBFGS:

  protein positions -> fragment positions (cap hydrogens on the acceptor->removed ray, ``distancefrag.py:34-54``)
  -> engine (energies/forces of every fragment) -> signed reduction to whole-protein energy / forces.

friction = 0 gives velocity Verlet; its energy conservation is a physics check of the analytic forces
(``tests/test_md_gpu.py``).  The reference's pre-equilibration and ``--constraints`` springs (ASE ``Hookean``) are
:mod:`ai2bmd_b200.restraints`: ``DeviceLangevin.set_restraints`` on the device, a wrapped ``force_fn`` on the host.  Units follow ASE: eV, Angstrom, amu, time in Angstrom*sqrt(amu/eV).
"""
from __future__ import annotations

import numpy as np

from .engine import Engine
from .fragment_data import FragmentData
from .pdbfrag import FragmentRecipe, ProteinMap

FS = 0.09822694788464063        # 1 fs in ASE time units
KB = 8.617330337217213e-05      # eV / K
MASSES = {1: 1.008, 6: 12.011, 7: 14.007, 8: 15.999, 16: 32.06}


class BondedForceField:
    """Whole-protein bonded energy/forces from the fragment batch (device-side reduction)."""

    def __init__(self, state_dict, frags: FragmentData, pm: ProteinMap, recipe: FragmentRecipe, device: int = 0, refine=None):
        """``refine(frag_pos) -> frag_pos``: optional host-side refinement of the placed fragment coordinates (the parity
        tests pass the CPU restatement of the cap-hydrogen LBFGS here to check the device loop that runs it in-kernel)."""
        import torch
        self.torch = torch
        self.recipe, self.pm, self.refine = recipe, pm, refine
        self.engine = Engine(state_dict, device)
        self.engine.set_topology(frags.z, frags.batch, n_graphs=len(frags))
        self.engine.set_protein_map(pm.n_protein, pm.src_atom, pm.dst_atom, pm.sign, pm.frag_sign)
        self.engine.forward_host(np.asarray(frags.pos, dtype=np.float32))       # start geometry: real edge count for the tile plan
        self.engine.set_option("calibrate", 1)
        dev = torch.device("cuda", device)
        self.pos_host = torch.empty((len(frags.z), 3), dtype=torch.float32).pin_memory()
        self.pos_dev = torch.empty((len(frags.z), 3), dtype=torch.float32, device=dev)
        self.ef_dev = torch.empty(3 * pm.n_protein + 1, dtype=torch.float32, device=dev)
        self.ef_host = torch.empty(3 * pm.n_protein + 1, dtype=torch.float32).pin_memory()
        self.stream = torch.cuda.current_stream(dev)

    def __call__(self, prot_pos: np.ndarray):
        """(E [eV], F [n_protein,3] eV/A) for the given protein coordinates."""
        frag_pos = self.recipe.positions(prot_pos)
        if getattr(self, "refine", None) is not None:
            frag_pos = self.refine(frag_pos)
        self.pos_host.numpy()[:] = frag_pos
        self.pos_dev.copy_(self.pos_host, non_blocking=True)
        self.engine.forward_protein_device(self.pos_dev.data_ptr(), self.ef_dev.data_ptr(), self.stream.cuda_stream)
        self.ef_host.copy_(self.ef_dev, non_blocking=True)
        self.stream.synchronize()
        ef = self.ef_host.numpy()
        return float(ef[-1]), ef[:-1].reshape(-1, 3).astype(np.float64)


class Langevin:
    """ASE-style Langevin integrator, restating ``ase/md/langevin.py`` ``Langevin.step`` of ASE 3.22 with
    ``fixcm=True`` (recalled; ASE is not in the image): half-kick, drift, centre of mass put back where it was,
    velocities recomputed from the positions, forces, half-kick, centre-of-mass velocity removed.
    ``friction=0`` reduces to velocity Verlet (no random numbers, no centre-of-mass handling)."""

    def __init__(self, positions, numbers, force_fn, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0,
                 normal_source=None, zero_com_momentum=False):
        """``normal_source(step) -> (xi, eta)`` overrides the numpy generator for the per-step normals (used to
        drive this host integrator with the device's Philox stream in the parity tests).  ``zero_com_momentum``
        removes the centre-of-mass momentum of the Maxwell-Boltzmann draw; the reference does not
        (``simulator.py:96`` calls ``MaxwellBoltzmannDistribution`` only, no ``Stationary``)."""
        self.normal_source = normal_source
        self.nsteps = 0
        self.x = np.array(positions, dtype=np.float64)
        self.m = np.array([MASSES[int(z)] for z in numbers], dtype=np.float64)[:, None]
        self.force_fn = force_fn
        self.dt = dt_fs * FS
        self.T = temperature_K * KB
        self.fr = friction_per_fs / FS
        self.rng = np.random.default_rng(seed)
        # Maxwell-Boltzmann start (simulator.py:96)
        self.v = self.rng.standard_normal(self.x.shape) * np.sqrt(self.T / self.m)
        if zero_com_momentum:
            self.v -= (self.v * self.m).sum(0) / self.m.sum()
        self.energy, self.f = force_fn(self.x)
        dt, fr = self.dt, self.fr
        sigma = np.sqrt(2 * self.T * fr / self.m)
        self.c1 = dt / 2.0 - dt * dt * fr / 8.0
        self.c2 = dt * fr / 2 - dt * dt * fr * fr / 8.0
        self.c3 = np.sqrt(dt) * sigma / 2.0 - dt ** 1.5 * fr * sigma / 8.0
        self.c5 = dt ** 1.5 * sigma / (2 * np.sqrt(3))
        self.c4 = fr / 2.0 * self.c5

    def kinetic_energy(self):
        return 0.5 * float((self.m * self.v * self.v).sum())

    def temperature(self):
        return 2.0 * self.kinetic_energy() / (3 * len(self.x)) / KB

    def step(self):
        if self.fr > 0 and self.normal_source is not None:
            xi, eta = self.normal_source(self.nsteps)
        else:
            xi = self.rng.standard_normal(self.x.shape) if self.fr > 0 else 0.0
            eta = self.rng.standard_normal(self.x.shape) if self.fr > 0 else 0.0
        self.v = self.v + (self.c1 * self.f / self.m - self.c2 * self.v + self.c3 * xi - self.c4 * eta)
        x_old = self.x
        self.x = self.x + self.dt * self.v + self.c5 * eta
        if self.fr > 0:     # fix_com: the centre of mass stays where it was before the drift (atoms.set_center_of_mass(old_com))
            msum = self.m.sum()
            self.x = self.x + ((self.m * x_old).sum(0) / msum - (self.m * self.x).sum(0) / msum)
        self.v = (self.x - x_old - self.c5 * eta) / self.dt
        self.energy, self.f = self.force_fn(self.x)
        self.v = self.v + (self.c1 * self.f / self.m - self.c2 * self.v + self.c3 * xi - self.c4 * eta)
        if self.fr > 0:
            self.v -= (self.v * self.m).sum(0) / self.m.sum()
        self.nsteps += 1
        return self.energy

    def run(self, n_steps):
        for _ in range(n_steps):
            self.step()


# ---------------------------------------------------------------------------------------------------------
# device-resident integrator (csrc/k_md.cuh behind include/visnet_b200.h vb_md_*)
# ---------------------------------------------------------------------------------------------------------
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) on arrays of 32-bit words held in uint64; returns the four output words."""
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1, c2, c3 = (np.atleast_1d(np.asarray(c, dtype=np.uint64)) for c in np.broadcast_arrays(c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m32, p0 & m32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
    return c0, c1, c2, c3


def philox_normals(seed: int, step: int, n_components: int):
    """Host restatement of the device's per-step normals (k_md.cuh ``md_normals``): Philox4x32-10 with counter
    (component, step_lo, step_hi, 0) and key (seed_lo, seed_hi), two 53-bit uniforms in (0, 1], Box-Muller.
    Returns (xi, eta), each ``[n_components]`` float64."""
    c0, c1, c2, c3 = philox4x32_10(np.arange(n_components, dtype=np.uint64), step & 0xFFFFFFFF, (step >> 32) & 0xFFFFFFFF, 0,
                                   seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u1 = ((((c0 << np.uint64(32)) | c1) >> np.uint64(11)).astype(np.float64) + 1.0) / 9007199254740992.0
    u2 = ((((c2 << np.uint64(32)) | c3) >> np.uint64(11)).astype(np.float64) + 1.0) / 9007199254740992.0
    r = np.sqrt(-2.0 * np.log(u1))
    return r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)


class DeviceLangevin:
    """The same integrator with positions, velocities, cap-hydrogen placement and the force evaluation all on the
    GPU: ``run(n)`` enqueues n replays of one captured CUDA graph and never touches the host.

    With ``group`` (a ``torch.distributed`` process group, one rank per GPU) every rank holds the whole-protein state
    and its own shard of fragments; the per-step exchange is the one all-reduce of the force/energy buffer."""

    def __init__(self, state_dict, frags: FragmentData, pm: ProteinMap, recipe: FragmentRecipe, positions, numbers,
                 dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0, device: int = 0, velocities=None,
                 group=None, engine: Engine = None, zero_com_momentum=False, caph=None):
        """``caph``: an :class:`ai2bmd_b200.caph.CapHProblem` -- the added hydrogens are then refined every step on the
        device (one LBFGS call on the Amber terms, ``csrc/k_caph.cuh``) between their placement and the evaluation."""
        import torch
        self.torch, self.group = torch, group
        self.n = pm.n_protein
        self.masses = np.array([MASSES[int(z)] for z in numbers], dtype=np.float64)
        self.kT = temperature_K * KB
        self.fr = friction_per_fs / FS
        dev = torch.device("cuda", device)
        if engine is None:
            engine = Engine(state_dict, device)
            engine.set_topology(frags.z, frags.batch, n_graphs=len(frags))
            engine.set_protein_map(pm.n_protein, pm.src_atom, pm.dst_atom, pm.sign, pm.frag_sign)
            engine.forward_host(np.asarray(frags.pos, dtype=np.float32))
            engine.set_option("calibrate", 1)
        self.engine = engine
        if caph is not None:
            engine.set_caph(caph)
        self.ef = torch.zeros(3 * self.n + 1, dtype=torch.float32, device=dev)
        self.stream = torch.cuda.current_stream(dev)
        engine.md_setup(self.masses, recipe.real, recipe.acc, recipe.rem, recipe.blen, dt_fs * FS, self.kT, self.fr,
                        seed, self.ef.data_ptr())
        x = np.array(positions, dtype=np.float64)
        if velocities is None:      # Maxwell-Boltzmann start, as Langevin above (simulator.py:96)
            rng = np.random.default_rng(seed)
            m = self.masses[:, None]
            velocities = rng.standard_normal(x.shape) * np.sqrt(self.kT / m)
            if zero_com_momentum:
                velocities -= (velocities * m).sum(0) / m.sum()
        engine.md_set_state(x, velocities, 0)
        from .restraints import RestraintSet
        self.restraints = RestraintSet()
        if engine.get_option("restraints_ready"):          # a caller-supplied engine may carry a set: start without one
            engine.clear_restraints()
        self._eval()

    @property
    def _native_comm(self):
        """True when the engine all-reduces the force buffer itself (peer-memory all-reduce inside the step graph)."""
        return self.group is not None and self.engine.get_option("comm_ready") == 1 and self.engine.get_option("comm_auto") == 1

    def _eval(self):
        sp = self.stream.cuda_stream
        self.engine.md_eval(sp)
        if self.group is not None and not self._native_comm:
            self.torch.distributed.all_reduce(self.ef, group=self.group)

    def set_restraints(self, rs):
        """Make ``rs`` (an :class:`ai2bmd_b200.restraints.RestraintSet`, or None for none) the restraint term of every
        following evaluation and recompute the forces at the current positions, so the next half-kick already uses it.
        With ``group`` every rank computes the forces of an even slice of the protein atoms; the all-reduce sums them."""
        from .restraints import RestraintSet
        rs = RestraintSet() if rs is None else rs
        dev = rs
        if self.group is not None:
            rank, world = self.torch.distributed.get_rank(self.group), self.torch.distributed.get_world_size(self.group)
            dev = rs.sliced(rank * self.n // world, (rank + 1) * self.n // world)
        dev.install(self.engine)
        self.restraints = rs
        self._eval()

    def set_normals(self, pool):
        """Externally supplied normals ``[steps, 2, n, 3]`` (float64) instead of the Philox stream (tests)."""
        if pool is None:
            self._pool = None
            self.engine.md_set_normals(0, 0)
            return
        self._pool = self.torch.as_tensor(np.ascontiguousarray(pool, dtype=np.float64)).to(self.ef.device)
        self.engine.md_set_normals(self._pool.data_ptr(), self._pool.shape[0])

    def run(self, n_steps: int):
        sp = self.stream.cuda_stream
        if self.group is None or self._native_comm:      # whole step (incl. the all-reduce) = one graph replay
            self.engine.md_run(n_steps, sp)
            return
        for _ in range(n_steps):
            self.engine.md_kick1(sp)
            self._eval()
            self.engine.md_kick2(sp)

    def state(self, n_hist: int = 0):
        """(positions, velocities, step, potential energies of the last n_hist steps); synchronises."""
        return self.engine.md_get_state(n_hist)

    @property
    def energy(self):
        self.stream.synchronize()
        return float(self.ef[-1].item())

    def kinetic_energy(self):
        _, v, _, _ = self.state()
        return 0.5 * float((self.masses[:, None] * v * v).sum())

    def temperature(self):
        return 2.0 * self.kinetic_energy() / (3 * self.n) / KB
