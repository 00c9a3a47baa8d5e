"""ctypes binding of the C-ABI library ``libvisnet_b200.so`` (``include/visnet_b200.h``).

PyTorch is used only as plumbing here (device tensors and streams owned by the caller); the binding
itself passes raw pointers.  There is no CPU path: constructing an :class:`Engine` without a usable
sm_100 device raises ``RuntimeError``, and a missing library raises at import of this module's users.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import numpy as np

from . import build as _build
from .weights import pack_weights

_lib = None


class _HParams(C.Structure):
    _fields_ = [("hidden_channels", C.c_int32), ("num_layers", C.c_int32), ("num_heads", C.c_int32),
                ("num_rbf", C.c_int32), ("max_num_neighbors", C.c_int32), ("cutoff", C.c_float)]


class _CaphProblem(C.Structure):
    _fields_ = [("n_h", C.c_int64), ("h_idx", C.c_void_p),
                ("n_bonds", C.c_int64), ("bond_ij", C.c_void_p), ("bond_k", C.c_void_p), ("bond_r0", C.c_void_p),
                ("n_angles", C.c_int64), ("angle_ijk", C.c_void_p), ("angle_k", C.c_void_p), ("angle_t0", C.c_void_p),
                ("n_dih", C.c_int64), ("dih_ijkl", C.c_void_p), ("dih_k", C.c_void_p), ("dih_n", C.c_void_p), ("dih_p", C.c_void_p),
                ("n_pairs", C.c_int64), ("pair_ij", C.c_void_p), ("pair_a", C.c_void_p), ("pair_b", C.c_void_p), ("pair_qq", C.c_void_p),
                ("n_mirror", C.c_int64), ("mirror_dst", C.c_void_p), ("mirror_src", C.c_void_p),
                ("scnb", C.c_float), ("scee", C.c_float), ("max_iter", C.c_int32),
                ("lr", C.c_float), ("tol_grad", C.c_float), ("tol_change", C.c_float)]


class _RestraintSet(C.Structure):
    _fields_ = [("n_point", C.c_int64), ("point_atom", C.c_void_p), ("point_anchor", C.c_void_p), ("point_k", C.c_void_p),
                ("point_rt", C.c_void_p), ("n_pair", C.c_int64), ("pair_ij", C.c_void_p), ("pair_k", C.c_void_p),
                ("pair_rt", C.c_void_p), ("atom_lo", C.c_int64), ("atom_hi", C.c_int64)]


# every symbol include/visnet_b200.h declares (tests check that the library exports each of them)
EXPORTED_SYMBOLS = [
    "vb_weight_manifest", "vb_create", "vb_destroy", "vb_last_error", "vb_set_topology", "vb_forward",
    "vb_forward_host", "vb_set_protein_map", "vb_forward_protein", "vb_get_edges", "vb_launches_per_forward",
    "vb_set_option", "vb_get_option", "vb_num_stages", "vb_stage_name", "vb_debug_run", "vb_debug_read", "vb_profile_stages", "vb_tc_selftest",
    "vb_md_setup", "vb_md_set_normals", "vb_md_set_state", "vb_md_kick1", "vb_md_eval", "vb_md_kick2", "vb_md_run", "vb_md_get_state",
    "vb_set_nonbonded", "vb_nonbonded", "vb_set_restraints", "vb_restraints",
    "vb_comm_init", "vb_comm_connect", "vb_comm_allreduce",
    "vb_set_caph", "vb_caph_relax",
]


def load_library(path: Optional[str] = None):
    """Load (never build) the shared library; raises if it is missing -- there is no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or _build.LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -m ai2bmd_b200.build` "
                           "(nvcc, sm_100a).  The engine has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    lib.vb_weight_manifest.restype = C.c_char_p
    lib.vb_weight_manifest.argtypes = []
    lib.vb_create.restype = C.c_int
    lib.vb_create.argtypes = [vp, C.c_size_t, C.POINTER(_HParams), C.c_int, C.POINTER(vp)]
    lib.vb_destroy.restype = None
    lib.vb_destroy.argtypes = [vp]
    lib.vb_last_error.restype = C.c_char_p
    lib.vb_last_error.argtypes = [vp]
    lib.vb_set_topology.restype = C.c_int
    lib.vb_set_topology.argtypes = [vp, i64, i64, vp, vp, i64]
    lib.vb_forward.restype = C.c_int
    lib.vb_forward.argtypes = [vp, vp, vp, vp, vp]
    lib.vb_forward_host.restype = C.c_int
    lib.vb_forward_host.argtypes = [vp, vp, vp, vp]
    lib.vb_set_protein_map.restype = C.c_int
    lib.vb_set_protein_map.argtypes = [vp, i64, i64, vp, vp, vp, vp]
    lib.vb_forward_protein.restype = C.c_int
    lib.vb_forward_protein.argtypes = [vp, vp, vp, vp]
    lib.vb_get_edges.restype = C.c_int
    lib.vb_get_edges.argtypes = [vp, vp, vp]
    lib.vb_launches_per_forward.restype = C.c_int
    lib.vb_launches_per_forward.argtypes = [vp]
    lib.vb_set_option.restype = C.c_int
    lib.vb_set_option.argtypes = [vp, C.c_char_p, i64]
    lib.vb_get_option.restype = i64
    lib.vb_get_option.argtypes = [vp, C.c_char_p]
    lib.vb_num_stages.restype = C.c_int
    lib.vb_num_stages.argtypes = [vp]
    lib.vb_stage_name.restype = C.c_char_p
    lib.vb_stage_name.argtypes = [vp, C.c_int]
    lib.vb_debug_run.restype = C.c_int
    lib.vb_debug_run.argtypes = [vp, vp, C.c_int]
    lib.vb_profile_stages.restype = C.c_int
    lib.vb_profile_stages.argtypes = [vp, vp, C.c_int, vp]
    lib.vb_tc_selftest.restype = C.c_int
    lib.vb_tc_selftest.argtypes = [C.c_int, vp, vp, vp, C.c_int, vp]
    lib.vb_debug_read.restype = i64
    lib.vb_debug_read.argtypes = [vp, C.c_char_p, C.c_int, vp, i64]
    lib.vb_md_setup.restype = C.c_int
    lib.vb_md_setup.argtypes = [vp, i64, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_double, C.c_uint64, vp]
    lib.vb_md_set_normals.restype = C.c_int
    lib.vb_md_set_normals.argtypes = [vp, vp, i64]
    lib.vb_md_set_state.restype = C.c_int
    lib.vb_md_set_state.argtypes = [vp, vp, vp, i64]
    for name in ("vb_md_kick1", "vb_md_eval", "vb_md_kick2"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [vp, vp]
    lib.vb_md_run.restype = C.c_int
    lib.vb_md_run.argtypes = [vp, i64, vp]
    lib.vb_set_nonbonded.restype = C.c_int
    lib.vb_set_nonbonded.argtypes = [vp, i64, vp, vp, vp, vp, vp, i64, i64]
    lib.vb_nonbonded.restype = C.c_int
    lib.vb_nonbonded.argtypes = [vp, vp, vp, vp]
    lib.vb_set_restraints.restype = C.c_int
    lib.vb_set_restraints.argtypes = [vp, C.POINTER(_RestraintSet)]
    lib.vb_restraints.restype = C.c_int
    lib.vb_restraints.argtypes = [vp, vp, vp, vp]
    lib.vb_comm_init.restype = C.c_int
    lib.vb_comm_init.argtypes = [vp, C.c_int, C.c_int, i64, vp]
    lib.vb_comm_connect.restype = C.c_int
    lib.vb_comm_connect.argtypes = [vp, vp]
    lib.vb_comm_allreduce.restype = C.c_int
    lib.vb_comm_allreduce.argtypes = [vp, vp, i64, vp]
    lib.vb_set_caph.restype = C.c_int
    lib.vb_set_caph.argtypes = [vp, C.POINTER(_CaphProblem)]
    lib.vb_caph_relax.restype = C.c_int
    lib.vb_caph_relax.argtypes = [vp, vp, vp]
    lib.vb_md_get_state.restype = C.c_int
    lib.vb_md_get_state.argtypes = [vp, vp, vp, vp, vp, i64]
    if path == _build.LIB_PATH:
        _lib = lib
    return lib


def weight_manifest() -> str:
    return load_library().vb_weight_manifest().decode()


class Engine:
    """One engine per CUDA device (the reference keeps one ``ViSNetModel`` per device,
    ``src/Calculators/bonded.py:40-44``)."""

    def __init__(self, state_dict: Dict[str, np.ndarray], device: int = 0, cutoff: float = 5.0):
        self.lib = load_library()
        blob = pack_weights(state_dict, self.lib.vb_weight_manifest().decode())
        hp = _HParams(128, 6, 8, 32, 32, cutoff)
        handle = C.c_void_p()
        rc = self.lib.vb_create(blob.ctypes.data, blob.size, C.byref(hp), int(device), C.byref(handle))
        if rc != 0:
            raise RuntimeError(f"vb_create failed ({rc}): {self.lib.vb_last_error(None).decode()}")
        self.h = handle
        self.device = int(device)
        self.n_atoms = 0
        self.n_graphs = 0
        self.n_protein = 0

    def _check(self, rc, what):
        if rc < 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.vb_last_error(self.h).decode()}")
        return rc

    def close(self):
        if getattr(self, "h", None):
            self.lib.vb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- topology ----
    def set_topology(self, z, batch, n_graphs: Optional[int] = None, max_edges: int = 0):
        z = np.ascontiguousarray(z, dtype=np.int64)
        batch = np.ascontiguousarray(batch, dtype=np.int64)
        if z.shape != batch.shape or z.ndim != 1 or z.size == 0:
            raise ValueError("z and batch must be non-empty 1-D arrays of equal length")
        g = int(batch.max()) + 1 if n_graphs is None else int(n_graphs)
        self._check(self.lib.vb_set_topology(self.h, z.size, g, z.ctypes.data, batch.ctypes.data, int(max_edges)),
                    "vb_set_topology")
        self.n_atoms, self.n_graphs = int(z.size), g

    def set_protein_map(self, n_protein, src_atom, dst_atom, sign, frag_sign):
        src_atom = np.ascontiguousarray(src_atom, dtype=np.int32)
        dst_atom = np.ascontiguousarray(dst_atom, dtype=np.int32)
        sign = np.ascontiguousarray(sign, dtype=np.float32)
        frag_sign = np.ascontiguousarray(frag_sign, dtype=np.float32)
        if frag_sign.size != self.n_graphs:
            raise ValueError("frag_sign must have one entry per fragment")
        self._check(self.lib.vb_set_protein_map(self.h, int(n_protein), src_atom.size, src_atom.ctypes.data,
                                                dst_atom.ctypes.data, sign.ctypes.data, frag_sign.ctypes.data),
                    "vb_set_protein_map")
        self.n_protein = int(n_protein)

    def set_option(self, key: str, value: int):
        self._check(self.lib.vb_set_option(self.h, key.encode(), int(value)), "vb_set_option")

    def get_option(self, key: str) -> int:
        return int(self.lib.vb_get_option(self.h, key.encode()))

    # ---- evaluation ----
    def forward_host(self, pos: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        """Host arrays in, host arrays out (H2D / D2H inside the call)."""
        pos = np.ascontiguousarray(pos, dtype=np.float32)
        if pos.shape != (self.n_atoms, 3):
            raise ValueError(f"pos must be [{self.n_atoms},3]")
        e = np.empty((self.n_graphs,), dtype=np.float32)
        f = np.empty((self.n_atoms, 3), dtype=np.float32)
        # __array_interface__ instead of .ctypes.data: no ctypes helper object per array (this call is the per-step path)
        rc = self.lib.vb_forward_host(self.h, pos.__array_interface__["data"][0], e.__array_interface__["data"][0],
                                      f.__array_interface__["data"][0])
        if rc < 0:
            self._check(rc, "vb_forward_host")
        return e, f

    def forward_device(self, pos_ptr: int, energy_ptr: int, forces_ptr: int, stream_ptr: int = 0):
        """Raw device pointers (e.g. ``tensor.data_ptr()``) and a ``cudaStream_t``; asynchronous."""
        self._check(self.lib.vb_forward(self.h, pos_ptr, energy_ptr, forces_ptr, stream_ptr), "vb_forward")

    def forward_protein_device(self, pos_ptr: int, ef_ptr: int, stream_ptr: int = 0):
        self._check(self.lib.vb_forward_protein(self.h, pos_ptr, ef_ptr, stream_ptr), "vb_forward_protein")

    # ---- cap-hydrogen refinement (include/visnet_b200.h: vb_set_caph / vb_caph_relax) ----
    def set_caph(self, problem):
        """``problem``: an :class:`ai2bmd_b200.caph.CapHProblem` (flat term arrays over the packed fragment atoms)."""
        keep, p = [], _CaphProblem()

        def arr(a, dtype):
            a = np.ascontiguousarray(a, dtype=dtype)
            keep.append(a)
            return a.ctypes.data if a.size else None

        p.n_h, p.h_idx = len(problem.h_idx), arr(problem.h_idx, np.int32)
        p.n_bonds, p.bond_ij, p.bond_k, p.bond_r0 = len(problem.bond_k), arr(problem.bond_ij, np.int32), arr(problem.bond_k, np.float32), arr(problem.bond_r0, np.float32)
        p.n_angles, p.angle_ijk, p.angle_k, p.angle_t0 = len(problem.angle_k), arr(problem.angle_ijk, np.int32), arr(problem.angle_k, np.float32), arr(problem.angle_t0, np.float32)
        p.n_dih, p.dih_ijkl, p.dih_k = len(problem.dih_k), arr(problem.dih_ijkl, np.int32), arr(problem.dih_k, np.float32)
        p.dih_n, p.dih_p = arr(problem.dih_n, np.float32), arr(problem.dih_p, np.float32)
        p.n_pairs, p.pair_ij, p.pair_a = len(problem.pair_a), arr(problem.pair_ij, np.int32), arr(problem.pair_a, np.float32)
        p.pair_b, p.pair_qq = arr(problem.pair_b, np.float32), arr(problem.pair_qq, np.float32)
        p.n_mirror, p.mirror_dst, p.mirror_src = len(problem.mirror_dst), arr(problem.mirror_dst, np.int32), arr(problem.mirror_src, np.int32)
        p.scnb, p.scee, p.max_iter = float(problem.scnb), float(problem.scee), int(problem.max_iter)
        p.lr, p.tol_grad, p.tol_change = float(problem.lr), float(problem.tol_grad), float(problem.tol_change)
        self._check(self.lib.vb_set_caph(self.h, C.byref(p)), "vb_set_caph")

    def caph_relax(self, pos_ptr: int, stream_ptr: int = 0):
        """Refine the added hydrogens of a packed fragment position buffer (device pointer) in place; asynchronous."""
        self._check(self.lib.vb_caph_relax(self.h, pos_ptr, stream_ptr), "vb_caph_relax")

    # ---- NVLink peer-memory all-reduce (include/visnet_b200.h: vb_comm_*) ----
    def comm_init(self, rank: int, world: int, max_floats: int) -> bytes:
        """Allocate this rank's window; returns its 64-byte CUDA IPC handle (exchange it with every other rank)."""
        buf = C.create_string_buffer(64)
        self._check(self.lib.vb_comm_init(self.h, int(rank), int(world), int(max_floats), buf), "vb_comm_init")
        return bytes(buf.raw)

    def comm_connect(self, handles) -> None:
        """``handles``: the IPC handles of all ranks in rank order (this rank's own included)."""
        blob = b"".join(bytes(x) for x in handles)
        self._check(self.lib.vb_comm_connect(self.h, C.c_char_p(blob)), "vb_comm_connect")

    def comm_allreduce(self, buf_ptr: int, n: int, stream_ptr: int = 0):
        self._check(self.lib.vb_comm_allreduce(self.h, buf_ptr, int(n), stream_ptr), "vb_comm_allreduce")

    # ---- non-bonded MM term ----
    def set_nonbonded(self, charges, sigmas_nm, epsilons_kj, excl_rowptr, excl_col, atom_lo: int = 0, atom_hi: int = -1):
        q = np.ascontiguousarray(charges, dtype=np.float32)
        sg = np.ascontiguousarray(sigmas_nm, dtype=np.float32)
        ep = np.ascontiguousarray(epsilons_kj, dtype=np.float32)
        rp = np.ascontiguousarray(excl_rowptr, dtype=np.int32)
        cl = np.ascontiguousarray(excl_col, dtype=np.int32)
        n = len(q)
        if not (len(sg) == len(ep) == n and len(rp) == n + 1 and int(rp[-1]) == len(cl)):
            raise ValueError("non-bonded parameter arrays / exclusion table have inconsistent lengths")
        self._check(self.lib.vb_set_nonbonded(self.h, n, q.ctypes.data, sg.ctypes.data, ep.ctypes.data, rp.ctypes.data,
                                              cl.ctypes.data if len(cl) else None, int(atom_lo),
                                              int(n if atom_hi < 0 else atom_hi)), "vb_set_nonbonded")

    def nonbonded_device(self, prot_pos_ptr: int, ef_ptr: int, stream_ptr: int = 0):
        self._check(self.lib.vb_nonbonded(self.h, prot_pos_ptr, ef_ptr, stream_ptr), "vb_nonbonded")

    # ---- Hookean restraints (include/visnet_b200.h: vb_set_restraints / vb_restraints) ----
    def set_restraints(self, point_atom=(), point_anchor=(), point_k=(), point_rt=(), pair_ij=(), pair_k=(), pair_rt=(),
                       atom_lo: int = 0, atom_hi: int = -1):
        """Install a restraint set (eV/A^2, A); replaces the previous one.  ``atom_hi < 0`` means every protein atom.
        :class:`ai2bmd_b200.restraints.RestraintSet` holds these arrays (``RestraintSet.install(engine)``)."""
        pa = np.ascontiguousarray(point_atom, dtype=np.int32).reshape(-1)
        px = np.ascontiguousarray(point_anchor, dtype=np.float64).reshape(-1, 3)
        pk = np.ascontiguousarray(point_k, dtype=np.float64).reshape(-1)
        pr = np.ascontiguousarray(point_rt, dtype=np.float64).reshape(-1)
        qij = np.ascontiguousarray(pair_ij, dtype=np.int32).reshape(-1, 2)
        qk = np.ascontiguousarray(pair_k, dtype=np.float64).reshape(-1)
        qr = np.ascontiguousarray(pair_rt, dtype=np.float64).reshape(-1)
        if not (len(pa) == len(px) == len(pk) == len(pr) and len(qij) == len(qk) == len(qr)):
            raise ValueError("restraint arrays have inconsistent lengths")
        ptr = lambda a: a.ctypes.data if a.size else None
        rs = _RestraintSet(len(pa), ptr(pa), ptr(px), ptr(pk), ptr(pr), len(qij), ptr(qij), ptr(qk), ptr(qr),
                           int(atom_lo), int(self.n_protein if atom_hi < 0 else atom_hi))
        self._check(self.lib.vb_set_restraints(self.h, C.byref(rs)), "vb_set_restraints")

    def clear_restraints(self):
        self.set_restraints()

    def restraints_device(self, prot_pos_ptr: int, ef_ptr: int, stream_ptr: int = 0):
        """ef[3n+1] += restraint forces / energy at the fp64 protein positions (device pointers); asynchronous."""
        self._check(self.lib.vb_restraints(self.h, prot_pos_ptr, ef_ptr, stream_ptr), "vb_restraints")

    # ---- device-resident MD (include/visnet_b200.h: vb_md_*) ----
    def md_setup(self, masses, real, acc, rem, blen, dt, kT, friction, seed, ef_ptr: int):
        self._md_keep = [np.ascontiguousarray(masses, dtype=np.float64), np.ascontiguousarray(real, dtype=np.int32),
                         np.ascontiguousarray(acc, dtype=np.int32), np.ascontiguousarray(rem, dtype=np.int32),
                         np.ascontiguousarray(blen, dtype=np.float32)]
        m, r, a, q, b = self._md_keep
        if not (len(r) == len(a) == len(q) == len(b)):
            raise ValueError("recipe arrays must have one entry per fragment atom")
        self._check(self.lib.vb_md_setup(self.h, len(m), m.ctypes.data, r.ctypes.data, a.ctypes.data, q.ctypes.data,
                                         b.ctypes.data, float(dt), float(kT), float(friction), int(seed), ef_ptr),
                    "vb_md_setup")
        self._md_n = len(m)

    def md_set_normals(self, pool_ptr: int, pool_steps: int):
        self._check(self.lib.vb_md_set_normals(self.h, pool_ptr, int(pool_steps)), "vb_md_set_normals")

    def md_set_state(self, x, v, step: int = 0):
        x = np.ascontiguousarray(x, dtype=np.float64)
        v = np.ascontiguousarray(v, dtype=np.float64)
        if x.size != 3 * self._md_n or v.size != 3 * self._md_n:
            raise ValueError("state arrays must be [n_protein, 3]")
        self._check(self.lib.vb_md_set_state(self.h, x.ctypes.data, v.ctypes.data, int(step)), "vb_md_set_state")

    def md_kick1(self, stream_ptr: int = 0):
        self._check(self.lib.vb_md_kick1(self.h, stream_ptr), "vb_md_kick1")

    def md_eval(self, stream_ptr: int = 0):
        self._check(self.lib.vb_md_eval(self.h, stream_ptr), "vb_md_eval")

    def md_kick2(self, stream_ptr: int = 0):
        self._check(self.lib.vb_md_kick2(self.h, stream_ptr), "vb_md_kick2")

    def md_run(self, n_steps: int, stream_ptr: int = 0):
        self._check(self.lib.vb_md_run(self.h, int(n_steps), stream_ptr), "vb_md_run")

    def md_get_state(self, n_hist: int = 0):
        """(x [n,3], v [n,3], step, epot history of the last n_hist steps) -- synchronises the device."""
        x = np.empty((self._md_n, 3), dtype=np.float64)
        v = np.empty((self._md_n, 3), dtype=np.float64)
        step = C.c_int64(0)
        hist = np.zeros(max(n_hist, 1), dtype=np.float64)
        self._check(self.lib.vb_md_get_state(self.h, x.ctypes.data, v.ctypes.data, C.byref(step), hist.ctypes.data,
                                             int(n_hist)), "vb_md_get_state")
        return x, v, int(step.value), hist[:n_hist]

    def get_edges(self) -> Tuple[np.ndarray, np.ndarray]:
        slots = np.empty((self.n_atoms, 32), dtype=np.int32)
        deg = np.empty((self.n_atoms,), dtype=np.int32)
        self._check(self.lib.vb_get_edges(self.h, slots.ctypes.data, deg.ctypes.data), "vb_get_edges")
        return slots, deg

    @property
    def launches_per_forward(self) -> int:
        return int(self.lib.vb_launches_per_forward(self.h))

    # ---- diagnostics ----
    def stage_names(self):
        return [self.lib.vb_stage_name(self.h, i).decode() for i in range(self.lib.vb_num_stages(self.h))]

    def debug_run(self, pos_ptr: int, n_stages: int):
        self._check(self.lib.vb_debug_run(self.h, pos_ptr, int(n_stages)), "vb_debug_run")

    def profile_stages(self, pos_ptr: int, n_iter: int = 5):
        """[(stage name, ms)] -- per-launch device time measured with CUDA events inside the library."""
        names = self.stage_names()
        ms = np.zeros(len(names), dtype=np.float32)
        self._check(self.lib.vb_profile_stages(self.h, pos_ptr, int(n_iter), ms.ctypes.data), "vb_profile_stages")
        return list(zip(names, ms.tolist()))

    def vecln_near_ties(self, rel_gap: float = 1e-5) -> np.ndarray:
        """Atoms of the LAST evaluation that sit on a derivative kink of the model (diagnostic).

        VecLayerNorm(max_min) (reference ``src/ViSNet/model/utils.py:165-215``) normalises the channel norms of an atom's
        vector features by their max and min over the 128 channels, so the gradient of the energy is routed through the
        argmax / argmin channel.  Where the two largest (or two smallest) channel norms agree to fp32 rounding the
        argmax flips with the rounding order and the force on that fragment jumps by up to ~1e-2 eV/A -- in the
        reference as much as here.  Returns the sorted atom indices whose top-two or bottom-two channel norms in any
        layer differ by less than ``rel_gap`` relative; callers comparing two evaluation orders (tests,
        plan-vs-plan checks) exclude the fragments of these atoms.
        """
        n = self.n_atoms
        hit = np.zeros(n, dtype=bool)
        for k in range(1, 6):                     # the vector features entering layer 0 are identically zero
            v = self.debug_read("V", k, (n, 3, 128)).astype(np.float64)
            srt = np.sort(np.sqrt((v * v).sum(1)), axis=1)
            hit |= ((srt[:, -1] - srt[:, -2]) < rel_gap * srt[:, -1]) | ((srt[:, 1] - srt[:, 0]) < rel_gap * srt[:, 1])
        return np.flatnonzero(hit)

    def debug_read(self, name: str, layer: int, shape, dtype=np.float32) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        n = self._check(self.lib.vb_debug_read(self.h, name.encode(), int(layer), out.ctypes.data, out.nbytes),
                        "vb_debug_read")
        if n != out.nbytes:
            raise RuntimeError(f"vb_debug_read({name}): got {n} bytes, wanted {out.nbytes}")
        return out


def tc_selftest(a: np.ndarray, w_nk: np.ndarray, reps: int = 1, device: int = 0):
    """Run D = A @ W^T (A [128,128], W [128 out,128 in]) through the tcgen05 pipeline; returns (D, ms)."""
    from .weights import tc_image
    lib = load_library()
    a = np.ascontiguousarray(a, dtype=np.float32)
    img = tc_image(w_nk)
    d = np.zeros((128, 128), dtype=np.float32)
    ms = C.c_float(0)
    rc = lib.vb_tc_selftest(int(device), a.ctypes.data, img.ctypes.data, d.ctypes.data, int(reps), C.byref(ms))
    if rc != 0:
        raise RuntimeError(f"vb_tc_selftest failed ({rc}): {lib.vb_last_error(None).decode()}")
    return d, float(ms.value)
