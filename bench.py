#!/usr/bin/env python
"""bench.py -- MD steps/s of the ViSNet energy/force hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload chig] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: neighbour build + ViSNet energy + analytic forces for
every fragment of the protein + signed reduction to whole-protein energy/forces (what one MD step of the
reference's ``FragmentCalculator`` asks of ``DLBondedCalculator``, bonded.py:102-123).  Workload at N=1:
BASELINE.json configs[1], Chignolin fully fragmented (19 fragments, 391 fragment atoms, ~6.7k edges,
175 protein atoms), real checkpoint weights (tests/golden/weights_2ef43f29.npz), the example-PDB geometry.

* ``value``  : steps/s with inputs resident in HBM (``vb_forward_protein`` on device buffers), each step
               timed with CUDA events on the launching stream, L2 flushed between timed steps.
* ``e2e``    : steps/s through the reference-facing call ``ViSNetModel.dl_potential_loader(FragmentData)``
               with HOST numpy buffers: H2D of the positions and D2H of energies/forces inside the timed region.
* ``roofline``: dominant kernel (per-launch device times measured live with CUDA events inside the library),
               algorithmic bytes per launch (SURVEY.md section 8d) / time, against MEASURED_PEAKS.json.
* ``cpu_baseline`` / ``--impl reference``: the CPU oracle (pure-PyTorch port of the reference model) on the
               host cores -- the reference itself cannot be imported on this image (its third-party graph
               packages are absent), so kind = "port".
N>1 (torchrun, one rank per GPU): fragments sharded over ranks (strong scaling: the protein is fixed), one
NCCL all-reduce of the [3*N_prot+1] buffer per step; time = max over ranks between barriers.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, L = 128, 6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chig", choices=["chig", "trpcage", "ww", "abd", "c4", "c4_20k", "c5"])
    ap.add_argument("--no-flush", action="store_true", help="keep L2 warm between timed steps (diagnostic)")
    ap.add_argument("--fragments", type=int, default=512, help="fragment count of the synthetic c4 batch")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--nccl", action="store_true", help="N > 1: torch.distributed all-reduce instead of the peer-memory one")
    ap.add_argument("--no-c4", action="store_true", help="N > 1: skip the 512-fragment strong-scaling leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the whole-protein forces and energy of the last timed step as DIR/forces.npy, DIR/energy.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; it does not apply to --impl reference")
    return args


def load_workload(name, n_fragments=512):
    from ai2bmd_b200.fixtures import load_fragments
    from ai2bmd_b200.synth import conformer_batch, synthetic_batch, synthetic_protein_map
    if name in ("chig", "trpcage", "ww", "abd"):
        fd, pm = load_fragments(name)
        desc = {"chig": "Chignolin (chig.pdb) full fragmentation", "trpcage": "Trp-cage full fragmentation",
                "ww": "WW domain full fragmentation", "abd": "ABD full fragmentation"}[name]
    elif name == "c4":
        fd = synthetic_batch(n_fragments, seed=0)
        pm, desc = synthetic_protein_map(fd), f"synthetic {n_fragments}-fragment batch (seed 0)"
    elif name == "c4_20k":
        fd = synthetic_batch(512, seed=0, min_atoms=20000)
        pm, desc = synthetic_protein_map(fd), "synthetic >=20k-atom batch (seed 0)"
    else:
        fd = conformer_batch(2048, seed=1)
        pm, desc = synthetic_protein_map(fd), "2048 dipeptide conformers (seed 1)"
    return fd, pm, desc


def load_weights():
    from ai2bmd_b200.fixtures import WEIGHTS
    from ai2bmd_b200.weights import load_state_dict
    return load_state_dict(WEIGHTS)


class ClockSampler:
    """SM clock and throttle reasons sampled every 20 ms through NVML (in-process thread; works the same under torchrun)
    while ``loaded`` is set, i.e. during the warm-up and the timed GPU regions; nvidia-smi is the fallback."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index=0):
        self.index, self.sm, self.mx, self.mask = index, [], [], 0
        self.loaded, self._stop, self.thread, self.how = False, False, None, None

    def _nvml_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.nv, self.how = pynvml, "nvml, 20 ms period"
            self.max_clock = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv, self.how = None, "nvidia-smi -lms 100"
        self.thread = threading.Thread(target=self._run_nvml if self.nv else self._run_smi, daemon=True)
        self.thread.start()

    def _run_nvml(self):
        nv = self.nv
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop:
            if self.loaded:
                try:
                    self.sm.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    self.mx.append(self.max_clock)
                    self.mask |= int(reasons(self.h))
                except Exception:
                    pass
            time.sleep(0.02)

    def _run_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
        try:
            proc = subprocess.Popen(["nvidia-smi", "-i", str(self._nvml_index()), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                     "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        for line in proc.stdout:
            if self._stop:
                break
            r = [x.strip() for x in line.split(",")]
            if self.loaded and len(r) >= 3 and r[0].isdigit():
                self.sm.append(int(r[0])); self.mx.append(int(r[1]) if r[1].isdigit() else 0)
                try:
                    self.mask |= int(r[2], 16)
                except ValueError:
                    pass
        proc.terminate()

    def stop(self):
        self._stop = True
        names = sorted(n for bit, n in self.REASONS.items() if self.mask & bit)
        return {"sm_mhz": int(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": names, "samples": len(self.sm), "how": self.how}


def algorithmic_bytes(stage, n_atoms, n_edges):
    """Algorithmic HBM bytes of one launch (SURVEY.md section 8d, fully fused lower bound)."""
    if stage.startswith("edge_fwd"):
        last = stage.endswith(str(L - 1))
        return n_edges * (1044 - (512 if last else 0)) + 4096 * n_atoms
    if stage.startswith("edge_bwd"):
        return 1572 * n_edges + 8192 * n_atoms
    if stage.startswith("node_fwd") or stage.startswith("node_bwd"):
        return 8192 * n_atoms
    if stage.startswith("head"):
        return 4096 * n_atoms
    return None


def tensor_roofline(stages, n_edges, seconds, edge_tc):
    """Tensor-pipe view of the tcgen05 edge stages (SURVEY 8d: report against the measured bf16 rate, TF32 = 1/2 of it).

    ``stages`` = names of the launches timed in ``seconds``.  Algorithmic MMA work per edge and layer: forward
    dk, dv, f (3 x 128x128) + s_proj (2 x 128x128), adjoint g_s.Ws (2) + g_P.W1 (3); the last layer has no f chunk.
    Each product runs as three TF32 MMAs (3xTF32: hi.hi + lo.hi + hi.lo) for fp32 parity, so the executed tensor
    flops are 3x the fp32-equivalent ones.  Returns None for stages that do not run on tensor cores."""
    fwd = [s for s in stages if s.startswith("edge_fwd")]
    bwd = [s for s in stages if s.startswith("edge_bwd")]
    if not ((fwd and (edge_tc & 1)) or (bwd and (edge_tc & 2))) or seconds <= 0:
        return None
    products = 0
    for s in fwd + bwd:
        products += 4 if s.endswith(str(L - 1)) else 5
    fp32_equiv = 2.0 * D * D * n_edges * products
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        bf16, kind = float(json.load(open(p))["bf16_tflops_sustained"]), "measured bf16 sustained / 2"
    else:
        bf16, kind = 1590.0, "fallback bf16 / 2"
    achieved = 3.0 * fp32_equiv / seconds / 1e12
    return {"bound": "tensor", "achieved": achieved, "peak": bf16 / 2, "peak_kind": kind, "unit": "TFLOP/s",
            "frac": achieved / (bf16 / 2), "fp32_equivalent_tflops": fp32_equiv / seconds / 1e12,
            "note": "executed TF32 MMA flops (3xTF32) of the algorithmic products; padded tile rows not counted"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def make_cpu_model(sd, sample):
    """The CPU oracle with the thread count that is fastest on this host for this workload: tiny per-fragment
    tensors do not scale to hundreds of threads, so a few candidates up to all host threads are timed once."""
    import torch
    from oracle import visnet_ref as O
    model = O.OracleCalculatorModel({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    avail = host_threads()
    cands = sorted({c for c in (4, 8, 16, 32, 64, avail) if c <= avail}) or [avail]
    torch.set_num_threads(cands[0])
    model.dl_potential_loader(sample)                   # warm-up (allocator, lazy init)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        dt = float("inf")
        for _ in range(2):                              # best of two: a single timing picked 8 threads (2.8 steps/s) where 16 give 4.0
            t0 = time.perf_counter()
            model.dl_potential_loader(sample)
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return model, best, avail


# ---------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port, on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fd, pm, desc = load_workload(args.workload, args.fragments)
    sd = load_weights()
    calib = fd if len(fd) <= 64 else fd[0:8]              # the whole workload when it is small: the thread optimum depends on the batch
    model, threads, avail = make_cpu_model(sd, calib)
    t0 = time.perf_counter()
    model.dl_potential_loader(fd)
    t1 = time.perf_counter() - t0
    # bounded sample: a contiguous prefix of fragments so that (steps+warmup) evaluations fit ~150 s
    budget = 150.0
    frac = min(1.0, budget / max(1e-9, (args.steps + args.warmup) * t1))
    n_frag = len(fd) if frac >= 1.0 else max(2, int(len(fd) * frac) // 2 * 2)
    sample = fd if n_frag >= len(fd) else fd[0:n_frag]
    scale = float(len(fd.z)) / float(len(sample.z))
    for _ in range(args.warmup):
        model.dl_potential_loader(sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.dl_potential_loader(sample)
    dt = (time.perf_counter() - t0) / args.steps * scale
    value = 1.0 / dt
    sample_desc = (f"{args.steps} evaluations of the first {n_frag}/{len(fd)} fragments ({len(sample.z)} atoms), "
                   f"time scaled by atoms x{scale:.2f}" if n_frag < len(fd) else f"{args.steps} full evaluations")
    line = {
        "impl": "reference", "metric": "MD steps/sec", "value": value, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "example-PDB geometry, shipped checkpoint weights",
        "config": {"workload": workload_string(desc, fd), "device": "host CPU"},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "host_threads_available": avail,
                         "kind": "port", "sample": sample_desc},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_string(desc, fd):
    """Identical in both arms (the driver compares the strings)."""
    return f"{desc}: G={len(fd)} N={len(fd.z)}"


def time_shard_steps(torch, dist, shard, steps, warmup, world, flush=None):
    """Device time of `steps` evaluations of a DeviceShard (CUDA events around each step, max over ranks), seconds."""
    stream = torch.cuda.current_stream()
    for _ in range(max(3, warmup)):
        shard.step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        if flush is not None:
            flush.fill_(1.0)
        a.record(stream)
        shard.step()
        b.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def golden_reference(workload):
    """Outputs of the reference's own model source on this workload (tests/golden/make_golden.py), if committed."""
    path = os.path.join(ROOT, "tests", "golden", "reference_outputs.npz")
    if workload not in ("chig", "trpcage") or not os.path.exists(path):
        return None
    r = np.load(path)
    return {"e": r[f"{workload}_ref_e"], "f": r[f"{workload}_ref_f"], "e64": r[f"{workload}_e64"], "f64": r[f"{workload}_f64"]}


DUMP_FORCE_BYTES = 60 << 20          # keeps a dump under 64 MB


def dump_outputs(out_dir, ef, n_protein):
    """Write what a caller of the timed path (``vb_forward_protein``) receives, float32: ``forces.npy`` [n_protein, 3]
    (eV/A) and ``energy.npy`` [1] (eV).  Forces above 60 MiB are a fixed sample of protein atoms, the rows
    ``sort(default_rng(0).choice(n_protein, k, replace=False))``, so that two runs write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    forces = ef[:-1].reshape(n_protein, 3)
    if forces.nbytes > DUMP_FORCE_BYTES:
        k = DUMP_FORCE_BYTES // forces[0].nbytes
        forces = forces[np.sort(np.random.default_rng(0).choice(n_protein, k, replace=False))]
    np.save(os.path.join(out_dir, "forces.npy"), forces)
    np.save(os.path.join(out_dir, "energy.npy"), ef[-1:])


def run_ours(args):
    import torch
    import torch.distributed as dist
    from ai2bmd_b200.calculator import ViSNetModel
    from ai2bmd_b200.parallel import DeviceShard, combine_local

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("BENCH_FAULT_AFTER"):       # debugging aid: dump every thread's stack and exit after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BENCH_FAULT_AFTER"]), exit=True)
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    fd, pm, desc = load_workload(args.workload, args.fragments)
    sd = load_weights()
    n_atoms, n_frag = len(fd.z), len(fd)

    shard = DeviceShard(sd, fd, pm, rank, world, local, native_comm=not args.nccl)
    stream = torch.cuda.current_stream()
    flush = None if args.no_flush else torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    clocks.loaded = True
    # ---- device-resident timing (value): CUDA events around each step, L2 flushed before each, max over ranks ----
    wall0 = time.perf_counter()
    t_dev = time_shard_steps(torch, dist, shard, args.steps, args.warmup, world, flush)
    wall = time.perf_counter() - wall0
    ef = shard.ef.clone()
    n_edges_local = int(shard.engine.get_edges()[1].sum()) if shard.engine is not None else 0   # edges of the timed positions
    # ---- warm-L2 variant (diagnostic) ----
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(args.steps):
        shard.step()
    b.record(stream)
    barrier()
    t_warm = torch.tensor([a.elapsed_time(b) / 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_warm, op=dist.ReduceOp.MAX)
    # ---- the collective alone (N > 1): all-reduce of the [3*N_prot + 1] buffer, device time per call ----
    comm = None
    if world > 1:
        buf = torch.zeros(3 * pm.n_protein + 1, dtype=torch.float32, device="cuda")

        def one_reduce():
            if shard.native:
                shard.comm_engine.comm_allreduce(buf.data_ptr(), buf.numel(), stream.cuda_stream)
            else:
                dist.all_reduce(buf)
        for _ in range(5):
            one_reduce()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(50):
            one_reduce()
        b.record(stream)
        barrier()
        t_c = torch.tensor([a.elapsed_time(b) / 50.0 * 1e3], dtype=torch.float64, device="cuda")
        dist.all_reduce(t_c, op=dist.ReduceOp.MAX)
        comm = {"us_per_allreduce": float(t_c.item()), "bytes": 4 * (3 * pm.n_protein + 1), "how": shard.collective}

    # ---- end-to-end through the reference-facing call, host buffers (rank-local shard + all-reduce) ----
    local_frags = shard.plan.local_fragments(fd)
    model = None
    if local_frags is not None:
        model = ViSNetModel.from_engine(shard.engine, f"cuda:{local}", local_frags)   # the shard's engine, topology already set
    ef_host = torch.zeros(3 * pm.n_protein + 1, dtype=torch.float32).pin_memory()
    ef_dev = torch.zeros(3 * pm.n_protein + 1, dtype=torch.float32, device="cuda")

    def e2e_step():
        if model is not None:
            e, f = model.dl_potential_loader(local_frags)         # H2D pos, kernels, D2H e/f (host numpy in/out)
        if world > 1:
            loc = combine_local(shard.plan.local_map, e, f) if model is not None else np.zeros(3 * pm.n_protein + 1, np.float32)
            ef_host.copy_(torch.from_numpy(loc))
            ef_dev.copy_(ef_host, non_blocking=True)
            if shard.native:
                shard.comm_engine.comm_allreduce(ef_dev.data_ptr(), ef_dev.numel(), stream.cuda_stream)
            else:
                dist.all_reduce(ef_dev)
            ef_host.copy_(ef_dev)
        return None

    for _ in range(max(3, args.warmup)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    n_loc = len(local_frags.z) if local_frags is not None else 0
    g_loc = len(local_frags) if local_frags is not None else 0
    e2e = {"value": args.steps / float(t_e2e.item()), "unit": "steps/s", "h2d_bytes_per_step": 12 * n_loc,
           "d2h_bytes_per_step": 12 * n_loc + 4 * g_loc, "api": "ViSNetModel.dl_potential_loader(FragmentData) (host numpy in/out)"}

    # ---- the same loop with the integrator on the device (vb_md_*): state never leaves the GPU ----
    md_device = None
    if args.workload in ("chig", "trpcage", "ww", "abd"):
        from ai2bmd_b200.fixtures import load_protein
        from ai2bmd_b200.md import DeviceLangevin
        from ai2bmd_b200.pdbfrag import FragmentRecipe
        have = torch.tensor([1 if shard.engine is not None else 0], device="cuda")
        if world > 1:
            dist.all_reduce(have, op=dist.ReduceOp.MIN)
        if int(have.item()) == 1:
            prot_pos, prot_z, recipe = load_protein(args.workload)
            lo, hi = (shard.plan.atom_lo, shard.plan.atom_hi) if world > 1 else (0, n_atoms)
            local_recipe = FragmentRecipe(recipe.real[lo:hi], recipe.acc[lo:hi], recipe.rem[lo:hi], recipe.blen[lo:hi])
            dmd = DeviceLangevin(None, None, pm, local_recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0,
                                 friction_per_fs=0.001, seed=0, device=local, group=dist.group.WORLD if world > 1 else None,
                                 engine=shard.engine)
            dmd.run(10)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            dmd.run(args.steps)
            b.record(stream)
            barrier()
            t_md = torch.tensor([a.elapsed_time(b) / 1e3], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t_md, op=dist.ReduceOp.MAX)
            one_graph = world == 1 or shard.native
            md_device = {"value": args.steps / float(t_md.item()), "unit": "steps/s", "temperature_K": dmd.temperature(),
                         "launches_per_step": shard.engine.launches_per_forward + 3 + (1 if world > 1 else 0),
                         "what": "Langevin (dt 1 fs, 300 K, friction 0.001/fs) entirely on the device: half-kick + drift, "
                                 "cap-H placement, engine, signed reduction" + (", all-reduce" if world > 1 else "") +
                                 ", half-kick; " + ("one CUDA graph replay per step" if one_graph else "phases enqueued by the host around the engine's graph") +
                                 ", no host synchronisation, L2 in the loop's steady state"}
    # ---- per-step cap-hydrogen refinement (SURVEY 8f rank 1): cost of the LBFGS kernel alone and of the MD step with it ----
    caph_info = None
    if world == 1 and md_device is not None and args.workload in ("chig", "trpcage"):
        from ai2bmd_b200 import caph as caph_mod
        from ai2bmd_b200.fixtures import load_capped_protein, load_caph_tables
        tables, _ = load_caph_tables(args.workload)
        problem = caph_mod.build_problem(load_capped_protein(args.workload), fd, recipe, tables)
        shard.engine.set_caph(problem)
        ptmp = shard.pos.clone()
        for _ in range(3):
            shard.engine.caph_relax(ptmp.data_ptr(), stream.cuda_stream)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(50):
            ptmp.copy_(shard.pos)
            shard.engine.caph_relax(ptmp.data_ptr(), stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        us = a.elapsed_time(b) / 50 * 1e3
        dmd.run(5)
        barrier()
        a.record(stream)
        dmd.run(args.steps)
        b.record(stream)
        barrier()
        caph_info = {"us_per_refinement": us, "hydrogens": int(len(problem.h_idx)), "terms": int(len(problem.bond_k) + len(problem.angle_k) + len(problem.dih_k) + len(problem.pair_a)),
                     "energy_evaluations": shard.engine.get_option("caph_evals"),
                     "md_device_with_refinement_steps_per_s": args.steps / (a.elapsed_time(b) / 1e3),
                     "what": "one LBFGS call (lr 0.1, max_iter 10, tolerances 0.1 / 0.01) on the Amber terms of all dipeptides, added "
                             "hydrogens only, one CTA (csrc/k_caph.cuh); folded into the device MD step after the placement"}
    clocks.loaded = False
    clock_info = clocks.stop() if rank == 0 else None

    # ---- parity of the N-GPU result against the reference-source golden vectors (same tolerance as the tests) ----
    gold = golden_reference(args.workload)
    parity = None
    if gold is not None:
        ref_ef = combine_local(pm, gold["e"].reshape(-1), gold["f"])
        got = ef.cpu().numpy()
        dF = np.abs(got[:-1] - ref_ef[:-1])
        tol_f = 5e-5 + 2e-5 * float(np.abs(ref_ef[:-1]).max())
        tol_e = 4e-3 * n_frag
        parity = {"against": "whole-protein E/F combined from the outputs of the reference's own model source "
                             "(tests/golden/reference_outputs.npz)",
                  "force_mae_eV_per_A": float(dF.mean()), "force_max_abs_eV_per_A": float(dF.max()),
                  "energy_abs_err_eV": float(abs(got[-1] - ref_ef[-1])), "tol_force": tol_f, "tol_energy": tol_e,
                  "parity_ok": bool(dF.max() <= tol_f and abs(got[-1] - ref_ef[-1]) <= tol_e)}

    # ---- N > 1: the synthetic 512-fragment batch (config C4) at N GPUs and at 1 GPU in the same run ----
    scale_c4 = None
    if world > 1 and not args.no_c4:
        fd4, pm4, desc4 = load_workload("c4", 512)
        sh4 = DeviceShard(sd, fd4, pm4, rank, world, local, native_comm=not args.nccl)
        t4n = time_shard_steps(torch, dist, sh4, 10, 3, world, flush) / 10.0
        t41 = None
        if rank == 0:
            one = DeviceShard(sd, fd4, pm4, 0, 1, local)
            t41 = time_shard_steps(torch, dist, one, 10, 3, 1, flush) / 10.0
            del one
        barrier()
        scale_c4 = {"workload": workload_string(desc4, fd4), "ms_per_step_n_gpus": t4n * 1e3,
                    "ms_per_step_1_gpu": t41 * 1e3 if t41 else None, "speedup": (t41 / t4n) if t41 else None,
                    "collective": sh4.collective}
        del sh4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ef.cpu().numpy(), pm.n_protein)

    # ---- per-kernel times + roofline (rank 0, its shard) ----
    n_edges = n_edges_local
    prof = shard.engine.profile_stages(shard.pos.data_ptr(), n_iter=5)
    total_ms = sum(ms for _, ms in prof)
    fam = {}
    for name, ms in prof:
        key = name.rstrip("0123456789")
        fam.setdefault(key, []).append((name, ms))
    fam_ms = {k: sum(ms for _, ms in v) for k, v in fam.items()}
    top_fam = max(fam_ms, key=fam_ms.get)                 # dominant kernel = the kernel with the largest share of the step
    launches = fam[top_fam]
    peak, peak_kind = peaks()
    loc_atoms = shard.engine.n_atoms
    ab = sum(algorithmic_bytes(n, loc_atoms, n_edges) or 0 for n, _ in launches)
    t_fam = fam_ms[top_fam] * 1e-3
    achieved = (ab / t_fam / 1e9) if ab else None
    traffic = None      # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and world == 1:
        traffic = json.load(open(tpath)).get(f"{args.workload}:{top_fam}")
    roofline = {"bound": "hbm", "kernel": top_fam, "launches_per_step": len(launches),
                "kernel_ms": fam_ms[top_fam] / len(launches), "algorithmic_bytes": ab / len(launches) if ab else None,
                "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "note": "algorithmic bytes = SURVEY 8d fused lower bound per launch (N, E of the timed positions); this stage is "
                        "contraction/latency bound, not HBM bound (DESIGN.md section 5); workloads below ~2k atoms are L2 resident",
                "share_of_step": fam_ms[top_fam] / total_ms,
                "tensor": tensor_roofline([n for n, _ in launches], n_edges, t_fam, shard.engine.get_option("edge_tc")),
                "family_ms": {k: round(v, 4) for k, v in sorted(fam_ms.items(), key=lambda x: -x[1])}}

    # ---- force / energy error against the reference-source golden vectors, per fragment atom (the metric's second half) ----
    accuracy = None
    if gold is not None and world == 1:
        e_h, f_h = shard.engine.forward_host(fd.pos)
        accuracy = {"force_mae_vs_reference_eV_per_A": float(np.abs(f_h - gold["f"]).mean()),
                    "force_max_abs_vs_reference_eV_per_A": float(np.abs(f_h - gold["f"]).max()),
                    "energy_mae_vs_reference_eV": float(np.abs(e_h.reshape(-1) - gold["e"].reshape(-1)).mean()),
                    "force_mae_vs_fp64_oracle_eV_per_A": float(np.abs(f_h - gold["f64"]).mean()),
                    "energy_mae_vs_fp64_oracle_eV": float(np.abs(e_h.reshape(-1) - gold["e64"].reshape(-1)).mean()),
                    "reference": "fp32 outputs of the reference's own ViSNet.forward source on the same fragments "
                                 "(tests/golden/make_golden.py); fp64 oracle = oracle/visnet_ref.py"}

    # ---- CPU baseline (bounded sample) ----
    cpu = None
    if not args.skip_cpu_baseline:
        sample = fd if len(fd.z) <= 800 else fd[0:24]
        model_cpu, threads, avail = make_cpu_model(sd, sample if len(sample) <= 64 else sample[0:8])
        n_eval = 3
        model_cpu.dl_potential_loader(sample)
        t0 = time.perf_counter()
        for _ in range(n_eval):
            model_cpu.dl_potential_loader(sample)
        sec = (time.perf_counter() - t0) / n_eval * (len(fd.z) / len(sample.z))
        cpu = {"value": 1.0 / sec, "unit": "steps/s", "cores": threads, "host_threads_available": avail, "kind": "port",
               "sample": f"{n_eval} evaluations of {len(sample)}/{len(fd)} fragments ({len(sample.z)} atoms) by the "
                         f"pure-PyTorch CPU oracle, fp32, {threads} threads (fastest of the candidates tried); "
                         f"scaled by atom count"}

    # ---- B1 (BASELINE.md section 3): the same oracle as eager PyTorch on this B200 -- "the reference on a modern GPU" ----
    gpu_eager = None
    if not args.skip_cpu_baseline and world == 1:
        from oracle import visnet_ref as O
        sample = fd if len(fd.z) <= 800 else fd[0:24]
        m_gpu = O.OracleCalculatorModel({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, device="cuda")
        for _ in range(2):
            m_gpu.dl_potential_loader(sample)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n_eval = 5
        for _ in range(n_eval):
            m_gpu.dl_potential_loader(sample)
        torch.cuda.synchronize()
        sec = (time.perf_counter() - t0) / n_eval * (len(fd.z) / len(sample.z))
        gpu_eager = {"value": 1.0 / sec, "unit": "steps/s", "kind": "port, eager PyTorch ops on cuda:0 (autograd forces), "
                     "host numpy in/out, neighbour list by the canonical CPU rule",
                     "sample": f"{n_eval} evaluations of {len(sample)}/{len(fd)} fragments, scaled by atom count"}

    # ---- the MD loop that drives the path (host integrator, 1 GPU, real example proteins only) ----
    md_loop = None
    if world == 1 and args.workload in ("chig", "trpcage", "ww", "abd"):
        from ai2bmd_b200.fixtures import load_protein
        from ai2bmd_b200.md import BondedForceField, Langevin
        prot_pos, prot_z, recipe = load_protein(args.workload)
        ff = BondedForceField.__new__(BondedForceField)
        ff.torch, ff.recipe, ff.pm, ff.engine = torch, recipe, pm, shard.engine
        ff.pos_host = torch.empty((n_atoms, 3), dtype=torch.float32).pin_memory()
        ff.pos_dev, ff.ef_dev = shard.pos, shard.ef
        ff.ef_host = torch.empty(3 * pm.n_protein + 1, dtype=torch.float32).pin_memory()
        ff.stream = stream
        md = Langevin(prot_pos, prot_z, ff, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0)
        md.run(10)
        t0 = time.perf_counter()
        md.run(args.steps)
        dt_md = time.perf_counter() - t0
        md_loop = {"value": args.steps / dt_md, "unit": "steps/s", "temperature_K": md.temperature(),
                   "what": "Langevin (dt 1 fs, 300 K, friction 0.001/fs) with a numpy integrator on the host: protein "
                           "positions -> cap-H placement -> H2D -> engine -> device reduction -> D2H, per step"}

    # ---- non-bonded MM term (reported separately, SURVEY 8d; synthetic amber-like parameters: OpenMM is absent) ----
    nonbonded = None
    if world == 1 and args.workload in ("chig", "trpcage", "ww", "abd"):
        from ai2bmd_b200.fixtures import load_protein
        from ai2bmd_b200.nonbonded import dipeptide_atom_sets, exclusion_table, synthetic_parameters
        prot_pos, prot_z, recipe = load_protein(args.workload)
        rowptr, col = exclusion_table(len(prot_z), dipeptide_atom_sets(fd, recipe, pm))
        q, sg, ep = synthetic_parameters(prot_z, seed=0)
        shard.engine.set_nonbonded(q, sg, ep, rowptr, col)
        ppos = torch.from_numpy(np.ascontiguousarray(prot_pos, dtype=np.float32)).cuda()
        nbef = torch.zeros(3 * len(prot_z) + 1, dtype=torch.float32, device="cuda")
        for _ in range(3):
            shard.engine.nonbonded_device(ppos.data_ptr(), nbef.data_ptr(), stream.cuda_stream)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(args.steps):
            shard.engine.nonbonded_device(ppos.data_ptr(), nbef.data_ptr(), stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        n_p = len(prot_z)
        nonbonded = {"us_per_eval": a.elapsed_time(b) * 1e3 / args.steps, "pairs": int(n_p * (n_p - 1) - rowptr[-1]),
                     "what": "all-pairs LJ + Coulomb with dipeptide exclusions (vb_nonbonded), not part of `value`"}

    value = args.steps / t_dev
    edge_tc = shard.engine.get_option("edge_tc")
    line = {
        "metric": "MD steps/sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "example-PDB geometry (real for chig/trpcage/ww/abd, synthetic rotations+jitter for c4/c5), shipped checkpoint weights",
        "config": {"workload": workload_string(desc, fd),
                   "edges": n_edges if world == 1 else f"{n_edges} on rank 0 (sharded)", "n_protein": pm.n_protein,
                   "step": "one hot-path evaluation (neighbour list, ViSNet energy + analytic forces of every fragment, signed "
                           "whole-protein reduction" + (", all-reduce" if world > 1 else "") + "); the integrator update is NOT in "
                           "`value` -- `md_device` is the same step with the Langevin update on the device",
                   "parallelism": f"fragments sharded over {world} GPU(s); {shard.collective}" if world > 1 else "single GPU",
                   "l2": "flushed (256 MiB write) before every timed step" if flush is not None else "warm",
                   "timing": "CUDA events around each step on the launching stream, max over ranks",
                   "cuda_graph": True,
                   "launch_plan": "fused per-layer kernels" if shard.engine.get_option("fused") == 1 else "separate node / edge stages",
                   "edge_kernels": "tcgen05 (TMEM accumulators, TMA weight ring, 3xTF32)" if edge_tc == 3
                                   else ("fp32 SIMT" if edge_tc == 0 else f"mixed ({edge_tc})")},
        "value_l2_warm": args.steps / float(t_warm.item()),
        "wall_s_timed_region": wall,
        "e2e": e2e,
        "gpu_launches": args.steps * (shard.engine.launches_per_forward + (1 if world > 1 and shard.native else 0)),
        "launches_per_step": shard.engine.launches_per_forward + (1 if world > 1 and shard.native else 0),
        "clocks": clock_info,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "gpu_eager_baseline": gpu_eager,
        "accuracy": accuracy,
        "parity": parity,
        "comm": comm,
        "scale_c4": scale_c4,
        "md_loop": md_loop,
        "md_device": md_device,
        "caph": caph_info,
        "nonbonded": nonbonded,
        "checksum": {"E_prot_eV": float(ef[-1].item()), "F_abs_sum": float(ef[:-1].abs().sum().item())},
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
