#!/usr/bin/env python
"""Cost of the PME non-bonded term in the device-resident MD loop (Chignolin, one GPU).

* steps/s of ``DeviceLangevin.run`` with no non-bonded term, with the MM term and with the PME term on the ``chig.pdb``
  cell (25 x 27 x 23 grid) and on the ``chig-preeq-nowat.pdb`` cell (55 x 59 x 53 grid); one engine per configuration,
  the configurations alternate for several rounds, each with its own warm-up (CUDA events around each timed window);
* time per eager ``vb_pme`` call on both cells (CUDA events around 1,000 calls; host launch rate included);
* device time of every PME kernel per call, from ``torch.profiler`` (CUDA activities) over 200 calls in a phase of its
  own after the timed windows;
* the GPU's name and power limit, read in the same run.

    python tools/md_pme_cost.py [--steps 2000] [--warmup 200] [--rounds 3] [--out profiles/r04_md_pme_cost.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from md_restraint_cost import gpu_info  # noqa: E402

CELLS = {"pme_chig": (25.939, 27.327, 23.669), "pme_preeq": (55.216, 59.157, 53.428)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("md_pme_cost: no CUDA device (this measures the GPU; there is no CPU fallback)")
    from ai2bmd_b200.fixtures import WEIGHTS, load_fragments, load_protein
    from ai2bmd_b200.md import DeviceLangevin
    from ai2bmd_b200.nonbonded import PMENonBondedCalculator, dipeptide_atom_sets, exclusion_table, synthetic_parameters
    from ai2bmd_b200.weights import load_state_dict

    sd = load_state_dict(WEIGHTS)
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    n = len(prot_z)
    rowptr, col = exclusion_table(n, dipeptide_atom_sets(fd, recipe, pm))
    q, sg, ep = synthetic_parameters(prot_z, seed=1)
    q *= 0.25                                        # synthetic charges: keep the toy system gentle over many steps
    prm = (q, sg, ep, rowptr, col)
    stream = torch.cuda.current_stream()

    mds = {}
    for name in ("none", "mm", *CELLS):
        md = DeviceLangevin(sd, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0)
        if name == "mm":
            md.engine.set_nonbonded(*prm)
        elif name in CELLS:
            md.engine.set_pme(*prm, CELLS[name], PMENonBondedCalculator(None).grid(CELLS[name]))
        md._eval()
        mds[name] = md
    rates = {k: [] for k in mds}
    for _ in range(args.rounds):
        for name, md in mds.items():
            md.run(args.warmup)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            md.run(args.steps)
            b.record(stream)
            b.synchronize()
            rates[name].append(args.steps / (a.elapsed_time(b) / 1e3))
    temps = {k: md.temperature() for k, md in mds.items()}

    calls, kernels = {}, {}
    x = torch.as_tensor(prot_pos.astype(np.float32), device="cuda:0")
    ef = torch.zeros(3 * n + 1, dtype=torch.float32, device="cuda:0")
    for name in CELLS:
        eng = mds[name].engine
        for _ in range(100):
            eng.pme_device(x.data_ptr(), ef.data_ptr(), stream.cuda_stream)
        n_call = 1000
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(n_call):
            eng.pme_device(x.data_ptr(), ef.data_ptr(), stream.cuda_stream)
        b.record(stream)
        b.synchronize()
        calls[name] = a.elapsed_time(b) * 1e3 / n_call
    for name in CELLS:
        eng = mds[name].engine
        n_prof = 200
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                eng.pme_device(x.data_ptr(), ef.data_ptr(), stream.cuda_stream)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if "pme_" in ev.name and ev.device_type == torch.autograd.DeviceType.CUDA:
                key = ev.name.split("(")[0].split("<")[0].replace("void ", "").replace("vb::", "")
                per[key] = per.get(key, 0.0) + ev.device_time / n_prof
        kernels[name] = dict(sorted(per.items()))

    res = {
        "gpu": gpu_info(),
        "workload": f"Chignolin, {n} protein atoms, {len(fd)} fragments, device-resident Langevin (dt 1 fs, 300 K, "
                    f"friction 0.001/fs), one GPU; synthetic amber-like parameters (charges x 0.25)",
        "grids": {k: list(PMENonBondedCalculator(None).grid(c)) for k, c in CELLS.items()},
        "steps_per_s": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": v}
                        for k, v in rates.items()},
        "temperature_K_end": temps,
        "timing": f"{args.rounds} alternating rounds, {args.warmup} warm-up + {args.steps} timed steps per configuration "
                  f"and round, CUDA events",
        "us_per_vb_pme_call": calls,                       # eager calls: host launch rate included
        "us_per_kernel_per_call": kernels,                 # torch.profiler device times, separate phase
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
