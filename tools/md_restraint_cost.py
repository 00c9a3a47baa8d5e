#!/usr/bin/env python
"""Cost of the Hookean restraint term in the device-resident MD loop (Chignolin, one GPU).

* steps/s of ``DeviceLangevin.run`` with no restraints, with the 175 position restraints of a pre-equilibration stage
  and with those plus the 78 hydrogen-bond springs of ``--constraints``; the three configurations alternate, each
  with its own warm-up, for several rounds (CUDA events around each timed window);
* time per eager ``vb_restraints`` call (175 + 78 restraints, events around 2,000 calls; host launch rate included);
* wall time of the reference's default protocol on the device: ``pre_equilibrate(md, 2000)`` (five restrained stages)
  and then 1,000 production steps with the hydrogen-bond springs, next to 11,000 unrestrained steps;
* the GPU's name and power limit, read in the same run.

    python tools/md_restraint_cost.py [--steps 2000] [--warmup 200] [--rounds 3] [--preeq-steps 2000] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        line = ""
    return dict(zip(q.split(","), [s.strip() for s in line.split(",")])) if line else {"name": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preeq-steps", type=int, default=2000)
    ap.add_argument("--prod-steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("md_restraint_cost: no CUDA device (this measures the GPU; there is no CPU fallback)")
    from ai2bmd_b200 import restraints as R
    from ai2bmd_b200.fixtures import WEIGHTS, load_capped_protein, load_fragments, load_protein
    from ai2bmd_b200.md import DeviceLangevin
    from ai2bmd_b200.weights import load_state_dict

    sd = load_state_dict(WEIGHTS)
    fd, pm = load_fragments("chig")
    prot_pos, prot_z, recipe = load_protein("chig")
    prot = load_capped_protein("chig")
    hb = R.hydrogen_bond_restraints(prot.names, prot.positions)
    stream = torch.cuda.current_stream()

    def make():
        return DeviceLangevin(sd, fd, pm, recipe, prot_pos, prot_z, dt_fs=1.0, temperature_K=300.0, friction_per_fs=0.001, seed=0)

    md = make()
    configs = {
        "none": lambda x: None,
        "position": lambda x: R.position_restraints(x, 10.0),
        "position+hbond": lambda x: R.position_restraints(x, 10.0) + hb,
    }
    rates = {k: [] for k in configs}
    for _ in range(args.rounds):
        for name, mk in configs.items():
            md.set_restraints(mk(md.state()[0]))
            md.run(args.warmup)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            md.run(args.steps)
            b.record(stream)
            b.synchronize()
            rates[name].append(args.steps / (a.elapsed_time(b) / 1e3))
    md.set_restraints(None)

    # one launch of the term alone
    eng = md.engine
    (R.position_restraints(prot_pos, 10.0) + hb).install(eng)
    x = torch.as_tensor(prot_pos + 0.05, device="cuda:0")
    ef = torch.zeros(3 * len(prot_pos) + 1, dtype=torch.float32, device="cuda:0")
    for _ in range(100):
        eng.restraints_device(x.data_ptr(), ef.data_ptr(), stream.cuda_stream)
    n_launch = 2000
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(n_launch):
        eng.restraints_device(x.data_ptr(), ef.data_ptr(), stream.cuda_stream)
    b.record(stream)
    b.synchronize()
    us_launch = a.elapsed_time(b) * 1e3 / n_launch
    eng.clear_restraints()
    del md

    # the reference's default protocol: 5 x preeq-steps restrained, then prod-steps with the hydrogen-bond springs
    total = 5 * args.preeq_steps + args.prod_steps
    walls = {}
    for name in ("plain", "protocol"):
        m = make()
        m.run(10)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if name == "plain":
            m.run(total)
        else:
            R.pre_equilibrate(m, args.preeq_steps)
            m.set_restraints(hb)
            m.run(args.prod_steps)
        _, _, step, _ = m.state()                 # synchronises
        walls[name] = {"seconds": time.perf_counter() - t0, "steps": step - 10, "temperature_K": m.temperature()}
        del m

    res = {
        "gpu": gpu_info(),
        "workload": f"Chignolin, {len(prot_pos)} protein atoms, {len(fd)} fragments, device-resident Langevin (dt 1 fs, 300 K, "
                    f"friction 0.001/fs), one GPU",
        "restraints": {"position": len(prot_pos), "hbond": hb.n_pair},
        "steps_per_s": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": v}
                        for k, v in rates.items()},
        "timing": f"{args.rounds} alternating rounds, {args.warmup} warm-up + {args.steps} timed steps per configuration "
                  f"and round, CUDA events",
        "us_per_restraint_launch": us_launch,             # eager calls: host launch rate included
        "protocol_wall_s": walls,
        "protocol": f"pre_equilibrate({args.preeq_steps}) (k = 10, 5, 1, 0.5, 0.1 kcal/mol/A^2) + {args.prod_steps} steps "
                    f"with hydrogen-bond springs, vs {total} unrestrained steps; host clock around work ending in a sync",
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
