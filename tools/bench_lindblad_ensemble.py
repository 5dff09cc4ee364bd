"""Throughput of Lindblad ensembles: evaluations/s and member-evaluations/s of `LindbladPlan.cost_and_grad` on the bench
Lindblad problems (`bench.lindblad_problem`) with seeded detuning and decay-rate spreads, for E members in one plan (one CTA
each) and, for E <= 16, for E sequential one-member plans in the same process.  Sampled members are checked bit for bit
against one-member plans.  Prints one JSON document (and writes it to --out) with the card's name and power limit.

    python tools/bench_lindblad_ensemble.py --out profiles/r05_bench_lindblad_ensemble.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["nvidia_smi"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        out["nvidia_smi"] = None
    return out


def members(q, E, seed):
    """seeded spreads: detuning delta_e sigma_z / 2-like diagonal shift of the drift, rates gamma * U(0.5, 1.5)."""
    rng = np.random.default_rng(seed)
    n = q["n"]
    det = np.diag(np.linspace(-0.5, 0.5, n)).astype(np.complex128)
    drifts = np.array([q["h0"] + rng.uniform(-0.05, 0.05) * det for _ in range(E)])
    rates = np.array([q["gam"] * rng.uniform(0.5, 1.5, q["gam"].shape[0]) for _ in range(E)])
    return drifts, rates


def make_plan(q, drift=None, rate=None, drifts=None, rates=None):
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan, extract_hamiltonian_structure
    from tests.problems import numpy_hamiltonian
    ham = numpy_hamiltonian(q["h0"], q["drive"], True)
    h0, a_ops = extract_hamiltonian_structure(ham, 1, True, q["T"])
    gam = q["gam"] if rate is None else rate
    return LindbladPlan(q["rho0"], [std.TargetDensityInfidelity(q["targ"])], q["T"], q["N"], hamiltonian=ham,
                        lindblad_data=lambda t: (gam, q["lops"]), control_eval_count=q["M"], control_count=1,
                        complex_controls=True, structure=(h0 if drift is None else drift, a_ops),
                        ensemble_drifts=drifts, ensemble_rates=rates)


def timed(fn, min_seconds, min_reps):
    import torch
    fn()
    torch.cuda.synchronize()
    reps, t0 = 0, time.perf_counter()
    while reps < min_reps or time.perf_counter() - t0 < min_seconds:
        fn()
        reps += 1
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps, reps


def run(name, sizes, min_seconds, samples, seed):
    from bench import lindblad_problem
    q = lindblad_problem(name)
    u = q["controls"]
    rows = []
    for E in sizes:
        drifts, rates = members(q, E, seed + E)
        plan = make_plan(q) if E == 1 else make_plan(q, drifts=drifts, rates=rates)
        sec, reps = timed(lambda: plan.cost_and_grad(u), min_seconds, 3)
        row = {"E": E, "ms_per_eval": sec * 1e3, "evals_per_s": 1.0 / sec, "member_evals_per_s": E / sec, "reps": reps,
               "accepted_steps_per_member": plan.stats()["accepted"] / E}
        if E > 1:
            costs, grads, stats = plan.member_results()
            pick = sorted(set(np.random.default_rng(seed).choice(E, min(samples, E), replace=False).tolist()))
            ok = True
            for e in pick:
                one = make_plan(q, drift=drifts[e], rate=rates[e])
                c1, g1, _ = one.cost_and_grad(u)
                ok = ok and c1 == costs[e] and np.array_equal(g1, grads[e]) and one.stats() == stats[e]
                one.close()
            row["bit_identical_members"] = {"checked": pick, "identical": bool(ok)}
        if 1 < E <= 16:
            singles = [make_plan(q, drift=drifts[e], rate=rates[e]) for e in range(E)]
            sec_s, reps_s = timed(lambda: [s.cost_and_grad(u) for s in singles], min_seconds, 2)
            row["sequential_single_plans"] = {"ms_per_E_evals": sec_s * 1e3, "member_evals_per_s": E / sec_s,
                                              "reps": reps_s}
            for s in singles:
                s.close()
        plan.close()
        rows.append(row)
        print(json.dumps({"workload": name, **row}), flush=True)
    base = rows[0]["member_evals_per_s"] if rows and rows[0]["E"] == 1 else None
    for r in rows:
        if base:
            r["scaling_vs_E1"] = r["member_evals_per_s"] / base
    return {"workload": name, "hilbert_dim": q["n"], "densities": q["D"], "intervals": q["N"] - 1, "rows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", default="1,16,148,592,1184")
    ap.add_argument("--workloads", default="cfg2_lindblad_n2,lindblad_n8_D2_N5")
    ap.add_argument("--min-seconds", type=float, default=1.5)
    ap.add_argument("--samples", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_lindblad_ensemble.py needs a CUDA device (no CPU path)")
    sizes = [int(s) for s in args.sizes.split(",")]
    doc = {"card": card(), "sizes": sizes, "min_seconds": args.min_seconds,
           "results": [run(w, sizes, args.min_seconds, args.samples, args.seed) for w in args.workloads.split(",")]}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
