"""Throughput of Lindblad control batches (multi-start GRAPE): `LindbladPlan(control_batch=B).cost_and_grad` on the bench
Lindblad problems (`bench.lindblad_problem`) with B seeded starts, each the workload's controls with a +-10 % per-entry
perturbation.  Per B: ms per batched call, start-evaluations/s, the ratio to B sequential one-member evaluations in the same
process, accepted Runge-Kutta steps per start (min / median / max), and sampled starts checked bit for bit against
one-member plans.  Prints one JSON document (and writes it to --out) with the card's name and power limit.

The sequential reference times one-member evaluations of every start for B <= 16 and of 16 sampled starts above that; its
time for B starts is then B times the sampled mean (the starts' step counts differ, so this is an estimate for B > 16).

    python tools/bench_lindblad_control_batch.py --out profiles/r09_bench_lindblad_control_batch.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.bench_lindblad_ensemble import card, timed  # noqa: E402


def starts(q, B, seed):
    rng = np.random.default_rng(seed)
    u = q["controls"]
    pert = rng.uniform(-0.1, 0.1, (B,) + u.shape) + 1j * rng.uniform(-0.1, 0.1, (B,) + u.shape)
    return u[None] * (1.0 + pert)


def make_plan(q, B=None):
    import qoc_b200.standard as std
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    return LindbladPlan(q["rho0"], [std.TargetDensityInfidelity(q["targ"])], q["T"], q["N"],
                        hamiltonian=numpy_hamiltonian(q["h0"], q["drive"], True),
                        lindblad_data=lambda t: (q["gam"], q["lops"]), control_eval_count=q["M"], control_count=1,
                        complex_controls=True, control_batch=B)


def run(name, sizes, min_seconds, samples, seed):
    from bench import lindblad_problem
    q = lindblad_problem(name)
    one = make_plan(q)
    rows = []
    for B in sizes:
        U = starts(q, B, seed + B)
        plan = make_plan(q, B)
        sec, reps = timed(lambda: plan.cost_and_grad(U), min_seconds, 3)
        errs, grads, finals = plan.cost_and_grad(U)
        costs, mgrads, stats = plan.member_results()
        acc = np.array([s["accepted"] for s in stats])
        pick = sorted(set(np.random.default_rng(seed).choice(B, min(samples, B), replace=False).tolist()))
        ok = True
        for b in pick:
            e1, g1, f1 = one.cost_and_grad(U[b])
            ok = ok and e1 == errs[b] and np.array_equal(g1, grads[b]) and np.array_equal(f1, finals[b])
            ok = ok and one.stats() == stats[b]
        seq = list(range(B)) if B <= 16 else sorted(np.random.default_rng(seed + 1).choice(B, 16, replace=False).tolist())
        one.cost_and_grad(U[seq[0]])
        import torch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in seq:
            one.cost_and_grad(U[b])
        torch.cuda.synchronize()
        seq_ms = (time.perf_counter() - t0) / len(seq) * 1e3
        row = {"B": B, "ms_per_batch_call": sec * 1e3, "start_evals_per_s": B / sec, "reps": reps,
               "sequential_one_member_ms_per_start": seq_ms, "sequential_starts_timed": len(seq),
               "speedup_vs_sequential": B * seq_ms / (sec * 1e3),
               "accepted_steps_per_start": {"min": int(acc.min()), "median": float(np.median(acc)), "max": int(acc.max())},
               "bit_identical_starts": {"checked": pick, "identical": bool(ok)}}
        plan.close()
        rows.append(row)
        print(json.dumps({"workload": name, **row}), flush=True)
    one.close()
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
        raise RuntimeError("tools/bench_lindblad_control_batch.py needs a CUDA device (no CPU path)")
    sizes = [int(s) for s in args.sizes.split(",")]
    doc = {"card": card(), "sizes": sizes, "min_seconds": args.min_seconds,
           "perturbation": "controls * (1 + U(-0.1, 0.1) + i U(-0.1, 0.1)) per entry, seeded per B",
           "results": [run(w, sizes, args.min_seconds, args.samples, args.seed) for w in args.workloads.split(",")]}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
