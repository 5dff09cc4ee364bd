"""Cost of per-member control operators: the same robust-control ensemble measured twice, once with a drift spread only
(`ensemble_drifts`, shared control operators) and once with a drive-amplitude spread (`ensemble_hamiltonians` with
H_e = H0 + (1 + eps_e) sum_k u_k H_k, eps_e ~ U(-0.1, 0.1): every member has its own operators).

  * Schroedinger: the cfg5 shape of bench.py (n = 32, 500 slices, K = 2, S = 64) with M2 and M4, device-resident
    evaluations (`time_resident`, L2 flushed before each) -> member-evaluations/s.
  * Lindblad: bench.py's `lindblad_n8_D2_N5`, host-facing `cost_and_grad` -> member-evaluations/s.

Also reports the device bytes of the per-member operators (G and, for the product-free M4, Cs).  Prints one JSON document
(and writes it to --out) with the card's name and power limit.

    python tools/bench_ensemble_member_ops.py --out profiles/r06_bench_ensemble_member_ops.json
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_lindblad_ensemble import card, timed  # noqa: E402


def _amplitudes(E, seed):
    return 1.0 + np.random.default_rng(seed).uniform(-0.1, 0.1, E)


def schroedinger(order, sizes, iters, warmup, seed):
    import qoc_b200.standard as std
    from bench import make_problem
    from qoc_b200.core.plan import SchroedingerPlan
    from qoc_b200.models import MagnusPolicy
    from tests.problems import numpy_hamiltonian
    p = make_problem("cfg5_n32_500_S64_E128_M2")          # the cfg5 shape; the members are built here
    p.order = order
    pol = {2: MagnusPolicy.M2, 4: MagnusPolicy.M4}[order]
    NP, KR = 32, p.K * (2 if p.complex_controls else 1)
    extra = KR * (KR - 1) // 2 if order == 4 else 0               # Cs of the product-free M4
    rows = []
    for E in sizes:
        z = np.diag(np.linspace(-1, 1, p.n)).astype(np.complex128) * np.abs(p.h0).max()
        drifts = np.stack([p.h0 + d * z for d in np.random.default_rng(12345).normal(0, 0.1, E)])
        members = [numpy_hamiltonian(p.h0, a * p.drives, p.complex_controls) for a in _amplitudes(E, seed + E)]
        row = {"E": E, "member_operator_bytes": E * (KR + extra) * 2 * NP * NP * 8}
        for label, kw in (("drift_spread", dict(ensemble_drifts=drifts)), ("amplitude_spread", dict(ensemble_hamiltonians=members))):
            plan = SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                                    control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol, **kw)
            plan.upload(p.controls)
            total_ms, _ = plan.time_resident(with_grad=True, warmup=warmup, iters=iters, flush_l2=True)
            row[label] = {"ms_per_eval": total_ms / iters, "member_evals_per_s": E * iters / (total_ms * 1e-3),
                          "launches": plan.launch_count(), "iters": iters}
            plan.close()
        row["amplitude_over_drift"] = row["amplitude_spread"]["member_evals_per_s"] / row["drift_spread"]["member_evals_per_s"]
        print(json.dumps({"workload": "cfg5_n32_500_S64_M%d" % order, **row}), flush=True)
        rows.append(row)
    return {"workload": "cfg5_n32_500_S64_M%d" % order, "hilbert_dim": p.n, "slices": p.N - 1, "states": p.S,
            "real_channels": KR, "rows": rows}


def lindblad(name, sizes, min_seconds, seed):
    import qoc_b200.standard as std
    from bench import lindblad_problem
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    q = lindblad_problem(name)
    u, n = q["controls"], q["n"]
    ham = numpy_hamiltonian(q["h0"], q["drive"], True)
    det = np.diag(np.linspace(-0.5, 0.5, n)).astype(np.complex128)
    rows = []
    for E in sizes:
        drifts = np.array([q["h0"] + d * det for d in np.random.default_rng(seed + E).uniform(-0.05, 0.05, E)])
        members = [numpy_hamiltonian(q["h0"], a * q["drive"], True) for a in _amplitudes(E, seed + E)]
        row = {"E": E, "member_operator_bytes": E * 2 * n * n * 16}
        for label, kw in (("drift_spread", dict(ensemble_drifts=drifts)), ("amplitude_spread", dict(ensemble_hamiltonians=members))):
            plan = LindbladPlan(q["rho0"], [std.TargetDensityInfidelity(q["targ"])], q["T"], q["N"], hamiltonian=ham,
                                lindblad_data=lambda t: (q["gam"], q["lops"]), control_eval_count=q["M"], control_count=1,
                                complex_controls=True, **kw)
            sec, reps = timed(lambda: plan.cost_and_grad(u), min_seconds, 3)
            row[label] = {"ms_per_eval": sec * 1e3, "member_evals_per_s": E / sec, "reps": reps,
                          "accepted_steps_per_member": plan.stats()["accepted"] / E}
            plan.close()
        row["amplitude_over_drift"] = row["amplitude_spread"]["member_evals_per_s"] / row["drift_spread"]["member_evals_per_s"]
        print(json.dumps({"workload": name, **row}), flush=True)
        rows.append(row)
    return {"workload": name, "hilbert_dim": n, "densities": q["D"], "intervals": q["N"] - 1, "rows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", default="16,148,1024")
    ap.add_argument("--lindblad-sizes", default="16,148,592")
    ap.add_argument("--orders", default="2,4")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--min-seconds", type=float, default=1.5)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_ensemble_member_ops.py needs a CUDA device (no CPU path)")
    sizes = [int(s) for s in args.sizes.split(",")]
    lsizes = [int(s) for s in args.lindblad_sizes.split(",")]
    results = [schroedinger(int(o), sizes, args.iters, args.warmup, args.seed) for o in args.orders.split(",")]
    results.append(lindblad("lindblad_n8_D2_N5", lsizes, args.min_seconds, args.seed))
    doc = {"card": card(), "results": results}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
