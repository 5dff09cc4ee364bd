"""Cost of per-member initial states and cost targets: the same robust-control ensemble (a drift spread) measured with shared
initial states and targets and with every member's own (`ensemble_initial_states` / `ensemble_initial_densities` and
`ensemble_costs`, Haar-random per member).

  * Schroedinger: the cfg5 shape of bench.py (n = 32, 500 slices, K = 2, S = 64, M2), device-resident evaluations
    (`time_resident`, L2 flushed before each) -> member-evaluations/s.  Two cost sets: the cfg5 target only, and the target
    plus ForbidStates with F = 6 forbidden states per state evaluated at every step (per-member vectors of E * S * 7 * 2 * 32
    doubles: about 235 MB at E = 1024, beyond the 126 MB L2).
  * Lindblad: bench.py's `lindblad_n8_D2_N5` and `cfg2_lindblad_n2`, host-facing `cost_and_grad` -> member-evaluations/s,
    with a third arm that forces identical data through the member path: distinct densities change the adaptive step
    counts, so only that arm isolates the cost of the path itself.

Prints one JSON document (and writes it to --out) with the card's name and power limit.

    python tools/bench_ensemble_member_targets.py --out profiles/r10_bench_ensemble_member_targets.json
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_lindblad_ensemble import card, timed  # noqa: E402


def _kets(rng, count, n):
    v = rng.standard_normal((count, n)) + 1j * rng.standard_normal((count, n))
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _dens(rng, count, n):
    v = _kets(rng, count, n)
    return np.einsum("di,dj->dij", v, v.conj())


def schroedinger(sizes, iters, warmup, seed, F):
    import qoc_b200.standard as std
    from bench import make_problem
    from qoc_b200.core.plan import SchroedingerPlan
    from qoc_b200.models import MagnusPolicy
    p = make_problem("cfg5_n32_500_S64_E128_M2")          # the cfg5 shape; the members are built here
    n, S, NP = p.n, p.S, 32

    def costs(targ, forb):
        out = [std.TargetStateInfidelity(targ)]
        if F:
            out.append(std.ForbidStates(forb, p.N, cost_multiplier=0.5))
        return out
    rows = []
    for E in sizes:
        rng = np.random.default_rng(seed + E)
        z = np.diag(np.linspace(-1, 1, n)).astype(np.complex128) * np.abs(p.h0).max()
        drifts = np.stack([p.h0 + d * z for d in rng.normal(0, 0.1, E)])
        psi0 = _kets(rng, E * S, n).reshape(E, S, n, 1)
        targ = _kets(rng, E * S, n).reshape(E, S, n, 1)
        forb = _kets(rng, E * S * F, n).reshape(E, S, F, n, 1) if F else [None] * E
        nominal_forb = forb[0] if F else None
        row = {"E": E, "member_vector_bytes": E * S * (1 + F) * 2 * NP * 8 + E * S * 2 * NP * 8}
        arms = (("shared", dict()),
                ("per_member", dict(ensemble_initial_states=psi0, ensemble_costs=[costs(targ[e], forb[e]) for e in range(E)])))
        for label, kw in arms:
            plan = SchroedingerPlan(p.hamiltonian_numpy(), psi0[0], costs(targ[0], nominal_forb), p.T, p.N,
                                    control_eval_count=p.M, control_count=p.K, complex_controls=p.complex_controls,
                                    magnus_policy=MagnusPolicy.M2, ensemble_drifts=drifts, **kw)
            plan.upload(p.controls)
            total_ms, _ = plan.time_resident(with_grad=True, warmup=warmup, iters=iters, flush_l2=True)
            row[label] = {"ms_per_eval": total_ms / iters, "member_evals_per_s": E * iters / (total_ms * 1e-3),
                          "launches": plan.launch_count(), "iters": iters}
            plan.close()
        row["per_member_over_shared"] = row["per_member"]["member_evals_per_s"] / row["shared"]["member_evals_per_s"]
        # the extra vector traffic per cost step: (per-member - shared) time over the cost steps of one evaluation
        cost_steps = (p.N - 1) if F else 1
        row["extra_us_per_cost_step"] = (row["per_member"]["ms_per_eval"] - row["shared"]["ms_per_eval"]) * 1e3 / cost_steps
        name = "cfg5_n32_500_S64_M2" + ("_forbid%d" % F if F else "")
        print(json.dumps({"workload": name, **row}), flush=True)
        rows.append(row)
    return {"workload": "cfg5_n32_500_S64_M2" + ("_forbid%d" % F if F else ""), "hilbert_dim": n, "slices": p.N - 1,
            "states": S, "forbidden_per_state": F, "rows": rows}


def lindblad(name, sizes, min_seconds, seed):
    import qoc_b200.standard as std
    from bench import lindblad_problem
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    q = lindblad_problem(name)
    u, n, D = q["controls"], q["n"], q["D"]
    ham = numpy_hamiltonian(q["h0"], q["drive"], True)
    det = np.diag(np.linspace(-0.5, 0.5, n)).astype(np.complex128)
    rows = []
    for E in sizes:
        rng = np.random.default_rng(seed + E)
        drifts = np.array([q["h0"] + d * det for d in rng.uniform(-0.05, 0.05, E)])
        rho0 = np.array([_dens(rng, D, n) for _ in range(E)])
        targ = np.array([_dens(rng, D, n) for _ in range(E)])
        row = {"E": E}
        arms = (("shared", dict()),
                ("identical_per_member", dict(ensemble_initial_densities=np.array([rho0[0]] * E),
                                              ensemble_costs=[[std.TargetDensityInfidelity(targ[0])]] * E)),
                ("per_member", dict(ensemble_initial_densities=rho0,
                                    ensemble_costs=[[std.TargetDensityInfidelity(t)] for t in targ])))
        for label, kw in arms:
            plan = LindbladPlan(rho0[0], [std.TargetDensityInfidelity(targ[0])], q["T"], q["N"], hamiltonian=ham,
                                lindblad_data=lambda t: (q["gam"], q["lops"]), control_eval_count=q["M"], control_count=1,
                                complex_controls=True, ensemble_drifts=drifts, **kw)
            sec, reps = timed(lambda: plan.cost_and_grad(u), min_seconds, 3)
            accepted = [s_["accepted"] for s_ in plan.member_results()[2]]
            row[label] = {"ms_per_eval": sec * 1e3, "member_evals_per_s": E / sec, "reps": reps,
                          "accepted_steps_per_member": float(np.mean(accepted)), "max_accepted_steps": int(max(accepted))}
            plan.close()
        # identical data through the member path isolates the path's own cost; distinct data also changes the adaptive step
        # counts (one CTA per member: the slowest member sets the time)
        row["identical_over_shared"] = row["identical_per_member"]["member_evals_per_s"] / row["shared"]["member_evals_per_s"]
        row["per_member_over_shared"] = row["per_member"]["member_evals_per_s"] / row["shared"]["member_evals_per_s"]
        print(json.dumps({"workload": name, **row}), flush=True)
        rows.append(row)
    return {"workload": name, "hilbert_dim": n, "densities": D, "intervals": q["N"] - 1, "rows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--sizes", default="16,148,1024")
    ap.add_argument("--lindblad-sizes", default="16,148,592")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--min-seconds", type=float, default=1.5)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_ensemble_member_targets.py needs a CUDA device (no CPU path)")
    sizes = [int(s) for s in args.sizes.split(",")]
    lsizes = [int(s) for s in args.lindblad_sizes.split(",")]
    results = [schroedinger(sizes, args.iters, args.warmup, args.seed, F) for F in (0, 6)]
    results += [lindblad(name, lsizes, args.min_seconds, args.seed) for name in ("lindblad_n8_D2_N5", "cfg2_lindblad_n2")]
    doc = {"card": card(), "results": results}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
