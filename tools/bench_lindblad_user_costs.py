"""Cost of user-defined costs on the Lindblad path.

For the `cfg2_lindblad_n2` and `lindblad_n8_D2_N5` problems of bench.py, times cost+gradient evaluations with
  builtin: TargetDensityInfidelity (final step) and ForbidDensities (every cost step) as device cost terms, and
  user:    the same two costs written as plain NumPy `Cost` subclasses (tests/test_gpu_lindblad_user_costs.py), which the
           plan evaluates on the host: forward pass with tape, central-difference cotangents of the densities (8 cost calls per
           complex density entry and cost step), reverse pass seeded with them,
alternately in one process (every evaluation returns its results to the host), and checks user against builtin (cost within
1e-12 relative, gradient within 1e-8).  For `user` it also splits one evaluation into device forward (with the D2H of the
densities), host cost and finite differences, and device backward.

    python tools/bench_lindblad_user_costs.py [--rounds 5] [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def split_evaluation(plan, controls):
    """seconds of (device forward, host costs + differences, device backward) of one user-cost evaluation, phase by phase as
    LindbladPlan.cost_and_grad runs them."""
    from qoc_b200 import _lib
    from qoc_b200.core.plan import explicit_control_grad
    x = plan._real_channels(controls)
    out, g = np.zeros(1), np.zeros((plan.M, plan.KR))
    fd = np.empty((plan.D, plan.n, plan.n), dtype=np.complex128)
    t0 = time.perf_counter()
    plan._evaluate(lambda h: plan.lib.qocb_lindblad_forward(h, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)))
    dens = plan._user_densities(fd)
    t1 = time.perf_counter()
    plan._user_value(controls, dens)
    seeds = plan._user_seeds(controls, dens)
    explicit_control_grad(lambda u: plan._user_value(u, dens), controls)
    t2 = time.perf_counter()
    plan._check(plan.lib.qocb_lindblad_backward(plan.handle, _lib.ptr(seeds), _lib.ptr(g)))
    t3 = time.perf_counter()
    return t1 - t0, t2 - t1, t3 - t2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("this benchmark needs a CUDA device")
    import qoc_b200.standard as std
    from bench import lindblad_problem
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    from tests.test_gpu_lindblad_user_costs import TwinForbid, TwinTarget
    from tools.bench_lindblad_timedep import card
    name, power = card()
    result = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": power, "rounds": args.rounds,
              "steps_per_round": args.steps, "workloads": {}}
    for wl in ("cfg2_lindblad_n2", "lindblad_n8_D2_N5"):
        q = lindblad_problem(wl)
        forb = q["rho0"][:, None]                             # forbid each initial density
        costs = {"builtin": [std.TargetDensityInfidelity(q["targ"]), std.ForbidDensities(forb, q["N"], cost_multiplier=0.5)],
                 "user": [TwinTarget(q["targ"]), TwinForbid(forb, q["N"], 1, 0.5)]}
        plans, rows, res = {}, {}, {}
        for key, cs in costs.items():
            plans[key] = LindbladPlan(q["rho0"], cs, q["T"], q["N"], hamiltonian=numpy_hamiltonian(q["h0"], q["drive"], True),
                                      lindblad_data=lambda t: (q["gam"], q["lops"]), control_eval_count=q["M"], control_count=1,
                                      complex_controls=True)
            for _ in range(3):
                res[key] = plans[key].cost_and_grad(q["controls"])
            rows[key] = {"user_costs": len(plans[key].user_costs), "sec": []}
        D, n, N = q["D"], q["n"], q["N"]
        rows["user"]["cost_calls_per_eval"] = sum(len(c) * (3 + 8 * D * n * n) for c in plans["user"]._user_at.values())
        for _ in range(args.rounds):                          # alternate the two variants
            for key in ("builtin", "user"):
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    plans[key].cost_and_grad(q["controls"])
                rows[key]["sec"].append((time.perf_counter() - t0) / args.steps)
        split = np.array([split_evaluation(plans["user"], q["controls"]) for _ in range(args.steps)])
        rows["user"]["split_ms_median"] = {k: float(np.median(split[:, i]) * 1e3)
                                           for i, k in enumerate(("device_forward", "host_costs_and_differences",
                                                                  "device_backward"))}
        for key in ("builtin", "user"):
            sec = np.array(rows[key].pop("sec"))
            rows[key]["evals_per_sec_median"] = float(1.0 / np.median(sec))
            rows[key]["evals_per_sec_rounds"] = [float(x) for x in 1.0 / sec]
            plans[key].close()
        (e_b, g_b, f_b), (e_u, g_u, f_u) = res["builtin"], res["user"]
        rows["parity"] = {"cost_rel": abs(e_u - e_b) / abs(e_b),
                          "grad_rel": float(np.linalg.norm(g_u - g_b) / np.linalg.norm(g_b)),
                          "final_densities_identical": bool(np.array_equal(f_u, f_b))}
        assert rows["parity"]["cost_rel"] <= 1e-12 and rows["parity"]["grad_rel"] <= 1e-8, rows["parity"]
        rows["problem"] = {"n": n, "D": D, "N": N}
        result["workloads"][wl] = rows
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
