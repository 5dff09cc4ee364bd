"""Throughput of control batches (multi-start GRAPE): B control sets of one problem evaluated per call
(`SchroedingerPlan(control_batch=B)`) against the same B starts evaluated one after another on a one-member plan.

  * workloads: cfg1 (n = 2, 10 slices, M2, complex controls) at B = 1, 16, 148, 1024; n = 16 x 500 slices M4 (K = 4, S = 4)
    at B = 1, 16, 148; n = 64 x 2000 slices M4 (bench.py's default workload) at B = 1, 2, 4;
  * each: device-resident cost_and_grad (`time_resident`, L2 flushed before each evaluation) -> start-evaluations/s of
    the batch, and of a one-member plan (B sequential plans run B times its time per start);
  * batch results are checked against the one-member plan on every start before timing (max relative deviation reported).

Prints one JSON line per row and one JSON document (also written to --out) with the card's name and power limit.

    python tools/bench_control_batch.py --out profiles/r07_bench_control_batch.json
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_lindblad_ensemble import card  # noqa: E402

WORKLOADS = [
    # name, (n, slices, K, S, order, complex_controls), batch sizes
    ("cfg1_n2_10_M2", (2, 10, 1, 1, 2, True), (1, 16, 148, 1024)),
    ("n16_500_M4", (16, 500, 4, 4, 4, False), (1, 16, 148)),
    ("n64_2000_M4", (64, 2000, 4, 4, 4, False), (1, 2, 4)),
]


def _controls(p, B, seed):
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((B, p.M, p.K)) * 0.5
    if p.complex_controls:
        u = (u + 1j * rng.standard_normal((B, p.M, p.K)) * 0.5) / np.sqrt(2)
    return u


def _rate(plan, controls, starts, iters, warmup):
    plan.upload(controls)
    total_ms, _ = plan.time_resident(with_grad=True, warmup=warmup, iters=iters, flush_l2=True)
    return {"ms_per_eval": total_ms / iters, "start_evals_per_s": starts * iters / (total_ms * 1e-3),
            "launches": plan.launch_count(), "iters": iters}


def run(name, shape, sizes, iters, warmup, seed):
    import qoc_b200.standard as std
    from qoc_b200.core.plan import SchroedingerPlan
    from qoc_b200.models import MagnusPolicy
    from tests.problems import Problem
    n, slices, K, S, order, cc = shape
    p = Problem(n, slices, K, S, order, complex_controls=cc, seed=0)
    pol = {2: MagnusPolicy.M2, 4: MagnusPolicy.M4}[order]

    def plan(**kw):
        return SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                                control_count=K, complex_controls=cc, magnus_policy=pol, **kw)
    one = plan()
    u = _controls(p, max(sizes), seed)
    single = _rate(one, u[0], 1, iters, warmup)
    print(json.dumps({"workload": name, "one_member_plan": single}), flush=True)
    rows = []
    for B in sizes:
        batch = plan(control_batch=B)
        errs, grads, finals = batch.cost_and_grad(u[:B])
        dev = 0.0
        for b in range(B):
            e1, g1, f1 = one.cost_and_grad(u[b])
            dev = max(dev, abs(errs[b] - e1) / abs(e1), np.linalg.norm(grads[b] - g1) / np.linalg.norm(g1),
                      np.linalg.norm(finals[b] - f1) / np.linalg.norm(f1))
        row = {"B": B, "batch": _rate(batch, u[:B], B, iters, warmup), "max_rel_dev_vs_one_member": dev}
        row["speedup_vs_sequential"] = row["batch"]["start_evals_per_s"] / single["start_evals_per_s"]
        batch.close()
        print(json.dumps({"workload": name, **row}), flush=True)
        rows.append(row)
    one.close()
    return {"workload": name, "hilbert_dim": n, "slices": slices, "real_channels": K * (2 if cc else 1), "states": S,
            "magnus_order": order, "one_member_plan": single, "rows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--workloads", default=",".join(w[0] for w in WORKLOADS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("tools/bench_control_batch.py needs a CUDA device (no CPU path)")
    wanted = args.workloads.split(",")
    results = [run(name, shape, sizes, args.iters, args.warmup, args.seed) for name, shape, sizes in WORKLOADS
               if name in wanted]
    doc = {"card": card(), "results": results}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
