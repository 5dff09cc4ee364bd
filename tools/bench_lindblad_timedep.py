"""Cost of time dependence on the Lindblad path.

For the `cfg2_lindblad_n2` and `lindblad_n8_D2_N5` problems of bench.py, times cost+gradient evaluations of
  TI: the problem as bench.py runs it (time-independent H = H0 + u a + conj(u) a^dag, constant dissipator), and
  TD: the same problem with a rotating-frame drive H(u, t) = H0 + u e^{i w t} a + conj(u e^{i w t}) a^dag and a decay
      rate modulated in time, so that the kernels evaluate piecewise Chebyshev series at every Runge-Kutta stage,
alternately in one process (device-synchronised: every evaluation returns its results to the host), and checks both
against the frozen-grid torch oracle.  The two variants take different step sequences, so besides evaluations/s it
reports the time per right-hand-side evaluation (7 per attempt in the forward pass, 14 per accepted step in the reverse
pass); the difference of those is the measured cost of the series evaluation per stage.

    python tools/bench_lindblad_timedep.py [--rounds 5] [--steps 40] [--out FILE]
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
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as exc:                                  # the name still comes from torch below
        return None, "unknown ({})".format(exc)


def variants(q, w=0.9):
    import torch
    from tests.problems import numpy_hamiltonian
    h0, a = q["h0"], q["drive"][0]
    ad = a.conj().T
    gam, lops = q["gam"], q["lops"]

    def h_td(u, t):
        ph = np.exp(1j * w * t)
        return h0 + u[0] * ph * a + np.conjugate(u[0] * ph) * ad

    def ld_td(t):
        return gam * (1.0 + 0.5 * np.sin(0.7 * t)), lops

    def oh_td(u, t):
        t = float(t)
        ph = complex(np.cos(w * t), np.sin(w * t))
        return torch.as_tensor(h0) + u[0] * ph * torch.as_tensor(a) + torch.conj(u[0] * ph) * torch.as_tensor(ad)

    def old_td(t):
        g, o = ld_td(float(t))
        return torch.as_tensor(g), torch.as_tensor(o)
    from oracle import qoc_oracle as orc
    return {"TI": (numpy_hamiltonian(h0, q["drive"], True), lambda t: (gam, lops),
                   orc.make_hamiltonian(h0, q["drive"], True), orc.make_lindblad_data(gam, lops)),
            "TD": (h_td, ld_td, oh_td, old_td)}


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("this benchmark needs a CUDA device")
    import qoc_b200.standard as std
    from bench import lindblad_problem
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    name, power = card()
    result = {"gpu": name or torch.cuda.get_device_name(0), "power_limit": power, "rounds": args.rounds,
              "steps_per_round": args.steps, "workloads": {}}
    for wl in ("cfg2_lindblad_n2", "lindblad_n8_D2_N5"):
        q = lindblad_problem(wl)
        plans, rows = {}, {}
        for key, (h, ld, oh, old) in variants(q).items():
            plans[key] = LindbladPlan(q["rho0"], [std.TargetDensityInfidelity(q["targ"])], q["T"], q["N"], hamiltonian=h,
                                      lindblad_data=ld, control_eval_count=q["M"], control_count=1, complex_controls=True)
            assert (plans[key].series is not None) == (key == "TD")
            for _ in range(3):
                err, grads, finals = plans[key].cost_and_grad(q["controls"])
            o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(q["controls"], oh, old, q["rho0"],
                                                              [orc.TargetDensityInfidelity(q["targ"])], q["T"], q["N"],
                                                              freeze_steps=True)
            st = plans[key].stats()
            s = plans[key].series
            rows[key] = {"rk_attempts": st["attempts"], "rk_accepted": st["accepted"],
                         "rhs_per_eval": 7 * st["attempts"] + 14 * st["accepted"],
                         "parity": {"cost_abs": abs(err - o_err), "final_rel": rel(finals, o_fin),
                                    "grad_rel": rel(grads, o_grad)},
                         "series": None if s is None else {"segments": s.segments, "degree": s.degree, "columns": s.series.shape[2],
                                                           "segments_per_step": s.m, "t_max": s.t_max},
                         "range_extensions": plans[key].range_extensions, "sec": []}
        for _ in range(args.rounds):                          # alternate the two variants
            for key in ("TI", "TD"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    plans[key].cost_and_grad(q["controls"])
                torch.cuda.synchronize()
                rows[key]["sec"].append((time.perf_counter() - t0) / args.steps)
        for key, r in rows.items():
            sec = np.array(r.pop("sec"))
            r["evals_per_sec_median"] = float(1.0 / np.median(sec))
            r["evals_per_sec_rounds"] = [float(x) for x in 1.0 / sec]
            r["ns_per_rhs_median"] = float(np.median(sec) / r["rhs_per_eval"] * 1e9)
            plans[key].close()
        rows["series_cost_ns_per_rhs"] = rows["TD"]["ns_per_rhs_median"] - rows["TI"]["ns_per_rhs_median"]
        result["workloads"][wl] = rows
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
