#!/usr/bin/env python
"""bench.py - GRAPE cost+gradient evaluations per second on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (see `dump_outputs`), so
that two builds can be compared output for output: every input is generated from fixed seeds.

A "step" is one cost+gradient evaluation of the hot path (Magnus assembly -> batched Pade-13 expm -> state /
costate sweeps -> cost reductions -> gradient) on one batch of synthetic random controls.  Default workload =
the shape BASELINE.json's target is quoted on: dim 64 x 2000 slices, Magnus M4, K = 4 real controls, S = 4
states, TargetStateInfidelity (SURVEY.md section 8d).  One JSON line is printed by rank 0.

  value        evals/s with the controls already resident in HBM (device timed, CUDA events on the plan stream)
  e2e          evals/s through the public API `SchroedingerPlan.cost_and_grad(controls)` = C-ABI
               `qocb_cost_and_grad` with HOST buffers: H2D of the controls and D2H of cost, gradient and final
               states are inside the timed region
  roofline     dominant kernel against the FP64 tensor (DMMA) pipe: algorithmic FLOPs / measured duration
  cpu_baseline the oracle (CPU restatement of the reference, torch complex128 + autograd) on the box's host
               cores, on a bounded sample of the same workload

N > 1 (torchrun): the time slices of ONE evaluation are sharded across the ranks (strong scaling) with an NCCL
exchange of the shard boundary propagators and costates.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.problems import Problem  # noqa: E402

FP64_TENSOR_PEAK_TFLOPS = 37.1   # measured on this pool's B200: DMMA m8n8k4 issue-bound loop and cuBLAS ZGEMM 4096
#                                  (profiles/r01_microbench_fp64.jsonl); MEASURED_PEAKS.json has no FP64 entry

WORKLOADS = {
    # name: (n, slices, K, S, order, complex_controls, F[, ensemble members])
    "n64_2000_M4": (64, 2000, 4, 4, 4, False, 0),
    "cfg3_n60_2000_M4": (60, 2000, 2, 4, 4, True, 6),
    "cfg1_n2_10_M2": (2, 10, 1, 1, 2, True, 0),
    "n32_2000_M4": (32, 2000, 4, 4, 4, False, 0),
    "n16_2000_M4": (16, 2000, 4, 4, 4, False, 0),
    "n8_2000_M2": (8, 2000, 2, 2, 2, False, 0),
    "n128_2000_M4": (128, 2000, 4, 4, 4, False, 0),
    "cfg4_n256_10000_M4": (256, 10000, 4, 4, 4, False, 0),
    "n256_1250_M4": (256, 1250, 4, 4, 4, False, 0),                     # one rank's share of cfg4 at 8 GPUs
    "cfg5_n32_500_S64_E1024_M2": (32, 500, 2, 64, 2, False, 0, 1024),
    "cfg5_n32_500_S64_E128_M2": (32, 500, 2, 64, 2, False, 0, 128),      # one rank's share of cfg5 at 8 GPUs
    "cfg5_n32_100_S64_E16_M2": (32, 100, 2, 64, 2, False, 0, 16),        # small ensemble (tests)
}


def flops_per_slice(n, S, order, s=0):
    """SURVEY.md 8(d): F = W (21 2/3 + 3 s + 3 c) + 24 n^2 S, W = 8 n^3, c = 0/2/6 commutator matmuls."""
    c = {2: 0, 4: 2, 6: 6}[order]
    W = 8.0 * n ** 3
    fwd = W * (c + 22.0 / 3 + s) + 8.0 * n * n * S
    bwd = W * (2 * c + 12 + 2 * s + 7.0 / 3) + 16.0 * n * n * S
    return fwd, bwd


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md).  NVML in a background thread
    (a few ms per sample, so short timed regions still get samples); falls back to `nvidia-smi -lms` when pynvml is absent."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    # nvmlClocksEventReason* bit masks
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []
        self.nvml, self.samples, self.stop_flag, self.thread = None, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.device]) if vis and vis.split(",")[self.device].isdigit() else self.device
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                try:
                    pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                except Exception:
                    pw = None
                self.samples.append((sm, mask, pw))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            if self.thread is not None:
                self.thread.join(timeout=2)
            sm = [x[0] for x in self.samples]
            reasons = sorted(k for k, bit in self.REASONS.items() if any(x[1] & bit for x in self.samples))
            pw = [x[2] for x in self.samples if x[2] is not None]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.sm_max,
                    "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons, "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi"}


def ncu_traffic(workload, kernel):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (or None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(workload, {}).get(kernel)
    except Exception:
        return None


DUMP_LIMIT_BYTES = 60 * 10 ** 6      # array data; with .npy headers and index files the dump stays below 64 MB


def dump_outputs(directory, arrays):
    """Write each array as `directory/<name>.npy`: real arrays as float64, complex ones as float64 with a trailing
    (real, imaginary) axis.  When the arrays together exceed DUMP_LIMIT_BYTES, each keeps a fixed, seeded sample of its
    leading-axis entries in proportion to its size, and the sampled indices go to `<name>_index.npy`."""
    os.makedirs(directory, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out[name] = np.stack([a.real, a.imag], axis=-1) if np.iscomplexobj(a) else a.astype(np.float64)
    total = sum(a.nbytes for a in out.values())
    for name, a in out.items():
        if total > DUMP_LIMIT_BYTES and a.ndim > 0 and a.shape[0] > 1:
            share = a.nbytes * DUMP_LIMIT_BYTES // total
            keep = max(1, share // (a.nbytes // a.shape[0] + 8))
            idx = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            np.save(os.path.join(directory, name + "_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def make_problem(name):
    w = WORKLOADS[name]
    n, slices, K, S, order, cc, F = w[:7]
    p = Problem(n, slices, K, S, order, complex_controls=cc, F=F, seed=0)
    p.E = w[7] if len(w) > 7 else 1
    p.drifts = None
    if p.E > 1:                         # SURVEY.md 8(d): H0^(e) = H0 + delta_e Z, delta_e ~ N(0, 0.1^2)
        rng = np.random.default_rng(12345)
        z = np.diag(np.linspace(-1, 1, n)).astype(np.complex128) * np.abs(p.h0).max()
        p.drifts = np.stack([p.h0 + d * z for d in rng.normal(0, 0.1, p.E)])
    return p


def oracle_time(p, sample_slices, reps, threads):
    """seconds per cost+gradient evaluation of a `sample_slices`-slice truncation of the workload (same dt,
    same operators, first sample_slices+1 control points), oracle = CPU restatement of the reference."""
    import torch
    from oracle import qoc_oracle as orc
    torch.set_num_threads(threads)
    N = sample_slices + 1
    controls = np.ascontiguousarray(p.controls[:N])
    ham = orc.make_hamiltonian(p.h0, p.drives, p.complex_controls)
    q = Problem.__new__(Problem)
    q.__dict__.update(p.__dict__)
    q.N = N
    times = []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        orc.schroedinger_cost_and_grad(controls, ham, p.initial_states, q.costs(orc), float(sample_slices), N,
                                       order=p.order, cost_eval_step=p.cost_eval_step)
        times.append(time.perf_counter() - t0)
    return float(np.median(times[1:]))


def cpu_sample(p, want):
    """bounded CPU sample: slices of ONE ensemble member; the cost per slice grows as n^3"""
    slices = p.N - 1
    cap = want if p.n <= 64 else (40 if p.n <= 128 else 12)
    return max(4, min(slices, cap))


def pick_threads(p):
    """the oracle's BLAS threading can hurt at small n (SURVEY.md section 6): calibrate 1 thread vs all cores on a
    few slices and use the faster."""
    allc = os.cpu_count() or 1
    t1 = oracle_time(p, 8, 1, 1)
    ta = oracle_time(p, 8, 1, allc) if allc > 1 else float("inf")
    return (1, t1, ta) if t1 <= ta else (allc, t1, ta)


def run_reference(args, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    p = make_problem(name)
    slices = p.N - 1
    threads, t1, ta = pick_threads(p)
    # the whole pulse whenever one evaluation of the oracle costs seconds (n <= 64: ~4 s for 2000 slices on 16 cores), a bounded
    # sample scaled linearly otherwise (cfg4: n = 256 x 10^4 slices would take hours)
    sample = slices if (p.n <= 64 and args.ref_slices <= 0) else cpu_sample(p, int(args.ref_slices) if args.ref_slices > 0 else 100)
    for _ in range(args.warmup):
        oracle_time(p, min(sample, 8), 0 + 1, threads)
    t0 = time.perf_counter()
    per = []
    for _ in range(args.steps):
        per.append(oracle_time(p, sample, 1, threads) * slices / sample * p.E)
    wall = time.perf_counter() - t0
    sec = float(np.mean(per))
    val = 1.0 / sec
    out = {"impl": "reference", "metric": "grape_cost_grad_evals_per_sec", "value": val, "unit": "evals/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "c128 (f64)",
           "data": "synthetic", "config": workload_config(name, p),
           "cpu_baseline": {"value": val, "unit": "evals/s", "cores": threads, "kind": "port",
                            "sample": "%d of %d slices (of one ensemble member) per step (fwd+bwd; scaled linearly when fewer than all); oracle = torch complex128 "
                                      "restatement of the reference (autograd absent in this image); 1 thread %.3fs vs %d "
                                      "threads %.3fs on an 8-slice calibration" % (sample, slices, t1, os.cpu_count() or 1, ta)},
           "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": wall}
    print(json.dumps(out))


def workload_config(name, p):
    return {"workload": name, "hilbert_dim": p.n, "slices": p.N - 1, "controls": p.K, "ensemble_members": p.E,
            "complex_controls": p.complex_controls, "states": p.S, "magnus": "M%d" % p.order,
            "costs": "TargetStateInfidelity" + ("+ForbidStates" if p.F else ""),
            "l2": "working set (propagators + tape) > 126 MB L2 and a 256 MiB flush write between timed iterations"}


def run_b200(args, name):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the GRAPE hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import qoc_b200.standard as std
    from qoc_b200.core.plan import SchroedingerPlan
    from qoc_b200.models import MagnusPolicy
    pol = {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}
    p = make_problem(name)
    slices = p.N - 1
    kw = {}
    if p.E > 1:                          # ensembles shard by members (independent units; the member set is fixed: strong)
        if world > 1:
            from qoc_b200.core.sharded import EnsembleShardedPlan as PlanCls
            kw["ensemble_drifts"] = p.drifts
        else:
            PlanCls = SchroedingerPlan
            kw["ensemble_drifts"] = p.drifts
    elif world > 1:
        from qoc_b200.core.sharded import ShardedSchroedingerPlan as PlanCls
    else:
        PlanCls = SchroedingerPlan
    plan = PlanCls(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                   control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order],
                   cost_eval_step=p.cost_eval_step, device=local, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ("value") -------------------------------------------------------------
    plan.upload(p.controls)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    total_ms, stages = plan.time_resident(with_grad=True, warmup=args.warmup, iters=args.steps, flush_l2=True)
    barrier()
    # ---- end-to-end timing through the public API with host buffers ----------------------------------------
    for _ in range(args.warmup):
        plan.cost_and_grad(p.controls)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        err, grads, finals = plan.cost_and_grad(p.controls)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"cost": err, "grads": grads, "final_states": finals})
    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])
    ms_per_step = total_ms / args.steps
    value = 1e3 / ms_per_step
    KR = plan.KR
    h2d = p.M * KR * 8
    d2h = p.M * KR * 8 + 8 + plan.E * p.S * p.n * 16
    if p.n > 64:
        stage_names_note = "n > 64: stages are not split (batched pipeline)"
    fwd_f, bwd_f = flops_per_slice(p.n, p.S, p.order)
    names = ["expm_fwd", "boundary_fwd", "sweep_fwd", "sweep_bwd", "expm_bwd", "gather", "finalize", "prop_tree"]
    stage_ms = {k: float(v) / args.steps for k, v in zip(names, stages)}
    total_flops = (fwd_f + bwd_f) * slices * p.E
    fwd_f, bwd_f = fwd_f * p.E, bwd_f * p.E
    if world == 1 or p.E > 1:
        dom = max(("expm_fwd", "expm_bwd"), key=lambda k: stage_ms[k])
        dom_flops = (fwd_f if dom == "expm_fwd" else bwd_f) * slices / (world if p.E > 1 else 1)
        achieved = dom_flops / (stage_ms[dom] * 1e-3) / 1e12
        dom_name = "k_backward (+ k_magnus_adj)" if dom == "expm_bwd" else "k_forward (+ k_magnus: the Magnus assembly is part of the slice's algorithmic FLOPs)"
    else:       # no per-kernel split across the collectives: whole evaluation, per GPU
        dom_flops = total_flops / world
        achieved = dom_flops / (ms_per_step * 1e-3) / 1e12
        dom_name = "whole evaluation incl. NCCL exchange (per GPU)"
        # per-phase breakdown from a SEPARATE short pass with one event per protocol phase (outside the timed region, so
        # the extra events cannot touch `value`); max over ranks per phase
        sn = ["forward_local", "gather_P", "forward_finish", "backward_particular", "gather_b", "backward_finish", "pack_reduce"]
        it = max(3, min(args.steps, 10))
        os.environ["QOCB_STAGE_TIMING"] = "1"
        _, st2 = plan.time_resident(with_grad=True, warmup=1, iters=it, flush_l2=True)
        os.environ.pop("QOCB_STAGE_TIMING")
        t2 = torch.tensor(np.asarray(st2[1:8]) / it, dtype=torch.float64, device="cuda")
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        stage_ms = {"total": ms_per_step, "phases_max_over_ranks": {k: float(v) for k, v in zip(sn, t2.tolist())},
                    "note": "phases timed in a separate pass of %d evaluations with per-phase events" % it}
    out = {"metric": "grape_cost_grad_evals_per_sec", "value": value, "unit": "evals/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "c128 (f64)", "data": "synthetic",
           "config": workload_config(name, p),
           "e2e": {"value": args.steps / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h},
           "gpu_launches": plan.launch_count(True) * args.steps,
           "roofline": {"bound": "tensor", "kernel": dom_name,
                        "achieved": achieved, "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s",
                        "frac": achieved / FP64_TENSOR_PEAK_TFLOPS, "traffic": ncu_traffic(name, "k_backward" if dom_name.startswith("k_backward") else "k_forward"),
                        "peak_source": "FP64 DMMA pipe measured on this pool (profiles/r01_microbench_fp64.jsonl); "
                                       "MEASURED_PEAKS.json has HBM and bf16 only",
                        "algorithmic_flops_per_launch": dom_flops,
                        "flop_model": "SURVEY 8(d): 4-real-multiplication complex products, c commutator products per slice, dense "
                                      "reverse pass; the kernels execute fewer (3M products = 0.75, constant commutators tabulated, "
                                      "Hermitian half products and the rank-S reverse pass at n = 64), so frac measures speed "
                                      "against the algorithmic work and may exceed the pipe utilisation ncu reports",
                        "whole_eval_tflops": total_flops / (ms_per_step * 1e-3) / 1e12,
                        "whole_eval_frac": total_flops / (ms_per_step * 1e-3) / 1e12 / FP64_TENSOR_PEAK_TFLOPS / world},
           "stage_ms": stage_ms, "clocks": clocks, "cost": err}
    if world > 1 and p.E == 1:
        # every N > 1 line proves itself: (a) the NCCL-sharded evaluation against the unsharded CUDA path on the SAME
        # full pulse, (b) the NCCL-sharded evaluation of a truncated pulse against the CPU oracle
        sample = max(world, 64 if p.n <= 64 else 8)
        gate = parity_gate(p, sample, std, PlanCls, pol, device=local)           # collective: all ranks take part
        if rank == 0:
            ref = SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                                   control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order],
                                   cost_eval_step=p.cost_eval_step, device=local)
            r_err, r_grad, r_fin = ref.cost_and_grad(p.controls)
            ref.close()
            gate["sharded_vs_unsharded"] = {"cost_rel": abs(err - r_err) / abs(r_err),
                                            "grad_rel": float(np.linalg.norm(grads - r_grad) / np.linalg.norm(r_grad)),
                                            "finals_rel": float(np.linalg.norm(finals - r_fin) / np.linalg.norm(r_fin))}
            gate["ok"] = bool(max(gate["sharded_vs_unsharded"].values()) < 1e-10 and gate["cost_rel_err"] < 1e-10
                              and gate["grad_rel_err"] < 1e-10)
            out["parity"] = gate
    elif world > 1:
        # ensemble sharding: the members of a small sub-ensemble against a python loop of the oracle over them
        out_par = ensemble_parity_gate(p, std, PlanCls, pol, local, world)
        if rank == 0:
            out["parity"] = out_par
    if rank == 0:
        if not args.no_cpu_baseline:
            threads, t1, ta = pick_threads(p)
            sample = cpu_sample(p, args.cpu_slices)
            sec = oracle_time(p, sample, 3, threads) * slices / sample * p.E
            out["cpu_baseline"] = {"value": 1.0 / sec, "unit": "evals/s", "cores": threads, "kind": "port",
                                   "sample": "%d of %d slices of one ensemble member (fwd+bwd), median of 3 after 1 warm-up, scaled linearly; "
                                             "1 thread %.3fs vs %d threads %.3fs on an 8-slice calibration; published "
                                             "reference figure: 0.187 evals/s at n=64 x 1000 slices on 1 core i7-6700K "
                                             "(report.tex:110)" % (sample, slices, t1, os.cpu_count() or 1, ta)}
            # parity gate on the same controls (bounded: first `sample` slices)
            if p.E == 1 and world == 1:
                out["parity"] = parity_gate(p, min(sample, 64 if p.n <= 64 else 8), std, SchroedingerPlan, pol)
            elif world == 1:
                out["parity"] = ensemble_parity_gate(p, std, SchroedingerPlan, pol, local, 1)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
    plan.close()
    if world > 1:
        dist.destroy_process_group()


def parity_gate(p, sample, std, Plan, pol, device=0):
    """cost and gradient of the first `sample` slices of the workload (same operators, same dt, same controls) through
    `Plan` (unsharded, or NCCL-sharded: then every rank must call this) against the CPU oracle (rank 0 computes it)."""
    from oracle import qoc_oracle as orc
    q = Problem.__new__(Problem)
    q.__dict__.update(p.__dict__)
    q.N = sample + 1
    controls = np.ascontiguousarray(p.controls[:q.N])
    plan = Plan(p.hamiltonian_numpy(), p.initial_states, q.costs(std), float(sample), q.N, control_eval_count=q.N,
                control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order],
                cost_eval_step=p.cost_eval_step, device=device)
    err, grads, _ = plan.cost_and_grad(controls)
    plan.close()
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    o_err, o_grad, _ = orc.schroedinger_cost_and_grad(controls, orc.make_hamiltonian(p.h0, p.drives, p.complex_controls),
                                                      p.initial_states, q.costs(orc), float(sample), q.N, order=p.order,
                                                      cost_eval_step=p.cost_eval_step)
    return {"slices": sample, "cost_rel_err": abs(err - o_err) / abs(o_err),
            "grad_rel_err": float(np.linalg.norm(grads - o_grad) / np.linalg.norm(o_grad)), "tolerance": 1e-10}


def ensemble_parity_gate(p, std, Plan, pol, device, world, members=None, slices=16):
    """ensemble workloads: the first `members` members (>= world) on a `slices`-slice truncation through `Plan` (member-
    sharded over NCCL when world > 1: every rank must call this) against a python loop of the CPU oracle over the members."""
    from oracle import qoc_oracle as orc
    members = members or max(world, 4)
    q = Problem.__new__(Problem)
    q.__dict__.update(p.__dict__)
    q.N = slices + 1
    controls = np.ascontiguousarray(p.controls[:q.N])
    drifts = p.drifts[:members]
    plan = Plan(p.hamiltonian_numpy(), p.initial_states, q.costs(std), float(slices), q.N, control_eval_count=q.N,
                control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order],
                cost_eval_step=p.cost_eval_step, device=device, ensemble_drifts=drifts)
    err, grads, _ = plan.cost_and_grad(controls)
    plan.close()
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    o_err, o_grad = 0.0, 0.0
    for e in range(members):
        v, g, _ = orc.schroedinger_cost_and_grad(controls, orc.make_hamiltonian(drifts[e], p.drives, p.complex_controls),
                                                 p.initial_states, q.costs(orc), float(slices), q.N, order=p.order,
                                                 cost_eval_step=p.cost_eval_step)
        o_err, o_grad = o_err + v / members, o_grad + g / members
    return {"slices": slices, "members": members, "cost_rel_err": abs(err - o_err) / abs(o_err),
            "grad_rel_err": float(np.linalg.norm(grads - o_grad) / np.linalg.norm(o_grad)), "tolerance": 1e-10}


# ---- Lindblad workloads (cfg2 and a denser variant): one step = one cost+gradient of the adaptive RKDP5 path -------------
LINDBLAD_WORKLOADS = {
    # name: (n, D, intervals, T, gamma, max control norm)
    "cfg2_lindblad_n2": (2, 1, 1, 10.0, 1e-3, 5.0),              # examples/1_transmon_pi_dechoerence.py:22-60
    "lindblad_n8_D2_N5": (8, 2, 4, 4.0, 5e-2, 1.0),
}


def lindblad_problem(name):
    n, D, intervals, T, gamma, mx = LINDBLAD_WORKLOADS[name]
    rng = np.random.default_rng(0)
    a = np.diag(np.sqrt(np.arange(1, n)), 1).astype(np.complex128)
    h0 = np.diag(np.arange(n) - (n - 1) / 2.0).astype(np.complex128) * (1.0 if n == 2 else 0.7)
    M = 11
    controls = (0.1 * mx * (1 - 1j) / np.sqrt(2)) * np.ones((M, 1), dtype=np.complex128)     # flat initial guess (common.py:110-142)
    if n > 2:
        controls = controls + 0.05 * (rng.standard_normal((M, 1)) + 1j * rng.standard_normal((M, 1)))
    rho0 = np.zeros((D, n, n), dtype=np.complex128)
    targ = np.zeros((D, n, n), dtype=np.complex128)
    for d in range(D):
        rho0[d, d, d] = 1.0
        targ[d, d + 1, d + 1] = 1.0
    return dict(n=n, D=D, N=intervals + 1, T=T, M=M, h0=h0, drive=a[None], controls=controls, gam=np.array([gamma]),
                lops=a[None], rho0=rho0, targ=targ)


def run_lindblad_reference(args, name):
    """reference arm of the Lindblad workloads: the oracle (torch restatement of lindbladdiscrete.py:357-495 with the adaptive
    RKDP5 of mathmethods.py:352-480, gradient by torch.autograd through the step-size controller as the reference's tape does)
    on the host, one full cost+gradient evaluation per step."""
    import torch
    from oracle import qoc_oracle as orc
    q = lindblad_problem(name)
    torch.set_num_threads(1)
    ocosts = [orc.TargetDensityInfidelity(q["targ"])]
    oh, old = orc.make_hamiltonian(q["h0"], q["drive"], True), orc.make_lindblad_data(q["gam"], q["lops"])
    for _ in range(args.warmup):
        orc.lindblad_cost_and_grad(q["controls"], oh, old, q["rho0"], ocosts, q["T"], q["N"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.lindblad_cost_and_grad(q["controls"], oh, old, q["rho0"], ocosts, q["T"], q["N"])
    sec = (time.perf_counter() - t0) / args.steps
    val = 1.0 / sec
    print(json.dumps({"impl": "reference", "metric": "grape_cost_grad_evals_per_sec", "value": val, "unit": "evals/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
                      "scaling": "replicas only", "vs_baseline": None, "dtype": "c128 (f64)", "data": "synthetic",
                      "config": {"workload": name, "hilbert_dim": q["n"], "densities": q["D"], "intervals": q["N"] - 1},
                      "cpu_baseline": {"value": val, "unit": "evals/s", "cores": 1, "kind": "port",
                                       "sample": "full cost+gradient evaluations of the oracle (every adaptive step, no truncation)"},
                      "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_lindblad(args, name):
    if args.impl == "reference":
        return run_lindblad_reference(args, name)
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the GRAPE hot path has no CPU fallback")
    import qoc_b200.standard as std
    from oracle import qoc_oracle as orc
    from qoc_b200.core.plan import LindbladPlan
    from tests.problems import numpy_hamiltonian
    q = lindblad_problem(name)
    plan = LindbladPlan(q["rho0"], [std.TargetDensityInfidelity(q["targ"])], q["T"], q["N"],
                        hamiltonian=numpy_hamiltonian(q["h0"], q["drive"], True), lindblad_data=lambda t: (q["gam"], q["lops"]),
                        control_eval_count=q["M"], control_count=1, complex_controls=True)
    for _ in range(max(3, args.warmup)):
        plan.cost_and_grad(q["controls"])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        err, grads, finals = plan.cost_and_grad(q["controls"])
    sec = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"cost": err, "grads": grads, "final_densities": finals})
    st = plan.stats()
    torch.set_num_threads(1)
    ocosts = [orc.TargetDensityInfidelity(q["targ"])]
    oh, old = orc.make_hamiltonian(q["h0"], q["drive"], True), orc.make_lindblad_data(q["gam"], q["lops"])
    t1 = time.perf_counter()
    o_err, o_grad, o_fin = orc.lindblad_cost_and_grad(q["controls"], oh, old, q["rho0"], ocosts, q["T"], q["N"], freeze_steps=True)
    cpu_sec = time.perf_counter() - t1
    # RHS evaluations: 7 per attempt (forward) + reverse replay of the accepted steps (7 recomputed + 7 adjoint)
    nn = q["n"] ** 2
    rhs_flops = 8.0 * q["n"] ** 3 * (2 + 2 * len(q["gam"])) * q["D"]
    flops = rhs_flops * (7 * st["attempts"] + 14 * st["accepted"])
    out = {"metric": "grape_cost_grad_evals_per_sec", "value": 1.0 / sec, "unit": "evals/s", "n_gpus": 1, "steps": args.steps,
           "warmup": max(3, args.warmup), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "replicas only",
           "vs_baseline": None, "dtype": "c128 (f64)", "data": "synthetic",
           "config": {"workload": name, "hilbert_dim": q["n"], "densities": q["D"], "intervals": q["N"] - 1,
                      "rk_attempts": st["attempts"], "rk_accepted": st["accepted"],
                      "l2": "latency-bound persistent CTA; working set in shared memory"},
           "e2e": {"value": 1.0 / sec, "unit": "evals/s", "h2d_bytes_per_step": q["M"] * 2 * 8,
                   "d2h_bytes_per_step": q["M"] * 2 * 8 + 8 + q["D"] * nn * 16},
           "gpu_launches": 2 * args.steps,
           "roofline": {"bound": "tensor", "kernel": "k_lindblad_forward + k_lindblad_backward", "achieved": flops / sec / 1e12,
                        "peak": FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": flops / sec / 1e12 / FP64_TENSOR_PEAK_TFLOPS,
                        "traffic": None, "note": "sequential adaptive integration on one SM: latency-bound by construction"},
           "clocks": clocks, "cost": err,
           "cpu_baseline": {"value": 1.0 / cpu_sec, "unit": "evals/s", "cores": 1, "kind": "port",
                            "sample": "one full cost+gradient evaluation of the oracle (torch, frozen step grid)"},
           "parity": {"cost_abs_err": abs(err - o_err), "grad_rel_err_vs_frozen_oracle":
                      float(np.linalg.norm(grads - o_grad) / np.linalg.norm(o_grad)), "tolerance": "1e-9 / 1e-7 (DESIGN.md section 5)"}}
    print(json.dumps(out))
    plan.close()


# ---- batched matrix exponential (BASELINE.json metric 2: "batched expm GFLOP/s"; SURVEY.md section 8d shapes) --------------------
EXPM_WORKLOADS = {
    # name: (n, batch): working sets (32 n^2 bytes per matrix) well above the 126 MB L2 for the HBM-bound sizes
    "expm_batched_n2": (2, 1 << 22), "expm_batched_n4": (4, 1 << 20), "expm_batched_n8": (8, 1 << 18),
    "expm_batched_n16": (16, 1 << 15), "expm_batched_n32": (32, 1 << 13), "expm_batched_n64": (64, 1 << 12),
}


def expm_flops(n, s=0):
    """SURVEY.md 8(d): W (6 + 4/3 + s), W = 8 n^3 (6 products, LU + two n-RHS triangular solves, s squarings)."""
    return 8.0 * n ** 3 * (6 + 4.0 / 3 + s)


def expm_sample(n, count, norm=1.5, seed=0):
    """anti-hermitian matrices -i H dt with ||.||_1 = norm (s = 0), as the GRAPE slices produce them"""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((count, n, n)) + 1j * rng.standard_normal((count, n, n))
    h = (x + x.conj().transpose(0, 2, 1)) / 2
    h *= (norm / np.abs(h).sum(axis=1).max(axis=1))[:, None, None]
    return np.ascontiguousarray(-1j * h)


def oracle_expm_rate(n, seconds=10.0, threads=1):
    """matrices/s of the oracle's expm_pade (torch complex128 restatement of expm.py:210-252) on the host, ~`seconds` of work"""
    import torch
    from oracle import qoc_oracle as orc
    torch.set_num_threads(threads)
    a = torch.as_tensor(expm_sample(n, 64))
    for k in range(4):
        orc.expm_pade(a[k])
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for k in range(64):
            orc.expm_pade(a[k])
        done += 64
    return done / (time.perf_counter() - t0)


def run_expm(args, name):
    import ctypes
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n, batch = EXPM_WORKLOADS[name]
    fl = expm_flops(n)
    cfg = {"workload": name, "hilbert_dim": n, "batch": batch, "norm": 1.5, "squarings": 0,
           "l2": "a 256 MiB flush write between launches (n <= 4); working set %.0f MB" % (32.0 * n * n * batch / 1e6)}
    if args.impl == "reference":
        t0 = time.perf_counter()
        rates = [oracle_expm_rate(n, seconds=max(2.0, 20.0 / max(1, args.steps)), threads=1) for _ in range(max(1, args.steps))]
        rate = float(np.mean(rates))
        val = rate * fl / 1e9
        print(json.dumps({"impl": "reference", "metric": "batched_expm_gflops", "value": val, "unit": "GFLOP/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * batch / rate, "higher_is_better": True,
                          "scaling": "replicas only", "vs_baseline": None, "dtype": "c128 (f64)", "data": "synthetic", "config": cfg,
                          "cpu_baseline": {"value": val, "unit": "GFLOP/s", "cores": 1, "kind": "port", "matrices_per_s": rate,
                                           "sample": "oracle expm_pade (torch complex128 restatement of expm.py:210-252) looped over 64 "
                                                     "matrices for a bounded time per step; ms_per_step is scaled to the batch"},
                          "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "wall_s": time.perf_counter() - t0}))
        return
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the expm kernels have no CPU fallback")
    from qoc_b200 import _lib
    from qoc_b200.standard.functions import expm
    lib = _lib.load()
    tot, best = ctypes.c_double(), ctypes.c_double()
    sampler = ClockSampler(0)
    sampler.start()
    _lib.check(lib.qocb_expm_batched_bench(n, batch, 1.5, max(3, args.warmup), args.steps, ctypes.byref(tot), ctypes.byref(best), 0))
    ms = tot.value / args.steps
    # end to end through the public call with host buffers (H2D of the batch, D2H of the result inside the timed region)
    eb = min(batch, 1 << 16 if n <= 8 else 1 << 12)
    a = expm_sample(n, eb)
    for _ in range(3):
        got = expm(a)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        got = expm(a)
    e2e_s = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"expm": got})
    rate = batch / (ms * 1e-3)
    gbs = 32.0 * n * n * rate / 1e9
    tfl = fl * rate / 1e12
    try:
        hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hsrc = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        hbm, hsrc = 6529.7, "fallback (round-1 MEASURED_PEAKS.json)"
    if n <= 4:
        roof = {"bound": "hbm", "kernel": "k_expm_thread" if n <= 2 else "k_expm_rows", "achieved": gbs, "peak": hbm, "unit": "GB/s",
                "frac": gbs / hbm, "traffic": None, "peak_source": hsrc, "algorithmic_bytes_per_launch": 32.0 * n * n * batch,
                "fp64_tflops": tfl, "fp64_frac": tfl / FP64_TENSOR_PEAK_TFLOPS}
    else:
        roof = {"bound": "tensor", "kernel": "k_expm", "achieved": tfl, "peak": FP64_TENSOR_PEAK_TFLOPS,
                "unit": "TFLOP/s", "frac": tfl / FP64_TENSOR_PEAK_TFLOPS, "traffic": None, "algorithmic_flops_per_launch": fl * batch,
                "peak_source": "FP64 pipe measured on this pool (profiles/r01_microbench_fp64.jsonl; tensor = vector peak on B200)",
                "hbm_gbs": gbs}
    out = {"metric": "batched_expm_gflops", "value": tfl * 1e3, "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps,
           "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None,
           "dtype": "c128 (f64)", "data": "synthetic", "config": cfg, "matrices_per_s": rate,
           "e2e": {"value": fl * eb / e2e_s / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": 16 * n * n * eb,
                   "d2h_bytes_per_step": 16 * n * n * eb, "batch": eb, "matrices_per_s": eb / e2e_s},
           "gpu_launches": args.steps, "roofline": roof, "clocks": clocks}
    if not args.no_cpu_baseline:
        crate = oracle_expm_rate(n, seconds=10.0, threads=1)
        out["cpu_baseline"] = {"value": crate * fl / 1e9, "unit": "GFLOP/s", "cores": 1, "kind": "port", "matrices_per_s": crate,
                               "sample": "oracle expm_pade looped over 64 matrices for 10 s; published reference figure: 2.18 ms per "
                                         "n = 64 matrix on 8 CPU cores (report.tex:250)"}
    import torch as _t
    from oracle import qoc_oracle as orc
    k = min(16, eb)
    want = np.stack([orc.expm_pade(_t.as_tensor(a[i])).numpy() for i in range(k)])
    out["parity"] = {"matrices": k, "rel_err": float(np.linalg.norm(got[:k] - want) / np.linalg.norm(want)), "tolerance": 1e-12}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="n64_2000_M4", choices=sorted(WORKLOADS) + sorted(LINDBLAD_WORKLOADS) + sorted(EXPM_WORKLOADS))
    ap.add_argument("--cpu-slices", type=int, default=400, help="slices of the bounded CPU-baseline sample")
    ap.add_argument("--ref-slices", type=int, default=0, help="slices per step of the --impl reference arm (0 = the whole pulse for n <= 64, "
                                                               "100 scaled linearly above)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--check", action="store_true", help="kept for compatibility: every N > 1 line now carries its parity block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (cost, gradient, final states; a seeded sample of the "
                         "batched expm) to DIR/<name>.npy as float64, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the outputs of the CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.workload in EXPM_WORKLOADS:
        run_expm(args, args.workload)
        return
    if args.workload in LINDBLAD_WORKLOADS:
        if int(os.environ.get("RANK", "0")) == 0:
            run_lindblad(args, args.workload)
        return
    if args.impl == "reference":
        run_reference(args, args.workload)
    else:
        run_b200(args, args.workload)


if __name__ == "__main__":
    main()
