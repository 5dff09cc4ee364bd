#!/usr/bin/env python
"""Per-phase clock64 breakdown of the expm kernels (CTA 0) on a B200.  Builds a -DQOCB_PROFILE variant of the
library into build/ (never the shipped .so; `--build-only` compiles it ahead of a GPU call), runs a workload and prints microseconds per slice and phase.
Usage (on the GPU box): python tools/phase_profile.py [workload]"""
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
out = os.path.join(ROOT, "build", "libqocb200_prof.so")      # git-ignored, travels with gpurun: build it before the GPU call
os.makedirs(os.path.dirname(out), exist_ok=True)
csrc = os.path.join(ROOT, "qoc_b200", "csrc")
srcs = [os.path.join(csrc, f) for f in os.listdir(csrc)]
if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(f) for f in srcs):
    subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-DQOCB_PROFILE",
                    "-shared", "-Xcompiler", "-fPIC", "-lcublas", "-o", out, os.path.join(csrc, "capi.cu"),
                    os.path.join(csrc, "lindblad.cu")], check=True)
if "--build-only" in sys.argv:
    sys.exit(0)
os.environ["QOCB200_LIB"] = out
import numpy as np  # noqa: E402
import bench  # noqa: E402
import qoc_b200.standard as std  # noqa: E402
from qoc_b200 import _lib  # noqa: E402
from qoc_b200.core.plan import SchroedingerPlan  # noqa: E402
from qoc_b200.models import MagnusPolicy  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
name = args[0] if args else "n64_2000_M4"
p = bench.make_problem(name)
pol = {2: MagnusPolicy.M2, 4: MagnusPolicy.M4, 6: MagnusPolicy.M6}
plan = SchroedingerPlan(p.hamiltonian_numpy(), p.initial_states, p.costs(std), p.T, p.N, control_eval_count=p.M,
                        control_count=p.K, complex_controls=p.complex_controls, magnus_policy=pol[p.order])
lib = _lib.load()
buf = (ctypes.c_longlong * 48)()
for _ in range(3):
    plan.cost_and_grad(p.controls)
lib.qocb_debug_profile(buf)
reps = 5
for _ in range(reps):
    plan.cost_and_grad(p.controls)
lib.qocb_debug_profile(buf)
v = np.array(list(buf), dtype=np.float64)
slices = v[0]
ghz = 1.965
us = v / slices / (ghz * 1e3)
names = {1: "fwd coefs+magnus", 2: "fwd one-norm/scale", 3: "fwd pade polynomial (6 products)", 4: "fwd LU factor (pivoted)",
         5: "fwd LU solve (pivoted)", 19: "fwd Q^-1, block Gauss-Jordan (pivot-free)", 25: "fwd R0 = Q^-1 P product (pivot-free)",
         6: "fwd squarings/copy", 7: "fwd pade total + stores + chunk product", 9: "bwd coefs + ubar", 10: "bwd reverse squarings + tape loads",
         11: "bwd transposed solve or Q^-T product", 14: "  LU: panels (warp 0; all 8 per LU)", 15: "  LU: swaps + U12 + trailing update",
         16: "  LU: writeback + diag inversion part of panels", 17: "  Q^-1: first diagonal tile inverse (warp 0)",
         18: "  Q^-1: block steps (NP / 8 per inverse)", 12: "bwd pade polynomial reverse", 13: "bwd pade total + magnus adjoint"}
print("workload", name, "slices sampled by CTA 0:", int(slices))
for k in sorted(names):
    print("  %-45s %8.2f us/slice" % (names[k], us[k]))

for k, nm in ((32, "scale A + store"), (33, "A2 product"), (34, "A2 store"), (35, "A4 product"), (36, "A4 store"), (37, "A6 product"),
              (38, "A6 store + epilogue"), (39, "A6 W1 product (half path: + A6 X1)"), (42, "epilogue + A6 X1 product (full path)"),
              (40, "epilogues + A reload"), (41, "Uo product"), (3, "Uo store + P, Q")):
    print("    poly: %-41s %8.2f us/slice" % (nm, us[k]))
for k, nm in ((43, "stage 0: thin blocks + wait for LU"), (44, "stage 1: l = Q^-T lam, thin product or solve + unpermute (+ wait A)"),
              (45, "stages 2-3: a = A^T l, chain start (+ wait A2)"), (46, "stage 4: two Krylov chains (6 steps)"),
              (47, "stage 5: rank-48 product + H = a2bar + a2bar^H (+ wait A)"), (12, "stage 6: dense product + anti-Hermitian part")):
    print("    krylov: %-50s %8.2f us/slice" % (nm, us[k]))
steps = max(v[24], 1.0)
print("boundary forward pass (CTA 0,0), per chunk step over %d steps:" % int(steps))
for k, nm in ((20, "issue prefetch of next propagator"), (21, "wait for current propagator + barrier"), (22, "mat-vec + barrier"), (23, "store boundary state")):
    print("  %-45s %8.3f us/step" % (nm, v[k] / steps / (ghz * 1e3)))
