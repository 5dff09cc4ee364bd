"""
_lib.py - ctypes binding of the C ABI in include/qocb200.h (libqocb200.so, built in-tree by
`__graft_entry__.build()` / `qoc_b200._lib.build_library()`).

There is no CPU fallback: if the shared library is missing or no CUDA device is present, every hot-path entry
point raises RuntimeError.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QOCB200_LIB", os.path.join(_HERE, "libqocb200.so"))
CSRC = os.path.join(_HERE, "csrc")
COMPILE_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-lcublas",
              "-Xlinker", "-rpath=/usr/local/cuda/lib64"]

EXPORTS = [
    "qocb_plan_create", "qocb_plan_destroy", "qocb_last_error", "qocb_set_operators", "qocb_set_node_map", "qocb_set_states",
    "qocb_add_cost", "qocb_clear_costs", "qocb_cost", "qocb_cost_and_grad", "qocb_forward", "qocb_backward", "qocb_get_states", "qocb_get_final_states", "qocb_get_node_grad",
    "qocb_get_propagators", "qocb_upload_controls", "qocb_run_resident", "qocb_sync", "qocb_download_result",
    "qocb_time_resident", "qocb_launch_count", "qocb_stream", "qocb_expm_batched", "qocb_expm_vjp_batched",
    "qocb_expm_batched_time", "qocb_expm_batched_bench", "qocb_version", "qocb_flush_l2", "qocb_shard_matrix_doubles",
    "qocb_shard_vector_doubles", "qocb_shard_forward_local", "qocb_shard_forward_finish",
    "qocb_shard_backward_particular", "qocb_shard_backward_finish", "qocb_shard_result_doubles",
    "qocb_shard_pack_result", "qocb_state_shard_coherent_doubles", "qocb_state_shard_forward", "qocb_state_shard_finish",
    "qocb_lindblad_create", "qocb_lindblad_destroy", "qocb_lindblad_last_error",
    "qocb_lindblad_set_operators", "qocb_lindblad_set_densities", "qocb_lindblad_add_cost", "qocb_lindblad_cost",
    "qocb_lindblad_cost_and_grad", "qocb_lindblad_stats", "qocb_lindblad_get_densities", "qocb_lindblad_set_time_series",
    "qocb_lindblad_max_stage_time", "qocb_lindblad_forward", "qocb_lindblad_backward", "qocb_lindblad_set_ensemble",
    "qocb_lindblad_member_results",
]


class Problem(C.Structure):
    """mirror of `qocb_problem` (include/qocb200.h)."""
    _fields_ = [("hilbert_size", C.c_int32), ("state_count", C.c_int32), ("control_count", C.c_int32),
                ("control_eval_count", C.c_int32), ("system_eval_count", C.c_int32), ("magnus_order", C.c_int32),
                ("cost_eval_step", C.c_int32), ("ensemble_count", C.c_int32), ("device", C.c_int32),
                ("store_tape", C.c_int32), ("chunks_per_member", C.c_int32), ("slice_begin", C.c_int32),
                ("slice_end", C.c_int32), ("channel_count", C.c_int32), ("state_total", C.c_int32), ("state_first", C.c_int32),
                ("evolution_time", C.c_double)]


class LindbladProblem(C.Structure):
    """mirror of `qocb_lindblad_problem` (include/qocb200.h)."""
    _fields_ = [("hilbert_size", C.c_int32), ("density_count", C.c_int32), ("control_count", C.c_int32),
                ("control_eval_count", C.c_int32), ("system_eval_count", C.c_int32), ("cost_eval_step", C.c_int32),
                ("lindblad_count", C.c_int32), ("have_hamiltonian", C.c_int32), ("device", C.c_int32),
                ("max_rk_steps", C.c_int32), ("channel_count", C.c_int32), ("time_dependent_rates", C.c_int32),
                ("ensemble_count", C.c_int32), ("evolution_time", C.c_double)]


def sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))]


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [os.path.join(os.path.dirname(_HERE), "include", "qocb200.h")]
    return any(os.path.getmtime(s) > t for s in deps)


def build_library(force=False, verbose=False):
    """nvcc cross-compiles for sm_100a without a GPU.  One object per .cu (compiled in parallel), then a link."""
    if not force and not needs_build():
        return LIB_PATH
    cus = [s for s in sources() if s.endswith(".cu")]
    hdrs = [s for s in sources() if s.endswith(".cuh")] + [os.path.join(os.path.dirname(_HERE), "include", "qocb200.h")]
    newest_hdr = max(os.path.getmtime(h) for h in hdrs)
    procs, objs = [], []
    for cu in cus:
        obj = cu[:-3] + ".o"
        objs.append(obj)
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(cu), newest_hdr)):
            continue
        cmd = ["nvcc"] + COMPILE_FLAGS + ["-c", "-o", obj, cu]
        if verbose:
            print(" ".join(cmd))
        procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, pr in procs:
        if pr.wait() != 0:
            raise subprocess.CalledProcessError(pr.returncode, cmd)
    cmd = ["nvcc"] + LINK_FLAGS + ["-o", LIB_PATH] + objs
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


_lib = None
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def load():
    """Load the shared library (fails loudly; no CPU path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("qoc_b200: {} is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the GRAPE hot path)".format(LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.qocb_plan_create.argtypes = [C.POINTER(Problem), C.POINTER(vp)]
    lib.qocb_plan_destroy.argtypes = [vp]
    lib.qocb_last_error.argtypes = [vp]
    lib.qocb_last_error.restype = C.c_char_p
    lib.qocb_set_operators.argtypes = [vp, vp, vp]
    lib.qocb_set_node_map.argtypes = [vp, vp, vp]
    lib.qocb_set_states.argtypes = [vp, vp]
    lib.qocb_add_cost.argtypes = [vp, i32, i32, dbl, vp, vp, i32]
    lib.qocb_clear_costs.argtypes = [vp]
    lib.qocb_cost.argtypes = [vp, vp, vp, vp]
    lib.qocb_cost_and_grad.argtypes = [vp, vp, vp, vp, vp]
    lib.qocb_forward.argtypes = [vp, vp, vp, vp]
    lib.qocb_backward.argtypes = [vp, vp, vp]
    lib.qocb_get_states.argtypes = [vp, vp]
    lib.qocb_get_final_states.argtypes = [vp, vp]
    lib.qocb_get_node_grad.argtypes = [vp, vp]
    lib.qocb_get_propagators.argtypes = [vp, vp]
    lib.qocb_upload_controls.argtypes = [vp, vp]
    lib.qocb_run_resident.argtypes = [vp, i32]
    lib.qocb_sync.argtypes = [vp]
    lib.qocb_download_result.argtypes = [vp, vp, vp]
    lib.qocb_time_resident.argtypes = [vp, i32, i32, i32, i32, vp, vp]
    lib.qocb_launch_count.argtypes = [vp, i32]
    lib.qocb_stream.argtypes = [vp]
    lib.qocb_stream.restype = vp
    lib.qocb_expm_batched.argtypes = [i32, i64, vp, vp, i32]
    lib.qocb_expm_vjp_batched.argtypes = [i32, i64, vp, vp, vp, vp, i32]
    lib.qocb_expm_batched_time.argtypes = [i32, i64, dbl, i32, vp, i32]
    lib.qocb_expm_batched_bench.argtypes = [i32, i64, dbl, i32, i32, vp, vp, i32]
    lib.qocb_version.restype = C.c_char_p
    lib.qocb_lindblad_create.argtypes = [C.POINTER(LindbladProblem), C.POINTER(vp)]
    lib.qocb_lindblad_destroy.argtypes = [vp]
    lib.qocb_lindblad_last_error.argtypes = [vp]
    lib.qocb_lindblad_last_error.restype = C.c_char_p
    lib.qocb_lindblad_set_operators.argtypes = [vp, vp, vp, vp, vp]
    lib.qocb_lindblad_set_densities.argtypes = [vp, vp]
    lib.qocb_lindblad_add_cost.argtypes = [vp, i32, i32, dbl, vp, vp, i32]
    lib.qocb_lindblad_cost.argtypes = [vp, vp, vp, vp]
    lib.qocb_lindblad_cost_and_grad.argtypes = [vp, vp, vp, vp, vp]
    lib.qocb_lindblad_forward.argtypes = [vp, vp, vp, vp]
    lib.qocb_lindblad_backward.argtypes = [vp, vp, vp]
    lib.qocb_lindblad_stats.argtypes = [vp, vp]
    lib.qocb_lindblad_get_densities.argtypes = [vp, vp]
    lib.qocb_lindblad_set_time_series.argtypes = [vp, i32, i32, dbl, vp]
    lib.qocb_lindblad_max_stage_time.argtypes = [vp, vp]
    lib.qocb_lindblad_set_ensemble.argtypes = [vp, vp, vp]
    lib.qocb_lindblad_member_results.argtypes = [vp, vp, vp, vp]
    lib.qocb_flush_l2.argtypes = [vp]
    lib.qocb_shard_matrix_doubles.argtypes = [vp]
    lib.qocb_shard_vector_doubles.argtypes = [vp]
    lib.qocb_shard_forward_local.argtypes = [vp, i32, vp]
    lib.qocb_shard_forward_finish.argtypes = [vp, vp, i32]
    lib.qocb_shard_backward_particular.argtypes = [vp, vp]
    lib.qocb_shard_backward_finish.argtypes = [vp, vp, vp, i32, i32]
    lib.qocb_shard_result_doubles.argtypes = [vp]
    lib.qocb_shard_pack_result.argtypes = [vp, i32, vp]
    lib.qocb_state_shard_coherent_doubles.argtypes = [vp]
    lib.qocb_state_shard_forward.argtypes = [vp, i32, vp]
    lib.qocb_state_shard_finish.argtypes = [vp, i32, vp]
    _lib = lib
    return lib


def ptr(a):
    """host pointer of a C-contiguous numpy array (or NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def check(rc, plan_handle=None):
    if rc != 0:
        msg = load().qocb_last_error(plan_handle)
        raise RuntimeError("qoc_b200 CUDA path failed (rc={}): {}".format(rc, msg.decode() if msg else "?"))
