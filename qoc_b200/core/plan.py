"""
plan.py - host side of the drop-in boundary: turns the reference's program state (user `hamiltonian`
callable, cost objects, states) into a device plan of the C ABI (include/qocb200.h) and evaluates
cost / cost+gradient on the GPU.

What happens here, once per `grape_*` / `evolve_*` call:
  * Hamiltonian structure extraction.  The reference calls the opaque Python callable `hamiltonian(controls, t)`
    at every Magnus node of every slice (qoc/core/schroedingerdiscrete.py:483-486) and differentiates through
    it.  The CUDA path needs the operator structure, so the callable is probed: H0 = h(0), A_k = h(e_k) - H0,
    B_k = h(i e_k) - H0 (complex controls), and real-linearity in (Re u, Im u) plus time-independence are
    verified with random probes.  Every hamiltonian in the reference's examples/tests has this form
    (examples/0_transmon_pi.py:24-26, examples/tutorial.py:101-106, tests/test_core.py:529-531,582).
    A callable that uses its `time` argument (SURVEY.md section 8f N3) is probed at every Magnus node of every
    slice instead and expanded over a small operator basis (`extract_time_dependent_structure`): the device
    then sees H = G0 + sum_c coef_c(node) A_c with per-node coefficients affine in the interpolated controls
    (qocb_set_node_map).  Anything else (non-linear in the controls, more than 16 operator channels) raises
    NotImplementedError - there is no CPU fallback.
  * cost recognition: the qoc cost classes provide device descriptors (`device_terms`) or, for control-only
    costs, an analytic host value+gradient (`control_value_and_grad`).
"""
import ctypes

import numpy as np

from qoc_b200 import _lib
from qoc_b200.models.enums import InterpolationPolicy, MagnusPolicy

_PROBE_RTOL = 1e-10


class NonlinearHamiltonian(NotImplementedError):
    """raised by the structure extraction when the callable is not affine in (Re u, Im u)."""


_MAX_CHANNELS = 16          # kMaxKR of the CUDA kernels
_NODES = {1: (0.5,), 2: (0.5 - np.sqrt(3.0) / 6, 0.5 + np.sqrt(3.0) / 6),
          3: (0.5 - np.sqrt(15.0) / 10, 0.5, 0.5 + np.sqrt(15.0) / 10)}          # mathmethods.py:88,113-114,148-150


def _unit_controls(control_count, complex_controls):
    dtype = np.complex128 if complex_controls else np.float64
    zero = np.zeros(control_count, dtype=dtype)
    units = []
    for part in ((1.0, 1j) if complex_controls else (1.0,)):
        for k in range(control_count):
            e = zero.copy()
            e[k] = part
            units.append(e)
    return zero, units


def _probe_times(evolution_time, system_eval_count=None, magnus_order=None, dense=64, seed=4321):
    """times at which a callable is checked for time dependence: the end points, `dense` evenly spread times, a few random
    ones and - when the slice grid is known - Magnus node times the reference evaluates the callable at
    (qoc/core/schroedingerdiscrete.py:483-497), including the first and last slices, so that windows, steps and envelopes
    that vanish at a handful of fixed probe times are still seen."""
    rng = np.random.default_rng(seed)
    T = float(evolution_time)
    times = [0.0, T, 0.37 * T, 0.731 * T]
    times += list(np.linspace(0.0, T, dense + 2)[1:-1])
    times += list(rng.uniform(0.0, T, 8))
    if system_eval_count is not None and magnus_order is not None and system_eval_count > 1:
        nsl = system_eval_count - 1
        dt = T / nsl
        picks = sorted(set([0, 1, nsl // 2, nsl - 2, nsl - 1] + [int(x) for x in rng.integers(0, nsl, 16)]))
        for j in picks:
            if 0 <= j < nsl:
                times += [(j + c) * dt for c in _NODES[magnus_order // 2]]
    return times


def _is_time_dependent(hamiltonian, zero, units, evolution_time, system_eval_count=None, magnus_order=None):
    times = _probe_times(evolution_time, system_eval_count, magnus_order)
    for u in [zero] + units:
        ref = np.asarray(hamiltonian(u, times[0]), dtype=np.complex128)
        tol = _PROBE_RTOL * max(1.0, np.abs(ref).max())
        for t in times[1:]:
            if not np.allclose(np.asarray(hamiltonian(u, t), dtype=np.complex128), ref, rtol=_PROBE_RTOL, atol=tol):
                return True
    return False


class _RealBasis(object):
    """Streaming rank-revealing Gram-Schmidt of complex matrices over the REALS (the device coefficients are real):
    `add(m)` returns the coefficient vector of m on the basis so far, extending the basis when the residual exceeds
    `tol` (1e-12) * scale.  Earlier samples have zero weight on later basis vectors by construction."""

    def __init__(self, limit, tol=1e-12):
        self.vecs, self.limit, self.scale, self.tol = [], limit, 1.0, tol

    def _too_many(self):
        return NotImplementedError("the time dependence of this hamiltonian needs more than {} operator channels; not "
                                   "supported by the CUDA path (no CPU fallback)".format(self.limit))

    def seed(self, mats):
        """starts the basis from a pool of samples by pivoted Gram-Schmidt (largest residual first), so that basis
        directions do not come from small samples dominated by cancellation."""
        R = np.array([np.concatenate([m.real.ravel(), m.imag.ravel()]) for m in mats])
        if R.size == 0:
            return
        self.scale = max(self.scale, np.abs(R).max())
        while True:
            norms = np.linalg.norm(R, axis=1)
            j = int(np.argmax(norms))
            if norms[j] <= self.tol * self.scale * np.sqrt(R.shape[1]):
                return
            if len(self.vecs) >= self.limit:
                raise self._too_many()
            r = R[j].copy()
            for _ in range(2):
                for b in self.vecs:
                    r -= np.dot(b, r) * b
            b = r / np.linalg.norm(r)
            self.vecs.append(b)
            R -= np.outer(R @ b, b)

    def add(self, m):
        v = np.concatenate([m.real.ravel(), m.imag.ravel()])
        self.scale = max(self.scale, np.abs(v).max())
        coef = np.zeros(len(self.vecs) + 1)
        r = v.copy()
        for _ in range(2):                       # re-orthogonalise once
            for k, b in enumerate(self.vecs):
                c = np.dot(b, r)
                coef[k] += c
                r -= c * b
        nr = np.linalg.norm(r)
        if nr > self.tol * self.scale * np.sqrt(v.size):
            if len(self.vecs) >= self.limit:
                raise self._too_many()
            self.vecs.append(r / nr)
            coef[-1] = nr
            return coef
        return coef[:-1]

    def matrices(self, shape):
        half = shape[0] * shape[1]
        return np.array([(b[:half] + 1j * b[half:]).reshape(shape) for b in self.vecs]).reshape((-1,) + tuple(shape))


def extract_time_dependent_structure(hamiltonian, control_count, complex_controls, evolution_time, system_eval_count,
                                     magnus_order, seed=1234):
    """Structure of a `hamiltonian(controls, time)` that is affine in the controls at every time:
    returns (G0, channels [KC x n x n], offset [N-1, q, KC], gain [N-1, q, KC, KR]) such that at Magnus node i of
    slice j   H = G0 + sum_c (offset[j,i,c] + sum_r gain[j,i,c,r] x_r) channels[c],   x = [Re u, Im u].
    The callable is evaluated at the node times the reference evaluates it at (schroedingerdiscrete.py:483-497);
    one shared real operator basis serves the drift variation and every control operator, built in one streaming
    pass (memory: the basis and the coefficients only)."""
    q = magnus_order // 2
    nsl = system_eval_count - 1
    dt = evolution_time / nsl
    times = np.array([[(j + c) * dt for c in _NODES[q]] for j in range(nsl)]).ravel()
    zero, units = _unit_controls(control_count, complex_controls) if control_count else (None, [])
    KR = len(units)
    g0 = np.array(hamiltonian(zero, times[0]), dtype=np.complex128)
    if g0.ndim != 2 or g0.shape[0] != g0.shape[1]:
        raise ValueError("hamiltonian(controls, time) must return a square matrix")
    basis = _RealBasis(_MAX_CHANNELS)
    rows = []                                   # per node: [offset coefficients, gain coefficients of control 0, ...]
    for t in times:
        d = np.asarray(hamiltonian(zero, t), dtype=np.complex128)
        row = [basis.add(d - g0)]
        for e in units:
            row.append(basis.add(np.asarray(hamiltonian(e, t), dtype=np.complex128) - d))
        rows.append(row)
    KC = len(basis.vecs)
    if KC == 0:                                 # H == G0 at every node
        return g0, np.zeros((KR,) + g0.shape, dtype=np.complex128)
    channels = basis.matrices(g0.shape)
    offset = np.zeros((len(times), KC))
    gain = np.zeros((len(times), KC, KR))
    for k, row in enumerate(rows):
        offset[k, :len(row[0])] = row[0]
        for r in range(KR):
            gain[k, :len(row[1 + r]), r] = row[1 + r]
    # affine in the controls?  (random controls at a few node times against the expansion)
    rng = np.random.default_rng(seed)
    scale = max(1.0, basis.scale, np.abs(g0).max())
    for trial in range(4 if KR else 0):
        k = int(rng.integers(len(times)))
        u = rng.standard_normal(control_count) * (1.0 + trial)
        if complex_controls:
            u = u + 1j * rng.standard_normal(control_count) * (1.0 + trial)
        x = np.concatenate([u.real, u.imag]) if complex_controls else u
        model = g0 + np.tensordot(offset[k] + gain[k] @ x, channels, axes=(0, 0))
        got = np.asarray(hamiltonian(u.astype(zero.dtype), times[k]), dtype=np.complex128)
        if not np.allclose(got, model, rtol=0, atol=_PROBE_RTOL * scale * (1 + np.abs(x).sum())):
            raise NonlinearHamiltonian(
                "hamiltonian(controls, time) is not affine in (Re u, Im u); a SchroedingerPlan needs that form - "
                "`make_schroedinger_plan` handles non-linear callables (no CPU fallback)")
    return (g0, channels, np.ascontiguousarray(offset.reshape(nsl, q, KC)),
            np.ascontiguousarray(gain.reshape(nsl, q, KC, KR)))


def extract_hamiltonian_structure(hamiltonian, control_count, complex_controls, evolution_time, hilbert_size=None,
                                  seed=1234, system_eval_count=None, magnus_order=None):
    """Returns (h0 [n x n], a_ops [KR x n x n]) with H(x) = H0 + sum_r x_r A_r, x = [Re u, Im u]; for a callable
    that depends on `time` (needs system_eval_count and magnus_order): the 4-tuple of
    `extract_time_dependent_structure`."""
    rng = np.random.default_rng(seed)
    t0, t1 = 0.0, 0.37 * evolution_time
    zero, units = _unit_controls(control_count, complex_controls) if control_count else (None, [])
    if _is_time_dependent(hamiltonian, zero, units, evolution_time, system_eval_count, magnus_order):
        if system_eval_count is None or magnus_order is None:
            raise NotImplementedError("time-dependent hamiltonian callables are not supported by this CUDA path yet "
                                      "(no CPU fallback)")
        return extract_time_dependent_structure(hamiltonian, control_count, complex_controls, evolution_time,
                                                system_eval_count, magnus_order, seed)
    if control_count == 0:
        h0 = np.asarray(hamiltonian(None, t0), dtype=np.complex128)
        return h0, np.zeros((0,) + h0.shape, dtype=np.complex128)
    dtype = zero.dtype
    h0 = np.array(hamiltonian(zero, t0), dtype=np.complex128)
    if h0.ndim != 2 or h0.shape[0] != h0.shape[1]:
        raise ValueError("hamiltonian(controls, time) must return a square matrix")
    a_ops = np.stack([np.array(hamiltonian(e, t0), dtype=np.complex128) - h0 for e in units])
    scale = max(1.0, np.abs(h0).max(), np.abs(a_ops).max())
    for trial in range(3):
        u = rng.standard_normal(control_count) * (1.0 + trial)
        if complex_controls:
            u = u + 1j * rng.standard_normal(control_count) * (1.0 + trial)
        x = np.concatenate([u.real, u.imag]) if complex_controls else u
        model = h0 + np.tensordot(x, a_ops, axes=(0, 0))
        for t in (t0, t1, float(rng.uniform(0.0, evolution_time)), float(evolution_time)):
            got = np.asarray(hamiltonian(u.astype(dtype), t), dtype=np.complex128)
            if not np.allclose(got, model, rtol=0, atol=_PROBE_RTOL * scale * (1 + np.abs(x).sum())):
                raise NonlinearHamiltonian(
                    "hamiltonian(controls, time) is not of the form H0 + sum_k Re(u_k) A_k + Im(u_k) B_k; a SchroedingerPlan "
                    "needs that form - `make_schroedinger_plan` handles non-linear callables (no CPU fallback)")
    return h0, a_ops


def central_differences(f, z):
    """4-point central differences (step 1e-3 max(1, |z_i|), error O(h^4)) of the real function `f` at every entry of the
    array `z`, of any shape: returns (df/dRe z, df/dIm z), the second None for real `z`.  Every entry is differentiated on its
    own, so a function that reads only one triangle of a matrix (eigvalsh and the like) gets the derivative of what it computes
    on general matrices, not of its Hermitian restriction.  Used for the cotangents of user-defined costs."""
    z = np.asarray(z)
    directions = (1.0, 1j) if np.iscomplexobj(z) else (1.0,)
    parts = [np.zeros(z.shape) for _ in directions]
    for idx in np.ndindex(*z.shape):
        h = 1e-3 * max(1.0, abs(z[idx]))
        for part, direction in zip(parts, directions):
            vals = []
            for k in (1.0, -1.0, 2.0, -2.0):
                q = z.copy()
                q[idx] += k * h * direction
                vals.append(f(q))
            part[idx] = (8.0 * (vals[0] - vals[1]) - (vals[2] - vals[3])) / (12.0 * h)
    return parts[0], (parts[1] if len(parts) > 1 else None)


def explicit_control_grad(f, controls):
    """df/dRe u + i df/dIm u (df/du for real controls) of a user-cost sum `f(controls)` whose densities or states are held
    fixed, or None when f does not move under one random probe of the controls (most user costs never read them)."""
    controls = np.asarray(controls)
    base = f(controls)
    rng = np.random.default_rng(0)
    probe = controls + 1e-3 * (rng.standard_normal(controls.shape) + (1j * rng.standard_normal(controls.shape)
                                                                        if np.iscomplexobj(controls) else 0))
    if abs(f(probe) - base) <= 1e-14 * max(1.0, abs(base)):
        return None
    dre, dim = central_differences(f, controls)
    g = np.zeros(controls.shape, dtype=controls.dtype)
    g[...] = dre if dim is None else dre + 1j * dim
    return g


def is_user_cost(cost):
    """a user-defined Cost subclass (qoc/models/cost.py:5-51): it overrides none of the B200 hooks (`device_terms`,
    `device_terms_density`, `control_value_and_grad`), so `cost(controls, states_or_densities, step)` is all it has."""
    from qoc_b200.models.cost import Cost
    t = type(cost)
    return (getattr(t, "device_terms", Cost.device_terms) is Cost.device_terms and getattr(t, "device_terms_density", None) is None
            and getattr(t, "control_value_and_grad", Cost.control_value_and_grad) is Cost.control_value_and_grad)


class SchroedingerPlan(object):
    """Device plan for `_evaluate_schroedinger_discrete` and its jacobian (schroedingerdiscrete.py:356-438,
    :318).  `cost(controls)` and `cost_and_grad(controls)` take controls in cost-function format
    ((M x K) float64 or complex128) and return what the reference seam returns."""

    def __init__(self, hamiltonian, initial_states, costs, evolution_time, system_eval_count,
                 control_eval_count=0, control_count=0, complex_controls=False,
                 magnus_policy=MagnusPolicy.M2, cost_eval_step=1,
                 interpolation_policy=InterpolationPolicy.LINEAR, device=0, store_tape=True,
                 chunks_per_member=0, ensemble_drifts=None, structure=None, slice_range=None, state_slice=None):
        if interpolation_policy != InterpolationPolicy.LINEAR:
            raise NotImplementedError("The interpolation policy {} is not yet supported for this method."
                                      "".format(interpolation_policy))
        if not isinstance(magnus_policy, MagnusPolicy):
            raise ValueError("Unrecognized magnus policy {}.".format(magnus_policy))
        self.lib = _lib.load()
        self._q = magnus_policy.order // 2
        initial_states = np.asarray(initial_states)
        # state sharding (qoc_b200/core/sharded.py): this plan holds states [s0, s1) of S_total; normalisations use S_total
        self.S_total = initial_states.shape[0]
        self.state_first = 0
        if state_slice is not None:
            s0, s1 = int(state_slice[0]), int(state_slice[1])
            if not 0 <= s0 < s1 <= self.S_total:
                raise ValueError("bad state slice {} of {} states".format(state_slice, self.S_total))
            if ensemble_drifts is not None or slice_range is not None:
                raise NotImplementedError("state sharding cannot be combined with ensembles or time-slice sharding")
            initial_states = initial_states[s0:s1]
            self.state_first = s0
        self.S, self.n = initial_states.shape[0], initial_states.shape[1]
        self.K = int(control_count)
        self.M = int(control_eval_count)
        self.N = int(system_eval_count)
        self.complex_controls = bool(complex_controls)
        self.KR = self.K * (2 if self.complex_controls else 1)
        self.costs = list(costs)
        if structure is None:
            structure = extract_hamiltonian_structure(hamiltonian, self.K, self.complex_controls, evolution_time,
                                                      system_eval_count=self.N, magnus_order=magnus_policy.order)
        self.structure = structure
        h0, a_ops = structure[0], structure[1]
        node_map = structure[2:] if len(structure) == 4 else None
        if node_map is not None and ensemble_drifts is not None:
            raise NotImplementedError("ensemble drifts with a time-dependent hamiltonian are not supported")
        if h0.shape[0] != self.n:
            raise ValueError("hamiltonian size {} does not match the states' hilbert size {}".format(h0.shape[0], self.n))
        if ensemble_drifts is not None:          # build-side extension: members differ in the drift only
            h0s = np.ascontiguousarray(ensemble_drifts, dtype=np.complex128)
        else:
            h0s = np.ascontiguousarray(h0[None], dtype=np.complex128)
        self.E = h0s.shape[0]
        pb = _lib.Problem(hilbert_size=self.n, state_count=self.S, control_count=self.KR,
                          control_eval_count=self.M, system_eval_count=self.N,
                          magnus_order=magnus_policy.order, cost_eval_step=int(cost_eval_step),
                          ensemble_count=self.E, device=int(device), store_tape=int(bool(store_tape)),
                          chunks_per_member=int(chunks_per_member),
                          slice_begin=0 if slice_range is None else int(slice_range[0]),
                          slice_end=0 if slice_range is None else int(slice_range[1]),
                          channel_count=0 if node_map is None else int(a_ops.shape[0]),
                          state_total=self.S_total if state_slice is not None else 0, state_first=self.state_first,
                          evolution_time=float(evolution_time))
        handle = ctypes.c_void_p()
        _lib.check(self.lib.qocb_plan_create(ctypes.byref(pb), ctypes.byref(handle)))
        self.handle = handle
        a_ops = np.ascontiguousarray(a_ops, dtype=np.complex128)
        _lib.check(self.lib.qocb_set_operators(handle, _lib.ptr(h0s), _lib.ptr(a_ops) if a_ops.shape[0] else None), handle)
        if node_map is not None:
            offset = np.ascontiguousarray(node_map[0], dtype=np.float64)
            gain = np.ascontiguousarray(node_map[1], dtype=np.float64)
            _lib.check(self.lib.qocb_set_node_map(handle, _lib.ptr(offset), _lib.ptr(gain) if self.KR else None), handle)
        psi0 = np.ascontiguousarray(initial_states.reshape(self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_set_states(handle, _lib.ptr(psi0)), handle)
        self.control_costs = []
        self.user_costs = []
        from qoc_b200.models.cost import Cost
        for c in self.costs:
            if (getattr(type(c), "device_terms", Cost.device_terms) is Cost.device_terms and
                    getattr(type(c), "control_value_and_grad", Cost.control_value_and_grad) is Cost.control_value_and_grad):
                # a user-defined Cost subclass (qoc/models/cost.py:5-51): only `cost(controls, states, step)` exists.  Its value and
                # a numeric cotangent of the final states are computed on the host around qocb_forward / qocb_backward.
                if getattr(c, "requires_step_evaluation", False):
                    raise NotImplementedError("The user-defined cost {} requires step evaluation; only final-step user costs are "
                                              "supported by the CUDA path (no CPU fallback).".format(c))
                if ensemble_drifts is not None or slice_range is not None or state_slice is not None:
                    raise NotImplementedError("user-defined costs cannot be combined with ensembles or sharded plans")
                self.user_costs.append(c)
                continue
            terms = c.device_terms(self.S_total, self.n)
            if state_slice is not None:                  # the vectors (and counts) of the local states only
                terms = [(kind, step, weight, np.asarray(vecs)[self.state_first:self.state_first + self.S],
                          None if counts is None else np.asarray(counts)[self.state_first:self.state_first + self.S])
                         for kind, step, weight, vecs, counts in terms]
            if not terms:
                if getattr(type(c), "control_value_and_grad", Cost.control_value_and_grad) is Cost.control_value_and_grad:
                    raise NotImplementedError("The cost {} has neither device terms nor an analytic control gradient "
                                              "(no CPU fallback).".format(c))
                self.control_costs.append(c)
            for kind, step, weight, vecs, counts in terms:
                vecs = np.ascontiguousarray(vecs, dtype=np.complex128)
                cnt = None if counts is None else np.ascontiguousarray(counts, dtype=np.int32)
                _lib.check(self.lib.qocb_add_cost(handle, kind, step, float(weight), _lib.ptr(vecs),
                                                  None if cnt is None else cnt.ctypes.data_as(ctypes.c_void_p),
                                                  vecs.shape[1]), handle)

    # -- helpers ------------------------------------------------------------------------------------
    def _real_channels(self, controls):
        if self.KR == 0:
            return None
        controls = np.asarray(controls)
        if controls.shape != (self.M, self.K):
            raise ValueError("controls must have shape {}".format((self.M, self.K)))
        if self.complex_controls:
            return np.ascontiguousarray(np.concatenate([controls.real, controls.imag], axis=1), dtype=np.float64)
        return np.ascontiguousarray(controls, dtype=np.float64)

    def _control_costs(self, controls, want_grad):
        value, grad = 0.0, None
        for c in self.control_costs:
            v, g = c.control_value_and_grad(controls)
            value += v
            if want_grad and g is not None:
                grad = g if grad is None else grad + g
        return value, grad

    def _final_states(self, buf):
        fs = buf.reshape(self.E, self.S, self.n, 1)
        return fs[0] if self.E == 1 else fs

    # -- user-defined costs: value and cotangents by 4-point central differences of `cost(controls, states, step)` ---------
    def _user_value(self, controls, finals):
        return float(sum(np.real(c.cost(controls, finals, self.N - 1)) for c in self.user_costs))

    def _user_seed(self, controls, finals):
        """d c / d Re psi - i d c / d Im psi of the summed user costs at the final states (autograd's cotangent convention)."""
        dre, dim = central_differences(lambda q: self._user_value(controls, q), np.array(finals, dtype=np.complex128))
        return (dre - 1j * dim).reshape(self.S, self.n)

    def _user_control_grad(self, controls, finals):
        """explicit dependence of the user costs on the controls (most have none: one probe decides)."""
        return explicit_control_grad(lambda u: self._user_value(u, finals), controls)

    def _eval_with_user_costs(self, controls, want_grad):
        x = self._real_channels(controls)
        out = np.zeros(1)
        fs = np.empty((self.E, self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_forward(self.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fs)), self.handle)
        finals = self._final_states(fs)
        err = float(out[0]) + self._user_value(controls, finals)
        extra, extra_grad = self._control_costs(np.asarray(controls), want_grad)
        if not want_grad:
            return err + extra, None, finals
        seed = np.ascontiguousarray(self._user_seed(controls, finals))
        g = np.zeros((self.M, self.KR))
        _lib.check(self.lib.qocb_backward(self.handle, _lib.ptr(seed), _lib.ptr(g)), self.handle)
        grads = g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g
        ug = self._user_control_grad(controls, finals)
        if ug is not None:
            grads = grads + ug
        if extra_grad is not None:
            grads = grads + extra_grad
        return err + extra, grads, finals

    # -- the seam ---------------------------------------------------------------------------------------
    def cost(self, controls):
        if self.user_costs:
            err, _, finals = self._eval_with_user_costs(controls, False)
            return err, finals
        x = self._real_channels(controls)
        out = np.zeros(1)
        fs = np.empty((self.E, self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_cost(self.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fs)), self.handle)
        extra, _ = self._control_costs(controls, False) if controls is not None else (0.0, None)
        return float(out[0]) + extra, self._final_states(fs)

    def cost_and_grad(self, controls):
        """returns (error, grads, final_states); grads has controls' shape and dtype and is
        dE/dRe(u) + i dE/dIm(u) for complex controls (the value after the wrapper's conjugate,
        schroedingerdiscrete.py:323-324)."""
        if self.user_costs:
            return self._eval_with_user_costs(controls, True)
        x = self._real_channels(controls)
        out = np.zeros(1)
        g = np.zeros((self.M, self.KR))
        fs = np.empty((self.E, self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_cost_and_grad(self.handle, _lib.ptr(x), _lib.ptr(out), _lib.ptr(g), _lib.ptr(fs)),
                   self.handle)
        grads = g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g
        extra, extra_grad = self._control_costs(np.asarray(controls), True)
        if extra_grad is not None:
            grads = grads + extra_grad
        return float(out[0]) + extra, grads, self._final_states(fs)

    def cost_and_grad_autograd(self, controls):
        """the same (error, grads, finals) through HIPS autograd: the GPU evaluation is registered as an autograd primitive
        with defvjp (`make_autograd_primitive`) and differentiated with the reference's own operator
        (`ans_jacobian`, qoc/core/schroedingerdiscrete.py:318, followed by the conjugate for complex controls, :323-324).
        Used by the `_value_and_jacobian_*` seams whenever `autograd` is importable."""
        from qoc_b200.standard.utils import ans_jacobian, make_autograd_primitive
        prim = getattr(self, "_autograd_primitive", None)
        if prim is None:
            def value_and_grad(c):
                err, g, fin = self.cost_and_grad(c)
                self._autograd_finals = fin
                return err, (np.conjugate(g) if np.iscomplexobj(g) else g)      # autograd convention: d/dx - i d/dy
            prim = self._autograd_primitive = make_autograd_primitive(value_and_grad)
        controls = np.asarray(controls)
        error, jac = ans_jacobian(prim, 0)(controls)
        grads = np.conjugate(jac) if np.iscomplexobj(controls) else jac
        return float(error), grads, self._autograd_finals

    def final_states(self):
        """final states of the last evaluation (also of one enqueued through the device-resident hooks)."""
        fs = np.empty((self.E, self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_get_final_states(self.handle, _lib.ptr(fs)), self.handle)
        return self._final_states(fs)

    def node_grad(self):
        """per-node cotangents of the operator-channel coefficients of the last cost_and_grad: [N-1][q][KC] (member 0)."""
        KC = self.structure[1].shape[0]
        buf = np.zeros((self.N - 1, self._q, KC))
        _lib.check(self.lib.qocb_get_node_grad(self.handle, _lib.ptr(buf)), self.handle)
        return buf

    def intermediate_states(self):
        """[N][S][n][1] states of the last evaluation (member 0 unless E > 1: then [E][N][S][n][1])."""
        buf = np.empty((self.E, self.N, self.S, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_get_states(self.handle, _lib.ptr(buf)), self.handle)
        buf = buf[..., None]
        return buf[0] if self.E == 1 else buf

    def propagators(self):
        buf = np.empty((self.E, self.N - 1, self.n, self.n), dtype=np.complex128)
        _lib.check(self.lib.qocb_get_propagators(self.handle, _lib.ptr(buf)), self.handle)
        return buf[0] if self.E == 1 else buf

    # -- device-resident benchmarking hooks --------------------------------------------------------------
    def upload(self, controls):
        _lib.check(self.lib.qocb_upload_controls(self.handle, _lib.ptr(self._real_channels(controls))), self.handle)

    def time_resident(self, with_grad=True, warmup=3, iters=10, flush_l2=True):
        total = np.zeros(1)
        stages = np.zeros(8)
        _lib.check(self.lib.qocb_time_resident(self.handle, int(with_grad), warmup, iters, int(flush_l2),
                                               _lib.ptr(total), _lib.ptr(stages)), self.handle)
        return float(total[0]), stages

    def launch_count(self, with_grad=True):
        return int(self.lib.qocb_launch_count(self.handle, int(with_grad)))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle:
            self.lib.qocb_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _interp_pair(x, xs):
    """the two control points and weights the reference's linear interpolation uses at time x, including its
    extrapolation rule outside [xs[0], xs[-1]] (qoc/core/mathmethods.py:54-65)."""
    M = len(xs)
    if x <= xs[0]:
        i0, i1 = 0, 1
    elif x >= xs[M - 1]:
        i0, i1 = M - 2, M - 1
    else:
        i1 = int(np.argmax(x <= xs))
        i0 = i1 - 1
    w1 = (x - xs[i0]) / (xs[i1] - xs[i0])
    return i0, i1, 1.0 - w1, w1


class NonlinearSchroedingerPlan(object):
    """`hamiltonian(controls, time)` callables that are NOT affine in the controls (SURVEY.md section 8f N3), e.g.
    H0 + u0^2 X + sin(u1 t) Y.  The reference differentiates through the callable with autograd; here

      * once per plan, the callable is sampled at random controls and node times and H - G0 is expanded over a small real
        operator basis {A_c}, c < 16 (anything that needs more channels raises NotImplementedError);
      * per evaluation the HOST calls the callable at every Magnus node of every slice - exactly where the reference calls it
        (qoc/core/schroedingerdiscrete.py:483-497) - with the linearly interpolated controls, projects H - G0 on the basis
        (residual checked) and uploads the channel coefficients; the same CUDA kernels propagate and differentiate with
        respect to those coefficients (`qocb_set_node_map` with control_count = 0, `qocb_get_node_grad`);
      * the chain rule through the callable uses a NUMERIC Jacobian of the coefficients with respect to (Re u, Im u) at each
        node: 4-point central differences (error O(h^4)), about 1e-11 relative for smooth callables.  Cost and final states
        keep the 1e-10 parity of the affine path; the gradient is as accurate as that Jacobian (tests assert 1e-8).

    The host work is O(nodes * control channels) Python calls per evaluation: a generality path, not a fast one."""

    def __init__(self, hamiltonian, initial_states, costs, evolution_time, system_eval_count, control_eval_count=0,
                 control_count=0, complex_controls=False, magnus_policy=MagnusPolicy.M2, cost_eval_step=1,
                 interpolation_policy=InterpolationPolicy.LINEAR, device=0, store_tape=True, seed=1234, **unused):
        from qoc_b200.models.cost import Cost
        self.hamiltonian = hamiltonian
        self.K, self.M, self.N = int(control_count), int(control_eval_count), int(system_eval_count)
        self.complex_controls = bool(complex_controls)
        self.KR = self.K * (2 if self.complex_controls else 1)
        self.T = float(evolution_time)
        self.q = magnus_policy.order // 2
        nsl = self.N - 1
        dt = self.T / nsl
        self.times = np.array([[(j + c) * dt for c in _NODES[self.q]] for j in range(nsl)])         # [N-1][q]
        xs = np.linspace(0, self.T, self.M)
        self.pairs = [[_interp_pair(t, xs) for t in row] for row in self.times]
        dtype = np.complex128 if self.complex_controls else np.float64
        rng = np.random.default_rng(seed)
        zero = np.zeros(self.K, dtype=dtype)
        self.g0 = np.array(hamiltonian(zero, float(self.times[0, 0])), dtype=np.complex128)
        n = self.g0.shape[0]
        basis = _RealBasis(_MAX_CHANNELS)
        probe_times = list(self.times.ravel()[np.linspace(0, self.times.size - 1, min(12, self.times.size)).astype(int)])
        for t in probe_times:
            basis.add(np.asarray(hamiltonian(zero, float(t)), dtype=np.complex128) - self.g0)
            for trial in range(10):
                u = rng.standard_normal(self.K) * (0.3 + 0.5 * trial)
                if self.complex_controls:
                    u = u + 1j * rng.standard_normal(self.K) * (0.3 + 0.5 * trial)
                basis.add(np.asarray(hamiltonian(u.astype(dtype), float(t)), dtype=np.complex128) - self.g0)
        self.KC = len(basis.vecs)
        if self.KC == 0:
            raise ValueError("the hamiltonian does not depend on controls or time: use a SchroedingerPlan")
        self.basis = np.array(basis.vecs)                                    # [KC][2 n^2] orthonormal over the reals
        self.scale = max(1.0, basis.scale)
        channels = basis.matrices(self.g0.shape)
        offset = np.zeros((nsl, self.q, self.KC))
        gain = np.zeros((nsl, self.q, self.KC, 0))
        for c in costs:
            if (getattr(type(c), "device_terms", Cost.device_terms) is Cost.device_terms and
                    getattr(type(c), "control_value_and_grad", Cost.control_value_and_grad) is Cost.control_value_and_grad):
                raise NotImplementedError("user-defined costs together with a non-linear hamiltonian are not supported")
        self.state_costs = [c for c in costs if getattr(type(c), "control_value_and_grad", Cost.control_value_and_grad)
                            is Cost.control_value_and_grad]
        self.control_costs = [c for c in costs if c not in self.state_costs]
        self.inner = SchroedingerPlan(None, initial_states, self.state_costs, evolution_time, system_eval_count,
                                      control_eval_count=0, control_count=0, complex_controls=False, magnus_policy=magnus_policy,
                                      cost_eval_step=cost_eval_step, interpolation_policy=interpolation_policy, device=device,
                                      store_tape=store_tape, structure=(self.g0, channels, offset, gain))
        self.S, self.n, self.E = self.inner.S, n, 1

    # -- host side of one evaluation ---------------------------------------------------------------------
    def _project(self, h):
        d = h - self.g0
        v = np.concatenate([d.real.ravel(), d.imag.ravel()])
        c = self.basis @ v
        if np.abs(v - c @ self.basis).max() > 1e-9 * self.scale:
            raise RuntimeError("hamiltonian(controls, time) left the operator basis found at plan creation (a term that the "
                               "probing did not excite): not representable on the CUDA path")
        return c

    def _coefficients(self, controls, want_jacobian):
        controls = np.asarray(controls)
        if controls.shape != (self.M, self.K):
            raise ValueError("controls must have shape {}".format((self.M, self.K)))
        nsl = self.N - 1
        coef = np.zeros((nsl, self.q, self.KC))
        jac = np.zeros((nsl, self.q, self.KC, self.KR)) if want_jacobian else None
        dirs = [1.0] * self.K + ([1j] * self.K if self.complex_controls else [])
        for j in range(nsl):
            for i in range(self.q):
                i0, i1, w0, w1 = self.pairs[j][i]
                u = controls[i0] * w0 + controls[i1] * w1
                t = float(self.times[j, i])
                coef[j, i] = self._project(np.asarray(self.hamiltonian(u, t), dtype=np.complex128))
                if not want_jacobian:
                    continue
                for r in range(self.KR):
                    k = r % self.K
                    h = 1e-3 * max(1.0, abs(u[k]))
                    e = np.zeros(self.K, dtype=u.dtype)
                    e[k] = dirs[r]

                    def f(s_, e=e, h=h):
                        return self._project(np.asarray(self.hamiltonian(u + s_ * h * e, t), dtype=np.complex128))
                    jac[j, i, :, r] = (8.0 * (f(1.0) - f(-1.0)) - (f(2.0) - f(-2.0))) / (12.0 * h)
        return coef, jac

    def _upload(self, coef):
        p = self.inner
        off = np.ascontiguousarray(coef, dtype=np.float64)
        _lib.check(p.lib.qocb_set_node_map(p.handle, _lib.ptr(off), None), p.handle)

    _control_costs = SchroedingerPlan._control_costs

    def cost(self, controls):
        coef, _ = self._coefficients(controls, False)
        self._upload(coef)
        err, finals = self.inner.cost(None)
        return err + self._control_costs(np.asarray(controls), False)[0], finals

    def cost_and_grad(self, controls):
        """(error, grads, final_states) as `SchroedingerPlan.cost_and_grad`."""
        controls = np.asarray(controls)
        coef, jac = self._coefficients(controls, True)
        self._upload(coef)
        err, _, finals = self.inner.cost_and_grad(None)
        gc = self.inner.node_grad()                                          # dE / d coef [N-1][q][KC]
        gx = np.zeros((self.M, self.KR))
        for j in range(self.N - 1):
            for i in range(self.q):
                i0, i1, w0, w1 = self.pairs[j][i]
                g = jac[j, i].T @ gc[j, i]
                gx[i0] += w0 * g
                gx[i1] += w1 * g
        grads = gx[:, :self.K] + 1j * gx[:, self.K:] if self.complex_controls else gx
        extra, extra_grad = self._control_costs(controls, True)
        if extra_grad is not None:
            grads = grads + extra_grad
        return err + extra, grads, finals

    cost_and_grad_autograd = SchroedingerPlan.cost_and_grad_autograd

    def intermediate_states(self):
        return self.inner.intermediate_states()

    def launch_count(self, with_grad=True):
        return self.inner.launch_count(with_grad)

    def close(self):
        self.inner.close()


def make_schroedinger_plan(hamiltonian, *args, **kw):
    """`SchroedingerPlan` when the callable is affine in the controls (time-dependent or not), `NonlinearSchroedingerPlan`
    otherwise - what the public programs (`grape_schroedinger_discrete`, `evolve_schroedinger_discrete`) build."""
    try:
        return SchroedingerPlan(hamiltonian, *args, **kw)
    except NonlinearHamiltonian:
        return NonlinearSchroedingerPlan(hamiltonian, *args, **kw)


# --- Lindblad --------------------------------------------------------------------------------------------
def extract_lindblad_structure(lindblad_data, evolution_time):
    """(gammas [L], operators [L x n x n]) of a time-independent `lindblad_data(time)` callable
    (qoc/core/lindbladdiscrete.py:486-492); time-dependent dissipation raises NotImplementedError."""
    if lindblad_data is None:
        return None, None
    g0, o0 = lindblad_data(0.0)
    g1, o1 = lindblad_data(0.37 * evolution_time)
    g0, o0 = np.asarray(g0, dtype=np.float64), np.asarray(o0, dtype=np.complex128)
    if not (np.allclose(g0, np.asarray(g1), rtol=_PROBE_RTOL, atol=0) and
            np.allclose(o0, np.asarray(o1), rtol=_PROBE_RTOL, atol=_PROBE_RTOL)):
        raise NotImplementedError("time-dependent lindblad_data callables are not supported by the CUDA path yet "
                                  "(no CPU fallback)")
    if o0.ndim != 3 or g0.shape[0] != o0.shape[0]:
        raise ValueError("lindblad_data(time) must return (dissipators [L], operators [L x n x n])")
    return np.ascontiguousarray(g0), np.ascontiguousarray(o0)


def _lindblad_is_time_dependent(lindblad_data, evolution_time):
    """True when `lindblad_data(time)` returns different rates, operators or operator counts at the probe times."""
    g0, o0 = lindblad_data(0.0)
    g0, o0 = np.asarray(g0, dtype=np.float64), np.asarray(o0, dtype=np.complex128)
    for t in _probe_times(evolution_time)[1:]:
        g, o = lindblad_data(t)
        g, o = np.asarray(g, dtype=np.float64), np.asarray(o, dtype=np.complex128)
        if g.shape != g0.shape or o.shape != o0.shape:
            return True
        if not (np.allclose(g, g0, rtol=_PROBE_RTOL, atol=0) and np.allclose(o, o0, rtol=_PROBE_RTOL, atol=_PROBE_RTOL)):
            return True
    return False


_SERIES_DEGREE = 24                   # highest Chebyshev degree per segment
_SERIES_RTOL = 1e-13                  # fit check: |reconstructed - callable| <= 1e-13 * scale
_SERIES_MAX_BYTES = 256 << 20         # table size beyond which the fit is refused


def _cheb_coefficients(values):
    """Chebyshev coefficients [.., deg+1, ..] (axis -2) of samples at the first-kind nodes x_k = cos(pi (k+1/2)/(deg+1)),
    constant term not halved: f(x) = sum_j c_j T_j(x)."""
    q = values.shape[-2]
    k = np.arange(q) + 0.5
    cosm = np.cos(np.pi * np.outer(np.arange(q), k) / q) * (2.0 / q)        # [j][k]
    cosm[0] *= 0.5
    return np.einsum("jk,...kc->...jc", cosm, values)


def _cheb_eval(coef, u):
    """Clenshaw for coef [deg+1][cols] at u in [-1, 1] (the same recurrence as the kernels)."""
    b1 = np.zeros(coef.shape[1])
    b2 = np.zeros(coef.shape[1])
    for k in range(coef.shape[0] - 1, 0, -1):
        b1, b2 = coef[k] + 2.0 * u * b1 - b2, b1
    return coef[0] + u * b1 - b2


class LindbladTimeStructure(object):
    """Time dependence of a Lindblad problem as piecewise Chebyshev series (see `extract_lindblad_time_structure`).

    g0 [n x n], channels [KC x n x n], rate_ops [L x n x n] (B_l; None without time-dependent dissipation) and
    series [segments][degree+1][NS] with NS = KC (1 + KR) + L columns [offset_c | gain_cr (c-major) | r_l] on uniform
    segments of width `width` that cover [0, t_max]."""

    def __init__(self, g0, channels, KR, rate_ops, series, width, m):
        self.g0, self.channels, self.KR, self.rate_ops = g0, channels, KR, rate_ops
        self.series, self.width, self.m = np.ascontiguousarray(series), float(width), m
        self.KC = channels.shape[0]
        self.L = 0 if rate_ops is None else rate_ops.shape[0]
        self.segments, self.degree = series.shape[0], series.shape[1] - 1
        self.t_max = self.segments * self.width

    def values(self, t):
        """all NS series at time t (clamped to [0, t_max], as the kernels do)."""
        t = min(max(float(t), 0.0), self.t_max)
        s = min(int(t / self.width), self.segments - 1)
        return _cheb_eval(self.series[s], 2.0 * (t - s * self.width) / self.width - 1.0)

    def coefficients(self, x, t):
        """channel coefficients offset_c(t) + sum_r gain_cr(t) x_r."""
        v = self.values(t)
        off, gain = v[:self.KC], v[self.KC:self.KC * (1 + self.KR)].reshape(self.KC, self.KR)
        return off + (gain @ np.asarray(x, dtype=np.float64) if self.KR else 0.0)

    def hamiltonian(self, x, t):
        """the reconstructed H(x, t) = G0 + sum_c coef_c A_c, x = [Re u, Im u]."""
        return self.g0 + np.tensordot(self.coefficients(x, t), self.channels, axes=(0, 0))

    def rates(self, t):
        return self.values(t)[self.KC * (1 + self.KR):]


def _rate_directions(lindblad_data, times):
    """fixed operator directions B_l (the largest sample of each operator, unit max-norm) of a time-dependent
    `lindblad_data`; raises NotImplementedError when the operator count changes."""
    best = None
    for t in times:
        g, o = lindblad_data(t)
        g, o = np.asarray(g, dtype=np.float64), np.asarray(o, dtype=np.complex128)
        if o.ndim != 3 or g.shape != (o.shape[0],):
            raise ValueError("lindblad_data(time) must return (dissipators [L], operators [L x n x n])")
        if best is None:
            best = o.copy()
        elif o.shape != best.shape:
            raise NotImplementedError("lindblad_data(time) changes its operator count over time; not supported by the CUDA "
                                      "Lindblad path (no CPU fallback)")
        for l in range(o.shape[0]):
            if np.abs(o[l]).max() > np.abs(best[l]).max():
                best[l] = o[l]
    for l in range(best.shape[0]):
        s = np.abs(best[l]).max()
        best[l] = best[l] / s if s > 0 else best[l]
    return best


def _rate_sample(lindblad_data, t, directions):
    """effective rates r_l(t) = gamma_l(t) |f_l(t)|^2 with L_l(t) = f_l(t) B_l; a dissipator that leaves its direction
    raises NotImplementedError."""
    g, o = lindblad_data(t)
    g, o = np.asarray(g, dtype=np.float64), np.asarray(o, dtype=np.complex128)
    if o.shape != directions.shape:
        raise NotImplementedError("lindblad_data(time) changes its operator count over time; not supported by the CUDA "
                                  "Lindblad path (no CPU fallback)")
    r = np.zeros(o.shape[0])
    for l in range(o.shape[0]):
        b = directions[l]
        f = np.vdot(b, o[l]) / max(np.vdot(b, b).real, 1e-300)
        if np.abs(o[l] - f * b).max() > _SERIES_RTOL * max(1.0, np.abs(o[l]).max()):
            raise NotImplementedError("lindblad operator {} changes direction over time (only L_l(t) = f_l(t) B_l with a fixed "
                                      "B_l is supported by the CUDA Lindblad path; no CPU fallback)".format(l))
        r[l] = g[l] * abs(f) ** 2
    return r


def extract_lindblad_time_structure(hamiltonian, control_count, complex_controls, evolution_time, system_eval_count, t_max,
                                    lindblad_data=None, seed=1234, min_m=1):
    """Time dependence of a Lindblad problem for the adaptive-step kernels, which evaluate it at data-dependent stage times.

    `hamiltonian(controls, time)` (time-dependent, affine in x = [Re u, Im u]; or None) becomes
        H(x, t) = G0 + sum_c (offset_c(t) + sum_r gain_cr(t) x_r) A_c
    over a shared real operator basis (`_RealBasis`, at most 16 channels), sampled as `extract_time_dependent_structure`
    does (zero and unit controls); `lindblad_data(time)` (time-dependent; or None) with operators L_l(t) = f_l(t) B_l becomes
    rates r_l(t) = gamma_l(t) |f_l(t)|^2.  Every scalar function is a Chebyshev series of degree <= 24 on uniform segments of
    width dt/m (aligned to the system grid) covering [0, t_max], fitted from samples at each segment's Chebyshev nodes.

    The fit is checked against the callables themselves at a random time in every segment, at the segment end points and at
    the probe times, to 1e-13 x scale; m doubles until it passes.  When it stops converging, or the table would exceed
    256 MB, NotImplementedError is raised: nothing is silently approximated.  Random controls check that the callable is
    affine (NonlinearHamiltonian otherwise).  Returns a `LindbladTimeStructure`."""
    T = float(evolution_time)
    dt = T / (system_eval_count - 1)
    rng = np.random.default_rng(seed)
    zero, units = _unit_controls(control_count, complex_controls) if control_count else (None, [])
    KR = len(units) if hamiltonian is not None else 0
    g0 = None
    if hamiltonian is not None:
        g0 = np.array(hamiltonian(zero, 0.0), dtype=np.complex128)
        if g0.ndim != 2 or g0.shape[0] != g0.shape[1]:
            raise ValueError("hamiltonian(controls, time) must return a square matrix")
    probe = [t for t in _probe_times(T) if t <= t_max]
    directions = None
    if lindblad_data is not None:
        directions = _rate_directions(lindblad_data, probe + list(np.linspace(0.0, t_max, 33)))
    L = 0 if directions is None else directions.shape[0]
    deg = _SERIES_DEGREE
    nodes = (np.cos(np.pi * (np.arange(deg + 1) + 0.5) / (deg + 1)) + 1.0) / 2.0          # on [0, 1] of a segment
    m, last_err = max(1, int(min_m)), None
    while True:
        w = dt / m
        segs = int(np.ceil(t_max / w - 1e-9))
        if segs * (deg + 1) * (KR + 1 + L) * 8 > _SERIES_MAX_BYTES:           # at least one channel or one rate
            raise NotImplementedError("the time dependence needs a Chebyshev table beyond 256 MB to reach 1e-13; not supported "
                                      "by the CUDA Lindblad path (no CPU fallback)")
        times = (np.arange(segs)[:, None] + nodes[None, :]) * w                              # [segs][deg+1]
        basis = _RealBasis(_MAX_CHANNELS, tol=1e-14)
        if hamiltonian is not None:
            pool = []
            for t in list(probe) + list(np.linspace(0.0, t_max, 17)):
                d = np.asarray(hamiltonian(zero, t), dtype=np.complex128)
                pool.append(d - g0)
                pool += [np.asarray(hamiltonian(e, t), dtype=np.complex128) - d for e in units]
            basis.seed(pool)
        rows = []
        for t in times.ravel():
            row = []
            if hamiltonian is not None:
                d = np.asarray(hamiltonian(zero, t), dtype=np.complex128)
                row.append(basis.add(d - g0))
                for e in units:
                    row.append(basis.add(np.asarray(hamiltonian(e, t), dtype=np.complex128) - d))
            rows.append(row)
        KC = len(basis.vecs)
        samples = np.zeros((segs * (deg + 1), KC * (1 + KR) + L))
        for k, row in enumerate(rows):
            if row:
                samples[k, :len(row[0])] = row[0]
                for r in range(KR):
                    samples[k, KC + np.arange(len(row[1 + r])) * KR + r] = row[1 + r]
            if L:
                samples[k, KC * (1 + KR):] = _rate_sample(lindblad_data, float(times.ravel()[k]), directions)
        coef = _cheb_coefficients(samples.reshape(segs, deg + 1, -1))
        # the lowest degree whose dropped tail is below rounding in every column and segment
        amp = (np.abs(coef) / np.maximum(1.0, np.abs(samples).max(axis=0))).max(axis=(0, 2))     # [deg+1]
        tail = np.r_[np.cumsum(amp[::-1])[::-1], 0.0]                                           # tail[j] = sum_{k >= j}
        coef = coef[:, :int(np.argmax(tail[1:] <= 1e-15)) + 1, :]
        if coef.nbytes > _SERIES_MAX_BYTES:
            raise NotImplementedError("the time dependence needs a Chebyshev table beyond 256 MB to reach 1e-13; not supported "
                                      "by the CUDA Lindblad path (no CPU fallback)")
        channels = basis.matrices(g0.shape) if KC else np.zeros((0,) + (g0.shape if g0 is not None else (0, 0)))
        st = LindbladTimeStructure(g0, channels, KR, directions, coef, w, m)
        err = _series_error(st, hamiltonian, zero, units, lindblad_data, probe, rng)
        if err <= _SERIES_RTOL:
            break
        if last_err is not None and m >= 16 and err > 0.25 * last_err:
            raise NotImplementedError("the time dependence is not reproduced by piecewise Chebyshev series (fit error {:.1e} "
                                      "relative at {} segments per system step, not converging): discontinuities inside a "
                                      "segment are not supported by the CUDA Lindblad path (no CPU fallback)".format(err, m))
        last_err, m = err, 2 * m
    _check_affine(st, hamiltonian, control_count, complex_controls, zero, rng)
    return st


def _series_error(st, hamiltonian, zero, units, lindblad_data, probe, rng):
    """largest relative deviation of the fitted series from the callables at off-node check times."""
    times = list((np.arange(st.segments) + rng.uniform(0.0, 1.0, st.segments)) * st.width)
    times += list(np.arange(st.segments + 1) * st.width) + list(probe)
    err = 0.0
    scale = 1.0 if hamiltonian is None else max(1.0, np.abs(st.g0).max(), np.abs(st.channels).max(initial=0.0))
    for t in times:
        t = min(float(t), st.t_max)
        if hamiltonian is not None:
            xs = [np.zeros(st.KR)] + [np.eye(st.KR)[r] for r in range(st.KR)]
            for u, x in zip([zero] + units, xs):
                got = np.asarray(hamiltonian(u, t), dtype=np.complex128)
                err = max(err, np.abs(got - st.hamiltonian(x, t)).max() / max(scale, np.abs(got).max()))
        if st.L:
            want = _rate_sample(lindblad_data, t, st.rate_ops)
            err = max(err, np.abs(want - st.rates(t)).max() / max(1.0, np.abs(want).max()))
    return err


def _check_affine(st, hamiltonian, control_count, complex_controls, zero, rng):
    if hamiltonian is None or not st.KR:
        return
    scale = max(1.0, np.abs(st.g0).max(), np.abs(st.channels).max(initial=0.0))
    for trial in range(4):
        t = float(rng.uniform(0.0, st.t_max))
        u = rng.standard_normal(control_count) * (1.0 + trial)
        if complex_controls:
            u = u + 1j * rng.standard_normal(control_count) * (1.0 + trial)
        x = np.concatenate([u.real, u.imag]) if complex_controls else u
        got = np.asarray(hamiltonian(u.astype(zero.dtype), t), dtype=np.complex128)
        if not np.allclose(got, st.hamiltonian(x, t), rtol=0, atol=_PROBE_RTOL * scale * (1 + np.abs(x).sum())):
            raise NonlinearHamiltonian("hamiltonian(controls, time) is not affine in (Re u, Im u); the CUDA Lindblad path "
                                       "needs that form (no CPU fallback)")


class LindbladPlan(object):
    """Device plan for `_evaluate_lindblad_discrete` and its jacobian (qoc/core/lindbladdiscrete.py:357-441, :322).

    Gradient semantics: the discrete adjoint of the Dormand-Prince map on the realised (accepted) step grid.  The
    reference's autograd tape also differentiates the step-size controller; those terms are rounding noise (see
    oracle/lindblad_adjoint_model.py and DESIGN.md section 5) and are deliberately not reproduced.

    Ensembles (robust control): `ensemble_drifts` [E][n][n] replaces the drift of `hamiltonian` and `ensemble_rates` [E][L]
    the decay rates of `lindblad_data`, member by member.  `cost` and `cost_and_grad` then return the member mean (control
    costs added once) with final densities [E][D][n][n], `intermediate_densities()` is [E][N][D][n][n] and `member_results()`
    returns every member's cost, gradient and stats.  One member is the plain plan."""

    def __init__(self, initial_densities, costs, evolution_time, system_eval_count, hamiltonian=None,
                 lindblad_data=None, control_eval_count=0, control_count=0, complex_controls=False, cost_eval_step=1,
                 interpolation_policy=InterpolationPolicy.LINEAR, device=0, max_rk_steps=0, structure=None,
                 ensemble_drifts=None, ensemble_rates=None):
        if interpolation_policy != InterpolationPolicy.LINEAR:
            raise ValueError("The interpolation policy {} is not implemented for this method."
                             "".format(interpolation_policy))
        self.lib = _lib.load()
        rho0 = np.ascontiguousarray(initial_densities, dtype=np.complex128)
        self.D, self.n = rho0.shape[0], rho0.shape[1]
        self.K, self.M, self.N = int(control_count), int(control_eval_count), int(system_eval_count)
        self.complex_controls = bool(complex_controls)
        self.have_h = hamiltonian is not None
        self.KR = self.K * (2 if self.complex_controls else 1) if self.have_h else 0
        self.costs = list(costs)
        self.T, self.dt = float(evolution_time), float(evolution_time) / (self.N - 1)
        # time dependence (hamiltonian reading `time`, lindblad_data varying with time): Chebyshev series evaluated on the
        # device at the stage times; a time-independent problem keeps the constant operators below and no series
        td_h = td_l = False
        if self.have_h and structure is None:
            zero, units = _unit_controls(self.K, self.complex_controls) if self.K else (None, [])
            td_h = _is_time_dependent(hamiltonian, zero, units, evolution_time)
        if lindblad_data is not None:
            td_l = _lindblad_is_time_dependent(lindblad_data, evolution_time)
        h0 = a_ops = gammas = lops = None
        if self.have_h and not td_h:
            if structure is None:
                structure = extract_hamiltonian_structure(hamiltonian, self.K, self.complex_controls, evolution_time)
            h0, a_ops = structure
        if not td_l:
            gammas, lops = extract_lindblad_structure(lindblad_data, evolution_time)
        self._td = (hamiltonian if td_h else None, lindblad_data if td_l else None)
        self.series = None
        if td_h or td_l:
            self.series = extract_lindblad_time_structure(self._td[0], self.K, self.complex_controls, evolution_time, self.N,
                                                          self.T + self.dt, lindblad_data=self._td[1])
            if td_h:
                h0, a_ops = self.series.g0, self.series.channels
            if td_l:
                lops = self.series.rate_ops
        if h0 is not None and h0.shape[0] != self.n:
            raise ValueError("hamiltonian size {} does not match the densities' hilbert size {}".format(h0.shape[0], self.n))
        self.L = 0 if lops is None else lops.shape[0]
        h0s, rates = self._ensemble_members(ensemble_drifts, ensemble_rates, td_h, td_l)
        self.E = 1 if h0s is None and rates is None else (h0s if h0s is not None else rates).shape[0]
        if self.E == 1:                                  # one member: the plain plan with that member's drift and rates
            h0 = h0 if h0s is None else h0s[0]
            gammas = gammas if rates is None else rates[0]
            h0s = rates = None
        self._members = (h0s, rates)
        self._last_extra = (0.0, None)
        self.range_extensions = 0
        self._setup = dict(rho0=rho0, h0=h0, a_ops=a_ops, gammas=gammas, lops=lops, cost_eval_step=int(cost_eval_step),
                           device=int(device), max_rk_steps=int(max_rk_steps))
        self.handle = None
        self._open()
        self.control_costs = []
        self.user_costs = []
        self._terms = []
        from qoc_b200.models.cost import Cost
        for c in self.costs:
            if is_user_cost(c):
                self.user_costs.append(c)
                continue
            terms = c.device_terms_density(self.D, self.n) if hasattr(c, "device_terms_density") else None
            if not terms:
                # only genuine control-only costs (classes that override the analytic hook) may skip the device: a state
                # cost passed by mistake must not be dropped silently
                hook = getattr(type(c), "control_value_and_grad", None)
                if terms is None or hook is None or hook is Cost.control_value_and_grad:
                    raise NotImplementedError("The cost {} has no B200 device descriptor for the Lindblad path (no CPU "
                                              "fallback): density costs need `device_terms_density`, control-only costs "
                                              "`control_value_and_grad`.".format(c))
                self.control_costs.append(c)
            for kind, step, weight, mats, counts in terms:
                term = (kind, step, float(weight), np.ascontiguousarray(mats, dtype=np.complex128),
                        None if counts is None else np.ascontiguousarray(counts, dtype=np.int32))
                self._terms.append(term)
                self._add_term(term)
        # user costs by system step, where the reference evaluates them (lindbladdiscrete.py:384-441): step costs at every
        # k % cost_eval_step == 0, k != 0, the others once on the final densities
        ces = int(cost_eval_step)
        self._user_at = {}
        for c in self.user_costs:
            for k in (range(ces, self.N, ces) if getattr(c, "requires_step_evaluation", False) else (self.N - 1,)):
                self._user_at.setdefault(k, []).append(c)

    def _ensemble_members(self, drifts, rates, td_h, td_l):
        """validated member drifts [E][n][n] and rates [E][L] (either may be None); raises before any device call."""
        if drifts is None and rates is None:
            return None, None
        if any(is_user_cost(c) for c in self.costs):
            raise NotImplementedError("user-defined costs cannot be combined with ensembles")
        if drifts is not None:
            if not self.have_h:
                raise ValueError("ensemble_drifts replace the drift of `hamiltonian`, which is None")
            if td_h:
                raise NotImplementedError("ensemble drifts with a time-dependent hamiltonian are not supported")
            drifts = np.ascontiguousarray(drifts, dtype=np.complex128)
            if drifts.ndim != 3 or drifts.shape[0] < 1 or drifts.shape[1:] != (self.n, self.n):
                raise ValueError("ensemble_drifts must have shape [E][{0}][{0}], got {1}".format(self.n, drifts.shape))
        if rates is not None:
            if self.L == 0:
                raise ValueError("ensemble_rates replace the rates of `lindblad_data`, which has no operators")
            if td_l:
                raise NotImplementedError("ensemble rates with a time-dependent lindblad_data are not supported")
            if np.iscomplexobj(rates):
                raise ValueError("ensemble_rates must be real")
            rates = np.ascontiguousarray(rates, dtype=np.float64)
            if rates.ndim != 2 or rates.shape[0] < 1 or rates.shape[1] != self.L:
                raise ValueError("ensemble_rates must have shape [E][{}], got {}".format(self.L, rates.shape))
        if drifts is not None and rates is not None and drifts.shape[0] != rates.shape[0]:
            raise ValueError("ensemble_drifts has {} members and ensemble_rates {}".format(drifts.shape[0], rates.shape[0]))
        return drifts, rates

    def _open(self):
        """creates the device plan and uploads operators, densities, the ensemble members and (time-dependent problems) the
        series table."""
        su, st = self._setup, self.series
        KC = st.KC if st is not None and self._td[0] is not None else 0
        tdr = int(st is not None and self._td[1] is not None)
        pb = _lib.LindbladProblem(hilbert_size=self.n, density_count=self.D, control_count=self.KR,
                                  control_eval_count=self.M if self.KR else 0, system_eval_count=self.N,
                                  cost_eval_step=su["cost_eval_step"], lindblad_count=self.L,
                                  have_hamiltonian=int(self.have_h), device=su["device"], max_rk_steps=su["max_rk_steps"],
                                  channel_count=KC, time_dependent_rates=tdr,
                                  ensemble_count=self.E if self.E > 1 else 0, evolution_time=self.T)
        handle = ctypes.c_void_p()
        rc = self.lib.qocb_lindblad_create(ctypes.byref(pb), ctypes.byref(handle))
        if rc != 0:
            raise RuntimeError("qoc_b200 CUDA Lindblad path failed (rc={}): {}".format(
                rc, self.lib.qocb_lindblad_last_error(None).decode()))
        self.handle = handle
        h0c = None if su["h0"] is None else np.ascontiguousarray(su["h0"], dtype=np.complex128)
        a_ops = su["a_ops"]
        aoc = None if a_ops is None or a_ops.shape[0] == 0 else np.ascontiguousarray(a_ops, dtype=np.complex128)
        lops = None if su["lops"] is None else np.ascontiguousarray(su["lops"], dtype=np.complex128)
        self._check(self.lib.qocb_lindblad_set_operators(handle, _lib.ptr(h0c), _lib.ptr(aoc), _lib.ptr(su["gammas"]),
                                                         _lib.ptr(lops)))
        if self.E > 1:
            self._check(self.lib.qocb_lindblad_set_ensemble(handle, _lib.ptr(self._members[0]), _lib.ptr(self._members[1])))
        self._check(self.lib.qocb_lindblad_set_densities(handle, _lib.ptr(su["rho0"])))
        if st is not None:
            self._check(self.lib.qocb_lindblad_set_time_series(handle, st.segments, st.degree, st.width, _lib.ptr(st.series)))

    def _add_term(self, term):
        kind, step, weight, mats, cnt = term
        self._check(self.lib.qocb_lindblad_add_cost(self.handle, kind, step, weight, _lib.ptr(mats),
                                                    None if cnt is None else cnt.ctypes.data_as(ctypes.c_void_p),
                                                    mats.shape[1]))

    _MAX_RANGE_EXTENSIONS = 4

    def _evaluate(self, call):
        """runs `call(handle)`; when a stage time left the series table (rc -5), refits the table to cover it with a margin
        (same segment width, so the covered range keeps its values), rebuilds the plan and evaluates again."""
        for _ in range(self._MAX_RANGE_EXTENSIONS + 1):
            rc = call(self.handle)
            if rc != -5 or self.series is None:
                return self._check(rc)
            tseen = np.zeros(1)
            self._check(self.lib.qocb_lindblad_max_stage_time(self.handle, _lib.ptr(tseen)))
            t_max = float(tseen[0]) + self.dt + 0.25 * max(0.0, float(tseen[0]) - self.T)
            self.series = extract_lindblad_time_structure(self._td[0], self.K, self.complex_controls, self.T, self.N, t_max,
                                                          lindblad_data=self._td[1], min_m=self.series.m)
            if self._td[0] is not None:
                self._setup.update(h0=self.series.g0, a_ops=self.series.channels)
            if self._td[1] is not None:
                self._setup.update(lops=self.series.rate_ops)
            self.close()
            self._open()
            for term in self._terms:
                self._add_term(term)
            self.range_extensions += 1
        raise RuntimeError("qoc_b200 CUDA Lindblad path: the Runge-Kutta stage times kept leaving the time series after {} "
                           "extensions".format(self._MAX_RANGE_EXTENSIONS))

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.qocb_lindblad_last_error(self.handle)
            raise RuntimeError("qoc_b200 CUDA Lindblad path failed (rc={}): {}".format(rc, msg.decode() if msg else "?"))

    _real_channels = SchroedingerPlan._real_channels
    _control_costs = SchroedingerPlan._control_costs
    cost_and_grad_autograd = SchroedingerPlan.cost_and_grad_autograd

    # -- user-defined costs: value and density cotangents by 4-point central differences of `cost(controls, densities, step)`
    def _user_value_at(self, controls, rho, k):
        return float(sum(np.real(c.cost(controls, rho, k)) for c in self._user_at[k]))

    def _user_densities(self, final_densities):
        """{step: densities of the last evaluation} for the steps that carry user costs."""
        if list(self._user_at) == [self.N - 1]:
            return {self.N - 1: final_densities}
        dens = self.intermediate_densities()
        return {k: dens[k] for k in self._user_at}

    def _user_value(self, controls, dens):
        return sum(self._user_value_at(controls, dens[k], k) for k in sorted(dens))

    def _user_seeds(self, controls, dens):
        """[N][D][n][n] seed table of qocb_lindblad_backward: row k = d c / d Re rho_k - i d c / d Im rho_k of the user
        costs evaluated at step k (each density entry differentiated on its own), zero elsewhere."""
        seeds = np.zeros((self.N, self.D, self.n, self.n), dtype=np.complex128)
        for k, rho in dens.items():
            dre, dim = central_differences(lambda r: self._user_value_at(controls, r, k), rho)
            seeds[k] = dre - 1j * dim
        return seeds

    def _final_buffer(self):
        shape = (self.D, self.n, self.n) if self.E == 1 else (self.E, self.D, self.n, self.n)
        return np.empty(shape, dtype=np.complex128)

    def cost(self, controls):
        x = self._real_channels(controls) if controls is not None else None
        out = np.zeros(1)
        fd = self._final_buffer()
        self._evaluate(lambda h: self.lib.qocb_lindblad_cost(h, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)))
        value = float(out[0])
        if self.user_costs:
            value += self._user_value(controls, self._user_densities(fd))
        extra, _ = self._control_costs(controls, False) if controls is not None else (0.0, None)
        self._last_extra = (extra, None)
        return value + extra, fd

    def cost_and_grad(self, controls):
        """(error, grads, final_densities); grads = dE/dRe(u) + i dE/dIm(u) for complex controls.  With user costs the
        forward pass keeps its tape, the host evaluates the user costs on the densities, and the reverse pass is seeded with
        their numeric cotangents (qocb_lindblad_forward / qocb_lindblad_backward)."""
        x = self._real_channels(controls)
        out = np.zeros(1)
        fd = self._final_buffer()
        controls = np.asarray(controls)
        g = np.zeros((self.M, self.KR))
        if self.KR == 0:                                   # hamiltonian = None: the densities do not see the controls
            self._evaluate(lambda h: self.lib.qocb_lindblad_cost(h, None, _lib.ptr(out), _lib.ptr(fd)))
        elif self.user_costs:
            self._evaluate(lambda h: self.lib.qocb_lindblad_forward(h, _lib.ptr(x), _lib.ptr(out), _lib.ptr(fd)))
        else:
            self._evaluate(lambda h: self.lib.qocb_lindblad_cost_and_grad(h, _lib.ptr(x), _lib.ptr(out), _lib.ptr(g), _lib.ptr(fd)))
        value, user_grad = float(out[0]), None
        if self.user_costs:
            dens = self._user_densities(fd)
            value += self._user_value(controls, dens)
            if self.KR:
                seeds = self._user_seeds(controls, dens)
                self._check(self.lib.qocb_lindblad_backward(self.handle, _lib.ptr(seeds), _lib.ptr(g)))
            if controls.ndim:
                user_grad = explicit_control_grad(lambda u: self._user_value(u, dens), controls)
        grads = self._controls_grad(g, controls)
        if user_grad is not None:
            grads = grads + user_grad
        extra, extra_grad = self._control_costs(controls, True)
        self._last_extra = (extra, (controls.shape, controls.dtype, extra_grad))
        if extra_grad is not None:
            grads = grads + extra_grad
        return value + extra, grads, fd

    def _controls_grad(self, g, controls):
        """dE/dRe u + i dE/dIm u in the controls' shape from the device gradient [M][KR]."""
        if self.KR == 0:
            return np.zeros(controls.shape, dtype=controls.dtype)
        return g[:, :self.K] + 1j * g[:, self.K:] if self.complex_controls else g

    def member_results(self):
        """every member's (cost, gradient, stats) of the last evaluation: costs [E], gradients [E] in the controls' shape and
        dtype (None after `cost`), stats [E] as {"attempts", "accepted"}; the control costs are included in each member's
        cost and gradient, so member e equals a one-member plan built with its drift and rates (and the same control
        operators)."""
        costs = np.zeros(self.E)
        g = np.zeros((self.E, self.M, self.KR))
        st = np.zeros((self.E, 2), dtype=np.int64)
        self._check(self.lib.qocb_lindblad_member_results(self.handle, _lib.ptr(costs), _lib.ptr(g),
                                                          st.ctypes.data_as(ctypes.c_void_p)))
        extra, grad_info = self._last_extra
        costs = costs + extra
        grads = None
        if grad_info is not None:
            shape, dtype, extra_grad = grad_info
            zero = np.zeros(shape, dtype=dtype)
            grads = []
            for e in range(self.E):
                ge = self._controls_grad(g[e], zero)
                grads.append(ge + extra_grad if extra_grad is not None else ge)
            grads = np.array(grads)
        return costs, grads, [{"attempts": int(a), "accepted": int(b)} for a, b in st]

    def stats(self):
        s = np.zeros(2, dtype=np.int64)
        self._check(self.lib.qocb_lindblad_stats(self.handle, s.ctypes.data_as(ctypes.c_void_p)))
        return {"attempts": int(s[0]), "accepted": int(s[1])}

    def intermediate_densities(self):
        shape = (self.N, self.D, self.n, self.n)
        buf = np.empty(shape if self.E == 1 else (self.E,) + shape, dtype=np.complex128)
        self._check(self.lib.qocb_lindblad_get_densities(self.handle, _lib.ptr(buf)))
        return buf

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle:
            self.lib.qocb_lindblad_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
