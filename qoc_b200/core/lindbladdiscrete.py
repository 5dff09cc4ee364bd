"""
lindbladdiscrete.py - `evolve_lindblad_discrete` and `grape_lindblad_discrete` with the reference's signatures
(qoc/core/lindbladdiscrete.py:31-40, :110-127).  Host-side wrappers follow `_eld_wrap` (:261-294) and `_eldj_wrap`
(:297-354); the evaluation inside them - the interval loop of `_evaluate_lindblad_discrete` (:357-441) with its
adaptive RKDP5 integration and the reverse pass - runs on the GPU through `LindbladPlan`.
"""
import numpy as np

from qoc_b200.core.common import (batch_initial_controls, clip_control_norms, grape_lockstep, initialize_controls,
                                  slap_controls, strip_controls)
from qoc_b200.core.plan import LindbladPlan
from qoc_b200.models import (Dummy, EvolveLindbladDiscreteState, EvolveLindbladResult, GrapeLindbladDiscreteState,
                             GrapeLindbladResult, InterpolationPolicy, ProgramType)
from qoc_b200.standard.optimizers import Adam
from qoc_b200.standard.utils import autograd_available


def _plan_for(pstate, control_count, complex_controls, device=0):
    plan = getattr(pstate, "_b200_plan", None)
    if plan is None:
        plan = LindbladPlan(pstate.initial_densities, pstate.costs, pstate.evolution_time, pstate.system_eval_count,
                            hamiltonian=pstate.hamiltonian, lindblad_data=pstate.lindblad_data,
                            control_eval_count=pstate.control_eval_count, control_count=control_count,
                            complex_controls=complex_controls, cost_eval_step=pstate.cost_eval_step,
                            interpolation_policy=pstate.interpolation_policy, device=device)
        pstate._b200_plan = plan
    return plan


def evolve_lindblad_discrete(evolution_time, initial_densities, system_eval_count, controls=None, cost_eval_step=1,
                             costs=list(), hamiltonian=None, interpolation_policy=InterpolationPolicy.LINEAR,
                             lindblad_data=None, save_file_path=None, save_intermediate_densities=False):
    """
    Evolve a set of density matrices under the lindblad equation and compute the optimization error.
    Arguments and result as in the reference (qoc/core/lindbladdiscrete.py:41-107).

    Returns:
    result :: EvolveLindbladResult (fields `error`, `final_densities`)
    """
    control_eval_count = controls.shape[0] if controls is not None else 0
    pstate = EvolveLindbladDiscreteState(control_eval_count, cost_eval_step, costs, evolution_time, hamiltonian,
                                         initial_densities, interpolation_policy, lindblad_data, save_file_path,
                                         save_intermediate_densities, system_eval_count)
    pstate.save_initial(controls)
    pstate._control_count = controls.shape[1] if controls is not None else 0
    pstate._complex_controls = bool(controls is not None and np.iscomplexobj(controls))
    result = EvolveLindbladResult()
    _evaluate_lindblad_discrete(controls, pstate, result)
    pstate._b200_plan.close()
    return result


def grape_lindblad_discrete(control_count, control_eval_count, costs, evolution_time, initial_densities,
                            system_eval_count, complex_controls=False, cost_eval_step=1, hamiltonian=None,
                            impose_control_conditions=None, initial_controls=None,
                            interpolation_policy=InterpolationPolicy.LINEAR, iteration_count=1000,
                            lindblad_data=None, log_iteration_step=10, max_control_norms=None, min_error=0,
                            optimizer=Adam(), save_file_path=None, save_intermediate_densities=False,
                            save_iteration_step=0):
    """
    Optimize the evolution of a set of density matrices under the lindblad equation for time-discrete control
    parameters.  Arguments and result as in the reference (qoc/core/lindbladdiscrete.py:128-256).

    Returns:
    result :: GrapeLindbladResult (best_controls, best_error, best_final_densities, best_iteration)
    """
    initial_controls, max_control_norms = initialize_controls(complex_controls, control_count, control_eval_count,
                                                              evolution_time, initial_controls, max_control_norms)
    pstate = GrapeLindbladDiscreteState(complex_controls, control_count, control_eval_count, cost_eval_step, costs,
                                        evolution_time, hamiltonian, impose_control_conditions, initial_controls,
                                        initial_densities, interpolation_policy, iteration_count, lindblad_data,
                                        log_iteration_step, max_control_norms, min_error, optimizer, save_file_path,
                                        save_intermediate_densities, save_iteration_step, system_eval_count)
    pstate.log_and_save_initial()
    reporter = Dummy()
    reporter.iteration = 0
    result = GrapeLindbladResult()
    x0 = strip_controls(pstate.complex_controls, pstate.initial_controls)
    try:
        pstate.optimizer.run(_eld_wrap, pstate.iteration_count, x0, _eldj_wrap, args=(pstate, reporter, result))
    finally:
        plan = getattr(pstate, "_b200_plan", None)
        if plan is not None:
            plan.close()
    return result


def grape_lindblad_discrete_batch(control_count, control_eval_count, costs, evolution_time, initial_densities,
                                  system_eval_count, initial_controls, complex_controls=False, cost_eval_step=1,
                                  hamiltonian=None, impose_control_conditions=None,
                                  interpolation_policy=InterpolationPolicy.LINEAR, iteration_count=1000, lindblad_data=None,
                                  log_iteration_step=10, max_control_norms=None, min_error=0, optimizer=Adam(),
                                  save_file_path=None):
    """
    Multi-start GRAPE on the Lindblad path: B optimisations of one problem from the initial pulses `initial_controls`
    [B][M][K], run in lockstep with one batched GPU evaluation (`LindbladPlan(control_batch=B)`, one CTA per start) per
    iteration.  Every other argument means what it means for `grape_lindblad_discrete`, and start b follows the trajectory
    that `grape_lindblad_discrete(..., initial_controls=initial_controls[b])` would: its controls are clipped in place to
    `max_control_norms` and passed through `impose_control_conditions` ([M][K] per call) before each evaluation, and its
    optimiser state is its own.  A start whose error reaches `min_error` stops updating and keeps its best result.  Adam and
    SGD are supported; L-BFGS-B, whose line search would couple the starts, and `save_file_path` raise NotImplementedError.

    Returns:
    results :: list of B GrapeLindbladResult (best_controls, best_error, best_final_densities, best_iteration)
    """
    controls0, max_control_norms = batch_initial_controls(
        "grape_lindblad_discrete_batch", complex_controls, control_count, control_eval_count, evolution_time,
        initial_controls, max_control_norms, optimizer, save_file_path)
    plan = LindbladPlan(initial_densities, costs, evolution_time, system_eval_count, hamiltonian=hamiltonian,
                        lindblad_data=lindblad_data, control_eval_count=control_eval_count, control_count=control_count,
                        complex_controls=complex_controls, cost_eval_step=cost_eval_step,
                        interpolation_policy=interpolation_policy, control_batch=controls0.shape[0])
    try:
        return grape_lockstep(plan.cost_and_grad, controls0, complex_controls, max_control_norms, impose_control_conditions,
                              iteration_count, log_iteration_step, min_error, optimizer, GrapeLindbladResult,
                              "best_final_densities")
    finally:
        plan.close()


def _prepare_controls(params, pstate):
    controls = slap_controls(pstate.complex_controls, params, pstate.controls_shape)
    clip_control_norms(controls, pstate.max_control_norms)
    if pstate.impose_control_conditions is not None:
        controls = pstate.impose_control_conditions(controls)
    return controls


def _eld_wrap(params, pstate, reporter, result):
    """`function` callback of the optimiser: (error, terminate)."""
    controls = _prepare_controls(params, pstate)
    error = _evaluate_lindblad_discrete(controls, pstate, reporter)
    return error, bool(error <= pstate.min_error)


def _eldj_wrap(params, pstate, reporter, result):
    """`jacobian` callback of the optimiser: (flat float64 grads, terminate) with the reference's side effects in
    the reference's order (best-so-far update, log/save, iteration counter)."""
    controls = _prepare_controls(params, pstate)
    error, grads = _value_and_jacobian_lindblad_discrete(controls, pstate, reporter)
    final_densities = reporter.final_densities
    if error < result.best_error:
        result.best_controls = controls
        result.best_error = error
        result.best_final_densities = final_densities
        result.best_iteration = reporter.iteration
    pstate.log_and_save(controls, error, final_densities, grads, reporter.iteration)
    reporter.iteration += 1
    return strip_controls(pstate.complex_controls, grads), bool(error <= pstate.min_error)


def _program_controls_meta(pstate):
    if pstate.program_type == ProgramType.GRAPE:
        return pstate.control_count, pstate.complex_controls
    return pstate._control_count, pstate._complex_controls


def _evaluate_lindblad_discrete(controls, pstate, reporter):
    """total cost of one evolution on the GPU; fills reporter.error / reporter.final_densities
    (qoc/core/lindbladdiscrete.py:357-441)."""
    control_count, complex_controls = _program_controls_meta(pstate)
    plan = _plan_for(pstate, control_count, complex_controls)
    error, final_densities = plan.cost(controls)
    _maybe_save_densities(pstate, reporter, plan)
    reporter.error = error
    reporter.final_densities = final_densities
    return error


def _value_and_jacobian_lindblad_discrete(controls, pstate, reporter):
    """(error, grads) of `ans_jacobian(_evaluate_lindblad_discrete, 0)` followed by the conjugate for complex
    controls (lindbladdiscrete.py:322-328): grads = dE/dRe(u) + i dE/dIm(u)."""
    control_count, complex_controls = _program_controls_meta(pstate)
    plan = _plan_for(pstate, control_count, complex_controls)
    # with HIPS autograd installed the GPU evaluation runs as an autograd primitive (defvjp) under the reference's own
    # ans_jacobian; without it the C ABI's value-and-gradient entry point is called directly (same numbers)
    evaluate = plan.cost_and_grad_autograd if (autograd_available() and plan.KR > 0) else plan.cost_and_grad
    error, grads, final_densities = evaluate(controls)
    _maybe_save_densities(pstate, reporter, plan)
    reporter.error = error
    reporter.final_densities = final_densities
    return error, grads


def _maybe_save_densities(pstate, reporter, plan):
    """the reference writes the densities of every system step from inside its interval loop
    (qoc/core/lindbladdiscrete.py:398-405, qoc/models/lindbladmodels.py:92-99, :315-334); the device keeps them all, so
    one D2H after the evaluation fills the same dataset."""
    if pstate.save_intermediate_densities_:
        iteration = reporter.iteration if pstate.program_type == ProgramType.GRAPE else 0
        pstate.save_all_intermediate_densities(iteration, plan.intermediate_densities())
