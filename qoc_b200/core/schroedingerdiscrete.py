"""
schroedingerdiscrete.py - `evolve_schroedinger_discrete` and `grape_schroedinger_discrete` with the reference's
signatures (qoc/core/schroedingerdiscrete.py:28-35, :106-122).  The optimiser protocol, control
transformations, best-so-far bookkeeping and logging stay on the host and follow the reference wrappers
(`_esd_wrap` :257-290, `_esdj_wrap` :293-353); the evaluation inside them - the time loop of
`_evaluate_schroedinger_discrete` (:356-438) and its reverse pass (`ans_jacobian`, :318) - runs on the GPU
through `SchroedingerPlan`.
"""
import numpy as np

from qoc_b200.core.common import (_adam_rows, batch_initial_controls, clip_control_norms, grape_lockstep,  # noqa: F401
                                  initialize_controls, slap_controls, strip_controls)
from qoc_b200.core.plan import SchroedingerPlan, make_schroedinger_plan
from qoc_b200.models import (Dummy, EvolveSchroedingerDiscreteState, EvolveSchroedingerResult,
                             GrapeSchroedingerDiscreteState, GrapeSchroedingerResult, InterpolationPolicy,
                             MagnusPolicy, ProgramType)
from qoc_b200.standard.optimizers import Adam
from qoc_b200.standard.utils import autograd_available


def _plan_for(pstate, control_count, complex_controls, device=0, store_tape=True):
    plan = getattr(pstate, "_b200_plan", None)
    if plan is None:
        plan = make_schroedinger_plan(pstate.hamiltonian, pstate.initial_states, pstate.costs, pstate.evolution_time,
                                pstate.system_eval_count, control_eval_count=pstate.control_eval_count,
                                control_count=control_count, complex_controls=complex_controls,
                                magnus_policy=pstate.magnus_policy, cost_eval_step=pstate.cost_eval_step,
                                interpolation_policy=pstate.interpolation_policy, device=device,
                                store_tape=store_tape)
        pstate._b200_plan = plan
    return plan


def evolve_schroedinger_discrete(evolution_time, hamiltonian, initial_states, system_eval_count,
                                 controls=None, cost_eval_step=1, costs=list(),
                                 interpolation_policy=InterpolationPolicy.LINEAR,
                                 magnus_policy=MagnusPolicy.M2, save_file_path=None,
                                 save_intermediate_states=False):
    """
    Evolve a set of state vectors under the schroedinger equation and compute the optimization error.
    Arguments and result as in the reference (qoc/core/schroedingerdiscrete.py:36-103).

    Returns:
    result :: EvolveSchroedingerResult (fields `error`, `final_states`)
    """
    control_eval_count = controls.shape[0] if controls is not None else 0
    pstate = EvolveSchroedingerDiscreteState(control_eval_count, cost_eval_step, costs, evolution_time,
                                             hamiltonian, initial_states, interpolation_policy, magnus_policy,
                                             save_file_path, save_intermediate_states, system_eval_count)
    pstate.save_initial(controls)
    pstate._control_count = controls.shape[1] if controls is not None else 0
    pstate._complex_controls = bool(controls is not None and np.iscomplexobj(controls))
    result = EvolveSchroedingerResult()
    _evaluate_schroedinger_discrete(controls, pstate, result)
    pstate._b200_plan.close()
    return result


# the north-star text calls the forward program `evaluate_schroedinger_discrete`; the reference's public name is
# `evolve_schroedinger_discrete`.  Both are exported.
evaluate_schroedinger_discrete = evolve_schroedinger_discrete


def grape_schroedinger_discrete(control_count, control_eval_count, costs, evolution_time, hamiltonian,
                                initial_states, system_eval_count, complex_controls=False, cost_eval_step=1,
                                impose_control_conditions=None, initial_controls=None,
                                interpolation_policy=InterpolationPolicy.LINEAR, iteration_count=1000,
                                log_iteration_step=10, magnus_policy=MagnusPolicy.M2, max_control_norms=None,
                                min_error=0, optimizer=Adam(), save_file_path=None,
                                save_intermediate_states=False, save_iteration_step=0):
    """
    Optimize the evolution of a set of states under the schroedinger equation for time-discrete control
    parameters.  Arguments and result as in the reference (qoc/core/schroedingerdiscrete.py:123-252).

    Returns:
    result :: GrapeSchroedingerResult (best_controls, best_error, best_final_states, best_iteration)
    """
    initial_controls, max_control_norms = initialize_controls(complex_controls, control_count,
                                                              control_eval_count, evolution_time,
                                                              initial_controls, max_control_norms)
    pstate = GrapeSchroedingerDiscreteState(complex_controls, control_count, control_eval_count, cost_eval_step,
                                            costs, evolution_time, hamiltonian, impose_control_conditions,
                                            initial_controls, initial_states, interpolation_policy,
                                            iteration_count, log_iteration_step, max_control_norms,
                                            magnus_policy, min_error, optimizer, save_file_path,
                                            save_intermediate_states, save_iteration_step, system_eval_count)
    pstate.log_and_save_initial()
    reporter = Dummy()
    reporter.iteration = 0
    result = GrapeSchroedingerResult()
    x0 = strip_controls(pstate.complex_controls, pstate.initial_controls)
    try:
        pstate.optimizer.run(_esd_wrap, pstate.iteration_count, x0, _esdj_wrap,
                             args=(pstate, reporter, result))
    finally:
        plan = getattr(pstate, "_b200_plan", None)
        if plan is not None:
            plan.close()
    return result


def grape_schroedinger_discrete_batch(control_count, control_eval_count, costs, evolution_time, hamiltonian,
                                      initial_states, system_eval_count, initial_controls, complex_controls=False,
                                      cost_eval_step=1, impose_control_conditions=None,
                                      interpolation_policy=InterpolationPolicy.LINEAR, iteration_count=1000,
                                      log_iteration_step=10, magnus_policy=MagnusPolicy.M2, max_control_norms=None,
                                      min_error=0, optimizer=Adam(), save_file_path=None):
    """
    Multi-start GRAPE: B optimisations of one problem from the initial pulses `initial_controls` [B][M][K], run in
    lockstep with one batched GPU evaluation (`SchroedingerPlan(control_batch=B)`) per iteration.  Every other argument
    means what it means for `grape_schroedinger_discrete`, and start b follows the trajectory that
    `grape_schroedinger_discrete(..., initial_controls=initial_controls[b])` would: its controls are clipped in place to
    `max_control_norms` and passed through `impose_control_conditions` ([M][K] per call) before each evaluation, and its
    optimiser state (Adam moments and step count, gradient scaling and clipping) is its own.  A start whose error reaches
    `min_error` stops updating and keeps its best result; the run ends when every start has stopped or after
    `iteration_count` iterations.  Adam and SGD are supported; L-BFGS-B, whose line search would couple the starts, and
    `save_file_path` raise NotImplementedError.

    Returns:
    results :: list of B GrapeSchroedingerResult (best_controls, best_error, best_final_states, best_iteration)
    """
    controls0, max_control_norms = batch_initial_controls(
        "grape_schroedinger_discrete_batch", complex_controls, control_count, control_eval_count, evolution_time,
        initial_controls, max_control_norms, optimizer, save_file_path)
    plan = SchroedingerPlan(hamiltonian, initial_states, costs, evolution_time, system_eval_count,
                            control_eval_count=control_eval_count, control_count=control_count,
                            complex_controls=complex_controls, magnus_policy=magnus_policy, cost_eval_step=cost_eval_step,
                            interpolation_policy=interpolation_policy, control_batch=controls0.shape[0])
    try:
        return grape_lockstep(plan.cost_and_grad, controls0, complex_controls, max_control_norms, impose_control_conditions,
                              iteration_count, log_iteration_step, min_error, optimizer, GrapeSchroedingerResult,
                              "best_final_states")
    finally:
        plan.close()


# --- optimiser callbacks ---------------------------------------------------------------------------------
def _prepare_controls(params, pstate):
    """optimiser format -> cost-function format, clip to the max norms in place, user conditions."""
    controls = slap_controls(pstate.complex_controls, params, pstate.controls_shape)
    clip_control_norms(controls, pstate.max_control_norms)
    if pstate.impose_control_conditions is not None:
        controls = pstate.impose_control_conditions(controls)
    return controls


def _esd_wrap(params, pstate, reporter, result):
    """`function` callback of the optimiser: (error, terminate)."""
    controls = _prepare_controls(params, pstate)
    error = _evaluate_schroedinger_discrete(controls, pstate, reporter)
    return error, bool(error <= pstate.min_error)


def _esdj_wrap(params, pstate, reporter, result):
    """`jacobian` callback of the optimiser: (flat float64 grads, terminate), with the reference's side
    effects in the reference's order: best-so-far update, log/save, iteration counter."""
    controls = _prepare_controls(params, pstate)
    error, grads = _value_and_jacobian_schroedinger_discrete(controls, pstate, reporter)
    final_states = reporter.final_states
    if error < result.best_error:
        result.best_controls = controls
        result.best_error = error
        result.best_final_states = final_states
        result.best_iteration = reporter.iteration
    pstate.log_and_save(controls, error, final_states, grads, reporter.iteration)
    reporter.iteration += 1
    return strip_controls(pstate.complex_controls, grads), bool(error <= pstate.min_error)


# --- the seam: these two replace the reference's python time loop and its autograd tape -------------------------
def _program_controls_meta(pstate):
    if pstate.program_type == ProgramType.GRAPE:
        return pstate.control_count, pstate.complex_controls
    return pstate._control_count, pstate._complex_controls


def _evaluate_schroedinger_discrete(controls, pstate, reporter):
    """total cost of one evolution on the GPU; fills reporter.error / reporter.final_states
    (qoc/core/schroedingerdiscrete.py:356-438)."""
    control_count, complex_controls = _program_controls_meta(pstate)
    # the plan is cached on pstate: a GRAPE run whose optimiser calls `function` before `jacobian` (L-BFGS-B) must not end up
    # with a recompute-mode plan for all its gradient evaluations
    plan = _plan_for(pstate, control_count, complex_controls, store_tape=pstate.program_type == ProgramType.GRAPE)
    error, final_states = plan.cost(controls)
    _maybe_save_states(pstate, reporter, plan)
    reporter.error = error
    reporter.final_states = final_states
    return error


def _value_and_jacobian_schroedinger_discrete(controls, pstate, reporter):
    """(error, grads) of `ans_jacobian(_evaluate_schroedinger_discrete, 0)` followed by the conjugate for
    complex controls (schroedingerdiscrete.py:318-324): grads = dE/dRe(u) + i dE/dIm(u)."""
    control_count, complex_controls = _program_controls_meta(pstate)
    plan = _plan_for(pstate, control_count, complex_controls)
    # with HIPS autograd installed the GPU evaluation runs as an autograd primitive (defvjp) under the reference's own
    # ans_jacobian; without it the C ABI's value-and-gradient entry point is called directly (same numbers)
    evaluate = plan.cost_and_grad_autograd if (autograd_available() and plan.KR > 0) else plan.cost_and_grad
    error, grads, final_states = evaluate(controls)
    _maybe_save_states(pstate, reporter, plan)
    reporter.error = error
    reporter.final_states = final_states
    return error, grads


def _maybe_save_states(pstate, reporter, plan):
    if pstate.save_intermediate_states_:
        iteration = reporter.iteration if pstate.program_type == ProgramType.GRAPE else 0
        pstate.save_all_intermediate_states(iteration, plan.intermediate_states())
