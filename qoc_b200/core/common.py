"""
common.py - control-array plumbing shared by the grape programs (host side of the drop-in boundary;
behaviour of qoc/core/common.py:8-30, :33-142, :146-198, :201-246).
"""
import numpy as np

from qoc_b200.standard.optimizers import SGD, Adam, LBFGSB

_NORM_TOLERANCE = 1e-10


def clip_control_norms(controls, max_control_norms):
    """rescale, IN PLACE, every control point whose modulus exceeds its column's maximum norm back onto
    that norm (for real controls: clipping to [-max, max])."""
    for k, max_norm in enumerate(max_control_norms):
        column = controls[:, k]
        norms = np.abs(column)
        over = np.nonzero(max_norm < norms)
        column[over] = column[over] / norms[over] * max_norm


def _complexify(controls, complex_controls):
    return (controls - 1j * controls) / np.sqrt(2) if complex_controls else controls


def gen_controls_cos(complex_controls, control_count, control_eval_count, evolution_time,
                     max_control_norms, periods=10.):
    """half-amplitude cosine with `periods` periods over the pulse; exact zeros replaced by max/10."""
    b = 2 * np.pi / (control_eval_count / periods)
    controls = np.zeros((control_eval_count, control_count))
    for k in range(control_count):
        wave = max_control_norms[k] / 2 * np.cos(b * np.arange(control_eval_count))
        controls[:, k] = np.where(wave, wave, max_control_norms[k] * 1e-1)
    return _complexify(controls, complex_controls)


def gen_controls_white(complex_controls, control_count, control_eval_count, evolution_time,
                       max_control_norms, periods=10.):
    """white noise with standard deviation max/5."""
    controls = np.zeros((control_eval_count, control_count))
    for k in range(control_count):
        controls[:, k] = np.random.normal(0, max_control_norms[k] / 5.0, control_eval_count)
    return _complexify(controls, complex_controls)


def gen_controls_flat(complex_controls, control_count, control_eval_count, evolution_time,
                      max_control_norms, periods=10.):
    """flat line at a tenth of the maximum norm (the default initial guess)."""
    controls = np.zeros((control_eval_count, control_count))
    for k in range(control_count):
        controls[:, k] = np.repeat(max_control_norms[k] * 1e-1, control_eval_count)
    return _complexify(controls, complex_controls)


def initialize_controls(complex_controls, control_count, control_eval_count, evolution_time,
                        initial_controls, max_control_norms):
    """default max norms (ones) / default flat controls, and validation of user-supplied controls against the
    declared dtype and the max norms (ValueError, as the reference)."""
    if max_control_norms is None:
        max_control_norms = np.ones(control_count)
    if initial_controls is None:
        return (gen_controls_flat(complex_controls, control_count, control_eval_count, evolution_time,
                                  max_control_norms), max_control_norms)
    is_complex = np.iscomplexobj(initial_controls)
    if complex_controls and not is_complex:
        raise ValueError("The program expected that the initial_controls specified by the user conformed to "
                         "complex_controls, but the program found that the initial_controls were not complex "
                         "and complex_controls was set to True.")
    if not complex_controls and is_complex:
        raise ValueError("The program expected that the initial_controls specified by the user conformed to "
                         "complex_controls, but the program found that the initial_controls were complex "
                         "and complex_controls was set to False.")
    for step, row in enumerate(initial_controls):
        if not np.less_equal(np.abs(row), max_control_norms + _NORM_TOLERANCE).all():
            raise ValueError("The program expected that the initial_controls specified by the user conformed to "
                             "max_control_norms, but the program found a conflict at initial_controls[{}]={} and "
                             "max_control_norms={}.".format(step, row, max_control_norms))
    return initial_controls, max_control_norms


def slap_controls(complex_controls, controls, controls_shape):
    """optimiser format (flat float64; complex as [real..., imag...]) -> cost-function format.  For real
    controls the result is a reshape VIEW, so the in-place clip reaches the optimiser's array, as in the
    reference."""
    if complex_controls:
        real, imag = np.split(controls, 2)
        controls = real + 1j * imag
    return np.reshape(controls, controls_shape)


def strip_controls(complex_controls, controls):
    """cost-function format -> optimiser format."""
    flat = np.ravel(controls)
    if complex_controls:
        flat = np.hstack((np.real(flat), np.imag(flat)))
    return flat


# --- multi-start GRAPE: B optimisations of one problem in lockstep, one batched evaluation per iteration -----------------
def batch_initial_controls(name, complex_controls, control_count, control_eval_count, evolution_time, initial_controls,
                           max_control_norms, optimizer, save_file_path):
    """the argument checks of the multi-start driver `name`: (initial controls [B][M][K], max_control_norms).  Raises
    NotImplementedError for `save_file_path` and optimisers other than Adam and SGD, ValueError for malformed controls."""
    if save_file_path is not None:
        raise NotImplementedError("{} does not save to files; run the best start again with {} to save it".format(
            name, name[:-len("_batch")]))
    if isinstance(optimizer, LBFGSB):
        raise NotImplementedError("L-BFGS-B is not supported for control batches: its line search would couple the starts")
    if not isinstance(optimizer, (Adam, SGD)):
        raise NotImplementedError("control batches run Adam or SGD, not {}".format(optimizer))
    controls0 = np.asarray(initial_controls)
    K, M = int(control_count), int(control_eval_count)
    if controls0.ndim != 3 or controls0.shape[0] < 1 or controls0.shape[1:] != (M, K):
        raise ValueError("initial_controls must have shape [B][{}][{}] with B >= 1, got {}".format(M, K, controls0.shape))
    if not np.issubdtype(controls0.dtype, np.number):
        raise ValueError("initial_controls must be numeric, got dtype {}".format(controls0.dtype))
    for b in range(controls0.shape[0]):      # the dtype and max-norm checks of the single-start program, per start
        _, max_control_norms = initialize_controls(complex_controls, K, M, evolution_time, controls0[b], max_control_norms)
    return controls0, max_control_norms


def grape_lockstep(evaluate, controls0, complex_controls, max_control_norms, impose_control_conditions, iteration_count,
                   log_iteration_step, min_error, optimizer, result_type, final_field):
    """runs B Adam or SGD optimisations from `controls0` [B][M][K] in lockstep.  Every iteration prepares each start's
    controls as the single-start program does (clip in place to `max_control_norms`, then `impose_control_conditions`),
    evaluates all of them with one call `evaluate(controls [B][M][K]) -> (errors [B], grads [B][M][K], finals [B][...])`,
    keeps each start's best-so-far in a `result_type` (its final states or densities in the field `final_field`) and updates
    each running start with its own optimiser state.  A start whose error reaches `min_error` stops; the loop ends when every
    start has stopped or after `iteration_count` iterations.  Returns the B results."""
    B, M, K = controls0.shape
    # optimiser format, one row per start: flat float64 ([Re | Im] for complex controls), as strip_controls
    params = np.stack([strip_controls(complex_controls, controls0[b]) for b in range(B)]).astype(np.float64)
    shape = (M, K)
    results = [result_type() for _ in range(B)]
    stopped = np.zeros(B, dtype=bool)
    adam = isinstance(optimizer, Adam)
    moment, square_moment, steps = np.zeros_like(params), np.zeros_like(params), np.zeros((B, 1))
    for iteration in range(iteration_count):
        controls = np.empty((B, M, K), dtype=np.complex128 if complex_controls else np.float64)
        for b in range(B):
            c = slap_controls(complex_controls, params[b], shape)      # a view of params[b] for real controls
            clip_control_norms(c, max_control_norms)
            if impose_control_conditions is not None:
                c = impose_control_conditions(c)
            controls[b] = c
        errors, grads, finals = evaluate(controls)
        active = np.nonzero(~stopped)[0]
        for b in active:
            if errors[b] < results[b].best_error:
                results[b].best_controls = controls[b].copy()
                results[b].best_error = float(errors[b])
                setattr(results[b], final_field, finals[b].copy())
                results[b].best_iteration = iteration
        stopped[active] = errors[active] <= min_error
        if log_iteration_step and iteration % log_iteration_step == 0:
            print("{:>6d} | best error {:.12e} | median error {:.12e} | stopped {}/{}".format(
                iteration, min(r.best_error for r in results), float(np.median(errors)), int(stopped.sum()), B))
        idx = np.nonzero(~stopped)[0]
        if idx.size == 0:
            break
        g = np.stack([strip_controls(complex_controls, grads[b]) for b in idx])
        if adam:
            params[idx], moment[idx], square_moment[idx], steps[idx] = _adam_rows(
                optimizer, params[idx], g, moment[idx], square_moment[idx], steps[idx])
        else:
            params[idx] = params[idx] - optimizer.learning_rate * g
    return results


def _adam_rows(opt, params, grads, moment, square_moment, steps):
    """`Adam.update` applied to every row on its own (one row per start; `steps` [rows][1] counts each row's updates):
    the gradient norm of `scale_grads` is the row's own."""
    lr = opt.initial_learning_rate
    if opt.apply_learning_rate_decay:
        lr = lr * np.exp(-np.divide(steps, opt.learning_rate_decay))
    if opt.apply_scale_grads:
        grads = grads / np.linalg.norm(grads, axis=1, keepdims=True) * opt.scale_grads
    if opt.apply_clip_grads:
        grads = np.clip(grads, -opt.clip_grads, opt.clip_grads)
    t = steps + 1
    moment = opt.beta_1 * moment + (1 - opt.beta_1) * grads
    square_moment = opt.beta_2 * square_moment + (1 - opt.beta_2) * np.square(grads)
    m_hat = moment / (1 - np.power(opt.beta_1, t))
    v_hat = square_moment / (1 - np.power(opt.beta_2, t))
    return params - lr * m_hat / (np.sqrt(v_hat) + opt.epsilon), moment, square_moment, t
