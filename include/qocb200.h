/*
 * qocb200.h - C ABI of the B200-native GRAPE propagate-and-differentiate hot path.
 *
 * The reference (SchusterLab/qoc) is pure Python and has no FFI; the seam this library replaces is
 *   (1) _evaluate_schroedinger_discrete(controls, pstate, reporter) -> error
 *       (qoc/core/schroedingerdiscrete.py:356-438, also used by evolve_schroedinger_discrete, :101), and
 *   (2) ans_jacobian(_evaluate_schroedinger_discrete, 0)(controls, pstate, reporter) -> (error, grads)
 *       (qoc/core/schroedingerdiscrete.py:318, qoc/standard/utils/autogradutil.py:10-31),
 * and the Lindblad twins (qoc/core/lindbladdiscrete.py:357-441, :322).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add at those two call sites.
 *
 * Conventions
 *   - every pointer is a HOST pointer unless the name ends in `_dev`; the caller owns all host buffers;
 *   - complex arrays are interleaved (re, im) doubles in NumPy C order (complex128);
 *   - controls are REAL channels: real controls -> KR = K; complex controls -> KR = 2K with
 *     x = [Re u_0..Re u_{K-1}, Im u_0..Im u_{K-1}] per control step, and the Hamiltonian is the real-linear form
 *     H(x) = H0 + sum_r x_r A_r (the Python layer extracts H0, A_r from the user's callable);
 *   - gradients are dE/dx_r (real).  For complex controls dE/dRe u + i dE/dIm u is what qoc's optimiser
 *     receives after the wrapper's conjugate (qoc/core/schroedingerdiscrete.py:320-324);
 *   - every function returns 0 on success; on failure a negative code, message via qocb_last_error();
 *   - a plan is not re-entrant; distinct plans are independent; calls block until outputs are on the host
 *     unless stated otherwise.  The plan owns all device memory and its stream.
 */
#ifndef QOCB200_H
#define QOCB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct qocb_plan qocb_plan;

typedef struct {
    int32_t hilbert_size;        /* n */
    int32_t state_count;         /* S */
    int32_t control_count;       /* KR: real control channels */
    int32_t control_eval_count;  /* M  (qoc/models/programstate.py:40-41) */
    int32_t system_eval_count;   /* N  (N-1 time slices, dt = T/(N-1), programstate.py:44) */
    int32_t magnus_order;        /* 2, 4 or 6  (qoc/models/magnuspolicy.py:8-26) */
    int32_t cost_eval_step;      /* >= 1 */
    int32_t ensemble_count;      /* E >= 1: members differ in the drift H0 only; cost = mean over members */
    int32_t device;              /* CUDA device ordinal */
    int32_t store_tape;          /* 1: keep Pade intermediates of the forward pass in HBM for the reverse pass;
                                    0: recompute them in the reverse pass (less memory, ~25% more flops) */
    int32_t chunks_per_member;   /* 0 = automatic */
    int32_t slice_begin;         /* time-slice sharding: this plan owns slices [slice_begin, slice_end) of the N-1 */
    int32_t slice_end;           /* (both 0 = the whole pulse, unsharded).  See the qocb_shard_* calls below */
    int32_t channel_count;       /* KC: operator channels of a time-dependent hamiltonian (qocb_set_node_map);
                                    0 = control_count (time-independent operators, one per real control channel) */
    int32_t state_total;         /* state sharding (qocb_state_shard_*): total number of initial states over all ranks; */
    int32_t state_first;         /* index of this plan's first state among them.  0 / 0 = all states are here */
    double evolution_time;       /* T */
} qocb_problem;

/* cost kinds (qoc/standard/costs): vectors are `state_count x fmax` column vectors of length n */
#define QOCB_COST_TARGET_COHERENT 0   /* w * (1 - |sum_s <t_s|psi_s>|^2 / S^2)   targetstateinfidelity.py:52-56 */
#define QOCB_COST_TARGET_INCOHERENT 1 /* w * (1 - sum_s |<t_s|psi_s>|^2 / S)     targetstateinfidelity.py:57-61 */
#define QOCB_COST_FORBID 2            /* w * sum_s (1/F_s) sum_f |<f_sf|psi_s>|^2  forbidstates.py:64-81         */

int qocb_plan_create(const qocb_problem *problem, qocb_plan **plan_out);
int qocb_plan_destroy(qocb_plan *plan);
const char *qocb_last_error(const qocb_plan *plan);           /* plan may be NULL: last creation error */

/* H0: [E][n][n] complex (E = ensemble_count), A: [KC][n][n] complex (KC = channel_count, or control_count if that is 0) */
int qocb_set_operators(qocb_plan *plan, const double *h0, const double *a_ops);
/* Time-dependent hamiltonian(controls, time) (the callable's `time` argument, qoc/core/schroedingerdiscrete.py:483-486),
   affine in the controls: at Magnus node i of slice j
       H = H0 + sum_c coef[j][i][c] A_c,   coef[j][i][c] = offset[j][i][c] + sum_r gain[j][i][c][r] x_r(t_ji),
   x_r = interpolated real control channel r.  offset: [N-1][q][KC], gain: [N-1][q][KC][KR] for ALL N-1 slices (a plan
   that owns a slice range reads its part); q = magnus_order / 2.  Requires channel_count > 0.  gain may be NULL when
   control_count is 0.  The gradient returned by qocb_cost_and_grad stays [M][KR]. */
int qocb_set_node_map(qocb_plan *plan, const double *offset, const double *gain);
/* psi0: [S][n] complex */
int qocb_set_states(qocb_plan *plan, const double *psi0);
/* vectors: [S][fmax][n] complex; counts: [S] number of valid vectors per state (NULL = fmax for all);
   weight = cost_multiplier / normalisation; step_cost != 0: evaluated at every cost step, else final step only */
int qocb_add_cost(qocb_plan *plan, int32_t kind, int32_t step_cost, double weight,
                  const double *vectors, const int32_t *counts, int32_t fmax);
int qocb_clear_costs(qocb_plan *plan);

/* controls: [M][KR] real.  cost: 1 double.  final_states: [E][S][n] complex or NULL. */
int qocb_cost(qocb_plan *plan, const double *controls, double *cost, double *final_states);
/* grad: [M][KR] real */
int qocb_cost_and_grad(qocb_plan *plan, const double *controls, double *cost, double *grad, double *final_states);
/* The same evaluation in two calls, for cost terms the host must evaluate itself (user-defined Cost subclasses,
   qoc/models/cost.py:5-51): qocb_forward runs the forward pass (keeping the reverse-pass tape) and returns the device costs'
   value and the final states; the host adds its own terms c(psi_N) and hands their cotangent to qocb_backward as
   final_seed[S][n] complex = d c / d Re psi - i d c / d Im psi (autograd's convention), or NULL; qocb_backward returns the
   gradient of (device costs + host terms) with respect to the controls.  Unsharded single-member plans only. */
int qocb_forward(qocb_plan *plan, const double *controls, double *cost, double *final_states);
int qocb_backward(qocb_plan *plan, const double *final_seed, double *grad);
/* all states of the last evaluation: [E][N][S][n] complex (the reference's save_intermediate_states payload,
   qoc/core/schroedingerdiscrete.py:395-402) */
int qocb_get_states(qocb_plan *plan, double *states);
/* final states of the last evaluation: [E][S][n] complex (reporter.final_states, qoc/core/schroedingerdiscrete.py:436);
   waits for the plan stream, so it also serves evaluations enqueued with qocb_run_resident */
int qocb_get_final_states(qocb_plan *plan, double *final_states);
/* per-node cotangents of the operator-channel coefficients of the last qocb_cost_and_grad: [E][N-1][q][KC], dE / d coef[j][i][c]
   (KC = channel_count, or control_count when that is 0).  With control_count = 0 and the coefficients uploaded as the offset
   table of qocb_set_node_map this is the device half of the chain rule through a hamiltonian(controls, time) callable that
   is not affine in the controls (qoc_b200/core/plan.py: NonlinearSchroedingerPlan). */
int qocb_get_node_grad(qocb_plan *plan, double *node_grad);
/* slice propagators U_j of the last evaluation: [E][N-1][n][n] complex */
int qocb_get_propagators(qocb_plan *plan, double *props);

/* device-resident pipeline for benchmarking: controls already in HBM, no host transfer, no sync.
   qocb_upload_controls stages them; qocb_run_resident enqueues the whole evaluation on the plan stream;
   qocb_sync waits; qocb_download_result copies cost/grad to the host. */
int qocb_upload_controls(qocb_plan *plan, const double *controls);
int qocb_run_resident(qocb_plan *plan, int32_t with_grad);
int qocb_sync(qocb_plan *plan);
int qocb_download_result(qocb_plan *plan, double *cost, double *grad);
/* time `iters` resident evaluations with CUDA events on the plan stream after `warmup` untimed ones.
   ms_total[0] = total ms; kernel_ms[8] = summed ms of each pipeline stage (expm forward = Magnus pass + k_forward, boundary
   fwd, sweep fwd, sweep bwd (all three), expm reverse (k_backward + Magnus adjoint pass), gather, finalize, propagator tree
   between the expm forward and the boundary pass); flush_l2 != 0 writes a 256 MiB buffer
   between evaluations (outside the stage timers, inside ms_total only if count_flush != 0). */
int qocb_time_resident(qocb_plan *plan, int32_t with_grad, int32_t warmup, int32_t iters, int32_t flush_l2,
                       double *ms_total, double *stage_ms);
/* enqueue a 256 MiB write on the plan stream (evicts the 126 MB L2 between timed iterations) */
int qocb_flush_l2(qocb_plan *plan);
/* number of kernel launches of one evaluation */
int qocb_launch_count(qocb_plan *plan, int32_t with_grad);
void *qocb_stream(qocb_plan *plan);                           /* cudaStream_t of the plan */

/* ---- time-slice sharding (SURVEY.md 8e; one plan per rank, created with a slice range) ---------------------
   The four phase calls only ENQUEUE work on the plan stream.  `*_dev` pointers are DEVICE buffers owned by the
   caller: the host language allocates them and runs the collectives between the phases on the same stream
   (qoc_b200/core/sharded.py uses torch.distributed / NCCL over NVLink):
     1. qocb_shard_forward_local(plan, with_grad, shardP_dev)   Magnus + expm of the local slices; product of the
        local propagators -> shardP_dev[qocb_shard_matrix_doubles]
        -- all-gather shardP_dev -> allP_dev[world][matrix_doubles]
     2. qocb_shard_forward_finish(plan, allP_dev, rank)         incoming boundary state P_{rank-1}..P_0 psi0, local
        state sweeps, cost partial
     3. qocb_shard_backward_particular(plan, b_dev)             costate at the shard's first state for a zero incoming
        costate -> b_dev[qocb_shard_vector_doubles]             (the affine recursion's particular part)
        -- all-gather b_dev -> allb_dev[world][vector_doubles]
     4. qocb_shard_backward_finish(plan, allP_dev, allb_dev, rank, world)
        incoming costate by suffix combination, local costate sweeps, expm/Magnus adjoints, gradient scatter
     5. qocb_shard_pack_result(plan, with_grad, result_dev)     result_dev[qocb_shard_result_doubles] =
        [partial gradient M*KR | partial cost | final states S*2*NP planar, zeros unless this shard owns the last
        slice] -- all-reduce(sum) it.  A forward-only evaluation runs phases 1, 2, 5 (with_grad = 0). */
int qocb_shard_matrix_doubles(qocb_plan *plan);
int qocb_shard_vector_doubles(qocb_plan *plan);
int qocb_shard_forward_local(qocb_plan *plan, int32_t with_grad, double *shardP_dev);
int qocb_shard_forward_finish(qocb_plan *plan, const double *allP_dev, int32_t rank);
int qocb_shard_backward_particular(qocb_plan *plan, double *b_dev);
int qocb_shard_backward_finish(qocb_plan *plan, const double *allP_dev, const double *allb_dev, int32_t rank,
                               int32_t world);
int qocb_shard_result_doubles(qocb_plan *plan);
int qocb_shard_pack_result(qocb_plan *plan, int32_t with_grad, double *result_dev);

/* ---- sharding of the initial STATES (SURVEY.md 8e: independent units; one plan per rank, created with state_count = the local
   states, state_total / state_first set, and the cost vectors of the local states only).  Every rank computes every slice
   propagator - they depend on the controls alone - and sweeps its own states; cost normalisations use state_total.  The only
   coupling is the coherent target infidelity 1 - |sum_s <t_s|psi_s>|^2 / S^2 (targetstateinfidelity.py:53-55):
     1. qocb_state_shard_forward(plan, with_grad, coh_dev)   expm + state sweeps; coh_dev[qocb_state_shard_coherent_doubles] =
        this rank's partial overlap sums (re, im per coherent term and cost step); the cost so far excludes those terms
        -- all-reduce(sum) coh_dev (skip when the count is 0)
     2. qocb_state_shard_finish(plan, with_grad, coh_dev)    coherent values from the totals (added once, by the rank with
        state_first = 0), then - with_grad - costate sweeps seeded from the totals, expm / Magnus adjoints, gradient
     3. qocb_shard_pack_result(plan, with_grad, result_dev)  [gradient | cost | ...] -- all-reduce(sum) the first M*KR + 1 doubles.
   The calls only enqueue on the plan stream.  Not combinable with time-slice sharding or ensembles. */
int qocb_state_shard_coherent_doubles(qocb_plan *plan);
int qocb_state_shard_forward(qocb_plan *plan, int32_t with_grad, double *coh_dev);
int qocb_state_shard_finish(qocb_plan *plan, int32_t with_grad, const double *coh_dev);

/* standalone batched matrix exponential (qoc/standard/functions/expm.py:210-252), bench / test hook.
   a, out: [batch][n][n] complex on the host. */
int qocb_expm_batched(int32_t n, int64_t batch, const double *a, double *out, int32_t device);
/* same with adjoint: given ubar [batch][n][n] (cotangent of the output, autograd convention) returns
   abar [batch][n][n] (cotangent of the input) - exercises the reverse pass in isolation */
int qocb_expm_vjp_batched(int32_t n, int64_t batch, const double *a, const double *ubar, double *out, double *abar,
                          int32_t device);
/* device-resident timing of the batched expm: returns ms per launch (best of `iters`) */
int qocb_expm_batched_time(int32_t n, int64_t batch, double norm_scale, int32_t iters, double *ms_best, int32_t device);

/* the same with `warmup` untimed launches and the total over exactly `iters` timed ones (bench.py --workload expm_batched_n*):
   ms_total / ms_best may be NULL.  n <= 4 runs the register-resident kernels (one matrix per thread for n <= 2, per 4-lane
   group for n = 3, 4) on [batch][n][n] interleaved complex128 with a 256 MiB L2 flush between launches. */
int qocb_expm_batched_bench(int32_t n, int64_t batch, double norm_scale, int32_t warmup, int32_t iters, double *ms_total,
                            double *ms_best, int32_t device);

/* ---- Lindblad path: _evaluate_lindblad_discrete (qoc/core/lindbladdiscrete.py:357-441) and its jacobian (:322) -------
   Densities are [D][n][n] complex128, interleaved (NumPy C order).  H(x) = H0 + sum_r x_r A_r as above; the dissipator is
   sum_l gamma_l (L_l rho L_l^dag - 1/2 {L_l^dag L_l, rho}).  Each of the N-1 intervals is a fresh adaptive Dormand-Prince
   5(4) integration (qoc/core/mathmethods.py:352-480).

   TIME DEPENDENCE.  The stage times of the adaptive integration depend on the data, so a time-dependent `hamiltonian` or
   `lindblad_data` is given to the device as piecewise Chebyshev series of scalar functions of t, evaluated in the kernels
   at every stage time:
     - channel_count = KC > 0:  H(x, t) = H0 + sum_c (offset_c(t) + sum_r gain_cr(t) x_r) A_c, and a_ops of
       qocb_lindblad_set_operators holds the KC channels A_c instead of KR control operators;
     - time_dependent_rates = 1:  L_l(t) = f_l(t) B_l with fixed B_l (lops holds B_l, gammas is unused) and the effective
       rate r_l(t) = gamma_l(t) |f_l(t)|^2.
   The series table (qocb_lindblad_set_time_series, required with either) holds NS = KC (1 + KR) + (rates ? L : 0)
   functions per row in the order [offset_c | gain_cr (c-major) | r_l], on `segments` uniform segments of width w that cover
   [0, segments * w].  Stage times beyond the table are never extrapolated: the forward pass records the largest stage time
   it needed (qocb_lindblad_max_stage_time), skips the reverse pass and the evaluation returns -5; the caller extends the
   table and evaluates again (the initial-step probe t0 + h0 and the overshooting last step of an interval can reach far
   beyond the evolution time).  The gradient maps the channel cotangents back, xbar_r = sum_c gain_cr(t) cbar_c, before
   the interpolation weights; offsets and rates receive none.  With KC = 0 and time_dependent_rates = 0 nothing changes.

   CONTRACT OF THE LINDBLAD RESULTS (tolerances are asserted in tests/test_gpu_lindblad.py):
     - cost and final densities: the reference's adaptive integration at atol = 1e-12, rtol = 0.  A rounding-level change of
       one error norm near the accept threshold moves the whole step sequence, so two correct implementations agree to the
       integrator's own tolerance, not to rounding: |cost - reference| and the final densities within 1e-9.
     - gradient: the DISCRETE ADJOINT OF THE DORMAND-PRINCE MAP ON THE REALISED STEP GRID - every accepted step (x, h) of the
       forward pass is held fixed and the Runge-Kutta stages, the 4th-order dense output at the interval end and the FSAL
       coupling are differentiated exactly.  The reference's autograd tape additionally differentiates the step-size
       controller (qoc/core/mathmethods.py:436-462), whose inputs are error norms taken at the rounding floor; those terms are
       noise (perturbing the controls by 1e-13 moves the reference-equivalent full gradient by 1e-5 .. 1e-4).  The gradient
       returned here matches the reference-equivalent gradient with the step grid frozen within 1e-7 relative, and the full
       one within its own reproducibility band.  It is NOT claimed at the 1e-10 of the Schroedinger path.

   ENSEMBLES (robust control over drifts and decay rates).  ensemble_count = E > 1 runs E members, one CTA each, in one launch
   of each kernel.  Members differ in the drift H0 and/or the rates gamma_l (qocb_lindblad_set_ensemble); rho0, control and
   Lindblad operators, cost terms, controls and the time series are shared.  Every member runs exactly the code and the launch
   layout of a one-member plan of the same shape, so its results are bit-identical to such a plan built with its drift and
   rates.  The cost and gradient are the member mean: sums in member order 0..E-1 divided by E (no atomics).  Each member has
   its own tape of max_rk_steps steps (0: max(4096, min(2^20, 8 GiB / (E * 2 * D n^2 * 16 B)))); a member whose forward
   pass fills its tape skips its reverse pass, and the evaluation returns -4. */
typedef struct qocb_lplan qocb_lplan;

typedef struct {
    int32_t hilbert_size;        /* n */
    int32_t density_count;       /* D */
    int32_t control_count;       /* KR real control channels (0 with have_hamiltonian = 0) */
    int32_t control_eval_count;  /* M */
    int32_t system_eval_count;   /* N */
    int32_t cost_eval_step;
    int32_t lindblad_count;      /* L (0: lindblad_data = None) */
    int32_t have_hamiltonian;    /* 0: hamiltonian = None (lindbladdiscrete.py:480-484) */
    int32_t device;
    int32_t max_rk_steps;        /* capacity of the accepted-step tape of one evaluation; 0 = automatic */
    int32_t channel_count;       /* KC in [0, 16]: time-dependent hamiltonian channels; 0 = time-independent H0 + x.A */
    int32_t time_dependent_rates;/* 0 or 1 (needs lindblad_count >= 1) */
    int32_t ensemble_count;      /* E members; 0 or 1: one member (no ensemble) */
    double evolution_time;
} qocb_lindblad_problem;

#define QOCB_LCOST_TARGET 0   /* w * (1 - sum_d |tr(T_d^dag rho_d)| / (D n))        targetdensityinfidelity.py:60-66 */
#define QOCB_LCOST_FORBID 1   /* w * sum_d (1/F_d) sum_f |tr(F_df^dag rho_d) / n|^2  forbiddensities.py:67-85        */

int qocb_lindblad_create(const qocb_lindblad_problem *problem, qocb_lplan **plan_out);
int qocb_lindblad_destroy(qocb_lplan *plan);
const char *qocb_lindblad_last_error(const qocb_lplan *plan);
/* h0: [n][n] (NULL without hamiltonian); a_ops: [KR][n][n]; gammas: [L]; lops: [L][n][n] */
int qocb_lindblad_set_operators(qocb_lplan *plan, const double *h0, const double *a_ops, const double *gammas,
                                const double *lops);
/* Members of an ensemble plan (E > 1), required before its first evaluation and again after qocb_lindblad_set_operators:
   h0s [E][n][n] (NULL: every member takes the h0 of qocb_lindblad_set_operators; needs have_hamiltonian = 1 and
   channel_count = 0), gammas [E][L] (NULL: every member takes the plan's; needs time_dependent_rates = 0).  Member e's
   1/2 sum_l gamma_el L_l^dag L_l is built on the host as qocb_lindblad_set_operators builds it.  Returns -1 on E <= 1. */
int qocb_lindblad_set_ensemble(qocb_lplan *plan, const double *h0s, const double *gammas);
/* series: [segments][degree+1][NS] Chebyshev coefficients per segment [s w, (s+1) w] (constant term not halved);
   degree <= 64; may be called again to replace the table */
int qocb_lindblad_set_time_series(qocb_lplan *plan, int32_t segments, int32_t degree, double segment_width,
                                  const double *series);
/* largest stage time of the last forward pass (plans with a series; the maximum over the members of an ensemble); an
   evaluation returns -5 when it lies beyond the table */
int qocb_lindblad_max_stage_time(qocb_lplan *plan, double *t);
int qocb_lindblad_set_densities(qocb_lplan *plan, const double *rho0);
/* mats: [D][fmax][n][n]; counts: [D] or NULL; weight = cost_multiplier / normalisation; step_cost as above */
int qocb_lindblad_add_cost(qocb_lplan *plan, int32_t kind, int32_t step_cost, double weight, const double *mats,
                           const int32_t *counts, int32_t fmax);
/* controls: [M][KR]; final_densities: [D][n][n] or NULL; grad: [M][KR].  Ensemble: member-mean cost and gradient, and
   final_densities [E][D][n][n] */
int qocb_lindblad_cost(qocb_lplan *plan, const double *controls, double *cost, double *final_densities);
int qocb_lindblad_cost_and_grad(qocb_lplan *plan, const double *controls, double *cost, double *grad,
                                double *final_densities);
/* The same evaluation in two calls, for cost terms the host evaluates itself on the densities (user-defined Cost subclasses,
   qoc/models/cost.py:5-51, on any subset of the system steps):
     - qocb_lindblad_forward runs the forward pass and keeps the reverse-pass tape.  `cost` is the value of the device cost
       terms only; the densities of every step are then available through qocb_lindblad_get_densities.  Return codes as
       qocb_lindblad_cost_and_grad, including -4 (tape full) and -5 (stage time beyond the series: extend and call again).
     - qocb_lindblad_backward runs the reverse pass of that forward pass and returns the gradient of (device costs + host
       terms).  seeds is NULL or [N][D][n][n] complex: row k = d c / d Re rho_k - i d c / d Im rho_k of the host terms at system
       step k (autograd's convention, the one the device costs use).  Row N-1 is added before the reverse sweep starts, row k
       next to the device step costs of step k; row 0 has no effect.  qocb_lindblad_forward followed by
       qocb_lindblad_backward(seeds = NULL) gives bit-identical results to qocb_lindblad_cost_and_grad.
   TAPE RULE: qocb_lindblad_backward needs a qocb_lindblad_forward that returned 0 as the plan's last evaluation, with no
   setter in between (qocb_lindblad_cost and qocb_lindblad_cost_and_grad overwrite the densities without that tape);
   otherwise it returns -1.  It may be called more than once on one tape.  With control_count = 0 it writes nothing and
   returns 0.  The seed buffer is allocated on first use: plans that never pass seeds allocate nothing for it.
   Both return -1 on an ensemble plan. */
int qocb_lindblad_forward(qocb_lplan *plan, const double *controls, double *cost, double *final_densities);
int qocb_lindblad_backward(qocb_lplan *plan, const double *seeds, double *grad);
/* stats[0] = Runge-Kutta attempts, stats[1] = accepted steps of the last evaluation (sums over the members of an ensemble) */
int qocb_lindblad_stats(qocb_lplan *plan, int64_t *stats);
/* each member's results of the last evaluation: costs [E], grads [E][M][KR], stats [E][2]; any may be NULL */
int qocb_lindblad_member_results(qocb_lplan *plan, double *costs, double *grads, int64_t *stats);
/* densities at every system step of the last evaluation: [N][D][n][n] (save_intermediate_densities payload); [E][N][D][n][n]
   for an ensemble */
int qocb_lindblad_get_densities(qocb_lplan *plan, double *densities);

const char *qocb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* QOCB200_H */
