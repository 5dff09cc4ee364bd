// lindblad.cu - Lindblad master-equation path of the GRAPE hot path on the GPU.
//
// Reference: _evaluate_lindblad_discrete (qoc/core/lindbladdiscrete.py:357-441) with the right-hand side of
// _get_rhs_lindbladian / get_lindbladian (:444-495, qoc/core/mathmethods.py:169-206) and, per interval, a fresh
// adaptive Dormand-Prince 5(4) integration (mathmethods.py:211-480: initial step heuristic :405-420, accept /
// reject and step factors :427-460, FSAL :477, 4th-order dense output at the interval end :263-304, :467-472),
// the density costs (qoc/standard/costs/targetdensityinfidelity.py:41-69, targetdensityinfidelitytime.py:47-76,
// forbiddensities.py:53-85) and the reverse pass.
//
// The integration is one sequential, data-dependent loop over tiny matrices: one persistent CTA walks all
// intervals and adaptive steps (all D densities share the step-size sequence through the rms norms), keeps its
// working set in shared memory when it fits, and records (x, h, y, k1) of every ACCEPTED step on a tape in HBM.
// The reverse pass replays the tape backwards: per step it recomputes the six stages and applies the
// hand-derived adjoint of the RK map, the dense output and the FSAL coupling on the realised grid
// (oracle/lindblad_adjoint_model.py is the NumPy statement of the same algebra and explains, with measurements,
// why the step-size controller itself is not differentiated).
//
// An ensemble plan (robust control over drifts and rates) launches E such CTAs at once: CTA e is member e and runs exactly
// the code of a one-member plan on its own drift, rates, densities, tape and result slots (member_args); a small kernel
// then forms the member mean in member order.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/qocb200.h"

namespace {

constexpr int LNT = 256;              // max threads of the persistent CTA (32 for tiny problems: barriers become warp-wide)
constexpr int kMaxKRL = 16;

__device__ __constant__ double cA[6][5] = {
    {0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
__device__ __constant__ double cC[6] = {0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1};
__device__ __constant__ double cB[7] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84, 0};
__device__ __constant__ double cBH[7] = {5179.0 / 57600, 0, 7571.0 / 16695, 393.0 / 640, -92097.0 / 339200, 187.0 / 2100, 1.0 / 40};
__device__ __constant__ double cD[7] = {-12715105075.0 / 11282082432.0, 0, 87487479700.0 / 32700410799.0,
                                        -10690763975.0 / 1880347072.0, 701980252875.0 / 199316789632.0,
                                        -1453857185.0 / 822651844.0, 69997945.0 / 29380423.0};
#define L_ATOL 1e-12

struct DTerm {
    int kind;      // 0: w * (1 - sum_d |tr(T_d^dag rho_d)| / (D n)),  1: w * sum_d (1/F_d) sum_f |tr(F_df^dag rho_d)/n|^2
    int step;      // 1: every cost step, 0: final step only
    int fmax, mat_off, cnt_off;
    double w;
};

struct LArgs {
    int n, D, KR, M, N, L, ces, have_h, nterms, cap;
    double T;
    const double2 *H0, *Aops, *Lops, *Khalf;   // [n*n], [KR][n*n], [L][n*n], 1/2 sum_l gamma_l L^dag L
    const double *gam, *controls, *xs;
    const double2 *rho0;
    const DTerm *terms; const double2 *mats; const int *counts;
    double2 *states;                            // [N][D*n*n] densities at every system step
    double *cost;
    double *tape_x, *tape_h; double2 *tape_y, *tape_k1;
    int *first;                                 // [N] first tape index of each interval; first[N-1] = total
    int *hit;                                   // [N-1] tape index of the step that produced the interval's output
    long long *stats;                           // attempts, accepted
    int *err_flag;
    double2 *work;                              // global work arrays (used when the working set exceeds shared memory)
    int work_in_smem, ops_in_smem;
    double *grad;                               // [M][KR]
    // time-dependent operators (0 series without them): piecewise Chebyshev series of the NS = KC*(1+KR) + L scalar
    // functions [offset_c | gain_cr | rate_l] on `segs` uniform segments of width `seg_w` covering [0, segs * seg_w]
    int KC, tdr, segs, deg, NS;
    double seg_w;
    const double *series;                       // [segs][deg+1][NS]
    const double2 *Kops;                        // [L][n*n] 1/2 B_l^dag B_l (tdr)
    double *tseen;                              // largest stage time of the forward pass
    const double2 *seeds;                       // [N][D*n*n] host-cost cotangents of the densities, or null
};

// the arguments of ensemble member blockIdx.x: per-member drift, K_half, rates, densities, tape, interval indices, global
// work, cost, gradient, stats, stage time and tape-overflow flag sit at member-major offsets; rho0, operators, cost terms,
// controls and the time series are shared.  Member 0 is the whole plan when E = 1.
__device__ __forceinline__ LArgs member_args(const LArgs &a0) {
    LArgs a = a0;
    const size_t e = blockIdx.x, nn = (size_t)a.n * a.n, DE = (size_t)a.D * nn;
    a.H0 += e * nn; a.Khalf += e * nn; a.gam += e * (size_t)max(a.L, 1);
    a.states += e * a.N * DE;
    a.tape_x += e * a.cap; a.tape_h += e * a.cap; a.tape_y += e * a.cap * DE; a.tape_k1 += e * a.cap * DE;
    a.first += e * a.N; a.hit += e * a.N;
    if (!a.work_in_smem) a.work += e * 24 * DE;
    a.cost += e; a.grad += e * (size_t)a.M * a.KR; a.stats += 2 * e; a.err_flag += e;
    if (a.tseen) a.tseen += e;
    return a;
}

// block-wide sum, result in all threads
__device__ double block_sum(double v, double *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double s = 0.;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;
}

// op codes for a matrix operand: 0 = M, 1 = M^T, 2 = conj(M), 3 = M^dagger
template <int OP> __device__ __forceinline__ double2 elem(const double2 *m, int n, int i, int j) {
    double2 v = (OP == 1 || OP == 3) ? m[j * n + i] : m[i * n + j];
    if (OP >= 2) v.y = -v.y;
    return v;
}

// out[d] = (ACC ? out[d] : 0) + alpha * opA(A[d or shared]) * opB(B[d or shared]); strides 0 = shared n x n operand
template <int OPA, int OPB, bool ACC>
__device__ void bmm(double2 *out, const double2 *A, int sA, const double2 *B, int sB, int n, int D, double alpha) {
    const int nn = n * n;
    for (int e = threadIdx.x; e < D * nn; e += blockDim.x) {
        const int d = e / nn, r = e - d * nn, i = r / n, j = r - i * n;
        const double2 *a = A + (size_t)d * sA, *b = B + (size_t)d * sB;
        double sr = 0., si = 0.;
        for (int k = 0; k < n; ++k) {
            const double2 x = elem<OPA>(a, n, i, k), y = elem<OPB>(b, n, k, j);
            sr += x.x * y.x - x.y * y.y;
            si += x.x * y.y + x.y * y.x;
        }
        if (ACC) { out[e].x += alpha * sr; out[e].y += alpha * si; }
        else { out[e].x = alpha * sr; out[e].y = alpha * si; }
    }
    __syncthreads();
}

struct Ctx {
    const LArgs &a;
    double2 *A1, *A2;       // shared: -iH - Khalf, +iH - Khalf at the current time
    double2 *tmp;           // [D*nn] scratch
    double *red;            // reduction scratch
    double *coef;           // interpolated controls [KR], then slot for (i0, i1, w)
    int *loc;               // i0, i1
    double *sv, *chan, *cbar;   // series values at t [NS], channel coefficients [KC], channel cotangents [KC] (series only)
    double tseen = 0.;      // largest stage time evaluated (uniform over the CTA)
    // operators, rates, controls and control times: shared-memory copies when they fit (a.ops_in_smem), else global
    const double2 *H0, *Aops, *Lops, *Khalf, *Kops;
    const double *gam, *controls, *xs;
    __device__ Ctx(const LArgs &a_) : a(a_), H0(a_.H0), Aops(a_.Aops), Lops(a_.Lops), Khalf(a_.Khalf), Kops(a_.Kops),
                                      gam(a_.gam), controls(a_.controls), xs(a_.xs) {}
};

// the NS series at t by Clenshaw, one series per thread.  A time beyond the table is recorded in c.tseen and evaluated at
// the table's end instead (never extrapolated); the host sees tseen, extends the table and runs the evaluation again.
__device__ void eval_series(Ctx &c, double t) {
    const LArgs &a = c.a;
    c.tseen = fmax(c.tseen, t);
    const double tc = fmin(fmax(t, 0.0), a.segs * a.seg_w);
    const int s = min(max((int)(tc / a.seg_w), 0), a.segs - 1);
    const double u = 2.0 * (tc - s * a.seg_w) / a.seg_w - 1.0, u2 = 2.0 * u;
    const double *tab = a.series + (size_t)s * (a.deg + 1) * a.NS;
    for (int j = threadIdx.x; j < a.NS; j += blockDim.x) {
        double b1 = 0., b2 = 0.;
        for (int k = a.deg; k >= 1; --k) {
            const double b0 = tab[(size_t)k * a.NS + j] + u2 * b1 - b2;
            b2 = b1; b1 = b0;
        }
        c.sv[j] = tab[j] + u * b1 - b2;
    }
    __syncthreads();
}

// controls at time t (qoc/core/mathmethods.py:36-67 on control_eval_times) and the effective generators.  TD: the plan has
// time series (a.NS > 0); the kernels are instantiated for both, so that plans without series run the code they always ran
template <bool TD> __device__ void set_time(Ctx &c, double t) {
    const LArgs &a = c.a;
    const int nn = a.n * a.n;
    if constexpr (TD) eval_series(c, t);
    if (a.have_h && a.KR > 0) {
        if (threadIdx.x == 0) {
            int i0, i1;
            if (t <= c.xs[0]) { i0 = 0; i1 = 1; }
            else if (t >= c.xs[a.M - 1]) { i0 = a.M - 2; i1 = a.M - 1; }
            else { i1 = 0; while (!(t <= c.xs[i1])) ++i1; i0 = i1 - 1; }
            c.loc[0] = i0; c.loc[1] = i1;
        }
        __syncthreads();
        const int i0 = c.loc[0], i1 = c.loc[1];
        for (int r = threadIdx.x; r < a.KR; r += blockDim.x) {
            const double y0 = c.controls[i0 * a.KR + r], y1 = c.controls[i1 * a.KR + r];
            c.coef[r] = y0 + ((y1 - y0) / (c.xs[i1] - c.xs[i0])) * (t - c.xs[i0]);
        }
        __syncthreads();
    }
    if (TD && a.KC > 0) {                                  // coef_c = offset_c(t) + sum_r gain_cr(t) x_r(t)
        for (int ch = threadIdx.x; ch < a.KC; ch += blockDim.x) {
            double v = c.sv[ch];
            for (int r = 0; r < a.KR; ++r) v += c.sv[a.KC + ch * a.KR + r] * c.coef[r];
            c.chan[ch] = v;
        }
        __syncthreads();
    }
    const int nch = (TD && a.KC > 0) ? a.KC : a.KR;
    const double *cf = (TD && a.KC > 0) ? c.chan : c.coef;
    for (int e = threadIdx.x; e < nn; e += blockDim.x) {
        double2 h = make_double2(0., 0.);
        if (a.have_h) {
            h = c.H0[e];
            for (int r = 0; r < nch; ++r) { const double2 g = c.Aops[(size_t)r * nn + e]; h.x += cf[r] * g.x; h.y += cf[r] * g.y; }
        }
        double2 k = make_double2(0., 0.);
        if (TD && a.tdr) {                                 // Khalf(t) = sum_l r_l(t) 1/2 B_l^dag B_l; c.gam points at r(t)
            for (int l = 0; l < a.L; ++l) { const double2 g = c.Kops[(size_t)l * nn + e]; k.x += c.gam[l] * g.x; k.y += c.gam[l] * g.y; }
        } else if (a.L > 0) k = c.Khalf[e];
        c.A1[e] = make_double2(h.y - k.x, -h.x - k.y);     // -i h - k
        c.A2[e] = make_double2(-h.y - k.x, h.x - k.y);     // +i h - k
    }
    __syncthreads();
}

// out = A1 rho + rho A2 + sum_l gamma_l L rho L^dag        (= get_lindbladian, mathmethods.py:187-204, regrouped)
template <bool TD> __device__ void rhs(Ctx &c, double t, const double2 *rho, double2 *out) {
    const LArgs &a = c.a;
    const int nn = a.n * a.n;
    set_time<TD>(c, t);
    bmm<0, 0, false>(out, c.A1, 0, rho, nn, a.n, a.D, 1.0);
    bmm<0, 0, true>(out, rho, nn, c.A2, 0, a.n, a.D, 1.0);
    for (int l = 0; l < a.L; ++l) {
        bmm<0, 0, false>(c.tmp, c.Lops + (size_t)l * nn, 0, rho, nn, a.n, a.D, 1.0);
        bmm<0, 3, true>(out, c.tmp, nn, c.Lops + (size_t)l * nn, 0, a.n, a.D, c.gam[l]);
    }
}

// reverse of rhs at (t, rho) for the output cotangent rbar: rho_bar += ..., control gradient scattered into a.grad
template <bool TD> __device__ void rhs_vjp(Ctx &c, double t, const double2 *rho, const double2 *rbar, double2 *rho_bar) {
    const LArgs &a = c.a;
    const int n = a.n, nn = n * n;
    set_time<TD>(c, t);
    bmm<1, 0, true>(rho_bar, c.A1, 0, rbar, nn, n, a.D, 1.0);
    bmm<0, 1, true>(rho_bar, rbar, nn, c.A2, 0, n, a.D, 1.0);
    for (int l = 0; l < a.L; ++l) {
        bmm<0, 2, false>(c.tmp, rbar, nn, c.Lops + (size_t)l * nn, 0, n, a.D, 1.0);
        bmm<1, 0, true>(rho_bar, c.Lops + (size_t)l * nn, 0, c.tmp, nn, n, a.D, c.gam[l]);
    }
    if (a.have_h && a.KR > 0) {
        // hbar = -i sum_d (rbar_d rho_d^T - rho_d^T rbar_d);  cbar_r = Re sum_ab hbar_ab (A_r)_ab
        // (with series the A are the KC channels, and xbar_r = sum_c gain_cr(t) cbar_c)
        const int nch = (TD && a.KC > 0) ? a.KC : a.KR;
        double part[kMaxKRL];
        for (int r = 0; r < nch; ++r) part[r] = 0.;
        for (int e = threadIdx.x; e < nn; e += blockDim.x) {
            const int i = e / n, j = e - i * n;
            double sr = 0., si = 0.;
            for (int d = 0; d < a.D; ++d) {
                const double2 *R = rbar + (size_t)d * nn, *P = rho + (size_t)d * nn;
                for (int k = 0; k < n; ++k) {
                    const double2 x = R[i * n + k], y = P[j * n + k];          // rbar rho^T
                    sr += x.x * y.x - x.y * y.y; si += x.x * y.y + x.y * y.x;
                    const double2 u = P[k * n + i], v = R[k * n + j];          // rho^T rbar
                    sr -= u.x * v.x - u.y * v.y; si -= u.x * v.y + u.y * v.x;
                }
            }
            const double hr = si, hi = -sr;                                    // -i (sr + i si)
            for (int r = 0; r < nch; ++r) {
                const double2 g = c.Aops[(size_t)r * nn + e];
                part[r] += hr * g.x - hi * g.y;
            }
        }
        const int i0 = c.loc[0], i1 = c.loc[1];
        const double w = (t - c.xs[i0]) / (c.xs[i1] - c.xs[i0]);
        if (TD && a.KC > 0) {
            for (int ch = 0; ch < a.KC; ++ch) {
                const double cb = block_sum(part[ch], c.red);
                if (threadIdx.x == 0) c.cbar[ch] = cb;
            }
            __syncthreads();
            if (threadIdx.x == 0)
                for (int r = 0; r < a.KR; ++r) {
                    double xb = 0.;
                    for (int ch = 0; ch < a.KC; ++ch) xb += c.sv[a.KC + ch * a.KR + r] * c.cbar[ch];
                    a.grad[i0 * a.KR + r] += xb * (1.0 - w);
                    a.grad[i1 * a.KR + r] += xb * w;
                }
        } else {
            for (int r = 0; r < a.KR; ++r) {
                const double cb = block_sum(part[r], c.red);
                if (threadIdx.x == 0) {
                    a.grad[i0 * a.KR + r] += cb * (1.0 - w);
                    a.grad[i1 * a.KR + r] += cb * w;
                }
            }
        }
        __syncthreads();
    }
}

__device__ double rms_of(const double2 *x, int count, double *red) {
    double s = 0.;
    for (int e = threadIdx.x; e < count; e += blockDim.x) s += x[e].x * x[e].x + x[e].y * x[e].y;
    return sqrt(block_sum(s, red) / count);
}

// the six stages of one attempt from (x0, y0, k[0]); fills k[1..6], y1 and returns err
template <bool TD> __device__ double rk_attempt(Ctx &c, double x0, double h, const double2 *y0, double2 *const *k, double2 *ytmp, double2 *y1) {
    const int DE = c.a.D * c.a.n * c.a.n;
    for (int i = 1; i < 6; ++i) {
        for (int e = threadIdx.x; e < DE; e += blockDim.x) {
            double2 acc = make_double2(0., 0.);
            for (int j = 0; j < i; ++j) { acc.x += cA[i][j] * k[j][e].x; acc.y += cA[i][j] * k[j][e].y; }
            ytmp[e] = make_double2(y0[e].x + h * acc.x, y0[e].y + h * acc.y);
        }
        __syncthreads();
        rhs<TD>(c, x0 + cC[i] * h, ytmp, k[i]);
    }
    for (int e = threadIdx.x; e < DE; e += blockDim.x) {
        double2 acc = make_double2(0., 0.);
        for (int j = 0; j < 6; ++j) { acc.x += cB[j] * k[j][e].x; acc.y += cB[j] * k[j][e].y; }
        y1[e] = make_double2(y0[e].x + h * acc.x, y0[e].y + h * acc.y);
    }
    __syncthreads();
    rhs<TD>(c, x0 + h, y1, k[6]);
    double s = 0.;
    for (int e = threadIdx.x; e < DE; e += blockDim.x) {
        double2 acc = make_double2(0., 0.);
        for (int j = 0; j < 7; ++j) { acc.x += cBH[j] * k[j][e].x; acc.y += cBH[j] * k[j][e].y; }
        const double er = (y1[e].x - (y0[e].x + h * acc.x)) / L_ATOL, ei = (y1[e].y - (y0[e].y + h * acc.y)) / L_ATOL;
        s += er * er + ei * ei;
    }
    return sqrt(block_sum(s, c.red) / DE);
}

// cost terms on a density set: returns the value (all threads) and, if seed != nullptr, adds d cost / d rho to it
__device__ double density_costs(Ctx &c, const double2 *rho, bool step_state, bool final_state, double2 *seed) {
    const LArgs &a = c.a;
    const int n = a.n, nn = n * n;
    double val = 0.;
    for (int t = 0; t < a.nterms; ++t) {
        const DTerm tm = a.terms[t];
        if (!((tm.step && step_state) || (!tm.step && final_state))) continue;
        double tot = 0.;
        for (int d = 0; d < a.D; ++d) {
            const int F = a.counts[tm.cnt_off + d];
            double sub = 0.;
            for (int f = 0; f < F; ++f) {
                const double2 *m = a.mats + ((size_t)tm.mat_off + (size_t)d * tm.fmax + f) * nn;
                double zr = 0., zi = 0.;                       // tr(M^dagger rho) = sum conj(M_ab) rho_ab
                for (int e = threadIdx.x; e < nn; e += blockDim.x) {
                    const double2 x = m[e], y = rho[(size_t)d * nn + e];
                    zr += x.x * y.x + x.y * y.y; zi += x.x * y.y - x.y * y.x;
                }
                zr = block_sum(zr, c.red); zi = block_sum(zi, c.red);
                double cr, ci;                                 // seed coefficient on conj(M)
                if (tm.kind == 0) {
                    const double az = sqrt(zr * zr + zi * zi);
                    sub += az;
                    const double kf = az > 0. ? -tm.w / ((double)a.D * n) / az : 0.;
                    cr = kf * zr; ci = -kf * zi;
                } else {
                    const double ir = zr / n, ii = zi / n;
                    sub += (ir * ir + ii * ii) / F;
                    const double kf = tm.w * 2.0 / F / n;
                    cr = kf * ir; ci = -kf * ii;
                }
                if (seed)
                    for (int e = threadIdx.x; e < nn; e += blockDim.x) {
                        const double2 x = m[e];                // conj(M) = (x.x, -x.y)
                        seed[(size_t)d * nn + e].x += cr * x.x + ci * x.y;
                        seed[(size_t)d * nn + e].y += -cr * x.y + ci * x.x;
                    }
            }
            tot += sub;
        }
        val += tm.kind == 0 ? tm.w * (1.0 - tot / ((double)a.D * n)) : tm.w * tot;
    }
    __syncthreads();
    return val;
}

__device__ __forceinline__ bool is_cost_step(int k, int ces) { return k != 0 && (k % ces) == 0; }

// rbar += seeds[step]: cotangents of costs the host evaluated on the densities of this step (qocb_lindblad_backward)
__device__ void add_seed(const LArgs &a, int step, double2 *rbar) {
    const int DE = a.D * a.n * a.n;
    const double2 *s = a.seeds + (size_t)step * DE;
    for (int e = threadIdx.x; e < DE; e += blockDim.x) { rbar[e].x += s[e].x; rbar[e].y += s[e].y; }
    __syncthreads();
}

struct Work {
    double2 *p[24];
};

template <bool TD> __device__ void carve(const LArgs &a, unsigned char *smem, Ctx &c, Work &w, int narr) {
    const int nn = a.n * a.n, DE = a.D * nn;
    double *d = reinterpret_cast<double *>(smem);
    c.A1 = reinterpret_cast<double2 *>(d); d += 2 * nn;
    c.A2 = reinterpret_cast<double2 *>(d); d += 2 * nn;
    c.red = d; d += 32;
    c.coef = d; d += kMaxKRL;
    c.loc = reinterpret_cast<int *>(d); d += 2;
    if (TD) {
        c.sv = d; d += (a.NS + 1) & ~1;
        c.chan = d; d += kMaxKRL;
        c.cbar = d; d += kMaxKRL;
    }
    if (a.ops_in_smem) {                           // the sequential loop re-reads these every stage: keep them on chip
        auto stage = [&](const double *src, int count) {
            double *dst = d;
            for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = src[i];
            d += (count + 1) & ~1;
            return dst;
        };
        c.H0 = reinterpret_cast<const double2 *>(stage(reinterpret_cast<const double *>(c.H0), 2 * nn));
        c.Khalf = reinterpret_cast<const double2 *>(stage(reinterpret_cast<const double *>(c.Khalf), 2 * nn));
        c.Aops = reinterpret_cast<const double2 *>(stage(reinterpret_cast<const double *>(a.Aops), 2 * nn * max(max(a.KR, a.KC), 1)));
        c.Lops = reinterpret_cast<const double2 *>(stage(reinterpret_cast<const double *>(a.Lops), 2 * nn * max(a.L, 1)));
        c.gam = stage(c.gam, max(a.L, 1));
        c.controls = stage(a.controls, max(a.M * a.KR, 1));
        c.xs = stage(a.xs, max(a.M, 1));
        if (TD && a.tdr) c.Kops = reinterpret_cast<const double2 *>(stage(reinterpret_cast<const double *>(a.Kops), 2 * nn * a.L));
        __syncthreads();
    }
    if (TD && a.tdr) c.gam = c.sv + a.KC * (1 + a.KR);  // rates r_l(t), refreshed by every set_time
    double2 *base = a.work_in_smem ? reinterpret_cast<double2 *>(d) : a.work;
    c.tmp = base;
    for (int i = 0; i < narr; ++i) w.p[i] = base + (size_t)(i + 1) * DE;
}

template <bool TD> __global__ void __launch_bounds__(LNT) k_lindblad_forward(LArgs a0, int keep_tape) {
    extern __shared__ __align__(16) unsigned char smem[];
    const LArgs a = member_args(a0);
    Ctx c(a);
    Work w;
    carve<TD>(a, smem, c, w, 12);
    const int DE = a.D * a.n * a.n;
    double2 *y = w.p[0], *y1 = w.p[1], *ytmp = w.p[2], *out = w.p[3];
    double2 *k[7] = {w.p[4], w.p[5], w.p[6], w.p[7], w.p[8], w.p[9], w.p[10]};
    for (int e = threadIdx.x; e < DE; e += blockDim.x) y[e] = a.rho0[e];
    __syncthreads();
    const double dt = a.T / (a.N - 1);
    double cost = 0.;
    long long attempts = 0, accepted = 0;
    int ntape = 0;
    for (int step = 0; step < a.N; ++step) {
        for (int e = threadIdx.x; e < DE; e += blockDim.x) a.states[(size_t)step * DE + e] = y[e];
        const bool st = is_cost_step(step, a.ces), fin = step == a.N - 1;
        if (a.nterms > 0 && (st || fin)) cost += density_costs(c, y, st, fin, nullptr);
        if (threadIdx.x == 0) a.first[step] = ntape;
        if (fin) break;
        const double t0 = step * dt, tf = step * dt + dt;
        // initial step size (mathmethods.py:405-420)
        rhs<TD>(c, t0, y, k[0]);
        const double d0 = rms_of(y, DE, c.red), d1 = rms_of(k[0], DE, c.red);
        const double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        for (int e = threadIdx.x; e < DE; e += blockDim.x) ytmp[e] = make_double2(y[e].x + h0 * k[0][e].x, y[e].y + h0 * k[0][e].y);
        __syncthreads();
        rhs<TD>(c, t0 + h0, ytmp, k[1]);
        double s = 0.;
        for (int e = threadIdx.x; e < DE; e += blockDim.x) { const double dr = k[1][e].x - k[0][e].x, di = k[1][e].y - k[0][e].y; s += dr * dr + di * di; }
        const double d2 = sqrt(block_sum(s, c.red) / DE) / h0;
        const double mx = fmax(d1, d2);
        const double h1 = (mx <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / mx, 1.0 / 6.0);
        double h = fmin(100.0 * h0, h1);
        double xc = t0;
        int hit_idx = -1;
        while (xc <= tf) {
            bool rejected = false;
            double hn;
            for (;;) {
                const double err = rk_attempt<TD>(c, xc, h, y, k, ytmp, y1);
                ++attempts;
                if (err < 1.0) {
                    double fac = (err == 0.0) ? 10.0 : fmin(10.0, 0.9 * pow(err, -0.2));
                    if (rejected) fac = fmin(1.0, fac);
                    hn = h * fac;
                    break;
                }
                rejected = true;
                h = h * fmax(0.2, 0.9 * pow(err, -0.2));
            }
            ++accepted;
            const double xn = xc + h;
            if (keep_tape) {
                if (ntape >= a.cap) { if (threadIdx.x == 0) *a.err_flag = 1; }
                else {
                    if (threadIdx.x == 0) { a.tape_x[ntape] = xc; a.tape_h[ntape] = h; }
                    for (int e = threadIdx.x; e < DE; e += blockDim.x) { a.tape_y[(size_t)ntape * DE + e] = y[e]; a.tape_k1[(size_t)ntape * DE + e] = k[0][e]; }
                }
            }
            if (xc <= tf && tf <= xn) {                                  // dense output (mathmethods.py:263-304)
                const double hh = xn - xc, th = (tf - xc) / hh;
                for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                    double o[2];
                    for (int q = 0; q < 2; ++q) {
                        const double y0v = q ? y[e].y : y[e].x, y1v = q ? y1[e].y : y1[e].x;
                        const double k0v = q ? k[0][e].y : k[0][e].x, k6v = q ? k[6][e].y : k[6][e].x;
                        double sd = 0.;
                        for (int j = 0; j < 7; ++j) sd += cD[j] * (q ? k[j][e].y : k[j][e].x);
                        const double r2 = y1v - y0v, r3 = y0v + hh * k0v - y1v, r4 = 2.0 * (y1v - y0v) - hh * (k0v + k6v), r5 = hh * sd;
                        o[q] = y0v + th * (r2 + r3) - th * th * (r3 - r4 - r5) - th * th * th * (r4 + 2.0 * r5) + th * th * th * th * r5;
                    }
                    out[e] = make_double2(o[0], o[1]);
                }
                hit_idx = ntape;
            }
            ++ntape;
            __syncthreads();
            double2 *t = y; y = y1; y1 = t;                               // y <- y1
            t = k[0]; k[0] = k[6]; k[6] = t;                              // FSAL (mathmethods.py:477)
            xc = xn; h = hn;
        }
        if (threadIdx.x == 0) a.hit[step] = hit_idx;
        for (int e = threadIdx.x; e < DE; e += blockDim.x) y[e] = out[e];
        __syncthreads();
    }
    if (threadIdx.x == 0) { *a.cost = cost; a.stats[0] = attempts; a.stats[1] = accepted; if (TD) *a.tseen = c.tseen; }
}

template <bool TD> __global__ void __launch_bounds__(LNT) k_lindblad_backward(LArgs a0) {
    extern __shared__ __align__(16) unsigned char smem[];
    const LArgs a = member_args(a0);
    Ctx c(a);
    Work w;
    if (*a.err_flag) return;                          // the forward pass overflowed this member's tape: hit[] is not valid
    if (TD && *a.tseen > a.segs * a.seg_w) return;    // the forward pass left the table: it is run again
    carve<TD>(a, smem, c, w, 22);
    const int DE = a.D * a.n * a.n;
    double2 *k[7] = {w.p[0], w.p[1], w.p[2], w.p[3], w.p[4], w.p[5], w.p[6]};
    double2 *kb[7] = {w.p[7], w.p[8], w.p[9], w.p[10], w.p[11], w.p[12], w.p[13]};
    double2 *y1 = w.p[14], *ytmp = w.p[15], *y0b = w.p[16], *y1b = w.p[17], *zb = w.p[18], *rbar = w.p[19], *k1b_next = w.p[20];
    for (int e = threadIdx.x; e < a.M * a.KR; e += blockDim.x) a.grad[e] = 0.;
    for (int e = threadIdx.x; e < DE; e += blockDim.x) rbar[e] = make_double2(0., 0.);
    __syncthreads();
    if (a.seeds) add_seed(a, a.N - 1, rbar);
    if (a.nterms > 0) density_costs(c, a.states + (size_t)(a.N - 1) * DE, is_cost_step(a.N - 1, a.ces), true, rbar);
    for (int step = a.N - 2; step >= 0; --step) {
        const int first = a.first[step], last = a.hit[step];
        const double tf = step * (a.T / (a.N - 1)) + a.T / (a.N - 1);
        for (int e = threadIdx.x; e < DE; e += blockDim.x) k1b_next[e] = make_double2(0., 0.);
        // rbar: cotangent of the interval's output; becomes ybar_next after the dense-output step
        for (int i = last; i >= first; --i) {
            const double x0 = a.tape_x[i], h = a.tape_h[i];
            const double2 *y0 = a.tape_y + (size_t)i * DE;
            for (int e = threadIdx.x; e < DE; e += blockDim.x) k[0][e] = a.tape_k1[(size_t)i * DE + e];
            __syncthreads();
            rk_attempt<TD>(c, x0, h, y0, k, ytmp, y1);
            for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                for (int j = 0; j < 6; ++j) kb[j][e] = make_double2(0., 0.);
                kb[6][e] = k1b_next[e];
                y0b[e] = make_double2(0., 0.);
            }
            if (i == last) {                                              // out = dense(...), seed rbar
                const double th = (tf - x0) / h;
                const double c2 = th, c3 = th - th * th, c4 = th * th - th * th * th, c5 = th * th - 2.0 * th * th * th + th * th * th * th;
                for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                    const double2 ob = rbar[e];
                    const double f0 = 1.0 - c2 + c3 - 2.0 * c4, f1 = c2 - c3 + 2.0 * c4;
                    y0b[e] = make_double2(f0 * ob.x, f0 * ob.y);
                    y1b[e] = make_double2(f1 * ob.x, f1 * ob.y);
                    const double g0 = h * (c3 - c4), g6 = -h * c4;
                    kb[0][e].x += g0 * ob.x; kb[0][e].y += g0 * ob.y;
                    kb[6][e].x += g6 * ob.x; kb[6][e].y += g6 * ob.y;
                    for (int j = 0; j < 7; ++j) { const double gj = h * cD[j] * c5; kb[j][e].x += gj * ob.x; kb[j][e].y += gj * ob.y; }
                }
            } else {
                for (int e = threadIdx.x; e < DE; e += blockDim.x) y1b[e] = rbar[e];      // ybar_next
            }
            __syncthreads();
            // ks[6] = rhs(x0 + h, y1)
            rhs_vjp<TD>(c, x0 + h, y1, kb[6], y1b);
            // y1 = y0 + h sum b_j k_j
            for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                y0b[e].x += y1b[e].x; y0b[e].y += y1b[e].y;
                for (int j = 0; j < 6; ++j) { kb[j][e].x += h * cB[j] * y1b[e].x; kb[j][e].y += h * cB[j] * y1b[e].y; }
            }
            __syncthreads();
            for (int s = 5; s >= 1; --s) {
                for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                    double2 acc = make_double2(0., 0.);
                    for (int j = 0; j < s; ++j) { acc.x += cA[s][j] * k[j][e].x; acc.y += cA[s][j] * k[j][e].y; }
                    ytmp[e] = make_double2(y0[e].x + h * acc.x, y0[e].y + h * acc.y);
                    zb[e] = make_double2(0., 0.);
                }
                __syncthreads();
                rhs_vjp<TD>(c, x0 + cC[s] * h, ytmp, kb[s], zb);
                for (int e = threadIdx.x; e < DE; e += blockDim.x) {
                    y0b[e].x += zb[e].x; y0b[e].y += zb[e].y;
                    for (int j = 0; j < s; ++j) { kb[j][e].x += h * cA[s][j] * zb[e].x; kb[j][e].y += h * cA[s][j] * zb[e].y; }
                }
                __syncthreads();
            }
            for (int e = threadIdx.x; e < DE; e += blockDim.x) { rbar[e] = y0b[e]; k1b_next[e] = kb[0][e]; }
            __syncthreads();
        }
        // k1 of the interval's first step = rhs(t0, y_in)
        rhs_vjp<TD>(c, step * (a.T / (a.N - 1)), a.states + (size_t)step * DE, k1b_next, rbar);
        if (a.nterms > 0 && is_cost_step(step, a.ces)) density_costs(c, a.states + (size_t)step * DE, true, false, rbar);
        if (a.seeds && step > 0) add_seed(a, step, rbar);     // row 0: the cotangent of rho0 is not needed
    }
}

// member mean of an ensemble: cost and gradient summed in member order 0..E-1 and divided by E, largest stage time
// over members (deterministic: no atomics).  Thread j < cnt owns gradient entry j; thread cnt the cost and stage time.
__global__ void k_lindblad_member_mean(int E, int cnt, const double *cost, const double *grad, const double *tseen,
                                       double *cost_mean, double *grad_mean, double *tseen_max) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < cnt) {
        double s = 0.;
        for (int e = 0; e < E; ++e) s += grad[(size_t)e * cnt + j];
        grad_mean[j] = s / E;
    } else if (j == cnt) {
        double s = 0.;
        for (int e = 0; e < E; ++e) s += cost[e];
        *cost_mean = s / E;
        if (tseen) {
            double t = tseen[0];
            for (int e = 1; e < E; ++e) t = fmax(t, tseen[e]);
            *tseen_max = t;
        }
    }
}

thread_local std::string g_lerr;

template <class T> struct Buf {
    T *p = nullptr; size_t n = 0;
    cudaError_t alloc(size_t count) {
        if (p) cudaFree(p);
        p = nullptr; n = count;
        if (!count) return cudaSuccess;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; n = 0; }
        return e;
    }
    ~Buf() { if (p) cudaFree(p); }
};

}  // namespace

struct qocb_lplan {
    qocb_lindblad_problem pb;
    int E = 1;                                     // ensemble members (one CTA each)
    bool ens_set = false;                          // qocb_lindblad_set_ensemble since the last qocb_lindblad_set_operators
    int cap = 0;                                   // tape capacity of one member
    bool ops_set = false, rho_set = false, costs_dirty = true, series_set = false;
    int NS = 0, segs = 0, deg = 0;                 // time series: NS = KC*(1+KR) + (time_dependent_rates ? L : 0)
    double seg_w = 0.;
    cudaStream_t stream = nullptr;
    bool tape_ok = false;                          // the last evaluation was a successful qocb_lindblad_forward
    Buf<double2> H0, Aops, Lops, Khalf, Kops, rho0, mats, states, tape_y, tape_k1, work, seeds;
    Buf<double> gam, controls, xs, cost, tape_x, tape_h, grad, series, tseen, cost_mean, grad_mean, tseen_max;
    Buf<int> counts, first, hit, err_flag;
    Buf<long long> stats;
    Buf<DTerm> terms;
    std::vector<DTerm> h_terms; std::vector<double2> h_mats; std::vector<int> h_counts;
    std::vector<double> h_h0, h_gam, h_lops;       // the plan's operators (E > 1): members without their own take these
    size_t smem_fwd = 0, smem_bwd = 0;
    int in_smem_fwd = 0, in_smem_bwd = 0, ops_in_smem = 0;
    std::string err;
};

namespace {
int lfail(qocb_lplan *p, const char *msg, int rc) { if (p) p->err = msg; g_lerr = msg; return rc; }
#define LTRY(p, expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { char b__[512]; snprintf(b__, sizeof(b__), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); return lfail(p, b__, -2); } } while (0)

LArgs make_largs(qocb_lplan *p) {
    LArgs a;
    a.n = p->pb.hilbert_size; a.D = p->pb.density_count; a.KR = p->pb.control_count; a.M = p->pb.control_eval_count;
    a.N = p->pb.system_eval_count; a.L = p->pb.lindblad_count; a.ces = p->pb.cost_eval_step; a.have_h = p->pb.have_hamiltonian;
    a.nterms = (int)p->h_terms.size(); a.cap = p->cap; a.T = p->pb.evolution_time;
    a.H0 = p->H0.p; a.Aops = p->Aops.p; a.Lops = p->Lops.p; a.Khalf = p->Khalf.p; a.gam = p->gam.p; a.controls = p->controls.p;
    a.xs = p->xs.p; a.rho0 = p->rho0.p; a.terms = p->terms.p; a.mats = p->mats.p; a.counts = p->counts.p;
    a.states = p->states.p; a.cost = p->cost.p; a.tape_x = p->tape_x.p; a.tape_h = p->tape_h.p; a.tape_y = p->tape_y.p;
    a.tape_k1 = p->tape_k1.p; a.first = p->first.p; a.hit = p->hit.p; a.stats = p->stats.p; a.err_flag = p->err_flag.p;
    a.work = p->work.p; a.work_in_smem = 0; a.ops_in_smem = p->ops_in_smem; a.grad = p->grad.p;
    a.KC = p->pb.channel_count; a.tdr = p->pb.time_dependent_rates; a.NS = p->NS; a.segs = p->segs; a.deg = p->deg;
    a.seg_w = p->seg_w; a.series = p->series.p; a.Kops = p->Kops.p; a.tseen = p->tseen.p; a.seeds = nullptr;
    return a;
}

// kh += 1/2 sum_l gammas_l L_l^dag L_l, or the per-operator 1/2 L_l^dag L_l into kh + l n^2 when gammas is null
void build_khalf(const double *lops, const double *gammas, int n, int L, double *kh) {
    const size_t nn = (size_t)n * n;
    for (int l = 0; l < L; ++l) {
        const double *Lm = lops + 2 * (size_t)l * nn;
        double *K = gammas ? kh : kh + 2 * (size_t)l * nn;
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) {
                double sr = 0., si = 0.;
                for (int k = 0; k < n; ++k) {                             // conj(L[k][i]) * L[k][j]
                    const double ar = Lm[2 * (k * n + i)], ai = -Lm[2 * (k * n + i) + 1], br = Lm[2 * (k * n + j)], bi = Lm[2 * (k * n + j) + 1];
                    sr += ar * br - ai * bi; si += ar * bi + ai * br;
                }
                if (gammas) { K[2 * (i * n + j)] += 0.5 * gammas[l] * sr; K[2 * (i * n + j) + 1] += 0.5 * gammas[l] * si; }
                else { K[2 * (i * n + j)] = 0.5 * sr; K[2 * (i * n + j) + 1] = 0.5 * si; }
            }
    }
}

int upload_lcosts(qocb_lplan *p) {
    if (!p->costs_dirty) return 0;
    LTRY(p, p->terms.alloc(std::max<size_t>(1, p->h_terms.size())));
    LTRY(p, p->mats.alloc(std::max<size_t>(1, p->h_mats.size())));
    LTRY(p, p->counts.alloc(std::max<size_t>(1, p->h_counts.size())));
    if (!p->h_terms.empty()) {
        LTRY(p, cudaMemcpy(p->terms.p, p->h_terms.data(), sizeof(DTerm) * p->h_terms.size(), cudaMemcpyHostToDevice));
        LTRY(p, cudaMemcpy(p->mats.p, p->h_mats.data(), sizeof(double2) * p->h_mats.size(), cudaMemcpyHostToDevice));
        LTRY(p, cudaMemcpy(p->counts.p, p->h_counts.data(), sizeof(int) * p->h_counts.size(), cudaMemcpyHostToDevice));
    }
    p->costs_dirty = false;
    return 0;
}

int lindblad_threads(const qocb_lplan *p) {
    const int DEl = p->pb.density_count * p->pb.hilbert_size * p->pb.hilbert_size;
    return DEl <= 64 ? 32 : (DEl <= 256 ? 128 : LNT);
}

// enqueues the forward pass (keep_tape: record the reverse-pass tape) after uploading the controls
int launch_forward(qocb_lplan *p, const double *controls, bool keep_tape) {
    if (!p->ops_set || !p->rho_set) return lfail(p, "operators and densities must be set before evaluation", -1);
    if (p->NS > 0 && !p->series_set) return lfail(p, "time-dependent operators need qocb_lindblad_set_time_series before evaluation", -1);
    if (p->E > 1 && !p->ens_set) return lfail(p, "an ensemble plan needs qocb_lindblad_set_ensemble after qocb_lindblad_set_operators", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    if (upload_lcosts(p)) return -2;
    const size_t cnt = (size_t)p->pb.control_eval_count * p->pb.control_count;
    if (cnt) {
        if (!controls) return lfail(p, "controls is null", -1);
        LTRY(p, cudaMemcpyAsync(p->controls.p, controls, sizeof(double) * cnt, cudaMemcpyHostToDevice, p->stream));
    }
    LTRY(p, cudaMemsetAsync(p->err_flag.p, 0, sizeof(int) * p->E, p->stream));
    LArgs a = make_largs(p);
    a.work_in_smem = p->in_smem_fwd;
    if (p->NS > 0) k_lindblad_forward<true><<<p->E, lindblad_threads(p), p->smem_fwd, p->stream>>>(a, keep_tape ? 1 : 0);
    else k_lindblad_forward<false><<<p->E, lindblad_threads(p), p->smem_fwd, p->stream>>>(a, keep_tape ? 1 : 0);
    LTRY(p, cudaGetLastError());
    return 0;
}

// enqueues the reverse pass over the tape of the last forward pass; seeds: device [N][D*n*n] or null
int launch_backward(qocb_lplan *p, const double2 *seeds) {
    LArgs a = make_largs(p);
    a.work_in_smem = p->in_smem_bwd;
    a.seeds = seeds;
    if (p->NS > 0) k_lindblad_backward<true><<<p->E, lindblad_threads(p), p->smem_bwd, p->stream>>>(a);
    else k_lindblad_backward<false><<<p->E, lindblad_threads(p), p->smem_bwd, p->stream>>>(a);
    LTRY(p, cudaGetLastError());
    return 0;
}

// enqueues the member mean of an ensemble evaluation (E > 1); with_grad: the reverse pass ran
int launch_mean(qocb_lplan *p, bool with_grad) {
    const int cnt = with_grad ? p->pb.control_eval_count * p->pb.control_count : 0;
    k_lindblad_member_mean<<<cnt / 256 + 1, 256, 0, p->stream>>>(p->E, cnt, p->cost.p, p->grad.p, p->NS > 0 ? p->tseen.p : nullptr,
                                                               p->cost_mean.p, p->grad_mean.p, p->tseen_max.p);
    LTRY(p, cudaGetLastError());
    return 0;
}

// copies the requested results to the host, waits for the stream and reports a stage time beyond the series (-5) or a
// full tape (-4) of the last forward pass.  An ensemble returns the member mean, every member's final densities [E][D][n][n],
// the largest stage time over members and -4 when any member's tape overflowed.
int finish_lindblad(qocb_lplan *p, double *cost, double *grad, double *final_densities) {
    const size_t cnt = (size_t)p->pb.control_eval_count * p->pb.control_count;
    const bool ens = p->E > 1;
    std::vector<int> flags(p->E, 0);
    LTRY(p, cudaMemcpyAsync(flags.data(), p->err_flag.p, sizeof(int) * p->E, cudaMemcpyDeviceToHost, p->stream));
    if (cost) LTRY(p, cudaMemcpyAsync(cost, ens ? p->cost_mean.p : p->cost.p, sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    if (grad && cnt) LTRY(p, cudaMemcpyAsync(grad, ens ? p->grad_mean.p : p->grad.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost, p->stream));
    const size_t DE = (size_t)p->pb.density_count * p->pb.hilbert_size * p->pb.hilbert_size, N = p->pb.system_eval_count;
    if (final_densities && !ens)
        LTRY(p, cudaMemcpyAsync(final_densities, p->states.p + (N - 1) * DE, sizeof(double2) * DE,
                                cudaMemcpyDeviceToHost, p->stream));
    if (final_densities && ens)                                  // row N-1 of every member's [N][DE] block
        LTRY(p, cudaMemcpy2DAsync(final_densities, sizeof(double2) * DE, p->states.p + (N - 1) * DE, sizeof(double2) * N * DE,
                                  sizeof(double2) * DE, p->E, cudaMemcpyDeviceToHost, p->stream));
    double tseen = 0.;
    if (p->NS > 0) LTRY(p, cudaMemcpyAsync(&tseen, ens ? p->tseen_max.p : p->tseen.p, sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    LTRY(p, cudaStreamSynchronize(p->stream));
    if (p->NS > 0 && tseen > p->segs * p->seg_w)
        return lfail(p, "a Runge-Kutta stage time lies beyond the time series: extend it (qocb_lindblad_max_stage_time)", -5);
    for (int f : flags)
        if (f) return lfail(p, "the Runge-Kutta tape is full: raise max_rk_steps", -4);
    return 0;
}

}  // namespace

extern "C" {

const char *qocb_lindblad_last_error(const qocb_lplan *p) { return p ? p->err.c_str() : g_lerr.c_str(); }

int qocb_lindblad_create(const qocb_lindblad_problem *pb, qocb_lplan **out) {
    if (!pb || !out) return lfail(nullptr, "null argument", -1);
    *out = nullptr;
    if (pb->hilbert_size < 1 || pb->hilbert_size > 64) return lfail(nullptr, "hilbert_size must be in [1, 64] for the Lindblad path", -1);
    if (pb->density_count < 1 || pb->system_eval_count < 2 || pb->cost_eval_step < 1) return lfail(nullptr, "density_count >= 1, system_eval_count >= 2, cost_eval_step >= 1 required", -1);
    if (pb->control_count < 0 || pb->control_count > kMaxKRL) return lfail(nullptr, "control_count (real channels) must be in [0, 16]", -1);
    if (pb->control_count > 0 && pb->control_eval_count < 2) return lfail(nullptr, "control_eval_count must be >= 2", -1);
    if (pb->lindblad_count < 0) return lfail(nullptr, "lindblad_count must be >= 0", -1);
    if (pb->channel_count < 0 || pb->channel_count > kMaxKRL) return lfail(nullptr, "channel_count must be in [0, 16]", -1);
    if (pb->channel_count > 0 && !pb->have_hamiltonian) return lfail(nullptr, "channel_count > 0 needs have_hamiltonian", -1);
    if (pb->time_dependent_rates != 0 && (pb->time_dependent_rates != 1 || pb->lindblad_count < 1))
        return lfail(nullptr, "time_dependent_rates must be 0 or 1, and 1 needs lindblad_count >= 1", -1);
    if (pb->ensemble_count < 0) return lfail(nullptr, "ensemble_count must be >= 0", -1);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return lfail(nullptr, "no CUDA device available (this library has no CPU path)", -2);
    qocb_lplan *p = new qocb_lplan();
    p->pb = *pb;
#define CTRY(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { char b__[512]; snprintf(b__, sizeof(b__), "%s failed: %s", #expr, cudaGetErrorString(e__)); g_lerr = b__; delete p; return -2; } } while (0)
    CTRY(cudaSetDevice(pb->device));
    CTRY(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    const int n = pb->hilbert_size, nn = n * n, D = pb->density_count, KR = pb->control_count, M = pb->control_eval_count;
    const int N = pb->system_eval_count, L = pb->lindblad_count, KC = pb->channel_count, tdr = pb->time_dependent_rates;
    const size_t DE = (size_t)D * nn;
    const size_t E = p->E = std::max(1, pb->ensemble_count);
    p->NS = KC * (1 + KR) + (tdr ? L : 0);
    // tape of one member: 512 MiB for one member, 8 GiB shared by the members of an ensemble, within [4096, 2^20] steps
    const size_t tape_bytes = E == 1 ? (size_t)512 << 20 : ((size_t)8 << 30) / E;
    p->cap = pb->max_rk_steps > 0 ? pb->max_rk_steps : (int)std::max<size_t>(4096, std::min<size_t>((size_t)1 << 20, tape_bytes / (2 * DE * sizeof(double2))));
    CTRY(p->H0.alloc(E * nn)); CTRY(p->Aops.alloc((size_t)std::max(1, std::max(KR, KC)) * nn)); CTRY(p->Lops.alloc((size_t)std::max(1, L) * nn));
    if (tdr) CTRY(p->Kops.alloc((size_t)L * nn));
    if (p->NS > 0) { CTRY(p->tseen.alloc(E)); CTRY(cudaMemset(p->tseen.p, 0, sizeof(double) * E)); }
    CTRY(p->Khalf.alloc(E * nn)); CTRY(p->gam.alloc(E * std::max(1, L))); CTRY(p->controls.alloc(std::max<size_t>(1, (size_t)M * KR)));
    CTRY(p->xs.alloc(std::max(1, M))); CTRY(p->rho0.alloc(DE)); CTRY(p->states.alloc(E * N * DE)); CTRY(p->cost.alloc(E));
    CTRY(p->tape_x.alloc(E * p->cap)); CTRY(p->tape_h.alloc(E * p->cap)); CTRY(p->tape_y.alloc(E * p->cap * DE)); CTRY(p->tape_k1.alloc(E * p->cap * DE));
    CTRY(p->first.alloc(E * N)); CTRY(p->hit.alloc(E * N)); CTRY(p->err_flag.alloc(E)); CTRY(p->stats.alloc(2 * E));
    CTRY(p->grad.alloc(E * std::max<size_t>(1, (size_t)M * KR)));
    if (E > 1) {
        CTRY(p->cost_mean.alloc(1)); CTRY(p->grad_mean.alloc(std::max<size_t>(1, (size_t)M * KR))); CTRY(p->tseen_max.alloc(1));
        CTRY(cudaMemset(p->tseen_max.p, 0, sizeof(double)));
    }
    CTRY(cudaMemset(p->H0.p, 0, sizeof(double2) * E * nn)); CTRY(cudaMemset(p->Khalf.p, 0, sizeof(double2) * E * nn));
    // control_eval_times = numpy.linspace(0, T, M) (qoc/models/programstate.py:41)
    if (M > 0) {
        std::vector<double> xs(M);
        const double T = pb->evolution_time;
        for (int m = 0; m < M; ++m) xs[m] = (M == 1) ? 0.0 : (m == M - 1 ? T : m * (T / (M - 1)));
        CTRY(cudaMemcpy(p->xs.p, xs.data(), sizeof(double) * M, cudaMemcpyHostToDevice));
    }
    size_t fixed = sizeof(double) * (4 * (size_t)nn + 32 + kMaxKRL + 2);
    if (p->NS > 0) fixed += sizeof(double) * (((size_t)p->NS + 1) / 2 * 2 + 2 * kMaxKRL);     // series values, coef_c, cbar_c
    const size_t limit = 200 * 1024;
    const size_t ops_doubles = 2 * (size_t)nn * (2 + std::max(std::max(KR, KC), 1) + std::max(L, 1) + (tdr ? L : 0)) + std::max(L, 1) +
                               std::max(M * KR, 1) + std::max(M, 1) + 16;
    p->ops_in_smem = ops_doubles * sizeof(double) <= 48 * 1024;
    if (p->ops_in_smem) fixed += ops_doubles * sizeof(double);
    const size_t need_f = fixed + sizeof(double2) * 13 * DE, need_b = fixed + sizeof(double2) * 23 * DE;
    p->in_smem_fwd = need_f <= limit; p->in_smem_bwd = need_b <= limit;
    p->smem_fwd = p->in_smem_fwd ? need_f : fixed; p->smem_bwd = p->in_smem_bwd ? need_b : fixed;
    if (fixed > limit) { g_lerr = "hilbert_size too large for the Lindblad kernels' shared-memory operators"; delete p; return -1; }
    CTRY(p->work.alloc((p->in_smem_fwd && p->in_smem_bwd ? 1 : E) * 24 * DE));   // one slice per member when it is used
    CTRY(cudaFuncSetAttribute(k_lindblad_forward<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    CTRY(cudaFuncSetAttribute(k_lindblad_backward<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    CTRY(cudaFuncSetAttribute(k_lindblad_forward<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
    CTRY(cudaFuncSetAttribute(k_lindblad_backward<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
#undef CTRY
    *out = p;
    return 0;
}

int qocb_lindblad_destroy(qocb_lplan *p) {
    if (!p) return 0;
    cudaSetDevice(p->pb.device);
    if (p->stream) { cudaStreamSynchronize(p->stream); cudaStreamDestroy(p->stream); }
    delete p;
    return 0;
}

/* h0: [n][n] or NULL (have_hamiltonian = 0); a_ops: [KR][n][n]; gammas: [L]; lops: [L][n][n] */
int qocb_lindblad_set_operators(qocb_lplan *p, const double *h0, const double *a_ops, const double *gammas, const double *lops) {
    if (!p) return -1;
    LTRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, nn = n * n, L = p->pb.lindblad_count;
    const int KA = p->pb.channel_count > 0 ? p->pb.channel_count : p->pb.control_count;     // operators in a_ops
    if (p->pb.have_hamiltonian) {
        if (!h0 || (KA > 0 && !a_ops)) return lfail(p, "h0 / a_ops missing", -1);
        LTRY(p, cudaMemcpy(p->H0.p, h0, sizeof(double2) * nn, cudaMemcpyHostToDevice));
        if (KA > 0) LTRY(p, cudaMemcpy(p->Aops.p, a_ops, sizeof(double2) * (size_t)KA * nn, cudaMemcpyHostToDevice));
    }
    if (L > 0 && p->pb.time_dependent_rates) {                              // per-operator 1/2 B_l^dag B_l; rates come from the series
        if (!lops) return lfail(p, "lops missing", -1);
        LTRY(p, cudaMemcpy(p->Lops.p, lops, sizeof(double2) * (size_t)L * nn, cudaMemcpyHostToDevice));
        std::vector<double> kh(2 * (size_t)L * nn, 0.0);
        build_khalf(lops, nullptr, n, L, kh.data());
        LTRY(p, cudaMemcpy(p->Kops.p, kh.data(), sizeof(double2) * (size_t)L * nn, cudaMemcpyHostToDevice));
    } else if (L > 0) {
        if (!gammas || !lops) return lfail(p, "gammas / lops missing", -1);
        LTRY(p, cudaMemcpy(p->gam.p, gammas, sizeof(double) * L, cudaMemcpyHostToDevice));
        LTRY(p, cudaMemcpy(p->Lops.p, lops, sizeof(double2) * (size_t)L * nn, cudaMemcpyHostToDevice));
        std::vector<double> kh(2 * (size_t)nn, 0.0);                         // 1/2 sum_l gamma_l L^dag L (mathmethods.py:193-194)
        build_khalf(lops, gammas, n, L, kh.data());
        LTRY(p, cudaMemcpy(p->Khalf.p, kh.data(), sizeof(double2) * nn, cudaMemcpyHostToDevice));
    }
    if (p->E > 1) {                                                         // kept for the members qocb_lindblad_set_ensemble leaves alone
        p->h_h0.assign(2 * (size_t)nn, 0.0);
        if (p->pb.have_hamiltonian) std::copy(h0, h0 + 2 * (size_t)nn, p->h_h0.begin());
        p->h_gam.assign(gammas && L > 0 && !p->pb.time_dependent_rates ? gammas : nullptr,
                        gammas && L > 0 && !p->pb.time_dependent_rates ? gammas + L : nullptr);
        p->h_lops.assign(lops ? lops : nullptr, lops ? lops + 2 * (size_t)L * nn : nullptr);
        p->ens_set = false;
    }
    p->ops_set = true;
    p->tape_ok = false;
    return 0;
}

/* h0s: [E][n][n] or NULL; gammas: [E][L] or NULL (NULL: every member takes the plan's from qocb_lindblad_set_operators) */
int qocb_lindblad_set_ensemble(qocb_lplan *p, const double *h0s, const double *gammas) {
    if (!p) return -1;
    if (p->E <= 1) return lfail(p, "qocb_lindblad_set_ensemble needs ensemble_count > 1", -1);
    if (!p->ops_set) return lfail(p, "qocb_lindblad_set_operators must come before qocb_lindblad_set_ensemble", -1);
    if (h0s && (!p->pb.have_hamiltonian || p->pb.channel_count > 0))
        return lfail(p, "member drifts need a time-independent hamiltonian (have_hamiltonian = 1, channel_count = 0)", -1);
    if (gammas && p->pb.time_dependent_rates) return lfail(p, "member rates need time_dependent_rates = 0", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, L = p->pb.lindblad_count, E = p->E;
    const size_t nn = (size_t)n * n, Lg = std::max(L, 1);
    std::vector<double> H(2 * E * nn), G(E * Lg, 0.0), K(2 * E * nn, 0.0);
    for (int e = 0; e < E; ++e) {
        const double *h = h0s ? h0s + 2 * e * nn : p->h_h0.data();
        std::copy(h, h + 2 * nn, H.begin() + 2 * e * nn);
        if (L > 0 && !p->pb.time_dependent_rates) {
            const double *g = gammas ? gammas + (size_t)e * L : p->h_gam.data();
            std::copy(g, g + L, G.begin() + e * Lg);
            build_khalf(p->h_lops.data(), g, n, L, K.data() + 2 * e * nn);
        }
    }
    LTRY(p, cudaStreamSynchronize(p->stream));
    LTRY(p, cudaMemcpy(p->H0.p, H.data(), sizeof(double) * H.size(), cudaMemcpyHostToDevice));
    LTRY(p, cudaMemcpy(p->gam.p, G.data(), sizeof(double) * G.size(), cudaMemcpyHostToDevice));
    LTRY(p, cudaMemcpy(p->Khalf.p, K.data(), sizeof(double) * K.size(), cudaMemcpyHostToDevice));
    p->ens_set = true;
    p->tape_ok = false;
    return 0;
}

/* series: [segments][degree+1][NS] Chebyshev coefficients (the constant one not halved) on [s w, (s+1) w] */
int qocb_lindblad_set_time_series(qocb_lplan *p, int32_t segments, int32_t degree, double segment_width, const double *series) {
    if (!p || !series) return lfail(p, "null argument", -1);
    if (p->NS == 0) return lfail(p, "this plan has neither operator channels nor time-dependent rates", -1);
    if (segments < 1 || degree < 0 || degree > 64 || !(segment_width > 0.0)) return lfail(p, "bad time series shape", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    const size_t count = (size_t)segments * (degree + 1) * p->NS;
    LTRY(p, cudaStreamSynchronize(p->stream));
    LTRY(p, p->series.alloc(count));
    LTRY(p, cudaMemcpy(p->series.p, series, sizeof(double) * count, cudaMemcpyHostToDevice));
    p->segs = segments; p->deg = degree; p->seg_w = segment_width;
    p->series_set = true;
    p->tape_ok = false;
    return 0;
}

/* largest Runge-Kutta stage time of the last forward pass (plans with a time series) */
int qocb_lindblad_max_stage_time(qocb_lplan *p, double *t) {
    if (!p || !t) return lfail(p, "null argument", -1);
    if (p->NS == 0) return lfail(p, "this plan has no time series", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    LTRY(p, cudaMemcpy(t, p->E > 1 ? p->tseen_max.p : p->tseen.p, sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

int qocb_lindblad_set_densities(qocb_lplan *p, const double *rho0) {
    if (!p || !rho0) return lfail(p, "null argument", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    const size_t DE = (size_t)p->pb.density_count * p->pb.hilbert_size * p->pb.hilbert_size;
    LTRY(p, cudaMemcpy(p->rho0.p, rho0, sizeof(double2) * DE, cudaMemcpyHostToDevice));
    p->rho_set = true;
    p->tape_ok = false;
    return 0;
}

/* mats: [D][fmax][n][n] complex; counts: [D] or NULL; kind: QOCB_LCOST_*; weight = cost_multiplier / normalisation */
int qocb_lindblad_add_cost(qocb_lplan *p, int32_t kind, int32_t step_cost, double weight, const double *mats, const int32_t *counts, int32_t fmax) {
    if (!p || !mats) return lfail(p, "null argument", -1);
    if (kind < 0 || kind > 1 || fmax < 1) return lfail(p, "bad cost kind or fmax", -1);
    const int n = p->pb.hilbert_size, nn = n * n, D = p->pb.density_count;
    DTerm t;
    t.kind = kind; t.step = step_cost ? 1 : 0; t.fmax = fmax; t.w = weight;
    t.mat_off = (int)(p->h_mats.size() / nn); t.cnt_off = (int)p->h_counts.size();
    for (int d = 0; d < D; ++d) {
        const int F = counts ? counts[d] : fmax;
        if (F < 1 || F > fmax) return lfail(p, "counts[d] must be in [1, fmax]", -1);
        p->h_counts.push_back(F);
    }
    const double2 *m = reinterpret_cast<const double2 *>(mats);
    p->h_mats.insert(p->h_mats.end(), m, m + (size_t)D * fmax * nn);
    p->h_terms.push_back(t);
    p->costs_dirty = true;
    p->tape_ok = false;
    return 0;
}

int qocb_lindblad_cost(qocb_lplan *p, const double *controls, double *cost, double *final_densities) {
    if (!p) return -1;
    p->tape_ok = false;
    if (int rc = launch_forward(p, controls, false)) return rc;
    if (p->E > 1)
        if (int rc = launch_mean(p, false)) return rc;
    return finish_lindblad(p, cost, nullptr, final_densities);
}

int qocb_lindblad_cost_and_grad(qocb_lplan *p, const double *controls, double *cost, double *grad, double *final_densities) {
    if (!p) return -1;
    p->tape_ok = false;
    if (int rc = launch_forward(p, controls, true)) return rc;
    const bool with_grad = (size_t)p->pb.control_eval_count * p->pb.control_count > 0;
    if (with_grad)
        if (int rc = launch_backward(p, nullptr)) return rc;
    if (p->E > 1)
        if (int rc = launch_mean(p, with_grad)) return rc;
    return finish_lindblad(p, cost, grad, final_densities);
}

int qocb_lindblad_forward(qocb_lplan *p, const double *controls, double *cost, double *final_densities) {
    if (!p) return -1;
    p->tape_ok = false;
    if (p->E > 1) return lfail(p, "qocb_lindblad_forward / qocb_lindblad_backward do not run ensemble plans", -1);
    if (int rc = launch_forward(p, controls, true)) return rc;
    const int rc = finish_lindblad(p, cost, nullptr, final_densities);
    p->tape_ok = rc == 0;
    return rc;
}

/* seeds: [N][D][n][n] complex or NULL; row k is added to the cotangent of the densities at system step k */
int qocb_lindblad_backward(qocb_lplan *p, const double *seeds, double *grad) {
    if (!p) return -1;
    if (p->E > 1) return lfail(p, "qocb_lindblad_forward / qocb_lindblad_backward do not run ensemble plans", -1);
    const size_t cnt = (size_t)p->pb.control_eval_count * p->pb.control_count;
    if (!cnt) return 0;
    if (!p->tape_ok) return lfail(p, "qocb_lindblad_backward needs a successful qocb_lindblad_forward as the last evaluation", -1);
    LTRY(p, cudaSetDevice(p->pb.device));
    if (seeds) {
        const size_t count = (size_t)p->pb.system_eval_count * p->pb.density_count * p->pb.hilbert_size * p->pb.hilbert_size;
        if (!p->seeds.p) LTRY(p, p->seeds.alloc(count));
        LTRY(p, cudaMemcpyAsync(p->seeds.p, seeds, sizeof(double2) * count, cudaMemcpyHostToDevice, p->stream));
    }
    if (int rc = launch_backward(p, seeds ? p->seeds.p : nullptr)) return rc;
    return finish_lindblad(p, nullptr, grad, nullptr);
}

/* stats[0] = Runge-Kutta attempts, stats[1] = accepted steps of the last evaluation (sums over the members of an ensemble) */
int qocb_lindblad_stats(qocb_lplan *p, int64_t *stats) {
    if (!p || !stats) return -1;
    LTRY(p, cudaSetDevice(p->pb.device));
    std::vector<long long> s(2 * (size_t)p->E);
    LTRY(p, cudaMemcpy(s.data(), p->stats.p, sizeof(long long) * s.size(), cudaMemcpyDeviceToHost));
    stats[0] = stats[1] = 0;
    for (int e = 0; e < p->E; ++e) { stats[0] += s[2 * e]; stats[1] += s[2 * e + 1]; }
    return 0;
}

/* per-member results of the last evaluation: costs [E], grads [E][M][KR], stats [E][2]; any may be NULL */
int qocb_lindblad_member_results(qocb_lplan *p, double *costs, double *grads, int64_t *stats) {
    if (!p) return -1;
    LTRY(p, cudaSetDevice(p->pb.device));
    LTRY(p, cudaStreamSynchronize(p->stream));
    const size_t E = p->E, cnt = (size_t)p->pb.control_eval_count * p->pb.control_count;
    if (costs) LTRY(p, cudaMemcpy(costs, p->cost.p, sizeof(double) * E, cudaMemcpyDeviceToHost));
    if (grads && cnt) LTRY(p, cudaMemcpy(grads, p->grad.p, sizeof(double) * E * cnt, cudaMemcpyDeviceToHost));
    if (stats) {
        std::vector<long long> s(2 * E);
        LTRY(p, cudaMemcpy(s.data(), p->stats.p, sizeof(long long) * s.size(), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < 2 * E; ++i) stats[i] = s[i];
    }
    return 0;
}

/* densities at every system step of the last evaluation: [N][D][n][n] complex, [E][N][D][n][n] for an ensemble */
int qocb_lindblad_get_densities(qocb_lplan *p, double *out) {
    if (!p || !out) return -1;
    LTRY(p, cudaSetDevice(p->pb.device));
    const size_t DE = (size_t)p->pb.density_count * p->pb.hilbert_size * p->pb.hilbert_size;
    LTRY(p, cudaMemcpy(out, p->states.p, sizeof(double2) * DE * p->pb.system_eval_count * p->E, cudaMemcpyDeviceToHost));
    return 0;
}

}  // extern "C"
