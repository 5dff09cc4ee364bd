// capi.cu - kernels' global entry points, the plan object and the C ABI declared in include/qocb200.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/qocb200.h"
#include "expm_slice.cuh"
#include "magnus.cuh"
#include "sweep.cuh"
#include "large.cuh"
#include "zgemm.cuh"
#include "small.cuh"

using namespace qocb;

namespace {

thread_local std::string g_last_error;

inline double kB_host(int i) {
    static const double b[14] = {64764752532480000., 32382376266240000., 7771770303897600., 1187353796428800.,
                                 129060195264000., 10559470521600., 670442572800., 33522128640., 1323241920.,
                                 40840800., 960960., 16380., 182., 1.};
    return b[i];
}

#define CU_TRY(plan, expr)                                                                              \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            char buf__[512];                                                                            \
            snprintf(buf__, sizeof(buf__), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            set_error(plan, buf__);                                                                     \
            return -2;                                                                                  \
        }                                                                                               \
    } while (0)

constexpr int kCtaTapeR = 16;            // squaring slots of the per-CTA (recompute) tape
constexpr int kStoredTapeR = 2;          // squaring slots of the stored per-slice tape

struct KArgs {
    GenArgs ga;                 // ga.G0 points at member 0
    int N, E, s_cap, tape_mats;
    const int *chunk_begin;
    double *U;                  // [E*(N-1)][GMAT]
    double *tape;               // stored tape or nullptr
    int *tape_piv;              // [E*(N-1)][NP]
    int *meta;                  // [E*(N-1)] squaring count of each slice
    double *scratch;            // [nchunks][S_COUNT][GMAT]
    double *cta_tape;           // [nchunks][8 + kCtaTapeR][GMAT]
    int *cta_piv;               // [nchunks][NP]
    double *chunkP;             // [nchunks][GMAT]
    const double *psi, *lam;    // [E][N][S][2][NP]
    double *node_grad;          // [E*(N-1)][q][KR]
    int S;
    int lowrank;                // 1: use the rank-S reverse pass where it applies (QOCB_NO_LOWRANK=1 disables it)
    int herm;                   // 1: every operator is Hermitian => anti-Hermitian Magnus matrices (pivot-free Pade inverse where safe)
    int tape_min;               // 1: slices without squarings keep {A, A2, LU} only (Krylov reverse pass, lowrank == 2)
    int post_adj;               // 1: slices replayed from the stored tape leave mbar in their A slot; k_magnus_adj does the Magnus adjoint
    int *err_flag;
};

// TMA feed of k_forward (tma.cuh): tensor maps of the propagator buffer U (whose slot j holds the Magnus matrix M_j, written
// by k_magnus, until slice j has consumed it) and of the chunk-propagator buffer.  Passed as a __grid_constant__ parameter:
// the maps must live in parameter / constant space for cp.async.bulk.tensor.
struct FeedMaps {
    CUtensorMap mapU, mapP;
    int tma;            // 1: both maps are valid, fetch asynchronously; 0: plain 16-byte loads at the point of use
    int premagnus;      // 1: U[w] holds M_w (magnus.cuh); 0: assemble the Magnus matrix in this kernel
};

// member e's control operators and their commutators (per-member operators only: the strides are 0 when they are
// shared).  Applied where the operators are read rather than once per slice, so that the pointers are not held in
// registers across the Pade passes (k_backward<64> sits at the register limit).
__device__ __forceinline__ GenArgs member_ops(GenArgs ga, int e) {
    ga.G += e * ga.g_stride;
    ga.Cs += e * ga.cs_stride;
    return ga;
}

template <class C>
__global__ void __launch_bounds__(C::NT) k_forward(KArgs a, const __grid_constant__ FeedMaps fm) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    const int c = blockIdx.x;
    const int wb = a.chunk_begin[c], we = a.chunk_begin[c + 1];
    double *scratch = a.scratch + (size_t)c * S_COUNT * C::GMAT;
    double *gP = a.chunkP + (size_t)c * C::GMAT;
    const bool tma = fm.tma != 0, premag = fm.premagnus != 0;
    uint64_t *barM = sm.bar, *barP = sm.bar + 1;
    uint32_t phM = 0, phP = 0;
    if (tma) {
        if (threadIdx.x == 0) { mbar_init(barM, 1); mbar_init(barP, 1); mbar_init_fence(); }
        __syncthreads();
        if (premag && wb < we && threadIdx.x == 0) tma_fetch_matrix<C::NP>(sm.X2, &fm.mapU, wb, barM);
    }
    bool parked = false;
    for (int w = wb; w < we; ++w) {
        const int e = w / (a.N - 1), j = w - e * (a.N - 1);
        GenArgs ga = a.ga;
        ga.G0 += e * ga.drift_stride;
        ga.C0 += e * ga.KR * ga.drift_stride;
        PROF_DECL
        double *gU = a.U + (size_t)w * C::GMAT;
        double *gMnext = scratch + (size_t)S_E * C::GMAT;            // parked Magnus matrix (slot unused by the forward of M2 / M4)
        if (premag) {                                                // M_w was written into U[w] by k_magnus
            if (tma) { mbar_wait(barM, phM); phM ^= 1; }
            else { g2s<C>(sm.X2, gU); __syncthreads(); }
        } else if (parked) {                                         // assembled together with the previous slice's
            g2s<C>(sm.X2, gMnext);
            __syncthreads();
            parked = false;
        } else {
            load_coefs<C>(sm, ga, j, e);
            if (magnus_pair_ok<C>(ga) && w + 1 < we) {
                load_coefs_to<C>(sm.red, ga, j + 1, e);                 // chunks never straddle members
                magnus_forward_pair<C>(sm, member_ops(ga, e), sm.coef, sm.red, gMnext);
                parked = true;
            } else {
                magnus_forward<C>(sm, member_ops(ga, e), scratch);
            }
        }
        PROF_MARK(1);
        double *tape = a.tape ? a.tape + (size_t)w * a.tape_mats * C::GMAT : nullptr;
        int *piv = a.tape ? a.tape_piv + (size_t)w * C::NP : nullptr;
        Feed feed;
        feed.mapM = &fm.mapU; feed.mapP = &fm.mapP; feed.barM = barM; feed.barP = barP; feed.fetchedP = false;
        feed.idxM = (tma && premag && w + 1 < we) ? (long long)w + 1 : -1;
        feed.idxP = (tma && w > wb) ? (long long)c : -1;
        const double *Ubuf = sm.X1;
        const int s = pade_forward<C>(sm, tape, piv, scratch + (size_t)S_T0 * C::GMAT, scratch + (size_t)S_T1 * C::GMAT, a.s_cap,
                                      &feed, &Ubuf, a.herm, a.tape_min);
        if (threadIdx.x == 0) a.meta[w] = s;
        if (w == wb) {
            for_owned<C>([&](int, int, int row, int col) {
                const c2 u = lds2<C>(Ubuf, row, col);
                stg2<C>(gU, row, col, u);
                stg2<C>(gP, row, col, u);
            });
            __syncthreads();                                         // X2 (LU -> tape) is rewritten by the next slice's Magnus matrix
        } else {
            double *Pbuf = Ubuf == sm.X0 ? sm.X1 : sm.X0;
            for_owned<C>([&](int, int, int row, int col) { stg2<C>(gU, row, col, lds2<C>(Ubuf, row, col)); });
            if (feed.fetchedP) { mbar_wait(barP, phP); phP ^= 1; }
            else { g2s<C>(Pbuf, gP); __syncthreads(); }
            Acc<C> acc; acc.zero();
            mma_smem<C, false, false, false>(acc, Ubuf, Pbuf);        // P <- U_j P
            for_owned<C>([&](int i, int jj, int row, int col) { stg2<C>(gP, row, col, accv<C>(acc, i, jj)); });
        }
        if (tma) fence_proxy_async_all();                            // the chunk propagator just written is fetched by TMA next slice
#ifdef QOCB_PROFILE
        { __syncthreads(); if (blockIdx.x == 0 && threadIdx.x == 0) { g_prof[7] += clock64() - prof_t0__; g_prof[0] += 1; } }
#endif
    }
}

// tensor maps of the stored tape and of the per-CTA recompute tape for the Krylov reverse pass
struct TapeMaps {
    CUtensorMap mapT, mapC;
    int tma;
};

template <class C>
__global__ void __launch_bounds__(C::NT) k_backward(KArgs a, const __grid_constant__ TapeMaps tmaps) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    const int c = blockIdx.x;
    const int wb = a.chunk_begin[c], we = a.chunk_begin[c + 1];
    double *scratch = a.scratch + (size_t)c * S_COUNT * C::GMAT;
    double *ctape = a.cta_tape + (size_t)c * (8 + kCtaTapeR) * C::GMAT;
    int *cpiv = a.cta_piv + (size_t)c * C::NP;
    const int VS = a.S * 2 * C::NP;
    uint32_t ph0 = 0, ph1 = 0;
    if (tmaps.tma) {
        if (threadIdx.x == 0) { mbar_init(sm.bar, 1); mbar_init(sm.bar + 1, 1); mbar_init_fence(); }
        __syncthreads();
    }
    for (int w = wb; w < we; ++w) {
        PROF_DECL
        const int e = w / (a.N - 1), j = w - e * (a.N - 1);
        GenArgs ga = a.ga;
        ga.G0 += e * ga.drift_stride;
        ga.C0 += e * ga.KR * ga.drift_stride;
        load_coefs<C>(sm, ga, j, e);
        const double *tape; const int *piv; int s;
        if (a.tape && a.meta[w] <= a.s_cap) {
            tape = a.tape + (size_t)w * a.tape_mats * C::GMAT;
            piv = a.tape_piv + (size_t)w * C::NP;
            s = a.meta[w];
        } else {
            magnus_forward<C>(sm, member_ops(ga, e), scratch);
            s = pade_forward<C>(sm, ctape, cpiv, scratch + (size_t)S_T0 * C::GMAT, scratch + (size_t)S_T1 * C::GMAT, kCtaTapeR,
                                nullptr, nullptr, a.herm, a.tape_min);
            if (s > kCtaTapeR && threadIdx.x == 0) *a.err_flag = 1;
            tape = ctape; piv = cpiv;
            if (tmaps.tma) fence_proxy_async_all();                    // this CTA's tape stores are read back by TMA
            __syncthreads();
        }
        const double *psi = a.psi + ((size_t)e * a.N + j) * VS;
        const double *lam = a.lam + ((size_t)e * a.N + j + 1) * VS;
        bool done = false;
        if constexpr (C::NP == 64 && C::NWARP == 8) {
            if (a.S <= 4 && s == 0 && a.lowrank == 2) {                // rank-S reverse pass on the Krylov basis of A2
                PROF_MARK(9);
                TapeFeed tf;
                tf.tape = tape; tf.bar0 = sm.bar; tf.bar1 = sm.bar + 1; tf.ph0 = &ph0; tf.ph1 = &ph1;
                const bool stored = tape != ctape;
                tf.map = tmaps.tma ? (stored ? &tmaps.mapT : &tmaps.mapC) : nullptr;
                tf.idx0 = stored ? (long long)w * a.tape_mats : (long long)c * (8 + kCtaTapeR);
                pade_backward_krylov<C>(sm, tf, piv, psi, psi + VS, lam, a.S, a.herm);
                done = true;
            } else if (a.S <= 4 && s == 0 && a.lowrank == 1) {         // rank-S reverse pass, re-associated form (lowrank.cuh)
                PROF_MARK(9);
                pade_backward_lowrank<C>(sm, tape, piv, psi, psi + VS, lam, a.S);
                done = true;
            }
        }
        if (!done) {
            // ubar = sum_s lam_{j+1,s} psi_{j,s}^T   (cotangent of U_j from states = U_j psi)
            for_owned<C>([&](int, int, int row, int col) {
                c2 u = czero();
                for (int s_ = 0; s_ < a.S; ++s_) {
                    const double lr = lam[s_ * 2 * C::NP + row], li = lam[s_ * 2 * C::NP + C::NP + row];
                    const double2 pr = *reinterpret_cast<const double2 *>(psi + s_ * 2 * C::NP + col);
                    const double2 pi = *reinterpret_cast<const double2 *>(psi + s_ * 2 * C::NP + C::NP + col);
                    u.r0 += lr * pr.x - li * pi.x; u.i0 += lr * pi.x + li * pr.x;
                    u.r1 += lr * pr.y - li * pi.y; u.i1 += lr * pi.y + li * pr.y;
                }
                sts2<C>(sm.X0, row, col, u);
            });
            __syncthreads();
            PROF_MARK(9);
            pade_backward<C>(sm, tape, piv, s, a.U + (size_t)w * C::GMAT, scratch);
        }
        if (a.post_adj && tape != ctape) {                          // the slice's tape is dead: its A slot takes mbar (magnus.cuh)
            double *gM = a.tape + ((size_t)w * a.tape_mats + T_A) * C::GMAT;
            for_owned<C>([&](int, int, int row, int col) { stg2<C>(gM, row, col, lds2<C>(sm.X0, row, col)); });
            __syncthreads();
        } else {
            magnus_backward<C>(sm, member_ops(ga, e), scratch, a.node_grad + (size_t)w * ga.q * ga.KR);
        }
        PROF_MARK(13);
    }
}

// grad[m][r] = (1/E) sum_e sum_{(j,i) using control point m} weight * node_grad[e][j][i][r]
__global__ void k_gather_grad(const int *csr_ptr, const int *csr_idx, const double *csr_w, const double *node_grad,
                              double *grad, int M, int KR, int q, int Nm1, int E) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= M * KR) return;
    const int m = t / KR, r = t % KR;
    double sum = 0.;
    for (int p = csr_ptr[m]; p < csr_ptr[m + 1]; ++p) {
        const int ji = csr_idx[p];
        const double w = csr_w[p];
        double sub = 0.;
        for (int e = 0; e < E; ++e) sub += node_grad[((size_t)e * Nm1 * q + ji) * KR + r];
        sum += w * sub;
    }
    grad[t] = sum / E;
}

// control batches: grad[b][m][r] = sum_{(j,i) using control point m} weight * node_grad[b][j][i][r], one thread per entry, the
// CSR order of k_gather_grad and no member mean (E = 1 gives k_gather_grad's bits)
__global__ void k_gather_grad_members(const int *csr_ptr, const int *csr_idx, const double *csr_w, const double *node_grad,
                                      double *grad, int M, int KR, int q, int Nm1, int E) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)E * M * KR) return;
    const int b = (int)(t / ((long long)M * KR)), mr = (int)(t - (long long)b * M * KR), m = mr / KR, r = mr % KR;
    const double *ng = node_grad + (size_t)b * Nm1 * q * KR;
    double sum = 0.;
    for (int p = csr_ptr[m]; p < csr_ptr[m + 1]; ++p) sum += csr_w[p] * ng[(size_t)csr_idx[p] * KR + r];
    grad[t] = sum;
}

// time-dependent operators: channel coefficients of every local node from the interpolated controls,
// coef[ji][c] = off[ji][c] + sum_r gain[ji][c][r] x_r(t_ji)
__global__ void k_node_coefs(const double *controls, const int *itab_idx, const double *itab_w, const double *off, const double *gain,
                             double *coef, int nodes, int KC, int KR) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nodes * KC) return;
    const int ji = t / KC;
    double v = off[t];
    for (int r = 0; r < KR; ++r) {
        const double x = controls[itab_idx[2 * ji] * KR + r] * itab_w[2 * ji] + controls[itab_idx[2 * ji + 1] * KR + r] * itab_w[2 * ji + 1];
        v += gain[(size_t)t * KR + r] * x;
    }
    coef[t] = v;
}
// ... and the transpose for the gradient: gx[e][ji][r] = sum_c gain[ji][c][r] gc[e][ji][c]
__global__ void k_node_grad_map(const double *gc, const double *gain, double *gx, int E, int nodes, int KC, int KR) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= E * nodes * KR) return;
    const int r = t % KR, eji = t / KR, ji = eji % nodes;
    double v = 0.;
    for (int c = 0; c < KC; ++c) v += gain[((size_t)ji * KC + c) * KR + r] * gc[(size_t)eji * KC + c];
    gx[t] = v;
}

__global__ void k_finalize_cost(const double *cost_part, int nchunks, int E, double *cost) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double s = 0.;
        for (int c = 0; c < nchunks; ++c) s += cost_part[c];
        *cost = s / E;
    }
}

// control batches: cost[e] = sum of member e's chunk costs in chunk order (E = 1 gives k_finalize_cost's bits)
__global__ void k_member_cost(const double *cost_part, const int *member_chunk0, int E, double *cost) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double s = 0.;
    for (int c = member_chunk0[e]; c < member_chunk0[e + 1]; ++c) s += cost_part[c];
    cost[e] = s;
}

template <class C>
__global__ void __launch_bounds__(C::NT) k_expm(const double *in, double *out, double *scratch, long long batch) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    double *sc = scratch + (size_t)blockIdx.x * 3 * C::GMAT;
    for (long long b = blockIdx.x; b < batch; b += gridDim.x) {
        __syncthreads();
        g2s<C>(sm.X2, in + (size_t)b * C::GMAT);
        __syncthreads();
        pade_forward<C>(sm, nullptr, nullptr, sc, sc + C::GMAT, 0);
        for_owned<C>([&](int, int, int row, int col) { stg2<C>(out + (size_t)b * C::GMAT, row, col, lds2<C>(sm.X1, row, col)); });
    }
}

template <class C>
__global__ void __launch_bounds__(C::NT) k_expm_vjp(const double *in, const double *ubar, double *out, double *abar,
                                                    double *scratch, double *cta_tape, int *cta_piv, long long batch) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    double *sc = scratch + (size_t)blockIdx.x * S_COUNT * C::GMAT;
    double *tape = cta_tape + (size_t)blockIdx.x * (8 + kCtaTapeR) * C::GMAT;
    int *piv = cta_piv + (size_t)blockIdx.x * C::NP;
    for (long long b = blockIdx.x; b < batch; b += gridDim.x) {
        __syncthreads();
        g2s<C>(sm.X2, in + (size_t)b * C::GMAT);
        __syncthreads();
        const int s = pade_forward<C>(sm, tape, piv, sc + (size_t)S_T0 * C::GMAT, sc + (size_t)S_T1 * C::GMAT, kCtaTapeR);
        double *gU = out + (size_t)b * C::GMAT;
        for_owned<C>([&](int, int, int row, int col) { stg2<C>(gU, row, col, lds2<C>(sm.X1, row, col)); });
        g2s<C>(sm.X0, ubar + (size_t)b * C::GMAT);
        __syncthreads();
        pade_backward<C>(sm, tape, piv, s, gU, sc);
        for_owned<C>([&](int, int, int row, int col) { stg2<C>(abar + (size_t)b * C::GMAT, row, col, lds2<C>(sm.X0, row, col)); });
    }
}

// [partial gradient | partial cost | final states (owner rank only, zeros elsewhere)] -> one all-reduce payload
__global__ void k_pack_result(const double *grad, const double *cost, const double *fin, double *out, int count, int VS) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < count) out[t] = grad ? grad[t] : 0.0;
    else if (t == count) out[t] = *cost;
    else if (t < count + 1 + VS) out[t] = fin ? fin[t - count - 1] : 0.0;
}

// pairwise product tree over propagators: out[i] = in[2i+1] * in[2i] (later slices on the left); an odd tail is copied
template <class C>
__global__ void __launch_bounds__(C::NT) k_reduce_props(const double *in, double *out, int count) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    const int i = blockIdx.x;
    const double *lo = in + (size_t)(2 * i) * C::GMAT;
    double *dst = out + (size_t)i * C::GMAT;
    if (2 * i + 1 >= count) {
        for (int idx = threadIdx.x; idx < C::GMAT / 2; idx += C::NT)
            reinterpret_cast<double2 *>(dst)[idx] = reinterpret_cast<const double2 *>(lo)[idx];
        return;
    }
    g2s<C>(sm.X0, lo);
    g2s<C>(sm.X1, lo + C::GMAT);
    __syncthreads();
    Acc<C> acc; acc.zero();
    mma_smem<C, false, false, false>(acc, sm.X1, sm.X0);
    for_owned<C>([&](int ii, int jj, int row, int col) { stg2<C>(dst, row, col, accv<C>(acc, ii, jj)); });
}

// radix-R version for the tail of the tree (shard propagator): out[i] = in[R i + R - 1] ... in[R i + 1] in[R i], the
// products chained inside one CTA - fewer dependent launches than the pairwise tree when only the root is wanted
template <class C>
__global__ void __launch_bounds__(C::NT) k_reduce_props_radix(const double *in, double *out, int count, int R) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem<C> sm(smem_raw);
    const int first = blockIdx.x * R, last = min(count, first + R);
    double *dst = out + (size_t)blockIdx.x * C::GMAT;
    if (last - first == 1) {
        const double *lo = in + (size_t)first * C::GMAT;
        for (int idx = threadIdx.x; idx < C::GMAT / 2; idx += C::NT)
            reinterpret_cast<double2 *>(dst)[idx] = reinterpret_cast<const double2 *>(lo)[idx];
        return;
    }
    g2s<C>(sm.X0, in + (size_t)first * C::GMAT);
    for (int k = first + 1; k < last; ++k) {
        g2s<C>(sm.X1, in + (size_t)k * C::GMAT);
        __syncthreads();
        Acc<C> acc; acc.zero();
        mma_smem<C, false, false, false>(acc, sm.X1, sm.X0);
        if (k + 1 == last) {
            for_owned<C>([&](int ii, int jj, int row, int col) { stg2<C>(dst, row, col, accv<C>(acc, ii, jj)); });
        } else {
            __syncthreads();
            for_owned<C>([&](int ii, int jj, int row, int col) { sts2<C>(sm.X0, row, col, accv<C>(acc, ii, jj)); });
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
int pad_dim(int n) {
    if (n <= 8) return 8;
    if (n <= 16) return 16;
    if (n <= 32) return 32;
    if (n <= 64) return 64;
    if (n <= 512) return n;          // large-dimension path (large.cuh): dense n x n, no padding
    return -1;
}

// interleaved complex n x n (host) -> planar padded NP x NP; generator: G = -1j * H
void to_planar(const double *src, double *dst, int n, int NP, bool generator) {
    std::fill(dst, dst + 2 * (size_t)NP * NP, 0.0);
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) {
            const double re = src[2 * ((size_t)r * n + c)], im = src[2 * ((size_t)r * n + c) + 1];
            dst[(size_t)r * NP + c] = generator ? im : re;
            dst[(size_t)NP * NP + (size_t)r * NP + c] = generator ? -re : im;
        }
}
void from_planar(const double *src, double *dst, int n, int NP) {
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) {
            dst[2 * ((size_t)r * n + c)] = src[(size_t)r * NP + c];
            dst[2 * ((size_t)r * n + c) + 1] = src[(size_t)NP * NP + (size_t)r * NP + c];
        }
}

// host-side commutators of the product-free M4 (qocb_set_operators, qocb_set_member_operators); interleaved complex n x n
typedef std::vector<double> HostMat;
HostMat host_generator(const double *h, int n) {             // G = -1j H
    HostMat g(2 * (size_t)n * n);
    for (size_t i = 0; i < (size_t)n * n; ++i) { g[2 * i] = h[2 * i + 1]; g[2 * i + 1] = -h[2 * i]; }
    return g;
}
HostMat host_commutator(const HostMat &x, const HostMat &y, int n) {   // [x, y]
    HostMat c(2 * (size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < n; ++k) {
            const double xr = x[2 * ((size_t)i * n + k)], xi = x[2 * ((size_t)i * n + k) + 1];
            const double yr = y[2 * ((size_t)i * n + k)], yi = y[2 * ((size_t)i * n + k) + 1];
            for (int j = 0; j < n; ++j) {
                const double br = y[2 * ((size_t)k * n + j)], bi = y[2 * ((size_t)k * n + j) + 1];
                const double ar = x[2 * ((size_t)k * n + j)], ai = x[2 * ((size_t)k * n + j) + 1];
                c[2 * ((size_t)i * n + j)] += (xr * br - xi * bi) - (yr * ar - yi * ai);
                c[2 * ((size_t)i * n + j) + 1] += (xr * bi + xi * br) - (yr * ai + yi * ar);
            }
        }
    return c;
}
// Hermitian to 1e-13 of the largest entry: selects the pivot-free Pade inverse where it is safe (tile.cuh)
bool host_is_hermitian(const double *h, int n) {
    double mx = 0., dev = 0.;
    for (int r = 0; r < n; ++r)
        for (int c = 0; c <= r; ++c) {
            const double ar = h[2 * ((size_t)r * n + c)], ai = h[2 * ((size_t)r * n + c) + 1];
            const double br = h[2 * ((size_t)c * n + r)], bi = h[2 * ((size_t)c * n + r) + 1];
            mx = std::max(mx, std::max(std::fabs(ar) + std::fabs(ai), std::fabs(br) + std::fabs(bi)));
            dev = std::max(dev, std::fabs(ar - br) + std::fabs(ai + bi));
        }
    return dev <= 1e-13 * mx;
}
bool no_nopiv() { const char *np_ = getenv("QOCB_NO_NOPIV"); return np_ && np_[0] == '1'; }

template <class T> struct DevBuf {
    T *p = nullptr; size_t n = 0;
    cudaError_t alloc(size_t count) {
        release();
        n = count;
        if (count == 0) return cudaSuccess;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; n = 0; }
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
};

}  // namespace

namespace {
// work arrays of the large-dimension path, each [batch][n*n] double2
enum { LA1 = 0, LA2N, LM, LA2, LA4, LA6, LW1, LX1, LY, LVE, LUO, LP, LQ, LT, LR0, LRS0,
       LRB = LRS0 + qocb::kLgMaxSq, LQB, LUOB, LVEB, LAB, LYB, LA6B, LA4B, LA2B, LTB, LXB, LA1B, LA2NB, LCOUNT };

struct LargeImpl {
    int n = 0, nn = 0, B = 0;
    cublasHandle_t blas = nullptr;
    DevBuf<double2> G0, G, C0, Cs, work, treeA, treeB, UT, lvl, PT, allPT, lr;   // lr: thin buffers of the rank-S reverse pass
    DevBuf<double2 *> ptrQ, ptrP, ptrRB, ptrPSI;
    bool lowrank = false;
    DevBuf<int> piv, info, sarr, cb;
    std::vector<int> h_smax;            // largest squaring count per batch, read back ONCE per evaluation (after the forward)
    DevBuf<int> smax_dev;               // [batches + 1]: per batch of the forward pass; last slot: scratch of recomputed batches
    int lstar = 0, nchunks = 0, lvl_count[24] = {}, lvl_off[24] = {};   // pairwise propagator tree levels 0..lstar
    bool use_cublas_gemm = false;       // QOCB_LARGE_CUBLAS=1: library ZGEMM instead of zgemm.cuh (A/B comparison)
    bool cluster_boundary = true;       // boundary passes on an 8-CTA cluster (QOCB_NO_CLUSTER=1: the single-CTA kernels)
    bool tma_gemm = true;               // operand panels by TMA (k_zgemm_tma); QOCB_NO_TMA=1: the cp.async kernel
    bool own_lu = false;                // block LU + block substitutions on the own GEMM (Hermitian operators, ||A||_1 < 2.5 checked on
                                        // the device; QOCB_LARGE_CUBLAS_LU=1 or a raised lu_flag: cuBLAS getrf / getrs)
    DevBuf<int> lu_flag;
    // reverse-pass tape (stored when it fits): M, A2, A4, A6, Y, LU(Q), R0 of every local slice + pivots + squaring counts.
    // tj >= 0 redirects those work arrays (and pivots / counts / LU pointers) to the tape entries of slices tj, tj+1, ...
    DevBuf<double2> tape;
    DevBuf<int> tpiv, tsarr;
    DevBuf<double2 *> tptrQ;
    bool taped = false;
    int tj = -1, Lsl = 0;
    std::vector<char> batch_taped;
    static int tslot(int id) {
        switch (id) { case LM: return 0; case LA2: return 1; case LA4: return 2; case LA6: return 3; case LY: return 4; case LQ: return 5; case LR0: return 6; }
        return -1;
    }
    double2 *arr(int i) {
        const int ts = tj >= 0 ? tslot(i) : -1;
        return ts >= 0 ? tape.p + ((size_t)ts * Lsl + tj) * nn : work.p + (size_t)i * B * nn;
    }
    int *cur_piv() { return tj >= 0 ? tpiv.p + (size_t)tj * n : piv.p; }
    int *cur_sarr() { return tj >= 0 ? tsarr.p + tj : sarr.p; }
    double2 **cur_ptrQ() { return tj >= 0 ? tptrQ.p + tj : ptrQ.p; }
    ~LargeImpl() { if (blas) cublasDestroy(blas); }
};
}  // namespace

struct qocb_plan {
    qocb_problem pb;
    LargeImpl *large = nullptr;
    int NP = 0, q = 0, nchunks = 0, tape_mats = 0, num_sms = 0;
    int j0 = 0, Nloc = 0;               // time sharding: first local slice (global index), local state count
    // operator channels (KC = pb.control_count unless a node map is set): the kernels see KC coefficient channels;
    // controls and gradients crossing the ABI keep pb.control_count real channels
    int KC = 0;
    bool mapped = false, map_set = false;
    bool particular_fresh = false;      // sharded: the boundary costates of this evaluation's particular pass are in `lam`
    const double *shardP_last = nullptr; // sharded: device buffer that received this shard's propagator in forward_local
    // sweep coarsening: the state / costate sweeps run on chunks merged pairwise `levels` times (propagator tree);
    // lvl_count[l] chunks at level l, their propagators at lvlP + lvl_off[l] matrices, boundaries at cb_lvl + cb_off[l]
    int levels = 0, lvl_count[16] = {}, lvl_off[16] = {}, cb_off[16] = {};
    // three-level scheme: the sequential boundary passes run on level `coarse` >= levels, k_mid_* fill in the sweep-chunk
    // boundaries (coarse == levels: two levels).  lv2 / lv3s, lv3c: the choices with / without step costs (pick_levels)
    int coarse = 0, lv2 = 0, lv3s = 0, lv3c = 0;
    DevBuf<double> part_coarse;         // [lvl_count[coarse]][S][2][NP] particular parts of the coarse chunks (step costs)
    bool sharded = false, owns_final = true;
    bool ops_set = false, states_set = false, have_step_costs = false, comm_ok = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[16] = {};
    DevBuf<double> C0, Cs, G0, G, controls, itab_w, U, tape, scratch, cta_tape, chunkP, psi, lam, part, cost_part, psi0,
        node_grad, grad, cost, csr_w, vecs, flush, redA, redB, psi_in, lam_in, lvlP, nodecoef, map_off, map_gain, node_grad_x;
    DevBuf<int> itab_idx, tape_piv, meta, cta_piv, chunk_begin, member_chunk0, csr_ptr, csr_idx, counts, err_flag, cb_lvl, mc0_lvl, one_chunk;
    DevBuf<CostTerm> terms;
    std::vector<CostTerm> h_terms;
    std::vector<double> h_vecs;
    std::vector<int> h_term_members;    // per term: 1 shared, E member term (h_vecs holds its [E][S][fmax] vectors)
    long long vecs_mstride = 0;         // doubles per member of the uploaded vector table (0: no member terms)
    std::vector<int> h_counts;
    int ip_total = 0;
    int coh_total = 0;                  // overlap-sum slots of the coherent target terms (state sharding)
    bool state_sharded = false;
    double *coh_out = nullptr;          // state sharding: device buffers of the current evaluation (caller-owned)
    const double *coh_in = nullptr;
    FeedMaps fm;                        // TMA tensor maps of U and chunkP (k_forward); fm.tma = 0 when TMA is unavailable
    TapeMaps tmaps;                     // ... of the stored tape and the per-CTA recompute tape (k_backward)
    bool post_adj_ok = false;           // Magnus adjoint as a streaming pass after k_backward (single member, stored tape)
    DevBuf<double> adj_partial;         // [slabs][W][kAdjMaxOps] slab sums of k_magnus_adj
    int lowrank_mode = 2;               // 0 dense reverse pass, 1 re-associated rank-S form, 2 Krylov basis of A2 (QOCB_LOWRANK=0/1/2)
    bool premagnus_ok = true;           // QOCB_NO_PREMAGNUS=1: assemble the Magnus matrices inside k_forward (A/B comparison)
    bool hermitian = false;             // H0 (every member) and every operator channel are Hermitian (QOCB_NO_NOPIV=1 clears it)
    bool drift_hermitian = false;       // H0 of every member is Hermitian (qocb_set_member_operators recomputes `hermitian`)
    bool member_ops = false;            // G, C0 and Cs hold every member's own control operators (qocb_set_member_operators)
    bool batch = false;                 // control batch (qocb_set_control_batch): member b has its own controls, cost and gradient
    bool member_states = false;         // psi0 holds [E][S][2][NP], every member's own initial states (qocb_set_member_states)
    double *h_pinned = nullptr;         // [ctl_doubles controls | ctl_doubles grad | cost_count costs]
    // CUDA graph of one whole host-facing evaluation (H2D controls, all kernels, D2H of gradient, cost, final states and the
    // error flag): replayed by qocb_cost / qocb_cost_and_grad from the third call on - launch-bound small problems gain 2x
    cudaGraphExec_t gexec[2] = {nullptr, nullptr};
    int host_calls[2] = {0, 0};
    double *h_fin = nullptr;            // pinned [E][S][2][NP] final states
    int *h_flag = nullptr;              // pinned device error flag
    bool use_graph = true;
    std::string err;
    ~qocb_plan() { delete large; }
};

namespace {

void set_error(qocb_plan *plan, const char *msg) {
    if (plan) plan->err = msg;
    g_last_error = msg;
}

template <class C> int launch_forward(qocb_plan *p, const KArgs &a) {
    FeedMaps fm = p->fm;
    fm.premagnus = 0;
    // Magnus matrices of all slices in one streaming pass (magnus.cuh) whenever the order needs no matrix products
    if (p->premagnus_ok && (a.ga.order == 2 || (a.ga.order == 4 && a.ga.comm))) {
        const long long W = (long long)a.E * (a.N - 1);
        const int slabs = (C::GMAT + kMagSlab - 1) / kMagSlab;
        const long long groups = std::max<long long>(1, std::min<long long>((W + 7) / 8, (3LL * p->num_sms + slabs - 1) / slabs));
        const long long per_block = (W + groups - 1) / groups;
        const size_t smem = magnus_smem_bytes(a.ga.order, a.ga.KR);
        CU_TRY(p, cudaFuncSetAttribute(k_magnus, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_magnus<<<dim3(slabs, (unsigned)((W + per_block - 1) / per_block)), kMagThreads, smem, p->stream>>>(a.ga, C::GMAT, a.N - 1, W, per_block, a.U);
        CU_TRY(p, cudaGetLastError());
        fm.premagnus = 1;
    }
    CU_TRY(p, cudaFuncSetAttribute(k_forward<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
    k_forward<C><<<p->nchunks, C::NT, Smem<C>::bytes(), p->stream>>>(a, fm);
    CU_TRY(p, cudaGetLastError());
    return 0;
}
template <class C> int launch_backward(qocb_plan *p, const KArgs &a) {
    CU_TRY(p, cudaFuncSetAttribute(k_backward<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
    k_backward<C><<<p->nchunks, C::NT, Smem<C>::bytes(), p->stream>>>(a, p->tmaps);
    CU_TRY(p, cudaGetLastError());
    if (a.post_adj) {                                               // Magnus adjoint of all slices in one streaming pass
        const long long W = (long long)a.E * (a.N - 1);
        const int slabs = (C::GMAT + kAdjSlab - 1) / kAdjSlab;
        const long long tiles = (W + 7) / 8;
        const long long groups = std::max<long long>(1, std::min<long long>(tiles, (3LL * p->num_sms + slabs - 1) / slabs));
        const long long per = (tiles + groups - 1) / groups;
        const size_t smem = magnus_adj_smem_bytes(a.ga.order, a.ga.KR);
        CU_TRY(p, cudaFuncSetAttribute(k_magnus_adj, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_magnus_adj<<<dim3(slabs, (unsigned)((tiles + per - 1) / per)), kAdjThreads, smem, p->stream>>>(
            a.ga, C::GMAT, C::GPLANE, W, per, a.tape + (size_t)T_A * C::GMAT, (long long)a.tape_mats * C::GMAT, p->adj_partial.p);
        const long long tot = W * a.ga.q * a.ga.KR;
        k_magnus_adj_final<<<(unsigned)((tot + 127) / 128), 128, 0, p->stream>>>(a.ga, p->adj_partial.p, slabs, W, a.meta, a.s_cap, a.node_grad);
        CU_TRY(p, cudaGetLastError());
    }
    return 0;
}

// run `stmt` with the compile-time constant NPc bound to the plan's padded dimension
#define SWEEP_NP(np, stmt)                                   \
    do {                                                     \
        switch (np) {                                        \
            case 8: { constexpr int NPc = 8; stmt; } break;   \
            case 16: { constexpr int NPc = 16; stmt; } break; \
            case 32: { constexpr int NPc = 32; stmt; } break; \
            case 64: { constexpr int NPc = 64; stmt; } break; \
        }                                                    \
    } while (0)

template <int NP> cudaError_t set_sweep_attrs(int big) {
    cudaError_t e;
    const auto A = cudaFuncAttributeMaxDynamicSharedMemorySize;
    if ((e = cudaFuncSetAttribute(k_boundary_fwd<NP>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_sweep_fwd<NP>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_sweep_bwd<NP, true>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_sweep_bwd<NP, false>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_boundary_bwd<NP>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_mid_fwd<NP>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_mid_bwd<NP, false>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_mid_bwd<NP, true>, A, big)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_prefix_states<NP>, A, big)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_suffix_costates<NP>, A, big);
}

using C8 = Cfg<8, 1, 1>;
using C16 = Cfg<16, 2, 2>;
using C32 = Cfg<32, 2, 2>;
using C64 = Cfg<64, 2, 4>;

template <class F8, class F16, class F32, class F64>
int dispatch(int NP, F8 f8, F16 f16, F32 f32, F64 f64) {
    switch (NP) {
        case 8: return f8();
        case 16: return f16();
        case 32: return f32();
        case 64: return f64();
    }
    return -3;
}

template <class C> int occupancy_fwd() {
    int occ = 0;
    cudaFuncSetAttribute(k_backward<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes());
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_backward<C>, C::NT, Smem<C>::bytes());
    return occ < 1 ? 1 : occ;
}

KArgs make_kargs(qocb_plan *p) {
    KArgs a;
    a.ga.G0 = p->G0.p; a.ga.G = p->G.p; a.ga.controls = p->controls.p;
    a.ga.itab_idx = p->itab_idx.p; a.ga.itab_w = p->itab_w.p;
    a.ga.KR = p->KC; a.ga.q = p->q; a.ga.order = p->pb.magnus_order;
    a.ga.nodecoef = p->mapped ? p->nodecoef.p : nullptr;
    a.ga.C0 = p->C0.p; a.ga.Cs = p->Cs.p; a.ga.comm = p->comm_ok ? 1 : 0;
    const long long GM = 2LL * p->NP * p->NP;
    a.ga.g_stride = p->member_ops ? p->KC * GM : 0;
    a.ga.cs_stride = p->member_ops && p->comm_ok ? p->KC * (p->KC - 1) / 2 * GM : 0;
    a.ga.ctl_stride = p->batch ? (long long)p->pb.control_eval_count * p->pb.control_count : 0;
    a.ga.drift_stride = p->batch ? 0 : GM;
    a.ga.dt = p->pb.evolution_time / (p->pb.system_eval_count - 1);
    a.N = p->Nloc; a.E = p->pb.ensemble_count;
    a.s_cap = kStoredTapeR; a.tape_mats = p->tape_mats;
    a.chunk_begin = p->chunk_begin.p;
    a.U = p->U.p; a.tape = p->tape.p; a.tape_piv = p->tape_piv.p; a.meta = p->meta.p;
    a.scratch = p->scratch.p; a.cta_tape = p->cta_tape.p; a.cta_piv = p->cta_piv.p; a.chunkP = p->chunkP.p;
    a.psi = p->psi.p; a.lam = p->lam.p; a.node_grad = p->node_grad.p; a.S = p->pb.state_count;
    a.err_flag = p->err_flag.p;
    a.lowrank = p->lowrank_mode;
    a.herm = p->hermitian ? 1 : 0;
    a.tape_min = (p->lowrank_mode == 2 && p->NP == 64 && p->pb.state_count <= 4) ? 1 : 0;
    a.post_adj = (p->post_adj_ok && p->tape.p && (a.ga.order == 2 || (a.ga.order == 4 && a.ga.comm)) && a.ga.KR > 0) ? 1 : 0;
    return a;
}

SweepArgs make_sargs(qocb_plan *p) {
    SweepArgs s;
    s.NP = p->NP; s.S = p->pb.state_count; s.N = p->Nloc; s.E = p->pb.ensemble_count;
    s.j_off = p->j0; s.Nglob = p->pb.system_eval_count; s.add_final_seed = p->owns_final ? 1 : 0;
    s.lam_in = nullptr; s.b_out = nullptr;
    s.ces = p->pb.cost_eval_step; s.nterms = (int)p->h_terms.size(); s.ip_total = p->ip_total;
    s.terms = p->terms.p; s.vecs = p->vecs.p; s.counts = p->counts.p;
    s.U = p->U.p; s.chunkP = p->chunkP.p; s.chunk_begin = p->chunk_begin.p; s.member_chunk0 = p->member_chunk0.p;
    if (p->levels > 0) {
        s.chunkP = p->lvlP.p + (size_t)p->lvl_off[p->levels] * 2 * p->NP * p->NP;
        s.chunk_begin = p->cb_lvl.p + p->cb_off[p->levels];
        s.member_chunk0 = p->mc0_lvl.p + 2 * p->levels;
    }
    s.psi = p->psi.p; s.lam = p->lam.p; s.part = p->part.p; s.cost_part = p->cost_part.p; s.psi_in = p->psi0.p;
    s.psi_mstride = p->member_states ? p->pb.state_count * 2 * p->NP : 0;
    s.vecs_mstride = p->vecs_mstride;
    s.S_norm = p->state_sharded ? p->pb.state_total : p->pb.state_count;
    s.const_on = (!p->state_sharded || p->pb.state_first == 0) ? 1 : 0;
    s.coh_out = p->state_sharded ? p->coh_out : nullptr;
    s.coh_in = p->state_sharded ? p->coh_in : nullptr;
    return s;
}

// the arguments of the sequential boundary passes: those of the sweeps with the chunks of level `coarse`
SweepArgs make_bargs(qocb_plan *p) {
    SweepArgs s = make_sargs(p);
    if (p->coarse > p->levels) {
        s.chunkP = p->lvlP.p + (size_t)p->lvl_off[p->coarse] * 2 * p->NP * p->NP;
        s.chunk_begin = p->cb_lvl.p + p->cb_off[p->coarse];
        s.member_chunk0 = p->mc0_lvl.p + 2 * p->coarse;
    }
    return s;
}
// called whenever the cost list changes.  With step costs the chunks of the costate pass are coupled through their particular
// parts: k_mid_bwd<PARTICULAR> combines those of the sweep chunks into one per coarse chunk before the coarse pass
void pick_levels(qocb_plan *p) {
    const char *n3 = getenv("QOCB_THREE_LEVEL_STEP");                // "0": step-cost plans stay on two levels (A/B)
    if (p->have_step_costs && n3 && n3[0] == '0') { p->levels = p->lv2; p->coarse = p->lv2; }
    else { p->levels = p->lv3s; p->coarse = p->lv3c; }
}

// with member terms (qocb_add_member_cost) the device table holds one block per member - its own vectors of member terms,
// copies of the shared ones - with the terms' offsets inside a block, so member e's kernels read block e exactly as a
// one-member plan reads its table
int upload_costs(qocb_plan *p) {
    if (p->terms.n == p->h_terms.size() && p->terms.n > 0) return 0;
    std::vector<CostTerm> terms = p->h_terms;
    std::vector<double> packed;
    const std::vector<double> *vecs = &p->h_vecs;
    p->vecs_mstride = 0;
    if (std::any_of(p->h_term_members.begin(), p->h_term_members.end(), [](int m) { return m > 1; })) {
        const size_t E = p->pb.ensemble_count, S = p->pb.state_count, V = 2 * (size_t)p->NP;
        size_t per = 0;                                                 // vectors of one member over all terms
        for (auto &t : terms) { t.vec_off = (int)per; per += S * t.fmax; }
        packed.resize(E * per * V);
        for (size_t e = 0; e < E; ++e)
            for (size_t i = 0; i < terms.size(); ++i) {
                const size_t cnt = S * terms[i].fmax * V;
                const double *src = p->h_vecs.data() + (size_t)p->h_terms[i].vec_off * V + (p->h_term_members[i] > 1 ? e * cnt : 0);
                std::copy(src, src + cnt, packed.begin() + (e * per + terms[i].vec_off) * V);
            }
        vecs = &packed;
        p->vecs_mstride = (long long)(per * V);
    }
    CU_TRY(p, p->terms.alloc(std::max<size_t>(1, terms.size())));
    CU_TRY(p, p->vecs.alloc(std::max<size_t>(1, vecs->size())));
    CU_TRY(p, p->counts.alloc(std::max<size_t>(1, p->h_counts.size())));
    if (!terms.empty()) {
        CU_TRY(p, cudaMemcpy(p->terms.p, terms.data(), sizeof(CostTerm) * terms.size(), cudaMemcpyHostToDevice));
        CU_TRY(p, cudaMemcpy(p->vecs.p, vecs->data(), sizeof(double) * vecs->size(), cudaMemcpyHostToDevice));
        CU_TRY(p, cudaMemcpy(p->counts.p, p->h_counts.data(), sizeof(int) * p->h_counts.size(), cudaMemcpyHostToDevice));
    }
    return 0;
}

template <class C> int launch_reduce(qocb_plan *p, const double *in, double *out, int count) {
    CU_TRY(p, cudaFuncSetAttribute(k_reduce_props<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
    k_reduce_props<C><<<(count + 1) / 2, C::NT, Smem<C>::bytes(), p->stream>>>(in, out, count);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

template <class C> int launch_reduce_radix(qocb_plan *p, const double *in, double *out, int count, int R) {
    CU_TRY(p, cudaFuncSetAttribute(k_reduce_props_radix<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
    k_reduce_props_radix<C><<<(count + R - 1) / R, C::NT, Smem<C>::bytes(), p->stream>>>(in, out, count, R);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// the chunk-boundary passes are chains of dependent mat-vecs: spread the states over CTAs unless the member axis
// already fills the machine
int boundary_state_groups(const qocb_plan *p) {
    const int S = p->pb.state_count;
    if (p->pb.ensemble_count >= p->num_sms) return 1;
    return std::min((S + 3) / 4, 8);        // the mat-vec works on groups of four states (sweep.cuh)
}

int ready(qocb_plan *p) {
    if (!p->ops_set || !p->states_set) { set_error(p, "operators and states must be set before evaluation"); return -1; }
    if (p->mapped && !p->map_set) { set_error(p, "channel_count > 0: qocb_set_node_map must be called before evaluation"); return -1; }
    return upload_costs(p);
}

// time-dependent operators: channel coefficients of the local nodes (first kernel of every evaluation) ...
int enqueue_node_coefs(qocb_plan *p) {
    if (!p->mapped) return 0;
    const int nodes = (p->Nloc - 1) * p->q, tot = nodes * p->KC;
    if (tot > 0)
        k_node_coefs<<<(tot + 127) / 128, 128, 0, p->stream>>>(p->controls.p, p->itab_idx.p, p->itab_w.p, p->map_off.p, p->map_gain.p,
                                                             p->nodecoef.p, nodes, p->KC, p->pb.control_count);
    CU_TRY(p, cudaGetLastError());
    return 0;
}
// ... and the per-node gradient with respect to the interpolated controls, which k_gather_grad scatters to the control points
int node_grad_for_gather(qocb_plan *p, const double **out) {
    *out = p->node_grad.p;
    if (!p->mapped) return 0;
    const int nodes = (p->Nloc - 1) * p->q, E = p->pb.ensemble_count, tot = E * nodes * p->pb.control_count;
    if (tot > 0)
        k_node_grad_map<<<(tot + 127) / 128, 128, 0, p->stream>>>(p->node_grad.p, p->map_gain.p, p->node_grad_x.p, E, nodes, p->KC,
                                                                p->pb.control_count);
    CU_TRY(p, cudaGetLastError());
    *out = p->node_grad_x.p;
    return 0;
}

// ==== large-dimension path (n > 64): batched level-3 pipeline, see large.cuh ======================================
#define BL_TRY(p, expr) do { cublasStatus_t s__ = (expr); if (s__ != CUBLAS_STATUS_SUCCESS) { char b__[640]; snprintf(b__, sizeof(b__), "%s failed: cuBLAS status %d (%s:%d)", #expr, (int)s__, __FILE__, __LINE__); set_error(p, b__); return -2; } } while (0)

inline int lg_blocks(size_t tot) { return (int)std::min<size_t>((tot + 255) / 256, 148 * 16); }

// own DMMA GEMM, general shapes: C (m x nc, ldc) = alpha op(A) (m x k) op(B) (k x nc) + beta C over `batch` matrices
int lg_gemm_rect(qocb_plan *p, bool ta, bool tb, const double2 *A, const double2 *B, double2 *C, int m, int nc, int k, int lda, int ldb,
                 int ldc, double alpha, double beta, int batch, long long sA, long long sB, long long sC, const int *gate = nullptr,
                 int gate_level = 0) {
    const bool thin = nc <= 16;
    const int bn = thin ? 16 : 64;
    const dim3 grid(((m + 63) / 64) * ((nc + bn - 1) / bn), batch);
    if (p->large && p->large->tma_gemm) {                          // TMA-fed variant (zgemm.cuh): operand tensor maps per call
        ZgMaps maps;
        const bool okA = ta ? qocb_host::make_zgemm_map(&maps.a, A, k, m, lda, sA, batch, ZG_LDT, ZG_BK)
                            : qocb_host::make_zgemm_map(&maps.a, A, m, k, lda, sA, batch, ZG_LDA, ZG_BM);
        const bool okB = tb ? qocb_host::make_zgemm_map(&maps.b, B, nc, k, ldb, sB, batch, ZG_LDA, bn)
                            : qocb_host::make_zgemm_map(&maps.b, B, k, nc, ldb, sB, batch, bn + 2, ZG_BK);
        if (okA && okB) {
#define ZT_LAUNCH(TA_, TB_, BN_) k_zgemm_tma<TA_, TB_, BN_><<<grid, ZG_NT, ZgTmaTile<TA_, TB_, BN_>::smem, p->stream>>>(maps, C, m, nc, k, ldc, alpha, beta, sC, gate, gate_level)
            if (thin) {
                if (!ta && !tb) ZT_LAUNCH(false, false, 16); else if (ta && !tb) ZT_LAUNCH(true, false, 16);
                else if (!ta && tb) ZT_LAUNCH(false, true, 16); else ZT_LAUNCH(true, true, 16);
            } else {
                if (!ta && !tb) ZT_LAUNCH(false, false, 64); else if (ta && !tb) ZT_LAUNCH(true, false, 64);
                else if (!ta && tb) ZT_LAUNCH(false, true, 64); else ZT_LAUNCH(true, true, 64);
            }
#undef ZT_LAUNCH
            CU_TRY(p, cudaGetLastError());
            return 0;
        }
    }
#define ZG_LAUNCH(TA_, TB_, BN_) k_zgemm<TA_, TB_, BN_><<<grid, ZG_NT, ZgTile<BN_>::smem, p->stream>>>(A, B, C, m, nc, k, lda, ldb, ldc, alpha, beta, sA, sB, sC, gate, gate_level)
    if (thin) {
        if (!ta && !tb) ZG_LAUNCH(false, false, 16); else if (ta && !tb) ZG_LAUNCH(true, false, 16);
        else if (!ta && tb) ZG_LAUNCH(false, true, 16); else ZG_LAUNCH(true, true, 16);
    } else {
        if (!ta && !tb) ZG_LAUNCH(false, false, 64); else if (ta && !tb) ZG_LAUNCH(true, false, 64);
        else if (!ta && tb) ZG_LAUNCH(false, true, 64); else ZG_LAUNCH(true, true, 64);
    }
#undef ZG_LAUNCH
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// row-major C = alpha op(A) op(B) + beta C over `batch` matrices (strides in elements)
int lg_gemm(qocb_plan *p, bool ta, bool tb, const double2 *A, const double2 *B, double2 *C, double alpha, double beta, int batch,
            long long sA = -1, long long sB = -1, long long sC = -1, const int *gate = nullptr, int gate_level = 0) {
    LargeImpl *L = p->large;
    const int n = L->n;
    if (sA < 0) sA = L->nn; if (sB < 0) sB = L->nn; if (sC < 0) sC = L->nn;
    if (!L->use_cublas_gemm || gate) {                 // own DMMA tile kernel (zgemm.cuh); gated launches exist only there
        return lg_gemm_rect(p, ta, tb, A, B, C, n, n, n, n, n, n, alpha, beta, batch, sA, sB, sC, gate, gate_level);
    }
    const cuDoubleComplex a = make_cuDoubleComplex(alpha, 0.), b = make_cuDoubleComplex(beta, 0.);
    BL_TRY(p, cublasZgemmStridedBatched(L->blas, tb ? CUBLAS_OP_T : CUBLAS_OP_N, ta ? CUBLAS_OP_T : CUBLAS_OP_N, n, n, n, &a,
                                        reinterpret_cast<const cuDoubleComplex *>(B), n, sB,
                                        reinterpret_cast<const cuDoubleComplex *>(A), n, sA, &b,
                                        reinterpret_cast<cuDoubleComplex *>(C), n, sC, batch));
    return 0;
}
int lg_axpby(qocb_plan *p, double2 *out, double al, const double2 *x, double be, const double2 *y, double ga, const double2 *z, int batch) {
    const size_t tot = (size_t)batch * p->large->nn;
    k_lg_axpby<<<lg_blocks(tot), 256, 0, p->stream>>>(out, al, x, be, y, ga, z, tot);
    CU_TRY(p, cudaGetLastError());
    return 0;
}
int lg_copy(qocb_plan *p, double2 *dst, const double2 *src, int batch) {
    CU_TRY(p, cudaMemcpyAsync(dst, src, sizeof(double2) * (size_t)batch * p->large->nn, cudaMemcpyDeviceToDevice, p->stream));
    return 0;
}

// out = alpha (a b - b a)
int lg_comm(qocb_plan *p, const double2 *a, const double2 *b, double2 *out, double alpha, int batch) {
    int rc = lg_gemm(p, false, false, a, b, out, alpha, 0., batch); if (rc) return rc;
    return lg_gemm(p, false, false, b, a, out, -alpha, 1., batch);
}
// cotangents of c = a b - b a (unconjugated convention): abar (+)= alpha (cbar b^T - b^T cbar), bbar (+)= alpha (a^T cbar - cbar a^T);
// beta = 0 overwrites, 1 accumulates; a null output is skipped
int lg_comm_bwd(qocb_plan *p, const double2 *a, const double2 *b, const double2 *cbar, double2 *abar, double2 *bbar, double alpha,
                double beta, int batch) {
    int rc;
    if (abar) {
        rc = lg_gemm(p, false, true, cbar, b, abar, alpha, beta, batch); if (rc) return rc;
        rc = lg_gemm(p, true, false, b, cbar, abar, -alpha, 1., batch); if (rc) return rc;
    }
    if (bbar) {
        rc = lg_gemm(p, true, false, a, cbar, bbar, alpha, beta, batch); if (rc) return rc;
        rc = lg_gemm(p, false, true, cbar, a, bbar, -alpha, 1., batch); if (rc) return rc;
    }
    return 0;
}

// Magnus M6 pieces of slices [jb, jb + Bc) (oracle/adjoint_model.py:magnus_fwd): b1 -> LA1, b2 -> LA2N, b3 -> LA1B,
// c12 = [b1, b2] -> LA2NB, e = 2 b3 + c12 -> LTB, p = -20 b1 - b3 + c12 -> LA6B, qm = b2 - [b1, e] / 60 -> LA4B
int lg_magnus6_pieces(qocb_plan *p, int jb, int Bc) {
    LargeImpl *L = p->large;
    const size_t tot = (size_t)Bc * L->nn;
    const double dt = p->pb.evolution_time / (p->pb.system_eval_count - 1);
    LgCoef cf{p->controls.p, p->itab_idx.p, p->itab_w.p, p->KC, p->q, p->mapped ? p->nodecoef.p : nullptr};
    double2 *b1 = L->arr(LA1), *b2 = L->arr(LA2N), *b3 = L->arr(LA1B), *c12 = L->arr(LA2NB), *e = L->arr(LTB), *d = L->arr(LXB);
    k_lg_assemble6<<<lg_blocks(tot), 256, 0, p->stream>>>(b1, b2, b3, L->G0.p, L->G.p, cf, jb, Bc, L->nn, dt);
    CU_TRY(p, cudaGetLastError());
    int rc = lg_comm(p, b1, b2, c12, 1., Bc); if (rc) return rc;
    rc = lg_axpby(p, e, 2., b3, 1., c12, 0., nullptr, Bc); if (rc) return rc;
    rc = lg_comm(p, b1, e, d, 1., Bc); if (rc) return rc;
    rc = lg_axpby(p, L->arr(LA4B), 1., b2, -1.0 / 60.0, d, 0., nullptr, Bc); if (rc) return rc;
    return lg_axpby(p, L->arr(LA6B), -20., b1, -1., b3, 1., c12, Bc);
}

// ---- own LU and block substitutions of the large-dimension path (large.cuh: k_lg_blockinv) ---------------------------------
constexpr int kLgBlk = 64;

// in-place block LU of the Bc matrices at Q (row-major n x n, batch stride nn)
int lg_block_lu(qocb_plan *p, double2 *Q, int Bc) {
    LargeImpl *L = p->large;
    const int n = L->n;
    const long long nn = L->nn;
    for (int k0 = 0; k0 < n; k0 += kLgBlk) {
        const int bs = std::min(kLgBlk, n - k0), rest = n - k0 - bs;
        k_lg_blockinv<C64><<<Bc, C64::NT, Smem<C64>::bytes(), p->stream>>>(Q, n, k0, bs, nn, L->lu_flag.p);
        CU_TRY(p, cudaGetLastError());
        if (rest <= 0) break;
        double2 *D = Q + (size_t)k0 * n + k0, *Q12 = D + bs, *Q21 = Q + (size_t)(k0 + bs) * n + k0, *Q22 = Q21 + bs;
        int rc = lg_gemm_rect(p, false, false, D, Q12, Q12, bs, rest, bs, n, n, n, 1., 0., Bc, nn, nn, nn); if (rc) return rc;      // U12 = D^-1 Q12 (in place)
        rc = lg_gemm_rect(p, false, false, Q21, Q12, Q22, rest, rest, bs, n, n, n, -1., 1., Bc, nn, nn, nn); if (rc) return rc;     // Q22 -= Q21 U12
    }
    return 0;
}

// X <- X Q^-1 (transposed = false) or X Q^-T (true) for the block factors at Q; X: m x n with row stride ldx, batch stride sX.
// T: scratch of Bc matrices (row stride n, batch stride nn, at least m rows each).
int lg_solve_right(qocb_plan *p, const double2 *Q, double2 *X, int m, int ldx, long long sX, double2 *T, int Bc, bool transposed) {
    LargeImpl *L = p->large;
    const int n = L->n;
    const long long nn = L->nn;
    const int nb = (n + kLgBlk - 1) / kLgBlk;
    int rc;
    if (!transposed) {
        // X L U = P:  Y = X L solves Y U = P (U unit block upper), then X L = Y (L block lower, inverted diagonal blocks stored)
        for (int j = 1; j < nb; ++j) {
            const int c0 = j * kLgBlk, bs = std::min(kLgBlk, n - c0);
            rc = lg_gemm_rect(p, false, false, X, Q + c0, X + c0, m, bs, c0, ldx, n, ldx, -1., 1., Bc, sX, nn, sX); if (rc) return rc;
        }
        for (int j = nb - 1; j >= 0; --j) {
            const int c0 = j * kLgBlk, bs = std::min(kLgBlk, n - c0), rest = n - c0 - bs;
            if (rest > 0) { rc = lg_gemm_rect(p, false, false, T + c0 + bs, Q + (size_t)(c0 + bs) * n + c0, X + c0, m, bs, rest, n, n, ldx, -1., 1., Bc, nn, nn, sX); if (rc) return rc; }
            rc = lg_gemm_rect(p, false, false, X + c0, Q + (size_t)c0 * n + c0, T + c0, m, bs, bs, ldx, n, n, 1., 0., Bc, sX, nn, nn); if (rc) return rc;
        }
    } else {
        // X U^T L^T = R:  Z = X U^T solves Z L^T = R (forward over the column blocks), then X U^T = Z (backward)
        for (int j = 0; j < nb; ++j) {
            const int c0 = j * kLgBlk, bs = std::min(kLgBlk, n - c0);
            if (j > 0) { rc = lg_gemm_rect(p, false, true, T, Q + (size_t)c0 * n, X + c0, m, bs, c0, n, n, ldx, -1., 1., Bc, nn, nn, sX); if (rc) return rc; }
            rc = lg_gemm_rect(p, false, true, X + c0, Q + (size_t)c0 * n + c0, T + c0, m, bs, bs, ldx, n, n, 1., 0., Bc, sX, nn, nn); if (rc) return rc;
        }
        for (int j = nb - 2; j >= 0; --j) {
            const int c0 = j * kLgBlk, bs = std::min(kLgBlk, n - c0), rest = n - c0 - bs;
            rc = lg_gemm_rect(p, false, true, T + c0 + bs, Q + (size_t)c0 * n + c0 + bs, T + c0, m, bs, rest, n, n, n, -1., 1., Bc, nn, nn, nn); if (rc) return rc;
        }
    }
    const size_t tot = (size_t)Bc * m * n;
    k_lg_copy_rect<<<lg_blocks(tot), 256, 0, p->stream>>>(X, T, m, n, ldx, n, sX, nn, Bc);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int large_init(qocb_plan *p) {
    LargeImpl *L = new LargeImpl();
    p->large = L;
    const int n = p->pb.hilbert_size;
    L->n = n; L->nn = n * n;
    const int Lsl = p->Nloc - 1;
    const size_t per = (size_t)LCOUNT * L->nn * sizeof(double2);
    L->B = (int)std::max<size_t>(1, std::min<size_t>((size_t)Lsl, std::min<size_t>(256, ((size_t)6 << 30) / per)));
    { const char *e = getenv("QOCB_LARGE_CUBLAS"); L->use_cublas_gemm = e && e[0] == '1'; }
#define ZG_ATTR(TA_, TB_, BN_) CU_TRY(p, cudaFuncSetAttribute(k_zgemm<TA_, TB_, BN_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZgTile<BN_>::smem))
    ZG_ATTR(false, false, 64); ZG_ATTR(true, false, 64); ZG_ATTR(false, true, 64); ZG_ATTR(true, true, 64);
    ZG_ATTR(false, false, 16); ZG_ATTR(true, false, 16); ZG_ATTR(false, true, 16); ZG_ATTR(true, true, 16);
#undef ZG_ATTR
#define ZT_ATTR(TA_, TB_, BN_) CU_TRY(p, cudaFuncSetAttribute(k_zgemm_tma<TA_, TB_, BN_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ZgTmaTile<TA_, TB_, BN_>::smem))
    ZT_ATTR(false, false, 64); ZT_ATTR(true, false, 64); ZT_ATTR(false, true, 64); ZT_ATTR(true, true, 64);
    ZT_ATTR(false, false, 16); ZT_ATTR(true, false, 16); ZT_ATTR(false, true, 16); ZT_ATTR(true, true, 16);
#undef ZT_ATTR
    { const char *nt = getenv("QOCB_NO_TMA"); L->tma_gemm = qocb_host::encode_tiled_fn() != nullptr && !(nt && nt[0] == '1'); }
    CU_TRY(p, cudaFuncSetAttribute(k_lg_blockinv<C64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C64>::bytes()));
    CU_TRY(p, L->lu_flag.alloc(1));
    CU_TRY(p, cudaMemset(L->lu_flag.p, 0, sizeof(int)));
    BL_TRY(p, cublasCreate(&L->blas));
    BL_TRY(p, cublasSetStream(L->blas, p->stream));
    CU_TRY(p, L->G0.alloc(L->nn)); CU_TRY(p, L->G.alloc((size_t)std::max(1, p->KC) * L->nn));
    CU_TRY(p, L->work.alloc((size_t)LCOUNT * L->B * L->nn));
    CU_TRY(p, L->piv.alloc((size_t)L->B * n)); CU_TRY(p, L->info.alloc(L->B)); CU_TRY(p, L->sarr.alloc(L->B));
    CU_TRY(p, L->ptrQ.alloc(L->B)); CU_TRY(p, L->ptrP.alloc(L->B)); CU_TRY(p, L->ptrRB.alloc(L->B));
    std::vector<double2 *> hq(L->B), hp(L->B), hr(L->B);
    for (int b = 0; b < L->B; ++b) { hq[b] = L->arr(LQ) + (size_t)b * L->nn; hp[b] = L->arr(LP) + (size_t)b * L->nn; hr[b] = L->arr(LRB) + (size_t)b * L->nn; }
    CU_TRY(p, cudaMemcpy(L->ptrQ.p, hq.data(), sizeof(double2 *) * L->B, cudaMemcpyHostToDevice));
    CU_TRY(p, cudaMemcpy(L->ptrP.p, hp.data(), sizeof(double2 *) * L->B, cudaMemcpyHostToDevice));
    CU_TRY(p, cudaMemcpy(L->ptrRB.p, hr.data(), sizeof(double2 *) * L->B, cudaMemcpyHostToDevice));
    // chunk level of the sweeps: first level of the pairwise tree with at most 160 propagators
    L->lvl_count[0] = Lsl;
    int off = 0;
    while (L->lvl_count[L->lstar] > 160) {
        const int nxt = (L->lvl_count[L->lstar] + 1) / 2;
        ++L->lstar;
        L->lvl_count[L->lstar] = nxt; L->lvl_off[L->lstar] = off; off += nxt;
    }
    L->nchunks = L->lvl_count[L->lstar];
    {
        std::vector<int> cb(L->nchunks + 1);
        for (int c = 0; c < L->nchunks; ++c) cb[c] = (int)std::min<long long>((long long)c << L->lstar, Lsl);
        cb[L->nchunks] = Lsl;
        CU_TRY(p, L->cb.alloc(cb.size()));
        CU_TRY(p, cudaMemcpy(L->cb.p, cb.data(), sizeof(int) * cb.size(), cudaMemcpyHostToDevice));
    }
    CU_TRY(p, L->UT.alloc((size_t)Lsl * L->nn));
    CU_TRY(p, L->lvl.alloc((size_t)std::max(1, off) * L->nn));
    if (L->lstar > 0) CU_TRY(p, L->PT.alloc((size_t)L->nchunks * L->nn));
    const size_t VSl = (size_t)p->pb.state_count * 2 * n;
    CU_TRY(p, p->part.alloc((size_t)L->nchunks * VSl)); CU_TRY(p, p->cost_part.alloc(L->nchunks));
    if (p->sharded) { CU_TRY(p, L->treeA.alloc((size_t)((L->nchunks + 1) / 2) * L->nn)); CU_TRY(p, L->treeB.alloc((size_t)((L->nchunks + 3) / 4) * L->nn)); }
    // rank-S reverse pass (S <= 4): PSI [B][4][n], LAM / LAMP / PT [B][n][4], TMPV [B][n][16], LEFT / RIGHT [B][n][48]
    { const char *nl = getenv("QOCB_NO_LOWRANK"); L->lowrank = p->pb.state_count <= 4 && !(nl && nl[0] == '1'); }
    if (L->lowrank) {
        CU_TRY(p, L->lr.alloc((size_t)L->B * n * (4 + 4 + 4 + 4 + 16 + 48 + 48)));
        CU_TRY(p, L->ptrPSI.alloc(L->B));
        std::vector<double2 *> hp2(L->B);
        for (int b = 0; b < L->B; ++b) hp2[b] = L->lr.p + (size_t)b * 4 * n;
        CU_TRY(p, cudaMemcpy(L->ptrPSI.p, hp2.data(), sizeof(double2 *) * L->B, cudaMemcpyHostToDevice));
    }
    L->h_smax.assign((Lsl + L->B - 1) / L->B + 1, 0);
    CU_TRY(p, L->smax_dev.alloc(L->h_smax.size()));
    CU_TRY(p, cudaMemset(L->smax_dev.p, 0, sizeof(int) * L->h_smax.size()));
    L->Lsl = Lsl;
    L->batch_taped.assign((Lsl + L->B - 1) / L->B, 0);
    if (p->pb.store_tape) {
        size_t free_b = 0, total_b = 0;
        CU_TRY(p, cudaMemGetInfo(&free_b, &total_b));
        const size_t need = (size_t)7 * Lsl * L->nn * sizeof(double2) + (size_t)Lsl * (n + 1) * sizeof(int) + (size_t)Lsl * sizeof(double2 *);
        if (need + ((size_t)6 << 30) <= free_b) {
            CU_TRY(p, L->tape.alloc((size_t)7 * Lsl * L->nn)); CU_TRY(p, L->tpiv.alloc((size_t)Lsl * n)); CU_TRY(p, L->tsarr.alloc(Lsl));
            CU_TRY(p, L->tptrQ.alloc(Lsl));
            std::vector<double2 *> hq2(Lsl);
            for (int j = 0; j < Lsl; ++j) hq2[j] = L->tape.p + ((size_t)LargeImpl::tslot(LQ) * Lsl + j) * L->nn;
            CU_TRY(p, cudaMemcpy(L->tptrQ.p, hq2.data(), sizeof(double2 *) * Lsl, cudaMemcpyHostToDevice));
            L->taped = true;
        }
    }
    const int big = 200 * 1024;
    CU_TRY(p, cudaFuncSetAttribute(k_lg_sweep_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_sweep_bwd<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_sweep_bwd<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_boundary_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_boundary_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_boundary_fwd_cl, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_boundary_bwd_cl, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    { const char *nc = getenv("QOCB_NO_CLUSTER"); L->cluster_boundary = !(nc && nc[0] == '1'); }
    CU_TRY(p, cudaFuncSetAttribute(k_lg_prefix, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CU_TRY(p, cudaFuncSetAttribute(k_lg_suffix, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    return 0;
}

// forward intermediates of slices [jb, jb + Bc); keep: also R0 and the squaring inputs for the reverse pass.
// Leaves U_j in arr(LP).  No host synchronisation: the squaring loop enqueues a fixed number of GATED launches that return at
// once beyond the largest squaring count of the batch (smax_slot, device).  keep: the capacity is that of the reverse pass.
constexpr int kLgFwdMaxSq = 10;          // forward-only capacity: ||M||_1 up to 5.37 * 2^10; beyond it the device error flag is raised
int lg_forward_batch(qocb_plan *p, int jb, int Bc, bool keep, int *smax_slot) {
    LargeImpl *L = p->large;
    const int nn = L->nn, order = p->pb.magnus_order;
    const size_t tot = (size_t)Bc * nn;
    const double dt = p->pb.evolution_time / (p->pb.system_eval_count - 1);
    LgCoef cf{p->controls.p, p->itab_idx.p, p->itab_w.p, p->KC, p->q, p->mapped ? p->nodecoef.p : nullptr};
    int rc;
    if (order == 4 && p->comm_ok) {
        k_lg_magnus4_comm<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LM), L->G0.p, L->G.p, L->C0.p, L->Cs.p, cf, jb, Bc, nn, dt);
    } else {
    if (order != 6) k_lg_assemble<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LA1), L->arr(LA2N), L->G0.p, L->G.p, cf, jb, Bc, nn);
    if (order == 2) { rc = lg_axpby(p, L->arr(LM), dt, L->arr(LA1), 0., nullptr, 0., nullptr, Bc); if (rc) return rc; }
    else if (order == 6) {
        rc = lg_magnus6_pieces(p, jb, Bc); if (rc) return rc;
        rc = lg_comm(p, L->arr(LA6B), L->arr(LA4B), L->arr(LA2B), 1., Bc); if (rc) return rc;                     // [p, qm]
        rc = lg_axpby(p, L->arr(LM), 1., L->arr(LA1), 0.5, L->arr(LA1B), 1.0 / 240.0, L->arr(LA2B), Bc); if (rc) return rc;
    } else {
        rc = lg_gemm(p, false, false, L->arr(LA2N), L->arr(LA1), L->arr(LT), 1., 0., Bc); if (rc) return rc;      // a2 a1
        rc = lg_gemm(p, false, false, L->arr(LA1), L->arr(LA2N), L->arr(LT), -1., 1., Bc); if (rc) return rc;     // - a1 a2
        k_lg_axpby<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LM), 0.5 * dt, L->arr(LA1), 0.5 * dt, L->arr(LA2N), (QOCB_S3 / 12.0) * dt * dt, L->arr(LT), tot);
    }
    }
    k_lg_norm_scale<<<Bc, 256, 0, p->stream>>>(L->arr(LM), L->cur_sarr(), L->n, L->own_lu ? L->lu_flag.p : nullptr);
    const int cap = keep ? kLgMaxSq : kLgFwdMaxSq;
    k_lg_batch_max<<<1, 256, 0, p->stream>>>(L->cur_sarr(), Bc, smax_slot, cap, p->err_flag.p);
    rc = lg_gemm(p, false, false, L->arr(LM), L->arr(LM), L->arr(LA2), 1., 0., Bc); if (rc) return rc;
    rc = lg_gemm(p, false, false, L->arr(LA2), L->arr(LA2), L->arr(LA4), 1., 0., Bc); if (rc) return rc;
    rc = lg_gemm(p, false, false, L->arr(LA2), L->arr(LA4), L->arr(LA6), 1., 0., Bc); if (rc) return rc;
    k_lg_poly<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LA2), L->arr(LA4), L->arr(LA6), L->arr(LW1), L->arr(LX1), L->arr(LY), L->arr(LVE), L->n, tot);
    rc = lg_gemm(p, false, false, L->arr(LA6), L->arr(LW1), L->arr(LY), 1., 1., Bc); if (rc) return rc;
    rc = lg_gemm(p, false, false, L->arr(LA6), L->arr(LX1), L->arr(LVE), 1., 1., Bc); if (rc) return rc;
    rc = lg_gemm(p, false, false, L->arr(LM), L->arr(LY), L->arr(LUO), 1., 0., Bc); if (rc) return rc;
    k_lg_pq<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LVE), L->arr(LUO), L->arr(LP), L->arr(LQ), tot);
    CU_TRY(p, cudaGetLastError());
    if (L->own_lu) {                                               // R0 = P Q^-1 by the block LU on the own GEMM
        rc = lg_block_lu(p, L->arr(LQ), Bc); if (rc) return rc;
        rc = lg_solve_right(p, L->arr(LQ), L->arr(LP), L->n, L->n, nn, L->arr(LT), Bc, false); if (rc) return rc;
    } else {
        BL_TRY(p, cublasZgetrfBatched(L->blas, L->n, reinterpret_cast<cuDoubleComplex **>(L->cur_ptrQ()), L->n, L->cur_piv(), L->info.p, Bc));
        int hinfo = 0;
        BL_TRY(p, cublasZgetrsBatched(L->blas, CUBLAS_OP_N, L->n, L->n, reinterpret_cast<const cuDoubleComplex *const *>(L->cur_ptrQ()), L->n, L->cur_piv(),
                                      reinterpret_cast<cuDoubleComplex **>(L->ptrP.p), L->n, &hinfo, Bc));   // R0 = P Q^-1 (row-major)
    }
    if (keep || L->tj >= 0) { rc = lg_copy(p, L->arr(LR0), L->arr(LP), Bc); if (rc) return rc; }
    for (int i = 0; i < cap; ++i) {                                 // expm.py:249-250, gated on the device
        if (keep) k_lg_copy_gated<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LRS0 + i), L->arr(LP), tot, smax_slot, i);
        rc = lg_gemm(p, false, false, L->arr(LP), L->arr(LP), L->arr(LT), 1., 0., Bc, -1, -1, -1, smax_slot, i); if (rc) return rc;
        k_lg_select<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LP), L->arr(LT), L->cur_sarr(), i, nn, tot, smax_slot);
    }
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int lg_expm_all(qocb_plan *p) {
    LargeImpl *L = p->large;
    const int Lsl = p->Nloc - 1;
    { int rc = enqueue_node_coefs(p); if (rc) return rc; }
    for (int attempt = 0; attempt < 2; ++attempt) {
        for (int jb = 0; jb < Lsl; jb += L->B) {
            const int Bc = std::min(L->B, Lsl - jb);
            L->tj = L->taped ? jb : -1;                             // forward intermediates go straight to the tape
            int rc = lg_forward_batch(p, jb, Bc, false, L->smax_dev.p + jb / L->B);
            L->tj = -1;
            if (rc) return rc;
            rc = lg_copy(p, reinterpret_cast<double2 *>(p->U.p) + (size_t)jb * L->nn, L->arr(LP), Bc); if (rc) return rc;
        }
        // the one host synchronisation of an evaluation on this path: squaring counts of the batches (the reverse pass
        // replays taped batches without squarings and recomputes the others) and the verdict on the own LU
        int lu_flag = 0;
        CU_TRY(p, cudaMemcpyAsync(L->h_smax.data(), L->smax_dev.p, sizeof(int) * L->h_smax.size(), cudaMemcpyDeviceToHost, p->stream));
        if (L->own_lu) CU_TRY(p, cudaMemcpyAsync(&lu_flag, L->lu_flag.p, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
        CU_TRY(p, cudaStreamSynchronize(p->stream));
        if (!(L->own_lu && lu_flag)) break;
        // a slice left the regime in which the unpivoted block LU is safe (||A||_1 >= 2.5 or an ill-conditioned diagonal block):
        // this plan factors with cuBLAS getrf / getrs from now on, and the forward pass is redone
        L->own_lu = false;
        CU_TRY(p, cudaMemsetAsync(L->lu_flag.p, 0, sizeof(int), p->stream));
    }
    // transposed copies for the costate sweeps; pairwise product tree up to the chunk level of the sweeps
    const double2 *U = reinterpret_cast<const double2 *>(p->U.p);
    k_lg_transpose<<<148 * 8, dim3(16, 16), 0, p->stream>>>(L->UT.p, U, L->n, Lsl);
    const double2 *in = U;
    for (int l = 1; l <= L->lstar; ++l) {
        double2 *out = L->lvl.p + (size_t)L->lvl_off[l] * L->nn;
        const int count = L->lvl_count[l - 1], pairs = count / 2;
        int rc = lg_gemm(p, false, false, in + L->nn, in, out, 1., 0., pairs, 2LL * L->nn, 2LL * L->nn, L->nn); if (rc) return rc;
        if (count & 1) { rc = lg_copy(p, out + (size_t)pairs * L->nn, in + (size_t)(count - 1) * L->nn, 1); if (rc) return rc; }
        in = out;
    }
    if (L->lstar > 0) k_lg_transpose<<<148 * 8, dim3(16, 16), 0, p->stream>>>(L->PT.p, in, L->n, L->nchunks);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

LgSweep lg_sweep_args(qocb_plan *p) {
    LgSweep g;
    g.a = make_sargs(p);
    LargeImpl *L = p->large;
    g.a.NP = L->n;
    g.a.chunk_begin = L->cb.p;
    g.U = reinterpret_cast<const double2 *>(p->U.p);
    g.UT = L->UT.p;
    g.P = L->lstar > 0 ? L->lvl.p + (size_t)L->lvl_off[L->lstar] * L->nn : g.U;
    g.PT = L->lstar > 0 ? L->PT.p : L->UT.p;
    g.nchunks = L->nchunks;
    return g;
}
size_t lg_sweep_smem(qocb_plan *p) {
    return sizeof(double) * ((size_t)4 * p->pb.state_count * p->large->n + 2 * (size_t)std::max(1, p->ip_total));
}

int lg_backward_all(qocb_plan *p) {
    LargeImpl *L = p->large;
    const int Lsl = p->Nloc - 1, nn = L->nn, order = p->pb.magnus_order, n = L->n;
    const double dt = p->pb.evolution_time / (p->pb.system_eval_count - 1);
    // squaring counts of the forward batches were read back at the end of lg_expm_all: taped batches without squarings are
    // replayed from the tape, the others recompute their forward pass
    for (size_t bi = 0; bi + 1 < L->h_smax.size(); ++bi) {
        if (L->h_smax[bi] > kLgMaxSq) { set_error(p, "scaling count exceeds the reverse-pass capacity of the large-dimension path"); return -4; }
        L->batch_taped[bi] = (L->taped && L->h_smax[bi] == 0) ? 1 : 0;
    }
    for (int jb = 0; jb < Lsl; jb += L->B) {
        const int Bc = std::min(L->B, Lsl - jb);
        const size_t tot = (size_t)Bc * nn;
        int smax = L->h_smax[jb / L->B], rc = 0;                    // same controls as the forward pass => same counts
        if (L->batch_taped[jb / L->B]) {
            // taped batch: only the cheap elementwise pieces are rebuilt (node generators for the Magnus adjoint, W1, X1)
            L->tj = jb;
            LgCoef cf{p->controls.p, p->itab_idx.p, p->itab_w.p, p->KC, p->q, p->mapped ? p->nodecoef.p : nullptr};
            if (!(order == 4 && p->comm_ok) && order != 6)
                k_lg_assemble<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LA1), L->arr(LA2N), L->G0.p, L->G.p, cf, jb, Bc, nn);
            k_lg_poly<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LA2), L->arr(LA4), L->arr(LA6), L->arr(LW1), L->arr(LX1), L->arr(LT), L->arr(LVE), L->n, tot);
        } else {
            L->tj = -1;
            rc = lg_forward_batch(p, jb, Bc, true, L->smax_dev.p + (L->h_smax.size() - 1)); if (rc) return rc;
        }
        struct TjReset { LargeImpl *l; ~TjReset() { l->tj = -1; } } tj_reset{L};
        double2 *RB = L->arr(LRB), *T = L->arr(LT), *M = L->arr(LM);
        if (L->lowrank && smax == 0) {
            // rank-S reverse pass: thin products through the own GEMM (64 x 16 tiles), one rank-48 recombination
            const int S = p->pb.state_count;
            const long long s4 = 4LL * n, s16 = 16LL * n, s48 = 48LL * n;
            double2 *PSI = L->lr.p, *LAM = PSI + (size_t)L->B * 4 * n, *LAMP = LAM + (size_t)L->B * 4 * n, *PTt = LAMP + (size_t)L->B * 4 * n;
            double2 *TMPV = PTt + (size_t)L->B * 4 * n, *LEFT = TMPV + (size_t)L->B * 16 * n, *RIGHT = LEFT + (size_t)L->B * 48 * n;
            const size_t tot4 = (size_t)Bc * n * 4;
            k_lr_load<<<lg_blocks(tot4), 256, 0, p->stream>>>(PSI, LAM, p->psi.p, p->lam.p, jb, Bc, n, S);
            CU_TRY(p, cudaMemsetAsync(LEFT, 0, sizeof(double2) * (size_t)Bc * 48 * n, p->stream));
            if (L->own_lu) {                                       // psit = Q^-1 psi: rows of PSI are the states, PSI <- PSI Q^-T
                rc = lg_solve_right(p, L->arr(LQ), PSI, 4, n, 4LL * n, L->arr(LT), Bc, true); if (rc) return rc;
            } else {
                int hinfo2 = 0;                                    // psit = Q^-1 psi (columns = states)
                BL_TRY(p, cublasZgetrsBatched(L->blas, CUBLAS_OP_T, n, S, reinterpret_cast<const cuDoubleComplex *const *>(L->cur_ptrQ()), n, L->cur_piv(),
                                              reinterpret_cast<cuDoubleComplex **>(L->ptrPSI.p), n, &hinfo2, Bc));
            }
            auto G = [&](bool ta, bool tb, const double2 *A_, const double2 *B_, double2 *C_, int m_, int nc_, int k_, int lda_, int ldb_, int ldc_,
                         double be, long long sa, long long sb, long long sc) {
                return lg_gemm_rect(p, ta, tb, A_, B_, C_, m_, nc_, k_, lda_, ldb_, ldc_, 1.0, be, Bc, sa, sb, sc);
            };
            rc = G(true, false, L->arr(LR0), LAM, LAMP, n, 4, n, n, 4, 4, 0., nn, s4, s4); if (rc) return rc;                 // lamp = R0^T lam
            k_lr_fill<<<lg_blocks(tot4), 256, 0, p->stream>>>(PSI, LAM, LAMP, PTt, TMPV, LEFT, RIGHT, Bc, n);
            rc = G(false, false, L->arr(LY), PTt, TMPV + 4, n, 4, n, n, 4, 16, 0., nn, s4, s16); if (rc) return rc;            // Y psit
            rc = G(true, false, M, TMPV, LEFT, n, 4, n, n, 16, 48, 0., nn, s16, s48); if (rc) return rc;                       // a = A^T pl
            rc = G(false, false, L->arr(LW1), PTt, RIGHT + 32, n, 4, n, n, 4, 48, 1., nn, s4, s48); if (rc) return rc;         // + W1 psit
            rc = G(false, false, L->arr(LX1), PTt, RIGHT + 36, n, 4, n, n, 4, 48, 1., nn, s4, s48); if (rc) return rc;         // + X1 psit
            rc = G(true, false, L->arr(LA6), LEFT, LEFT + 8, n, 8, n, n, 48, 48, 0., nn, s48, s48); if (rc) return rc;         // A6^T [a | ml]
            rc = G(false, false, L->arr(LA4), RIGHT + 32, RIGHT, n, 16, n, n, 48, 48, 1., nn, s48, s48); if (rc) return rc;    // X_a += A4 R6
            rc = G(false, false, L->arr(LA2), RIGHT + 16, RIGHT, n, 16, n, n, 48, 48, 1., nn, s48, s48); if (rc) return rc;    // X_a += A2 R4
            rc = G(false, false, L->arr(LA2), RIGHT + 32, RIGHT + 16, n, 16, n, n, 48, 48, 1., nn, s48, s48); if (rc) return rc; // X_b += A2 R6
            rc = G(true, false, L->arr(LA2), LEFT, LEFT + 16, n, 16, n, n, 48, 48, 0., nn, s48, s48); if (rc) return rc;       // Lb2
            rc = G(true, false, L->arr(LA2), LEFT + 16, LEFT + 32, n, 16, n, n, 48, 48, 0., nn, s48, s48); if (rc) return rc;  // Lb3
            rc = G(false, true, LEFT, RIGHT, L->arr(LA2B), n, n, 48, 48, 48, n, 0., s48, s48, nn); if (rc) return rc;          // a2bar
            rc = G(false, true, TMPV, TMPV + 4, L->arr(LAB), n, n, 4, 16, 16, n, 0., s16, s16, nn); if (rc) return rc;         // pl (Y psit)^T
            rc = lg_gemm(p, false, true, L->arr(LA2B), M, L->arr(LAB), 1., 1., Bc); if (rc) return rc;
            rc = lg_gemm(p, true, false, M, L->arr(LA2B), L->arr(LAB), 1., 1., Bc); if (rc) return rc;
        } else {
        k_lg_ubar<<<lg_blocks(tot), 256, 0, p->stream>>>(RB, p->psi.p, p->lam.p, jb, Bc, n, p->pb.state_count);
        for (int i = smax - 1; i >= 0; --i) {                      // R_{i+1} = R_i^2
            rc = lg_gemm(p, false, true, RB, L->arr(LRS0 + i), T, 1., 0., Bc); if (rc) return rc;
            rc = lg_gemm(p, true, false, L->arr(LRS0 + i), RB, T, 1., 1., Bc); if (rc) return rc;
            k_lg_select<<<lg_blocks(tot), 256, 0, p->stream>>>(RB, T, L->cur_sarr(), i, nn, tot);
        }
        if (L->own_lu) {                                           // pbar = rbar Q^-T
            rc = lg_solve_right(p, L->arr(LQ), RB, n, n, nn, T, Bc, true); if (rc) return rc;
        } else {
            int hinfo = 0;
            BL_TRY(p, cublasZgetrsBatched(L->blas, CUBLAS_OP_T, n, n, reinterpret_cast<const cuDoubleComplex *const *>(L->cur_ptrQ()), n, L->cur_piv(),
                                          reinterpret_cast<cuDoubleComplex **>(L->ptrRB.p), n, &hinfo, Bc));
        }
        rc = lg_gemm(p, true, false, L->arr(LR0), RB, L->arr(LQB), -1., 0., Bc); if (rc) return rc;       // qbar = -R0^T pbar
        rc = lg_axpby(p, L->arr(LUOB), 1., RB, -1., L->arr(LQB), 0., nullptr, Bc); if (rc) return rc;
        rc = lg_axpby(p, L->arr(LVEB), 1., RB, 1., L->arr(LQB), 0., nullptr, Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LUOB), L->arr(LY), L->arr(LAB), 1., 0., Bc); if (rc) return rc;  // abar = uobar Y^T
        rc = lg_gemm(p, true, false, M, L->arr(LUOB), L->arr(LYB), 1., 0., Bc); if (rc) return rc;           // ybar = A^T uobar
        rc = lg_axpby(p, L->arr(LA6B), kB_host(7), L->arr(LYB), kB_host(6), L->arr(LVEB), 0., nullptr, Bc); if (rc) return rc;
        rc = lg_axpby(p, L->arr(LA4B), kB_host(5), L->arr(LYB), kB_host(4), L->arr(LVEB), 0., nullptr, Bc); if (rc) return rc;
        rc = lg_axpby(p, L->arr(LA2B), kB_host(3), L->arr(LYB), kB_host(2), L->arr(LVEB), 0., nullptr, Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LYB), L->arr(LW1), L->arr(LA6B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LVEB), L->arr(LX1), L->arr(LA6B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, true, false, L->arr(LA6), L->arr(LYB), L->arr(LTB), 1., 0., Bc); if (rc) return rc;  // w1bar
        rc = lg_gemm(p, true, false, L->arr(LA6), L->arr(LVEB), L->arr(LXB), 1., 0., Bc); if (rc) return rc; // x1bar
        rc = lg_axpby(p, L->arr(LA6B), 1., L->arr(LA6B), kB_host(13), L->arr(LTB), kB_host(12), L->arr(LXB), Bc); if (rc) return rc;
        rc = lg_axpby(p, L->arr(LA4B), 1., L->arr(LA4B), kB_host(11), L->arr(LTB), kB_host(10), L->arr(LXB), Bc); if (rc) return rc;
        rc = lg_axpby(p, L->arr(LA2B), 1., L->arr(LA2B), kB_host(9), L->arr(LTB), kB_host(8), L->arr(LXB), Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LA6B), L->arr(LA4), L->arr(LA2B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, true, false, L->arr(LA2), L->arr(LA6B), L->arr(LA4B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LA4B), L->arr(LA2), L->arr(LA2B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, true, false, L->arr(LA2), L->arr(LA4B), L->arr(LA2B), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, false, true, L->arr(LA2B), M, L->arr(LAB), 1., 1., Bc); if (rc) return rc;
        rc = lg_gemm(p, true, false, M, L->arr(LA2B), L->arr(LAB), 1., 1., Bc); if (rc) return rc;
        }
        k_lg_unscale<<<lg_blocks(tot), 256, 0, p->stream>>>(L->arr(LAB), L->cur_sarr(), nn, tot);                // mbar
        double2 *AB = L->arr(LAB);
        if (order == 4 && p->comm_ok) {
            if (p->KC > 0) {
                LgCoef cf2{p->controls.p, p->itab_idx.p, p->itab_w.p, p->KC, p->q, p->mapped ? p->nodecoef.p : nullptr};
                k_lg_contract_comm<<<Bc, 256, 0, p->stream>>>(AB, L->G.p, L->C0.p, L->Cs.p, cf2, p->node_grad.p, jb, nn, dt);
            }
            CU_TRY(p, cudaGetLastError());
            continue;
        }
        if (order == 6) {
            // oracle/adjoint_model.py:magnus_bwd; the forward pieces are rebuilt (the Pade reverse pass reused their arrays)
            rc = lg_magnus6_pieces(p, jb, Bc); if (rc) return rc;
            double2 *b1 = L->arr(LA1), *b2 = L->arr(LA2N), *e = L->arr(LTB), *pm = L->arr(LA6B), *qm = L->arr(LA4B);
            double2 *pb = L->arr(LW1), *qb = L->arr(LX1), *db = L->arr(LVE), *t1 = L->arr(LUO), *eb = L->arr(LP);
            double2 *b1b = L->arr(LRB), *b3b = L->arr(LQB), *c12b = L->arr(LUOB);
            rc = lg_comm_bwd(p, pm, qm, AB, pb, qb, 1.0 / 240.0, 0., Bc); if (rc) return rc;              // pbar, qbar (= b2bar so far)
            rc = lg_axpby(p, db, -1.0 / 60.0, qb, 0., nullptr, 0., nullptr, Bc); if (rc) return rc;       // dbar
            rc = lg_comm_bwd(p, b1, e, db, t1, eb, 1., 0., Bc); if (rc) return rc;                        // t1, ebar
            rc = lg_axpby(p, b1b, 1., AB, 1., t1, -20., pb, Bc); if (rc) return rc;
            rc = lg_axpby(p, b3b, 0.5, AB, 2., eb, -1., pb, Bc); if (rc) return rc;
            rc = lg_axpby(p, c12b, 1., eb, 1., pb, 0., nullptr, Bc); if (rc) return rc;
            rc = lg_comm_bwd(p, b1, b2, c12b, b1b, qb, 1., 1., Bc); if (rc) return rc;                    // b1bar +=, b2bar +=
            double2 *n0 = L->arr(LVEB), *n1 = L->arr(LYB), *n2 = L->arr(LT);
            rc = lg_axpby(p, n0, -(QOCB_S15 / 3.0) * dt, qb, (10.0 / 3.0) * dt, b3b, 0., nullptr, Bc); if (rc) return rc;
            rc = lg_axpby(p, n1, dt, b1b, -(20.0 / 3.0) * dt, b3b, 0., nullptr, Bc); if (rc) return rc;
            rc = lg_axpby(p, n2, (QOCB_S15 / 3.0) * dt, qb, (10.0 / 3.0) * dt, b3b, 0., nullptr, Bc); if (rc) return rc;
            if (p->KC > 0)
                k_lg_contract<<<dim3(Bc, 3), 256, 0, p->stream>>>(n0, n1, n2, L->G.p, p->node_grad.p, jb, nn, p->KC, 3);
            CU_TRY(p, cudaGetLastError());
            continue;
        }
        if (order == 2) { rc = lg_axpby(p, L->arr(LA1B), dt, AB, 0., nullptr, 0., nullptr, Bc); if (rc) return rc; }
        else {
            const double f = (QOCB_S3 / 12.0) * dt * dt;
            rc = lg_gemm(p, false, true, AB, L->arr(LA1), T, 1., 0., Bc); if (rc) return rc;                 // a2bar
            rc = lg_gemm(p, true, false, L->arr(LA1), AB, T, -1., 1., Bc); if (rc) return rc;
            rc = lg_axpby(p, L->arr(LA2NB), 0.5 * dt, AB, f, T, 0., nullptr, Bc); if (rc) return rc;
            rc = lg_gemm(p, true, false, L->arr(LA2N), AB, T, 1., 0., Bc); if (rc) return rc;                // a1bar
            rc = lg_gemm(p, false, true, AB, L->arr(LA2N), T, -1., 1., Bc); if (rc) return rc;
            rc = lg_axpby(p, L->arr(LA1B), 0.5 * dt, AB, f, T, 0., nullptr, Bc); if (rc) return rc;
        }
        if (p->KC > 0)
            k_lg_contract<<<dim3(Bc, p->q), 256, 0, p->stream>>>(L->arr(LA1B), L->arr(LA2NB), nullptr, L->G.p, p->node_grad.p, jb, nn, p->KC, p->q);
        CU_TRY(p, cudaGetLastError());
    }
    const int totg = p->pb.control_eval_count * p->pb.control_count;
    const double *ng = nullptr;
    { int rc = node_grad_for_gather(p, &ng); if (rc) return rc; }
    if (totg > 0)
        k_gather_grad<<<(totg + 127) / 128, 128, 0, p->stream>>>(p->csr_ptr.p, p->csr_idx.p, p->csr_w.p, ng, p->grad.p,
                                                               p->pb.control_eval_count, p->pb.control_count, p->q, p->Nloc - 1, 1);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int lg_states_forward(qocb_plan *p, const double *psi_in_dev) {
    LgSweep g = lg_sweep_args(p);
    g.a.psi_in = psi_in_dev;
    const size_t sm = lg_sweep_smem(p);
    if (p->large->cluster_boundary) k_lg_boundary_fwd_cl<<<kLgCluster, kLgThreads, sm, p->stream>>>(g);
    else k_lg_boundary_fwd<<<1, kLgThreads, sm, p->stream>>>(g);
    k_lg_sweep_fwd<<<g.nchunks, kLgThreads, sm, p->stream>>>(g);
    k_finalize_cost<<<1, 32, 0, p->stream>>>(p->cost_part.p, g.nchunks, 1, p->cost.p);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int lg_costates(qocb_plan *p, const double *lam_in_dev, double *b_out_dev, bool do_particular, bool do_sweeps, bool do_boundary = true) {
    LgSweep g = lg_sweep_args(p);
    g.a.lam_in = lam_in_dev; g.a.b_out = b_out_dev;
    const size_t sm = lg_sweep_smem(p);
    if (do_particular && p->have_step_costs) k_lg_sweep_bwd<true><<<g.nchunks, kLgThreads, sm, p->stream>>>(g);
    if (do_boundary) {
        if (p->large->cluster_boundary) k_lg_boundary_bwd_cl<<<kLgCluster, kLgThreads, sm, p->stream>>>(g, p->have_step_costs ? 1 : 0);
        else k_lg_boundary_bwd<<<1, kLgThreads, sm, p->stream>>>(g, p->have_step_costs ? 1 : 0);
    }
    if (do_sweeps) k_lg_sweep_bwd<false><<<g.nchunks, kLgThreads, sm, p->stream>>>(g);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// ev != nullptr: stage boundaries as in enqueue_eval (1 expm forward incl. the propagator tree, 2-3 state sweeps,
// 4 costate sweeps, 5-6 expm reverse + gather)
int lg_eval(qocb_plan *p, bool with_grad, cudaEvent_t *ev) {
    auto rec = [&](int i) { if (ev) cudaEventRecord(ev[i], p->stream); };
    int rc = lg_expm_all(p); if (rc) return rc;
    rec(1); rec(2);
    rc = lg_states_forward(p, p->psi0.p); if (rc) return rc;
    rec(3);
    if (with_grad) {
        rc = lg_costates(p, nullptr, nullptr, true, true); if (rc) return rc;
        rec(4);
        rc = lg_backward_all(p); if (rc) return rc;
        rec(5);
    } else { rec(4); rec(5); }
    rec(6); rec(7);
    return 0;
}

// product of all local propagators (pairwise tree of batched GEMMs) -> out_dev[n*n] (interleaved)
int lg_shard_propagator(qocb_plan *p, double2 *out_dev) {
    LargeImpl *L = p->large;
    const int nn = L->nn;
    const double2 *in = L->lstar > 0 ? L->lvl.p + (size_t)L->lvl_off[L->lstar] * nn : reinterpret_cast<const double2 *>(p->U.p);
    int count = L->nchunks;
    double2 *bufs[2] = {L->treeA.p, L->treeB.p};
    int which = 0;
    if (count == 1) return lg_copy(p, out_dev, in, 1);
    while (count > 1) {
        double2 *out = (count <= 2) ? out_dev : bufs[which];
        const int pairs = count / 2;
        int rc = lg_gemm(p, false, false, in + nn, in, out, 1., 0., pairs, 2LL * nn, 2LL * nn, nn); if (rc) return rc;   // later * earlier
        if (count & 1) { rc = lg_copy(p, out + (size_t)pairs * nn, in + (size_t)(count - 1) * nn, 1); if (rc) return rc; }
        in = out; count = (count + 1) / 2; which ^= 1;
    }
    return 0;
}

// ---- pipeline phases (each only enqueues on the plan stream) -----------------------------------------------
int reduce_level(qocb_plan *p, const double *in, double *out, int count) {
    return dispatch(p->NP, [&] { return launch_reduce<C8>(p, in, out, count); }, [&] { return launch_reduce<C16>(p, in, out, count); },
                    [&] { return launch_reduce<C32>(p, in, out, count); }, [&] { return launch_reduce<C64>(p, in, out, count); });
}

// mid (optional): recorded after the Magnus pass + k_forward, before the propagator tree
int enqueue_expm_forward(qocb_plan *p, bool with_grad, cudaEvent_t mid = nullptr) {
    KArgs ka = make_kargs(p);
    if (!with_grad) ka.tape = nullptr;
    int rc = enqueue_node_coefs(p); if (rc) return rc;
    rc = dispatch(p->NP, [&] { return launch_forward<C8>(p, ka); }, [&] { return launch_forward<C16>(p, ka); },
                      [&] { return launch_forward<C32>(p, ka); }, [&] { return launch_forward<C64>(p, ka); });
    if (rc) return rc;
    if (mid) cudaEventRecord(mid, p->stream);
    // propagator tree up to the level the sweeps run on
    const size_t GM = 2 * (size_t)p->NP * p->NP;
    const double *in = p->chunkP.p;
    for (int l = 1; l <= p->coarse; ++l) {
        double *out = p->lvlP.p + (size_t)p->lvl_off[l] * GM;
        rc = reduce_level(p, in, out, p->lvl_count[l - 1]);
        if (rc) return rc;
        in = out;
    }
    return 0;
}

// product of all chunk propagators of this shard (member 0) -> out_dev[GMAT]
int enqueue_shard_propagator(qocb_plan *p, double *out_dev) {
    const size_t GM = 2 * (size_t)p->NP * p->NP;
    const double *in = p->coarse > 0 ? p->lvlP.p + (size_t)p->lvl_off[p->coarse] * GM : p->chunkP.p;   // continue the tree
    int count = p->lvl_count[p->coarse];
    double *bufs[2] = {p->redA.p, p->redB.p};
    int which = 0;
    if (count == 1) {
        CU_TRY(p, cudaMemcpyAsync(out_dev, in, sizeof(double) * GM, cudaMemcpyDeviceToDevice, p->stream));
        return 0;
    }
    const int R = 4;                                                 // 148 chunks: 148 -> 37 -> 10 -> 3 -> 1
    while (count > 1) {
        double *out = (count <= R) ? out_dev : bufs[which];
        int rc = dispatch(p->NP, [&] { return launch_reduce_radix<C8>(p, in, out, count, R); }, [&] { return launch_reduce_radix<C16>(p, in, out, count, R); },
                          [&] { return launch_reduce_radix<C32>(p, in, out, count, R); }, [&] { return launch_reduce_radix<C64>(p, in, out, count, R); });
        if (rc) return rc;
        in = out; count = (count + R - 1) / R; which ^= 1;
    }
    return 0;
}

int enqueue_state_forward(qocb_plan *p, const double *psi_in_dev, cudaEvent_t mid) {
    SweepArgs sa = make_sargs(p);
    sa.psi_in = psi_in_dev;
    const size_t sw_smem = sweep_smem_bytes(p->NP, sa.S, p->ip_total);
    const dim3 bgrid(sa.E, boundary_state_groups(p));
    SweepArgs ba = make_bargs(p);
    ba.psi_in = psi_in_dev;
    SWEEP_NP(p->NP, (k_boundary_fwd<NPc><<<bgrid, kSwThreads, sw_smem, p->stream>>>(ba)));
    if (p->coarse > p->levels) {
        const dim3 mgrid(p->lvl_count[p->coarse], boundary_state_groups(p));
        SWEEP_NP(p->NP, (k_mid_fwd<NPc><<<mgrid, kSwThreads, sw_smem, p->stream>>>(sa, p->lvl_count[p->levels], 1 << (p->coarse - p->levels))));
    }
    if (mid) cudaEventRecord(mid, p->stream);
    SWEEP_NP(p->NP, (k_sweep_fwd<NPc><<<p->lvl_count[p->levels], kSwThreads, sw_smem, p->stream>>>(sa)));
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// costate pass.  particular_only: chunk particular parts (if step costs) + boundary pass with `lam_in_dev`
// (nullptr = zero) writing the costate at the first local state to b_out_dev; otherwise also the local sweeps.
int enqueue_costate(qocb_plan *p, const double *lam_in_dev, double *b_out_dev, bool do_particular, bool do_sweeps, bool do_boundary = true) {
    SweepArgs sa = make_sargs(p);
    sa.lam_in = lam_in_dev; sa.b_out = b_out_dev;
    const size_t sw_smem = sweep_smem_bytes(p->NP, sa.S, p->ip_total);
    if (do_particular && p->have_step_costs) SWEEP_NP(p->NP, (k_sweep_bwd<NPc, true><<<p->lvl_count[p->levels], kSwThreads, sw_smem, p->stream>>>(sa)));
    const dim3 bgrid(sa.E, boundary_state_groups(p));
    const bool three = p->coarse > p->levels;
    const dim3 mgrid(p->lvl_count[p->coarse], boundary_state_groups(p));
    const int nfine = p->lvl_count[p->levels], span = 1 << (p->coarse - p->levels), hp = p->have_step_costs ? 1 : 0;
    if (three && do_particular && p->have_step_costs)
        SWEEP_NP(p->NP, (k_mid_bwd<NPc, true><<<mgrid, kSwThreads, sw_smem, p->stream>>>(sa, nfine, span, 1, p->part_coarse.p)));
    if (do_boundary) {
        SweepArgs ba = make_bargs(p);
        ba.lam_in = lam_in_dev; ba.b_out = b_out_dev;
        if (three) ba.part = p->part_coarse.p;
        SWEEP_NP(p->NP, (k_boundary_bwd<NPc><<<bgrid, kSwThreads, sw_smem, p->stream>>>(ba, hp)));
    }
    if (do_sweeps && three)
        SWEEP_NP(p->NP, (k_mid_bwd<NPc, false><<<mgrid, kSwThreads, sw_smem, p->stream>>>(sa, nfine, span, hp, nullptr)));
    if (do_sweeps) SWEEP_NP(p->NP, (k_sweep_bwd<NPc, false><<<p->lvl_count[p->levels], kSwThreads, sw_smem, p->stream>>>(sa)));
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int enqueue_expm_backward(qocb_plan *p, cudaEvent_t mid) {
    KArgs ka = make_kargs(p);
    int rc = dispatch(p->NP, [&] { return launch_backward<C8>(p, ka); }, [&] { return launch_backward<C16>(p, ka); },
                      [&] { return launch_backward<C32>(p, ka); }, [&] { return launch_backward<C64>(p, ka); });
    if (rc) return rc;
    if (mid) cudaEventRecord(mid, p->stream);
    const int tot = p->pb.control_eval_count * p->pb.control_count;
    const double *ng = nullptr;
    rc = node_grad_for_gather(p, &ng); if (rc) return rc;
    if (tot > 0 && p->batch) {
        const long long bt = (long long)tot * p->pb.ensemble_count;
        k_gather_grad_members<<<(unsigned)((bt + 127) / 128), 128, 0, p->stream>>>(p->csr_ptr.p, p->csr_idx.p, p->csr_w.p, ng,
                                                                              p->grad.p, p->pb.control_eval_count,
                                                                              p->pb.control_count, p->q, p->Nloc - 1,
                                                                              p->pb.ensemble_count);
    } else if (tot > 0) {
        k_gather_grad<<<(tot + 127) / 128, 128, 0, p->stream>>>(p->csr_ptr.p, p->csr_idx.p, p->csr_w.p, ng,
                                                              p->grad.p, p->pb.control_eval_count, p->pb.control_count,
                                                              p->q, p->Nloc - 1, p->pb.ensemble_count);
    }
    CU_TRY(p, cudaGetLastError());
    return 0;
}

int enqueue_finalize(qocb_plan *p) {
    if (p->batch) {
        const int E = p->pb.ensemble_count;
        k_member_cost<<<(E + 127) / 128, 128, 0, p->stream>>>(p->cost_part.p, make_sargs(p).member_chunk0, E, p->cost.p);
    } else {
        k_finalize_cost<<<1, 32, 0, p->stream>>>(p->cost_part.p, p->lvl_count[p->levels], p->pb.ensemble_count, p->cost.p);
    }
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// enqueue one (unsharded) evaluation on the plan stream; ev != nullptr records stage boundaries (8 events)
int enqueue_eval(qocb_plan *p, bool with_grad, cudaEvent_t *ev) {
    if (p->sharded) { set_error(p, "this plan covers a slice range: use the qocb_shard_* phase calls"); return -1; }
    if (p->state_sharded) { set_error(p, "this plan holds a share of the states: use the qocb_state_shard_* phase calls"); return -1; }
    int rc = ready(p); if (rc) return rc;
    auto rec = [&](int i) { if (ev) cudaEventRecord(ev[i], p->stream); };
    rec(0);
    if (p->large) {
        return lg_eval(p, with_grad, ev);
    }
    rc = enqueue_expm_forward(p, with_grad, ev ? ev[8] : nullptr); if (rc) return rc;
    rec(1);
    rc = enqueue_state_forward(p, p->psi0.p, ev ? ev[2] : nullptr); if (rc) return rc;
    rec(3);
    if (with_grad) {
        rc = enqueue_costate(p, nullptr, nullptr, true, true); if (rc) return rc;
        rec(4);
        rc = enqueue_expm_backward(p, ev ? ev[5] : nullptr); if (rc) return rc;
        rec(6);
    } else {
        rec(4); rec(5); rec(6);
    }
    rc = enqueue_finalize(p); if (rc) return rc;
    rec(7);
    return 0;
}

// doubles of the controls (and of the gradient) crossing the ABI, and the number of costs: [B][M][KR] and B for a control
// batch, [M][KR] and 1 otherwise
size_t ctl_doubles(const qocb_plan *p) {
    return (size_t)(p->batch ? p->pb.ensemble_count : 1) * p->pb.control_eval_count * p->pb.control_count;
}
int cost_count(const qocb_plan *p) { return p->batch ? p->pb.ensemble_count : 1; }

int check_device_flag(qocb_plan *p) {
    int flag = 0;
    CU_TRY(p, cudaMemcpy(&flag, p->err_flag.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) { set_error(p, "device error flag set: scaling count exceeded the recompute tape capacity"); return -4; }
    return 0;
}

}  // namespace

extern "C" {

const char *qocb_version(void) { return "qocb200 0.1 (sm_100a, complex128)"; }

#ifdef QOCB_PROFILE
/* profiling build only: cumulative clock64 ticks per phase id of CTA 0 (then reset) */
int qocb_debug_profile(long long *out32) {
    long long zero[48] = {0};
    if (cudaMemcpyFromSymbol(out32, qocb::g_prof, sizeof(zero)) != cudaSuccess) return -2;
    if (cudaMemcpyToSymbol(qocb::g_prof, zero, sizeof(zero)) != cudaSuccess) return -2;
    return 0;
}
#endif

const char *qocb_last_error(const qocb_plan *plan) { return plan ? plan->err.c_str() : g_last_error.c_str(); }

void *qocb_stream(qocb_plan *plan) { return plan ? (void *)plan->stream : nullptr; }

int qocb_plan_create(const qocb_problem *pb, qocb_plan **out) {
    if (!pb || !out) { set_error((qocb_plan *)nullptr, "null argument"); return -1; }
    *out = nullptr;
    const int NP = pad_dim(pb->hilbert_size);
    if (pb->hilbert_size < 1 || NP < 0) { set_error((qocb_plan *)nullptr, "hilbert_size must be in [1, 512]"); return -1; }
    const bool is_large = NP > 64;
    if (is_large && pb->ensemble_count != 1) { set_error((qocb_plan *)nullptr, "ensembles are not implemented for hilbert_size > 64"); return -1; }
    if (pb->magnus_order != 2 && pb->magnus_order != 4 && pb->magnus_order != 6) { set_error((qocb_plan *)nullptr, "magnus_order must be 2, 4 or 6"); return -1; }
    if (pb->system_eval_count < 2) { set_error((qocb_plan *)nullptr, "system_eval_count must be >= 2"); return -1; }
    if (pb->control_count < 0 || pb->control_count > kMaxKR) { set_error((qocb_plan *)nullptr, "control_count (real channels) must be in [0, 16]"); return -1; }
    if (pb->control_count > 0 && pb->control_eval_count < 2) { set_error((qocb_plan *)nullptr, "control_eval_count must be >= 2"); return -1; }
    if (pb->channel_count < 0 || pb->channel_count > kMaxKR) { set_error((qocb_plan *)nullptr, "channel_count must be in [0, 16]"); return -1; }
    if (pb->state_count < 1 || pb->cost_eval_step < 1 || pb->ensemble_count < 1) { set_error((qocb_plan *)nullptr, "state_count, cost_eval_step, ensemble_count must be >= 1"); return -1; }
    const bool sliced = !(pb->slice_begin == 0 && pb->slice_end == 0);
    if (sliced && (pb->slice_begin < 0 || pb->slice_end <= pb->slice_begin || pb->slice_end > pb->system_eval_count - 1)) { set_error((qocb_plan *)nullptr, "bad slice range: need 0 <= slice_begin < slice_end <= system_eval_count - 1"); return -1; }
    const bool st_sharded = pb->state_total > 0;                    // also a single-rank "shard" of all states goes through the phase calls
    if (pb->state_total < 0 || pb->state_first < 0 || (pb->state_total > 0 && pb->state_first + pb->state_count > pb->state_total)) { set_error((qocb_plan *)nullptr, "bad state range: need state_first + state_count <= state_total"); return -1; }
    if (st_sharded && (sliced || pb->ensemble_count != 1)) { set_error((qocb_plan *)nullptr, "state sharding cannot be combined with time-slice sharding or ensembles"); return -1; }
    if (sliced && pb->ensemble_count != 1) { set_error((qocb_plan *)nullptr, "time-slice sharding and ensembles are mutually exclusive (shard the members instead)"); return -1; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error((qocb_plan *)nullptr, "no CUDA device available (this library has no CPU path)"); return -2; }
    qocb_plan *p = new qocb_plan();
    p->pb = *pb;
    p->NP = NP;
    p->q = pb->magnus_order / 2;
    p->sharded = sliced;
    p->state_sharded = st_sharded;
    p->j0 = sliced ? pb->slice_begin : 0;
    p->Nloc = (sliced ? pb->slice_end - pb->slice_begin : pb->system_eval_count - 1) + 1;
    p->owns_final = !sliced || pb->slice_end == pb->system_eval_count - 1;
    auto fail = [&](int rc) { std::string m = p->err; delete p; g_last_error = m; return rc; };
#define PTRY(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { char b__[512]; snprintf(b__, sizeof(b__), "%s failed: %s", #expr, cudaGetErrorString(e__)); p->err = b__; return fail(-2); } } while (0)
    PTRY(cudaSetDevice(pb->device));
    cudaDeviceProp prop;
    PTRY(cudaGetDeviceProperties(&prop, pb->device));
    p->num_sms = prop.multiProcessorCount;
    PTRY(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    for (auto &e : p->ev) PTRY(cudaEventCreate(&e));
    const int N = p->Nloc, Nm1 = N - 1, E = pb->ensemble_count, M = pb->control_eval_count;   // LOCAL counts
    const int KR = pb->control_count, S = pb->state_count, q = p->q;
    p->mapped = pb->channel_count > 0;
    p->KC = p->mapped ? pb->channel_count : KR;
    const int KC = p->KC;
    const size_t GM = 2 * (size_t)NP * NP;
    // ---- chunks -------------------------------------------------------------------------------------
    int occ = is_large ? 1 : dispatch(NP, [] { return occupancy_fwd<C8>(); }, [] { return occupancy_fwd<C16>(); },
                                      [] { return occupancy_fwd<C32>(); }, [] { return occupancy_fwd<C64>(); });
    int cpm = is_large ? 1 : pb->chunks_per_member;
    // automatic: fill the machine, but keep the sequential chunk-boundary pass (one step per chunk) short: beyond
    // two CTAs per SM the extra boundary steps cost more than the expm kernels gain at small dims
    if (cpm <= 0) cpm = (p->num_sms * std::min(occ, 2) + E - 1) / E;
    cpm = std::max(1, std::min(cpm, Nm1));
    if (is_large) cpm = 1;
    p->nchunks = cpm * E;
    std::vector<int> cb(p->nchunks + 1), mc0(E + 1);
    for (int e = 0; e < E; ++e) {
        mc0[e] = e * cpm;
        for (int c = 0; c < cpm; ++c) cb[e * cpm + c] = e * Nm1 + (int)(((long long)c * Nm1) / cpm);
    }
    mc0[E] = E * cpm; cb[p->nchunks] = E * Nm1;
    PTRY(p->chunk_begin.alloc(cb.size())); PTRY(p->member_chunk0.alloc(mc0.size()));
    PTRY(cudaMemcpy(p->chunk_begin.p, cb.data(), sizeof(int) * cb.size(), cudaMemcpyHostToDevice));
    PTRY(cudaMemcpy(p->member_chunk0.p, mc0.data(), sizeof(int) * mc0.size(), cudaMemcpyHostToDevice));
    // ---- sweep coarsening levels (single member only: pairs must not straddle members) -------------------
    {
        p->lvl_count[0] = p->nchunks;
        std::vector<int> cbl, mcl = {0, p->nchunks};
        std::vector<int> cur = cb;
        int maxl = 0, off = 0;
        p->cb_off[0] = 0; p->lvl_off[0] = 0;
        if (E == 1)
            while (p->lvl_count[maxl] > 1 && maxl < 15) {
                const int cnt = p->lvl_count[maxl], nxt = (cnt + 1) / 2;
                std::vector<int> nb(nxt + 1);
                for (int i = 0; i < nxt; ++i) nb[i] = cur[2 * i];
                nb[nxt] = cur[cnt];
                ++maxl;
                p->lvl_count[maxl] = nxt;
                p->lvl_off[maxl] = off; off += nxt;
                p->cb_off[maxl] = (int)cbl.size();
                cbl.insert(cbl.end(), nb.begin(), nb.end());
                mcl.push_back(0); mcl.push_back(nxt);
                cur = nb;
            }
        // pick the level: boundary passes cost one step per chunk (two directions), local sweeps one step per slice of
        // the longest chunk (two to three passes), every level one small product kernel
        const double r = (double)NP / 64.0;
        const double t_b = 0.4 + 1.4 * r * r, t_s = 0.8 + 2.8 * r * r, t_l = 4.0 + 8.0 * r * r * r;
        int best = 0; double best_t = 1e300;
        for (int l = 0; l <= maxl; ++l) {
            const double len = (double)Nm1 / p->lvl_count[l];
            const double t = 2.0 * p->lvl_count[l] * t_b + 2.5 * len * t_s + l * t_l;
            if (t < best_t) { best_t = t; best = l; }
        }
        if (pb->chunks_per_member > 0 || is_large) best = 0;   // explicit chunking: no coarsening
        p->lv2 = p->lv3s = p->lv3c = best;
        // three levels (one member, unsharded): boundary passes on level lc, the fill-in passes 2^(lc - ls) steps, sweeps
        // on level ls - in as many waves as its chunks need (one CTA per SM)
        if (E == 1 && !st_sharded && !is_large && pb->chunks_per_member <= 0) {
            double best3 = best_t;
            for (int ls = 0; ls <= maxl; ++ls)
                for (int lc = ls + 1; lc <= maxl; ++lc) {
                    const double len = (double)Nm1 / p->lvl_count[ls];
                    const int waves = (p->lvl_count[ls] + p->num_sms - 1) / p->num_sms;
                    const double t = 2.0 * p->lvl_count[lc] * t_b + 2.0 * (double)(1 << (lc - ls)) * t_b + 2.5 * len * waves * t_s + lc * t_l;
                    if (t < best3) { best3 = t; p->lv3s = ls; p->lv3c = lc; }
                }
            const char *n3 = getenv("QOCB_NO_THREE_LEVEL");
            if (n3 && n3[0] == '1') { p->lv3s = p->lv3c = best; }
        }
        pick_levels(p);
        PTRY(p->lvlP.alloc((size_t)std::max(1, off) * GM));
        PTRY(p->cb_lvl.alloc(std::max<size_t>(1, cbl.size()))); PTRY(p->mc0_lvl.alloc(mcl.size()));
        if (!cbl.empty()) PTRY(cudaMemcpy(p->cb_lvl.p, cbl.data(), sizeof(int) * cbl.size(), cudaMemcpyHostToDevice));
        PTRY(cudaMemcpy(p->mc0_lvl.p, mcl.data(), sizeof(int) * mcl.size(), cudaMemcpyHostToDevice));
    }
    // ---- interpolation table (qoc/core/mathmethods.py:36-67 on linspace(0, T, M), programstate.py:41) ----
    {
        const double T = pb->evolution_time, dt = T / (pb->system_eval_count - 1);
        const double s3 = std::sqrt(3.0), s15 = std::sqrt(15.0);
        double nodes[3];
        if (q == 1) nodes[0] = 0.5;
        else if (q == 2) { nodes[0] = 0.5 - s3 / 6; nodes[1] = 0.5 + s3 / 6; }
        else { nodes[0] = 0.5 - s15 / 10; nodes[1] = 0.5; nodes[2] = 0.5 + s15 / 10; }
        std::vector<int> idx((size_t)Nm1 * q * 2, 0);
        std::vector<double> w((size_t)Nm1 * q * 2, 0.0);
        std::vector<std::vector<std::pair<int, double>>> inv(std::max(M, 1));
        if (KR > 0) {
            std::vector<double> xs(M);
            for (int m = 0; m < M; ++m) xs[m] = (M == 1) ? 0.0 : (m == M - 1 ? T : m * (T / (M - 1)));   // numpy.linspace
            for (int j = 0; j < Nm1; ++j)
                for (int i = 0; i < q; ++i) {
                    const double x = (p->j0 + j) * dt + dt * nodes[i];
                    int i0, i1;
                    if (x <= xs[0]) { i0 = 0; i1 = 1; }
                    else if (x >= xs[M - 1]) { i0 = M - 2; i1 = M - 1; }
                    else { i1 = 0; while (!(x <= xs[i1])) ++i1; i0 = i1 - 1; }
                    const double w1 = (x - xs[i0]) / (xs[i1] - xs[i0]);
                    const size_t o = ((size_t)j * q + i) * 2;
                    idx[o] = i0; idx[o + 1] = i1; w[o] = 1.0 - w1; w[o + 1] = w1;
                    inv[i0].push_back({j * q + i, 1.0 - w1});
                    inv[i1].push_back({j * q + i, w1});
                }
        }
        PTRY(p->itab_idx.alloc(idx.size())); PTRY(p->itab_w.alloc(w.size()));
        PTRY(cudaMemcpy(p->itab_idx.p, idx.data(), sizeof(int) * idx.size(), cudaMemcpyHostToDevice));
        PTRY(cudaMemcpy(p->itab_w.p, w.data(), sizeof(double) * w.size(), cudaMemcpyHostToDevice));
        std::vector<int> ptr(std::max(M, 1) + 1, 0), ci; std::vector<double> cw;
        for (int m = 0; m < std::max(M, 1); ++m) {
            for (auto &pr : inv[m]) { ci.push_back(pr.first); cw.push_back(pr.second); }
            ptr[m + 1] = (int)ci.size();
        }
        PTRY(p->csr_ptr.alloc(ptr.size())); PTRY(p->csr_idx.alloc(std::max<size_t>(1, ci.size()))); PTRY(p->csr_w.alloc(std::max<size_t>(1, cw.size())));
        PTRY(cudaMemcpy(p->csr_ptr.p, ptr.data(), sizeof(int) * ptr.size(), cudaMemcpyHostToDevice));
        if (!ci.empty()) {
            PTRY(cudaMemcpy(p->csr_idx.p, ci.data(), sizeof(int) * ci.size(), cudaMemcpyHostToDevice));
            PTRY(cudaMemcpy(p->csr_w.p, cw.data(), sizeof(double) * cw.size(), cudaMemcpyHostToDevice));
        }
    }
    // ---- buffers -------------------------------------------------------------------------------------
    const size_t W = (size_t)E * Nm1;
    p->tape_mats = 8 + kStoredTapeR;
    PTRY(p->G0.alloc((size_t)E * GM)); PTRY(p->G.alloc(std::max<size_t>(1, (size_t)KC) * GM));
    PTRY(p->controls.alloc(std::max<size_t>(1, (size_t)M * KR)));
    PTRY(p->U.alloc(W * GM));
    PTRY(p->meta.alloc(W));
    PTRY(p->scratch.alloc((size_t)p->nchunks * S_COUNT * GM));
    PTRY(p->cta_tape.alloc((size_t)p->nchunks * (8 + kCtaTapeR) * GM));
    PTRY(p->cta_piv.alloc((size_t)p->nchunks * NP));
    PTRY(p->chunkP.alloc((size_t)p->nchunks * GM));
    const size_t VS = (size_t)S * 2 * NP;
    PTRY(p->psi.alloc((size_t)E * N * VS)); PTRY(p->lam.alloc((size_t)E * N * VS));
    PTRY(p->part.alloc((size_t)p->nchunks * VS)); PTRY(p->part_coarse.alloc((size_t)p->nchunks * VS)); PTRY(p->cost_part.alloc(p->nchunks)); PTRY(p->psi0.alloc(VS));
    if (sliced) {
        PTRY(p->redA.alloc((size_t)((p->nchunks + 1) / 2) * GM)); PTRY(p->redB.alloc((size_t)((p->nchunks + 3) / 4) * GM));
        PTRY(p->psi_in.alloc(VS)); PTRY(p->lam_in.alloc(VS));
        const int oc[4] = {0, Nm1, 0, 1};                           // the whole shard as one chunk: chunk_begin | member_chunk0
        PTRY(p->one_chunk.alloc(4));
        PTRY(cudaMemcpy(p->one_chunk.p, oc, sizeof(oc), cudaMemcpyHostToDevice));
    }
    if (!is_large) {
        std::memset(&p->fm, 0, sizeof(p->fm));
        const char *nt = getenv("QOCB_NO_TMA"), *npm = getenv("QOCB_NO_PREMAGNUS");
        if (!(nt && nt[0] == '1'))
            p->fm.tma = (qocb_host::make_matrix_map(&p->fm.mapU, p->U.p, (long long)W, NP) &&
                         qocb_host::make_matrix_map(&p->fm.mapP, p->chunkP.p, p->nchunks, NP)) ? 1 : 0;
        p->premagnus_ok = !(npm && npm[0] == '1');
    }
    PTRY(p->node_grad.alloc(std::max<size_t>(1, W * q * KC)));
    if (p->mapped) {
        PTRY(p->nodecoef.alloc(std::max<size_t>(1, (size_t)Nm1 * q * KC))); PTRY(p->map_off.alloc(std::max<size_t>(1, (size_t)Nm1 * q * KC)));
        PTRY(p->map_gain.alloc(std::max<size_t>(1, (size_t)Nm1 * q * KC * KR))); PTRY(p->node_grad_x.alloc(std::max<size_t>(1, W * q * KR)));
    }
    PTRY(p->grad.alloc(std::max<size_t>(1, (size_t)M * KR)));
    PTRY(p->cost.alloc(1)); PTRY(p->err_flag.alloc(1));
    PTRY(cudaMemset(p->err_flag.p, 0, sizeof(int)));
    PTRY(cudaMemset(p->controls.p, 0, sizeof(double) * p->controls.n));
    PTRY(cudaMemset(p->grad.p, 0, sizeof(double) * p->grad.n));
    PTRY(cudaMemset(p->psi.p, 0, sizeof(double) * p->psi.n)); PTRY(cudaMemset(p->lam.p, 0, sizeof(double) * p->lam.n));
    PTRY(cudaMallocHost(&p->h_pinned, sizeof(double) * (2 * std::max<size_t>(1, (size_t)M * KR) + 8)));
    PTRY(cudaMallocHost(&p->h_fin, sizeof(double) * (size_t)E * S * 2 * NP));
    PTRY(cudaMallocHost(&p->h_flag, sizeof(int)));
    { const char *ng = getenv("QOCB_NO_GRAPH"); p->use_graph = !(ng && ng[0] == '1') && !is_large && !sliced && !st_sharded; }
    // sweep kernels may need > 48 KB of dynamic shared memory
    {
        const int big = 200 * 1024;
        cudaError_t ae = cudaSuccess;
        SWEEP_NP(NP, (ae = set_sweep_attrs<NPc>(big)));
        PTRY(ae);
        if (is_large && large_init(p) != 0) return fail(-2);
    }
    // the reverse-pass tape goes last: if it does not fit beside everything else (and 4 GiB of head-room), the plan
    // runs in recompute mode on the GPU instead
    if (pb->store_tape && !is_large) {
        size_t free_b = 0, total_b = 0;
        PTRY(cudaMemGetInfo(&free_b, &total_b));
        const size_t need = W * p->tape_mats * GM * sizeof(double) + W * NP * sizeof(int);
        if (need + ((size_t)4 << 30) <= free_b) {
            cudaError_t e = p->tape.alloc(W * p->tape_mats * GM);
            if (e != cudaSuccess) { cudaGetLastError(); p->tape.release(); }
            else PTRY(p->tape_piv.alloc(W * NP));
        }
    }
    // Krylov reverse pass: tensor maps of the tapes; reverse-pass variant (QOCB_NO_LOWRANK=1: dense, QOCB_LOWRANK=1: the
    // re-associated rank-S form of round 1, default: Krylov basis of A2)
    std::memset(&p->tmaps, 0, sizeof(p->tmaps));
    if (!is_large && p->fm.tma) {
        bool ok = qocb_host::make_matrix_map(&p->tmaps.mapC, p->cta_tape.p, (long long)p->nchunks * (8 + kCtaTapeR), NP);
        if (p->tape.p) ok = ok && qocb_host::make_matrix_map(&p->tmaps.mapT, p->tape.p, (long long)W * p->tape_mats, NP);
        p->tmaps.tma = ok ? 1 : 0;
    }
    if (!is_large && E == 1 && p->tape.p && p->premagnus_ok && KC <= kMaxCommKR) {
        const size_t slabs = (GM + kAdjSlab - 1) / kAdjSlab;
        PTRY(p->adj_partial.alloc(slabs * W * kAdjMaxOps));
        p->post_adj_ok = true;
    }
    {
        const char *nl = getenv("QOCB_NO_LOWRANK"), *lm = getenv("QOCB_LOWRANK");
        p->lowrank_mode = (nl && nl[0] == '1') ? 0 : ((lm && lm[0] >= '0' && lm[0] <= '2') ? lm[0] - '0' : 2);
    }
#undef PTRY
    *out = p;
    return 0;
}

int qocb_plan_destroy(qocb_plan *p) {
    if (!p) return 0;
    cudaSetDevice(p->pb.device);
    if (p->stream) { cudaStreamSynchronize(p->stream); cudaStreamDestroy(p->stream); }
    for (auto &e : p->ev) if (e) cudaEventDestroy(e);
    if (p->h_pinned) cudaFreeHost(p->h_pinned);
    if (p->h_fin) cudaFreeHost(p->h_fin);
    if (p->h_flag) cudaFreeHost(p->h_flag);
    for (auto &g : p->gexec) if (g) cudaGraphExecDestroy(g);
    delete p;
    return 0;
}

static void drop_graphs(qocb_plan *p) {
    for (auto &g : p->gexec) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    p->host_calls[0] = p->host_calls[1] = 0;
}

int qocb_set_operators(qocb_plan *p, const double *h0, const double *a_ops) {
    if (!p || !h0) { set_error(p, "null argument"); return -1; }
    drop_graphs(p);
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, NP = p->NP, KR = p->KC;   // operator channels
    const int E = p->batch ? 1 : p->pb.ensemble_count;           // drifts: the members of a control batch share one
    const size_t GM = 2 * (size_t)NP * NP;
    auto is_hermitian = [&](const double *h) { return host_is_hermitian(h, n); };
    if (p->large) {                                    // interleaved generators G = -1j * H
        {   // Hermitian operators: the Pade denominator may be factored by the own block LU (large.cuh) while ||A||_1 < 2.5
            bool herm = is_hermitian(h0);
            for (int r = 0; r < KR && herm && a_ops; ++r) herm = is_hermitian(a_ops + (size_t)r * 2 * n * n);
            const char *cl = getenv("QOCB_LARGE_CUBLAS_LU");
            p->hermitian = herm;
            p->large->own_lu = herm && !(cl && cl[0] == '1');
        }
        auto gen = [&](const double *src, double2 *dst_dev) -> cudaError_t {
            std::vector<double> g(2 * (size_t)n * n);
            for (size_t e = 0; e < (size_t)n * n; ++e) { g[2 * e] = src[2 * e + 1]; g[2 * e + 1] = -src[2 * e]; }
            return cudaMemcpy(dst_dev, g.data(), sizeof(double) * g.size(), cudaMemcpyHostToDevice);
        };
        CU_TRY(p, gen(h0, p->large->G0.p));
        if (KR > 0) {
            if (!a_ops) { set_error(p, "a_ops is null but the operator channel count is > 0"); return -1; }
            for (int r = 0; r < KR; ++r) CU_TRY(p, gen(a_ops + (size_t)r * 2 * n * n, p->large->G.p + (size_t)r * n * n));
        }
        p->comm_ok = false;
        { const char *nc = getenv("QOCB_NO_COMM"); if (p->pb.magnus_order == 4 && KR <= kMaxCommKR && !(nc && nc[0] == '1')) p->comm_ok = true; }
        if (p->comm_ok) {                                // commutators [G0, G_r], [G_s, G_r] on the device (own ZGEMM)
            LargeImpl *L = p->large;
            const int npair = KR * (KR - 1) / 2;
            CU_TRY(p, L->C0.alloc((size_t)std::max(1, KR) * L->nn)); CU_TRY(p, L->Cs.alloc((size_t)std::max(1, npair) * L->nn));
            for (int r = 0; r < KR; ++r) {
                int rc = lg_gemm(p, false, false, L->G0.p, L->G.p + (size_t)r * L->nn, L->C0.p + (size_t)r * L->nn, 1., 0., 1); if (rc) return rc;
                rc = lg_gemm(p, false, false, L->G.p + (size_t)r * L->nn, L->G0.p, L->C0.p + (size_t)r * L->nn, -1., 1., 1); if (rc) return rc;
            }
            for (int s_ = 0; s_ < KR; ++s_)
                for (int r = s_ + 1; r < KR; ++r) {
                    double2 *dst = L->Cs.p + (size_t)comm_pair(s_, r, KR) * L->nn;
                    int rc = lg_gemm(p, false, false, L->G.p + (size_t)s_ * L->nn, L->G.p + (size_t)r * L->nn, dst, 1., 0., 1); if (rc) return rc;
                    rc = lg_gemm(p, false, false, L->G.p + (size_t)r * L->nn, L->G.p + (size_t)s_ * L->nn, dst, -1., 1., 1); if (rc) return rc;
                }
            CU_TRY(p, cudaStreamSynchronize(p->stream));
        }
        p->ops_set = true;
        return 0;
    }
    {   // Hermitian operators => anti-Hermitian generators: selects the pivot-free Pade inverse where it is safe (tile.cuh)
        auto is_herm = is_hermitian;
        bool herm = true;
        for (int e = 0; e < E && herm; ++e) herm = is_herm(h0 + (size_t)e * 2 * n * n);
        p->drift_hermitian = herm;
        for (int r = 0; r < KR && herm && a_ops; ++r) herm = is_herm(a_ops + (size_t)r * 2 * n * n);
        p->hermitian = herm && !no_nopiv();
    }
    p->member_ops = false;
    std::vector<double> buf((size_t)std::max(E, KR) * GM);
    for (int e = 0; e < E; ++e) to_planar(h0 + (size_t)e * 2 * n * n, buf.data() + (size_t)e * GM, n, NP, true);
    CU_TRY(p, cudaMemcpy(p->G0.p, buf.data(), sizeof(double) * E * GM, cudaMemcpyHostToDevice));
    if (KR > 0) {
        if (!a_ops) { set_error(p, "a_ops is null but the operator channel count is > 0"); return -1; }
        for (int r = 0; r < KR; ++r) to_planar(a_ops + (size_t)r * 2 * n * n, buf.data() + (size_t)r * GM, n, NP, true);
        CU_TRY(p, cudaMemcpy(p->G.p, buf.data(), sizeof(double) * KR * GM, cudaMemcpyHostToDevice));
    }
    // commutators of the generators G = -1j H for the product-free Magnus M4: C0[e][r] = [G0_e, G_r], Cs[s<r] = [G_s, G_r]
    p->comm_ok = false;
    { const char *nc = getenv("QOCB_NO_COMM"); if (p->pb.magnus_order == 4 && KR <= kMaxCommKR && !(nc && nc[0] == '1')) p->comm_ok = true; }
    if (p->comm_ok) {
        std::vector<HostMat> g(KR);
        for (int r = 0; r < KR; ++r) g[r] = host_generator(a_ops + (size_t)r * 2 * n * n, n);
        const int npair = KR * (KR - 1) / 2;
        CU_TRY(p, p->C0.alloc(std::max<size_t>(1, (size_t)E * KR) * GM)); CU_TRY(p, p->Cs.alloc(std::max<size_t>(1, (size_t)npair) * GM));
        std::vector<double> pl(GM);
        for (int e = 0; e < E; ++e) {
            const HostMat g0 = host_generator(h0 + (size_t)e * 2 * n * n, n);
            for (int r = 0; r < KR; ++r) {
                const HostMat c = host_commutator(g0, g[r], n);
                to_planar(c.data(), pl.data(), n, NP, false);
                CU_TRY(p, cudaMemcpy(p->C0.p + ((size_t)e * KR + r) * GM, pl.data(), sizeof(double) * GM, cudaMemcpyHostToDevice));
            }
        }
        for (int s_ = 0; s_ < KR; ++s_)
            for (int r = s_ + 1; r < KR; ++r) {
                const HostMat c = host_commutator(g[s_], g[r], n);
                to_planar(c.data(), pl.data(), n, NP, false);
                CU_TRY(p, cudaMemcpy(p->Cs.p + (size_t)comm_pair(s_, r, KR) * GM, pl.data(), sizeof(double) * GM, cudaMemcpyHostToDevice));
            }
    }
    p->ops_set = true;
    return 0;
}

int qocb_set_member_operators(qocb_plan *p, const double *a_ops) {
    if (!p || !a_ops) { set_error(p, "null argument"); return -1; }
    if (!p->ops_set) { set_error(p, "qocb_set_member_operators needs qocb_set_operators first"); return -1; }
    if (p->mapped) { set_error(p, "per-member operators need a plan without a node map (time-dependent or non-linear structure)"); return -1; }
    if (p->large || p->sharded || p->state_sharded) { set_error(p, "per-member operators are not implemented for time-sharded, state-sharded or hilbert_size > 64 plans"); return -1; }
    if (p->batch) { set_error(p, "the members of a control batch share their operators"); return -1; }
    drop_graphs(p);
    CU_TRY(p, cudaSetDevice(p->pb.device));
    CU_TRY(p, cudaStreamSynchronize(p->stream));                          // no evaluation in flight reads G, C0 or Cs
    const int n = p->pb.hilbert_size, NP = p->NP, E = p->pb.ensemble_count, KR = p->KC;
    const size_t GM = 2 * (size_t)NP * NP, nn2 = 2 * (size_t)n * n;
    bool herm = p->drift_hermitian;
    for (size_t m = 0; m < (size_t)E * KR && herm; ++m) herm = host_is_hermitian(a_ops + m * nn2, n);
    p->hermitian = herm && !no_nopiv();
    std::vector<double> buf(std::max<size_t>(1, (size_t)E * KR) * GM);
    for (size_t m = 0; m < (size_t)E * KR; ++m) to_planar(a_ops + m * nn2, buf.data() + m * GM, n, NP, true);
    CU_TRY(p, p->G.alloc(buf.size()));
    CU_TRY(p, cudaMemcpy(p->G.p, buf.data(), sizeof(double) * buf.size(), cudaMemcpyHostToDevice));
    // product-free M4: C0[e][r] = [G0_e, G_{e,r}], Cs[e][s<r] = [G_{e,s}, G_{e,r}] from each member's own operators
    if (p->comm_ok) {
        const int npair = KR * (KR - 1) / 2;
        CU_TRY(p, p->Cs.alloc(std::max<size_t>(1, (size_t)E * npair) * GM));
        std::vector<double> g0p(GM), pl(GM), g0(nn2);
        for (int e = 0; e < E; ++e) {
            CU_TRY(p, cudaMemcpy(g0p.data(), p->G0.p + (size_t)e * GM, sizeof(double) * GM, cudaMemcpyDeviceToHost));
            from_planar(g0p.data(), g0.data(), n, NP);                     // G0_e = -1j H0_e, as qocb_set_operators stored it
            std::vector<HostMat> g(KR);
            for (int r = 0; r < KR; ++r) g[r] = host_generator(a_ops + ((size_t)e * KR + r) * nn2, n);
            for (int r = 0; r < KR; ++r) {
                const HostMat c = host_commutator(g0, g[r], n);
                to_planar(c.data(), pl.data(), n, NP, false);
                CU_TRY(p, cudaMemcpy(p->C0.p + ((size_t)e * KR + r) * GM, pl.data(), sizeof(double) * GM, cudaMemcpyHostToDevice));
            }
            for (int s_ = 0; s_ < KR; ++s_)
                for (int r = s_ + 1; r < KR; ++r) {
                    const HostMat c = host_commutator(g[s_], g[r], n);
                    to_planar(c.data(), pl.data(), n, NP, false);
                    CU_TRY(p, cudaMemcpy(p->Cs.p + ((size_t)e * npair + comm_pair(s_, r, KR)) * GM, pl.data(), sizeof(double) * GM, cudaMemcpyHostToDevice));
                }
        }
    }
    p->member_ops = true;
    return 0;
}

int qocb_set_control_batch(qocb_plan *p) {
    if (!p) { set_error(p, "null argument"); return -1; }
    if (p->batch) return 0;
    if (p->ops_set) { set_error(p, "qocb_set_control_batch must be called before qocb_set_operators"); return -1; }
    if (p->mapped) { set_error(p, "control batches need a plan without a node map (time-dependent or non-linear structure)"); return -1; }
    if (p->large || p->sharded || p->state_sharded) { set_error(p, "control batches are not implemented for time-sliced, state-sharded or hilbert_size > 64 plans"); return -1; }
    drop_graphs(p);
    CU_TRY(p, cudaSetDevice(p->pb.device));
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    const int B = p->pb.ensemble_count;
    const size_t GM = 2 * (size_t)p->NP * p->NP, cnt = std::max<size_t>(1, (size_t)B * p->pb.control_eval_count * p->pb.control_count);
    // one shared drift (qocb_set_operators then takes h0 [1][n][n] and builds KR commutators); per start: controls, gradient, cost
    CU_TRY(p, p->G0.alloc(GM));
    CU_TRY(p, p->controls.alloc(cnt)); CU_TRY(p, p->grad.alloc(cnt)); CU_TRY(p, p->cost.alloc(B));
    CU_TRY(p, cudaMemset(p->controls.p, 0, sizeof(double) * cnt));
    CU_TRY(p, cudaMemset(p->grad.p, 0, sizeof(double) * cnt));
    double *hp = nullptr;
    CU_TRY(p, cudaMallocHost(&hp, sizeof(double) * (2 * cnt + B + 8)));
    cudaFreeHost(p->h_pinned);
    p->h_pinned = hp;
    p->batch = true;
    return 0;
}

int qocb_set_node_map(qocb_plan *p, const double *offset, const double *gain) {
    if (!p || !offset) { set_error(p, "null argument"); return -1; }
    if (!p->mapped) { set_error(p, "qocb_set_node_map needs a plan created with channel_count > 0"); return -1; }
    const int KR = p->pb.control_count, KC = p->KC, q = p->q, Nm1 = p->Nloc - 1;
    if (KR > 0 && !gain) { set_error(p, "gain is null but control_count > 0"); return -1; }
    drop_graphs(p);
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const size_t o0 = (size_t)p->j0 * q * KC;                       // local slices [j0, j0 + Nloc - 1)
    CU_TRY(p, cudaMemcpy(p->map_off.p, offset + o0, sizeof(double) * (size_t)Nm1 * q * KC, cudaMemcpyHostToDevice));
    if (KR > 0)
        CU_TRY(p, cudaMemcpy(p->map_gain.p, gain + o0 * KR, sizeof(double) * (size_t)Nm1 * q * KC * KR, cudaMemcpyHostToDevice));
    p->map_set = true;
    return 0;
}

int qocb_set_states(qocb_plan *p, const double *psi0) {
    if (!p || !psi0) { set_error(p, "null argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count;
    std::vector<double> buf((size_t)S * 2 * NP, 0.0);
    for (int s = 0; s < S; ++s)
        for (int a = 0; a < n; ++a) {
            buf[(size_t)s * 2 * NP + a] = psi0[2 * ((size_t)s * n + a)];
            buf[(size_t)s * 2 * NP + NP + a] = psi0[2 * ((size_t)s * n + a) + 1];
        }
    CU_TRY(p, cudaMemcpy(p->psi0.p, buf.data(), sizeof(double) * buf.size(), cudaMemcpyHostToDevice));
    p->states_set = true;
    if (p->member_states) { p->member_states = false; drop_graphs(p); }      // shared states again
    return 0;
}

// per-member data (qocb_set_member_states, qocb_add_member_cost) needs the unsharded n <= 64 path and an ensemble plan
static bool refuse_member_data(qocb_plan *p, const char *call) {
    const char *why = p->batch ? "control batches share their initial states and cost targets"
                      : p->large ? "is not implemented for hilbert_size > 64"
                      : (p->sharded || p->state_sharded) ? "is not implemented for time-sharded or state-sharded plans" : nullptr;
    if (!why) return false;
    set_error(p, (std::string(call) + ": " + why).c_str());
    return true;
}

int qocb_set_member_states(qocb_plan *p, const double *psi0) {
    if (!p || !psi0) { set_error(p, "null argument"); return -1; }
    if (refuse_member_data(p, "qocb_set_member_states")) return -1;
    if (!p->states_set) { set_error(p, "qocb_set_member_states needs qocb_set_states first"); return -1; }
    drop_graphs(p);
    CU_TRY(p, cudaSetDevice(p->pb.device));
    CU_TRY(p, cudaStreamSynchronize(p->stream));                          // no evaluation in flight reads psi0
    const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count, E = p->pb.ensemble_count;
    const size_t VS = (size_t)S * 2 * NP;
    std::vector<double> buf((size_t)E * VS, 0.0);
    for (size_t es = 0; es < (size_t)E * S; ++es)
        for (int a = 0; a < n; ++a) {
            buf[es * 2 * NP + a] = psi0[2 * (es * n + a)];
            buf[es * 2 * NP + NP + a] = psi0[2 * (es * n + a) + 1];
        }
    CU_TRY(p, p->psi0.alloc(buf.size()));
    CU_TRY(p, cudaMemcpy(p->psi0.p, buf.data(), sizeof(double) * buf.size(), cudaMemcpyHostToDevice));
    p->member_states = true;
    return 0;
}

int qocb_clear_costs(qocb_plan *p) {
    if (!p) return -1;
    drop_graphs(p);
    p->h_terms.clear(); p->h_vecs.clear(); p->h_counts.clear(); p->h_term_members.clear(); p->ip_total = 0; p->coh_total = 0;
    p->have_step_costs = false;
    pick_levels(p);
    p->terms.release();
    return 0;
}

// members: 1 for a shared term (vectors [S][fmax][n]), E for a member term (vectors [E][S][fmax][n]; upload_costs lays
// them out per member)
static int add_cost_term(qocb_plan *p, int32_t kind, int32_t step_cost, double weight, const double *vectors, const int32_t *counts,
                  int32_t fmax, int members) {
    if (!p || !vectors) { set_error(p, "null argument"); return -1; }
    if (kind < 0 || kind > 2 || fmax < 1) { set_error(p, "bad cost kind or fmax"); return -1; }
    if (kind != QOCB_COST_FORBID && fmax != 1) { set_error(p, "target costs take one vector per state"); return -1; }
    const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count;
    for (int s = 0; s < S; ++s) {
        const int F = counts ? counts[s] : fmax;
        if (F < 1 || F > fmax) { set_error(p, "counts[s] must be in [1, fmax]"); return -1; }
    }
    CostTerm t;
    t.kind = kind; t.step = step_cost ? 1 : 0; t.fmax = fmax; t.w = weight;
    t.vec_off = (int)(p->h_vecs.size() / (2 * (size_t)NP));
    t.cnt_off = (int)p->h_counts.size();
    t.ip_off = p->ip_total;
    p->ip_total += S * fmax;
    t.coh_off = p->coh_total;
    if (kind == QOCB_COST_TARGET_COHERENT) p->coh_total += t.step ? (p->pb.system_eval_count - 1) / p->pb.cost_eval_step : 1;
    const size_t base = p->h_vecs.size(), nvec = (size_t)members * S * fmax;
    p->h_vecs.resize(base + nvec * 2 * NP, 0.0);
    for (int s = 0; s < S; ++s) p->h_counts.push_back(counts ? counts[s] : fmax);
    for (size_t v = 0; v < nvec; ++v)                               // [members][S][fmax] vectors of n, planar with padding
        for (int a = 0; a < n; ++a) {
            p->h_vecs[base + v * 2 * NP + a] = vectors[2 * (v * n + a)];
            p->h_vecs[base + v * 2 * NP + NP + a] = vectors[2 * (v * n + a) + 1];
        }
    p->h_terms.push_back(t);
    p->h_term_members.push_back(members);
    if (t.step) p->have_step_costs = true;
    pick_levels(p);
    p->terms.release();          // force re-upload
    drop_graphs(p);
    return 0;
}

int qocb_add_cost(qocb_plan *p, int32_t kind, int32_t step_cost, double weight, const double *vectors,
                  const int32_t *counts, int32_t fmax) {
    return add_cost_term(p, kind, step_cost, weight, vectors, counts, fmax, 1);
}

int qocb_add_member_cost(qocb_plan *p, int32_t kind, int32_t step_cost, double weight, const double *vectors,
                         const int32_t *counts, int32_t fmax) {
    if (!p) { set_error(p, "null argument"); return -1; }
    if (refuse_member_data(p, "qocb_add_member_cost")) return -1;
    return add_cost_term(p, kind, step_cost, weight, vectors, counts, fmax, p->pb.ensemble_count);
}

int qocb_upload_controls(qocb_plan *p, const double *controls) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const size_t cnt = ctl_doubles(p);
    if (cnt == 0) return 0;
    if (!controls) { set_error(p, "controls is null"); return -1; }
    std::memcpy(p->h_pinned, controls, sizeof(double) * cnt);
    CU_TRY(p, cudaMemcpyAsync(p->controls.p, p->h_pinned, sizeof(double) * cnt, cudaMemcpyHostToDevice, p->stream));
    return 0;
}

int qocb_run_resident(qocb_plan *p, int32_t with_grad) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    return enqueue_eval(p, with_grad != 0, nullptr);
}

int qocb_sync(qocb_plan *p) {
    if (!p) return -1;
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    return 0;
}

int qocb_download_result(qocb_plan *p, double *cost, double *grad) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const size_t cnt = ctl_doubles(p);
    const int nc = cost_count(p);
    double *hg = p->h_pinned + std::max<size_t>(1, cnt), *hc = hg + std::max<size_t>(1, cnt);
    if (grad && cnt) CU_TRY(p, cudaMemcpyAsync(hg, p->grad.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost, p->stream));
    CU_TRY(p, cudaMemcpyAsync(hc, p->cost.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, p->stream));
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    if (grad && cnt) std::memcpy(grad, hg, sizeof(double) * cnt);
    if (cost) std::memcpy(cost, hc, sizeof(double) * nc);
    return check_device_flag(p);
}

static int fetch_final_states(qocb_plan *p, double *final_states) {
    if (!final_states) return 0;
    const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count, N = p->Nloc, E = p->pb.ensemble_count;
    const size_t VS = (size_t)S * 2 * NP;
    std::vector<double> buf(VS);
    for (int e = 0; e < E; ++e) {
        CU_TRY(p, cudaMemcpy(buf.data(), p->psi.p + ((size_t)e * N + (N - 1)) * VS, sizeof(double) * VS, cudaMemcpyDeviceToHost));
        for (int s = 0; s < S; ++s)
            for (int a = 0; a < n; ++a) {
                final_states[2 * (((size_t)e * S + s) * n + a)] = buf[(size_t)s * 2 * NP + a];
                final_states[2 * (((size_t)e * S + s) * n + a) + 1] = buf[(size_t)s * 2 * NP + NP + a];
            }
    }
    return 0;
}

// everything one host-facing evaluation puts on the stream, in capture-safe form (async copies through pinned buffers)
static int enqueue_host_eval(qocb_plan *p, bool with_grad) {
    const size_t cnt = ctl_doubles(p);
    const size_t VS = (size_t)p->pb.state_count * 2 * p->NP;
    const int N = p->Nloc, E = p->pb.ensemble_count;
    double *hg = p->h_pinned + std::max<size_t>(1, cnt), *hc = hg + std::max<size_t>(1, cnt);
    if (cnt) CU_TRY(p, cudaMemcpyAsync(p->controls.p, p->h_pinned, sizeof(double) * cnt, cudaMemcpyHostToDevice, p->stream));
    int rc = enqueue_eval(p, with_grad, nullptr); if (rc) return rc;
    if (with_grad && cnt) CU_TRY(p, cudaMemcpyAsync(hg, p->grad.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost, p->stream));
    CU_TRY(p, cudaMemcpyAsync(hc, p->cost.p, sizeof(double) * cost_count(p), cudaMemcpyDeviceToHost, p->stream));
    CU_TRY(p, cudaMemcpy2DAsync(p->h_fin, sizeof(double) * VS, p->psi.p + (size_t)(N - 1) * VS, sizeof(double) * N * VS,
                                sizeof(double) * VS, E, cudaMemcpyDeviceToHost, p->stream));
    CU_TRY(p, cudaMemcpyAsync(p->h_flag, p->err_flag.p, sizeof(int), cudaMemcpyDeviceToHost, p->stream));
    return 0;
}

static int host_eval(qocb_plan *p, bool with_grad, const double *controls, double *cost, double *grad, double *final_states) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    if (!p->use_graph) {
        int rc = qocb_upload_controls(p, controls); if (rc) return rc;
        rc = enqueue_eval(p, with_grad, nullptr); if (rc) return rc;
        rc = qocb_download_result(p, cost, with_grad ? grad : nullptr); if (rc) return rc;
        return fetch_final_states(p, final_states);
    }
    int rc = ready(p); if (rc) return rc;                          // synchronous uploads of changed cost tables: never captured
    const size_t cnt = ctl_doubles(p);
    if (cnt) {
        if (!controls) { set_error(p, "controls is null"); return -1; }
        std::memcpy(p->h_pinned, controls, sizeof(double) * cnt);
    }
    const int wg = with_grad ? 1 : 0;
    if (p->gexec[wg]) {
        CU_TRY(p, cudaGraphLaunch(p->gexec[wg], p->stream));
    } else if (p->host_calls[wg]++ < 1) {
        rc = enqueue_host_eval(p, with_grad); if (rc) return rc;    // first call: plain launches (function attributes, lazy init)
    } else {
        cudaGraph_t graph = nullptr;
        CU_TRY(p, cudaStreamBeginCapture(p->stream, cudaStreamCaptureModeThreadLocal));
        rc = enqueue_host_eval(p, with_grad);
        const cudaError_t ce = cudaStreamEndCapture(p->stream, &graph);
        if (rc || ce != cudaSuccess || !graph) {                    // capture refused: fall back to plain launches for good
            cudaGetLastError();
            if (graph) cudaGraphDestroy(graph);
            p->use_graph = false;
            return host_eval(p, with_grad, controls, cost, grad, final_states);
        }
        const cudaError_t ie = cudaGraphInstantiate(&p->gexec[wg], graph, 0);
        cudaGraphDestroy(graph);
        if (ie != cudaSuccess) { cudaGetLastError(); p->gexec[wg] = nullptr; p->use_graph = false; return host_eval(p, with_grad, controls, cost, grad, final_states); }
        CU_TRY(p, cudaGraphLaunch(p->gexec[wg], p->stream));
    }
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    double *hg = p->h_pinned + std::max<size_t>(1, cnt), *hc = hg + std::max<size_t>(1, cnt);
    if (with_grad && grad && cnt) std::memcpy(grad, hg, sizeof(double) * cnt);
    if (cost) std::memcpy(cost, hc, sizeof(double) * cost_count(p));
    if (*p->h_flag) { set_error(p, "device error flag set: scaling count exceeded the recompute tape capacity"); return -4; }
    if (final_states) {
        const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count, E = p->pb.ensemble_count;
        for (int e = 0; e < E; ++e)
            for (int s_ = 0; s_ < S; ++s_)
                for (int a = 0; a < n; ++a) {
                    const double *b = p->h_fin + ((size_t)e * S + s_) * 2 * NP;
                    final_states[2 * (((size_t)e * S + s_) * n + a)] = b[a];
                    final_states[2 * (((size_t)e * S + s_) * n + a) + 1] = b[NP + a];
                }
    }
    return 0;
}

static bool refuse_batch(qocb_plan *p, const char *call) {
    if (!p || !p->batch) return false;
    set_error(p, (std::string(call) + " serves [M][KR] controls and one cost: a control batch takes qocb_batch_cost / "
                  "qocb_batch_cost_and_grad").c_str());
    return true;
}

int qocb_cost(qocb_plan *p, const double *controls, double *cost, double *final_states) {
    if (refuse_batch(p, "qocb_cost")) return -1;
    return host_eval(p, false, controls, cost, nullptr, final_states);
}

int qocb_cost_and_grad(qocb_plan *p, const double *controls, double *cost, double *grad, double *final_states) {
    if (refuse_batch(p, "qocb_cost_and_grad")) return -1;
    return host_eval(p, true, controls, cost, grad, final_states);
}

int qocb_batch_cost(qocb_plan *p, const double *controls, double *costs, double *final_states) {
    if (p && !p->batch) { set_error(p, "qocb_batch_cost needs a control batch (qocb_set_control_batch)"); return -1; }
    return host_eval(p, false, controls, costs, nullptr, final_states);
}

int qocb_batch_cost_and_grad(qocb_plan *p, const double *controls, double *costs, double *grads, double *final_states) {
    if (p && !p->batch) { set_error(p, "qocb_batch_cost_and_grad needs a control batch (qocb_set_control_batch)"); return -1; }
    return host_eval(p, true, controls, costs, grads, final_states);
}

// ---- split evaluation: forward pass now, reverse pass later with an extra cotangent of the final states -------------------
int qocb_forward(qocb_plan *p, const double *controls, double *cost, double *final_states) {
    if (!p || refuse_batch(p, "qocb_forward")) return -1;
    if (p->sharded || p->state_sharded || p->pb.ensemble_count != 1) { set_error(p, "qocb_forward / qocb_backward need an unsharded single-member plan"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    int rc = qocb_upload_controls(p, controls); if (rc) return rc;
    rc = ready(p); if (rc) return rc;
    if (p->large) {
        rc = lg_expm_all(p); if (rc) return rc;
        rc = lg_states_forward(p, p->psi0.p); if (rc) return rc;
    } else {
        rc = enqueue_expm_forward(p, true); if (rc) return rc;      // with the reverse-pass tape
        rc = enqueue_state_forward(p, p->psi0.p, nullptr); if (rc) return rc;
        rc = enqueue_finalize(p); if (rc) return rc;
    }
    rc = qocb_download_result(p, cost, nullptr); if (rc) return rc;
    return fetch_final_states(p, final_states);
}

int qocb_backward(qocb_plan *p, const double *final_seed, double *grad) {
    if (!p || refuse_batch(p, "qocb_backward")) return -1;
    if (p->sharded || p->state_sharded || p->pb.ensemble_count != 1) { set_error(p, "qocb_forward / qocb_backward need an unsharded single-member plan"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, NP = p->large ? n : p->NP, S = p->pb.state_count;
    const double *lam_in = nullptr;
    if (final_seed) {                                               // extra cotangent of the final states, autograd convention
        const size_t VS = (size_t)S * 2 * NP;
        if (p->lam_in.n < VS) CU_TRY(p, p->lam_in.alloc(VS));
        std::vector<double> buf(VS, 0.0);
        for (int s_ = 0; s_ < S; ++s_)
            for (int a = 0; a < n; ++a) {
                buf[(size_t)s_ * 2 * NP + a] = final_seed[2 * ((size_t)s_ * n + a)];
                buf[(size_t)s_ * 2 * NP + NP + a] = final_seed[2 * ((size_t)s_ * n + a) + 1];
            }
        CU_TRY(p, cudaMemcpyAsync(p->lam_in.p, buf.data(), sizeof(double) * VS, cudaMemcpyHostToDevice, p->stream));
        CU_TRY(p, cudaStreamSynchronize(p->stream));                // buf is pageable and dies with this scope
        lam_in = p->lam_in.p;
    }
    int rc;
    if (p->large) {
        rc = lg_costates(p, lam_in, nullptr, true, true); if (rc) return rc;
        rc = lg_backward_all(p); if (rc) return rc;
    } else {
        rc = enqueue_costate(p, lam_in, nullptr, true, true); if (rc) return rc;
        rc = enqueue_expm_backward(p, nullptr); if (rc) return rc;
    }
    double dummy = 0.;
    return qocb_download_result(p, &dummy, grad);
}

int qocb_get_states(qocb_plan *p, double *states) {
    if (!p || !states) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, NP = p->NP, S = p->pb.state_count, N = p->Nloc, E = p->pb.ensemble_count;
    const size_t VS = (size_t)S * 2 * NP, tot = (size_t)E * N * VS;
    std::vector<double> buf(tot);
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    CU_TRY(p, cudaMemcpy(buf.data(), p->psi.p, sizeof(double) * tot, cudaMemcpyDeviceToHost));
    for (size_t en = 0; en < (size_t)E * N; ++en)
        for (int s = 0; s < S; ++s)
            for (int a = 0; a < n; ++a) {
                states[2 * ((en * S + s) * n + a)] = buf[en * VS + (size_t)s * 2 * NP + a];
                states[2 * ((en * S + s) * n + a) + 1] = buf[en * VS + (size_t)s * 2 * NP + NP + a];
            }
    return 0;
}

int qocb_get_final_states(qocb_plan *p, double *final_states) {
    if (!p || !final_states) { set_error(p, "null argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    return fetch_final_states(p, final_states);
}

int qocb_get_node_grad(qocb_plan *p, double *out) {
    if (!p || !out) { set_error(p, "null argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    const size_t cnt = (size_t)p->pb.ensemble_count * (p->Nloc - 1) * p->q * p->KC;
    if (cnt) CU_TRY(p, cudaMemcpy(out, p->node_grad.p, sizeof(double) * cnt, cudaMemcpyDeviceToHost));
    return 0;
}

int qocb_get_propagators(qocb_plan *p, double *props) {
    if (!p || !props) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int n = p->pb.hilbert_size, NP = p->NP;
    const size_t W = (size_t)p->pb.ensemble_count * (p->Nloc - 1), GM = 2 * (size_t)NP * NP;
    std::vector<double> buf(GM);
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    if (p->large) {
        CU_TRY(p, cudaMemcpy(props, p->U.p, sizeof(double) * W * GM, cudaMemcpyDeviceToHost));
        return 0;
    }
    for (size_t w = 0; w < W; ++w) {
        CU_TRY(p, cudaMemcpy(buf.data(), p->U.p + w * GM, sizeof(double) * GM, cudaMemcpyDeviceToHost));
        from_planar(buf.data(), props + w * 2 * n * n, n, NP);
    }
    return 0;
}

static int launch_count_unmapped(qocb_plan *p, int32_t with_grad);
int qocb_launch_count(qocb_plan *p, int32_t with_grad) {
    if (!p) return -1;
    return launch_count_unmapped(p, with_grad) + (p->mapped ? (with_grad ? 2 : 1) : 0);   // k_node_coefs, k_node_grad_map
}
static int launch_count_unmapped(qocb_plan *p, int32_t with_grad) {
    if (p->large) {
        const int batches = (p->Nloc - 2 + p->large->B) / p->large->B;
        const int o = p->pb.magnus_order;
        const int fwd = o == 6 ? 21 : o == 4 ? 14 : 11;                      // own kernels + library calls per batch
        return batches * (fwd + (with_grad ? fwd + (o == 6 ? 60 : o == 4 ? 38 : 30) : 0)) + (with_grad ? 3 : 1);
    }
    const int pm = (p->premagnus_ok && (p->pb.magnus_order == 2 || (p->pb.magnus_order == 4 && p->comm_ok))) ? 1 : 0;   // k_magnus
    const int pa = (with_grad && pm && p->post_adj_ok && p->pb.control_count > 0) ? 2 : 0;                            // k_magnus_adj, k_magnus_adj_final
    const int mids = p->coarse > p->levels ? (with_grad ? 2 + (p->have_step_costs ? 1 : 0) : 1) : 0;                  // k_mid_fwd, k_mid_bwd (+ particular)
    if (!p->sharded) return (with_grad ? (p->have_step_costs ? 9 : 8) : 4) + p->coarse + mids + pm + pa;
    int levels = p->coarse + mids + pm;                                   // pairwise levels for the sweeps, then radix 4 to the root
    for (int c = p->lvl_count[p->coarse]; c > 1; c = (c + 3) / 4) ++levels;
    // forward: expm, tree, prefix, boundary, sweep; backward: [particular sweeps], boundary (twice only with step costs on a
    // shard that is not the last), suffix, sweep, expm, gather, finalize, pack
    const int nb = (p->have_step_costs && !p->owns_final) ? 2 : 1;
    return with_grad ? 1 + levels + 3 + (p->have_step_costs ? 1 : 0) + nb + 6 + pa : 1 + levels + 3 + 2;
}

int qocb_time_resident(qocb_plan *p, int32_t with_grad, int32_t warmup, int32_t iters, int32_t flush_l2,
                       double *ms_total, double *stage_ms) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const size_t flush_bytes = 256ull << 20;
    if (flush_l2 && p->flush.n == 0) CU_TRY(p, p->flush.alloc(flush_bytes / sizeof(double)));
    for (int i = 0; i < warmup; ++i) { int rc = enqueue_eval(p, with_grad != 0, nullptr); if (rc) return rc; }
    CU_TRY(p, cudaStreamSynchronize(p->stream));
    double tot = 0.;
    double st[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < iters; ++i) {
        if (flush_l2) CU_TRY(p, cudaMemsetAsync(p->flush.p, i & 0xff, flush_bytes, p->stream));
        int rc = enqueue_eval(p, with_grad != 0, p->ev);
        if (rc) return rc;
        CU_TRY(p, cudaStreamSynchronize(p->stream));
        float ms = 0.f;
        CU_TRY(p, cudaEventElapsedTime(&ms, p->ev[0], p->ev[7]));
        tot += ms;
        for (int s = 0; s < 7; ++s) { CU_TRY(p, cudaEventElapsedTime(&ms, p->ev[s], p->ev[s + 1])); st[s] += ms; }
        if (!p->large) {                                            // split stage 0: Magnus pass + k_forward | propagator tree (-> stage 7)
            CU_TRY(p, cudaEventElapsedTime(&ms, p->ev[8], p->ev[1]));
            st[7] += ms; st[0] -= ms;
        }
    }
    if (ms_total) *ms_total = tot;
    if (stage_ms) for (int s = 0; s < 8; ++s) stage_ms[s] = st[s];
    return check_device_flag(p);
}

int qocb_flush_l2(qocb_plan *p) {
    if (!p) return -1;
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const size_t flush_bytes = 256ull << 20;
    if (p->flush.n == 0) CU_TRY(p, p->flush.alloc(flush_bytes / sizeof(double)));
    CU_TRY(p, cudaMemsetAsync(p->flush.p, 0x5a, flush_bytes, p->stream));
    return 0;
}

// ---- time-slice sharding phases ------------------------------------------------------------------------
int qocb_shard_matrix_doubles(qocb_plan *p) { return p ? 2 * p->NP * p->NP : -1; }
int qocb_shard_vector_doubles(qocb_plan *p) { return p ? p->pb.state_count * 2 * p->NP : -1; }

int qocb_shard_forward_local(qocb_plan *p, int32_t with_grad, double *shardP_dev) {
    if (!p || !shardP_dev) { set_error(p, "null argument"); return -1; }
    if (!p->sharded) { set_error(p, "plan has no slice range"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    int rc = ready(p); if (rc) return rc;
    p->particular_fresh = false;
    if (p->large) {
        rc = lg_expm_all(p); if (rc) return rc;
        return lg_shard_propagator(p, reinterpret_cast<double2 *>(shardP_dev));
    }
    rc = enqueue_expm_forward(p, with_grad != 0); if (rc) return rc;
    p->shardP_last = shardP_dev;
    return enqueue_shard_propagator(p, shardP_dev);
}

int qocb_shard_forward_finish(qocb_plan *p, const double *allP_dev, int32_t rank) {
    if (!p || !allP_dev || rank < 0) { set_error(p, "bad argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    if (p->large) {
        k_lg_prefix<<<1, kLgThreads, lg_sweep_smem(p), p->stream>>>(reinterpret_cast<const double2 *>(allP_dev), p->psi0.p, p->psi_in.p, rank,
                                                                   p->large->n, p->pb.state_count);
        CU_TRY(p, cudaGetLastError());
        return lg_states_forward(p, p->psi_in.p);
    }
    const size_t sm = prefix_smem_bytes(p->NP, p->pb.state_count);
    SWEEP_NP(p->NP, (k_prefix_states<NPc><<<1, kSweepThreads, sm, p->stream>>>(allP_dev, p->psi0.p, p->psi_in.p, rank, p->pb.state_count)));
    CU_TRY(p, cudaGetLastError());
    int rc = enqueue_state_forward(p, p->psi_in.p, nullptr); if (rc) return rc;
    return enqueue_finalize(p);
}

int qocb_shard_backward_particular(qocb_plan *p, double *b_dev) {
    if (!p || !b_dev) { set_error(p, "null argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    // without step costs a shard that does not hold the final state has no particular part: b = 0, nothing to run
    if (!p->have_step_costs && !p->owns_final) {
        CU_TRY(p, cudaMemsetAsync(b_dev, 0, sizeof(double) * (size_t)qocb_shard_vector_doubles(p), p->stream));
        return 0;
    }
    if (!p->have_step_costs && !p->large && p->shardP_last) {
        // last shard, final-step costs only: b = P_shard^T seed.  One mat-vec with the shard propagator (already built
        // for the exchange) instead of the pass over all chunk boundaries - the other ranks wait for this value
        SweepArgs sa = make_sargs(p);
        sa.chunkP = p->shardP_last; sa.chunk_begin = p->one_chunk.p; sa.member_chunk0 = p->one_chunk.p + 2;
        sa.lam_in = nullptr; sa.b_out = b_dev;
        const size_t sw_smem = sweep_smem_bytes(p->NP, sa.S, p->ip_total);
        const dim3 bgrid(1, boundary_state_groups(p));
        SWEEP_NP(p->NP, (k_boundary_bwd<NPc><<<bgrid, kSwThreads, sw_smem, p->stream>>>(sa, 0)));
        CU_TRY(p, cudaGetLastError());
        return 0;                                                   // particular_fresh stays false: the finish phase runs the full pass
    }
    p->particular_fresh = true;
    if (p->large) return lg_costates(p, nullptr, b_dev, true, false);
    return enqueue_costate(p, nullptr, b_dev, true, false);
}

int qocb_shard_backward_finish(qocb_plan *p, const double *allP_dev, const double *allb_dev, int32_t rank, int32_t world) {
    if (!p || !allP_dev || !allb_dev || rank < 0 || rank >= world) { set_error(p, "bad argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    // the last shard receives a zero costate: its boundary costates are those of the particular pass already in `lam`
    const bool reuse = rank == world - 1 && p->owns_final && p->particular_fresh;
    p->particular_fresh = false;
    if (p->large) {
        LargeImpl *L = p->large;
        if (L->allPT.n < (size_t)world * L->nn) CU_TRY(p, L->allPT.alloc((size_t)world * L->nn));
        k_lg_transpose<<<world * 64, dim3(16, 16), 0, p->stream>>>(L->allPT.p, reinterpret_cast<const double2 *>(allP_dev), L->n, world);
        k_lg_suffix<<<1, kLgThreads, lg_sweep_smem(p), p->stream>>>(L->allPT.p, allb_dev, p->lam_in.p, rank, world, L->n, p->pb.state_count);
        CU_TRY(p, cudaGetLastError());
        int rc = lg_costates(p, p->lam_in.p, nullptr, false, true, !reuse); if (rc) return rc;
        return lg_backward_all(p);
    }
    const size_t sm = prefix_smem_bytes(p->NP, p->pb.state_count);
    SWEEP_NP(p->NP, (k_suffix_costates<NPc><<<1, kSweepThreads, sm, p->stream>>>(allP_dev, allb_dev, p->lam_in.p, rank, world, p->pb.state_count)));
    CU_TRY(p, cudaGetLastError());
    int rc = enqueue_costate(p, p->lam_in.p, nullptr, false, true, !reuse); if (rc) return rc;
    return enqueue_expm_backward(p, nullptr);
}

// ---- state sharding phases -------------------------------------------------------------------------------------
int qocb_state_shard_coherent_doubles(qocb_plan *p) { return p ? 2 * p->coh_total : -1; }

int qocb_state_shard_forward(qocb_plan *p, int32_t with_grad, double *coh_dev) {
    if (!p || (p->coh_total > 0 && !coh_dev)) { set_error(p, "null argument"); return -1; }
    if (!p->state_sharded) { set_error(p, "plan was not created with a state range (state_total / state_first)"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    int rc = ready(p); if (rc) return rc;
    p->coh_out = coh_dev; p->coh_in = nullptr;
    if (p->coh_total > 0) CU_TRY(p, cudaMemsetAsync(coh_dev, 0, sizeof(double) * 2 * p->coh_total, p->stream));
    if (p->large) {
        rc = lg_expm_all(p); if (rc) return rc;
        return lg_states_forward(p, p->psi0.p);                    // includes the sum of the chunk costs
    }
    rc = enqueue_expm_forward(p, with_grad != 0); if (rc) return rc;
    rc = enqueue_state_forward(p, p->psi0.p, nullptr); if (rc) return rc;
    return enqueue_finalize(p);
}

int qocb_state_shard_finish(qocb_plan *p, int32_t with_grad, const double *coh_dev) {
    if (!p || (p->coh_total > 0 && !coh_dev)) { set_error(p, "null argument"); return -1; }
    if (!p->state_sharded) { set_error(p, "plan was not created with a state range (state_total / state_first)"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    p->coh_out = nullptr; p->coh_in = p->coh_total > 0 ? coh_dev : nullptr;
    if (p->coh_total > 0 && p->pb.state_first == 0) {
        k_coherent_value<<<1, 32, 0, p->stream>>>(p->terms.p, (int)p->h_terms.size(), coh_dev, p->pb.cost_eval_step, p->pb.system_eval_count,
                                                 p->pb.state_total, 1, p->cost.p);
        CU_TRY(p, cudaGetLastError());
    }
    if (!with_grad) return 0;
    if (p->large) {
        int rc = lg_costates(p, nullptr, nullptr, true, true); if (rc) return rc;
        return lg_backward_all(p);
    }
    int rc = enqueue_costate(p, nullptr, nullptr, true, true); if (rc) return rc;
    return enqueue_expm_backward(p, nullptr);
}

int qocb_shard_result_doubles(qocb_plan *p) {
    return p ? p->pb.control_eval_count * p->pb.control_count + 1 + p->pb.state_count * 2 * p->NP : -1;
}

int qocb_shard_pack_result(qocb_plan *p, int32_t with_grad, double *result_dev) {
    if (!p || !result_dev) { set_error(p, "null argument"); return -1; }
    CU_TRY(p, cudaSetDevice(p->pb.device));
    const int cnt = p->pb.control_eval_count * p->pb.control_count, VS = p->pb.state_count * 2 * p->NP;
    const double *fin = p->owns_final ? p->psi.p + (size_t)(p->Nloc - 1) * VS : nullptr;
    k_pack_result<<<(cnt + 1 + VS + 127) / 128, 128, 0, p->stream>>>(with_grad ? p->grad.p : nullptr, p->cost.p, fin,
                                                                   result_dev, cnt, VS);
    CU_TRY(p, cudaGetLastError());
    return 0;
}

// ---- standalone batched expm --------------------------------------------------------------------------
}  // extern "C"

// n <= 4: register-resident kernels of small.cuh on the caller's layout ([batch][n][n] interleaved complex128, device).
// (The lane-per-row kernel also instantiates for n = 5 .. 8 with 8-lane groups, but there it needs 250+ registers per thread and
// measured 3.8 TFLOP/s at n = 8 against 4.9 for the one-warp DMMA tile path of k_expm<Cfg<8,1,1>>, so 5 <= n <= 8 stays there.)
constexpr int kSmallMaxDim = 4;
static cudaError_t expm_small_launch(int n, long long batch, const double2 *din, double2 *dout, cudaStream_t st) {
    int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    const int threads = 128;
    const int T = n <= 2 ? 1 : 4;
    const long long units = (batch * T + threads - 1) / threads;          // blocks needed for one matrix per thread / group
    const int grid = (int)std::max<long long>(1, std::min<long long>(units, (long long)sms * 32));
    switch (n) {
        case 1: k_expm_thread<1><<<grid, threads, 0, st>>>(din, dout, batch); break;
        case 2: k_expm_thread<2><<<grid, threads, 0, st>>>(din, dout, batch); break;
        case 3: k_expm_rows<3, 4><<<grid, threads, 0, st>>>(din, dout, batch); break;
        case 4: k_expm_rows<4, 4><<<grid, threads, 0, st>>>(din, dout, batch); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

static int expm_small_impl(int n, long long batch, const double *a, double *out) {
    qocb_plan *np = nullptr;
    DevBuf<double2> din, dout;
    const size_t cnt = (size_t)batch * n * n;
    CU_TRY(np, din.alloc(cnt)); CU_TRY(np, dout.alloc(cnt));
    CU_TRY(np, cudaMemcpy(din.p, a, sizeof(double2) * cnt, cudaMemcpyHostToDevice));
    CU_TRY(np, expm_small_launch(n, batch, din.p, dout.p, 0));
    CU_TRY(np, cudaDeviceSynchronize());
    CU_TRY(np, cudaMemcpy(out, dout.p, sizeof(double2) * cnt, cudaMemcpyDeviceToHost));
    return 0;
}

// persistent grid of the standalone expm kernels: every CTA slot the SM can hold (small dimensions are latency-bound: one
// 8 x 8 problem per warp needs many warps in flight)
template <class C>
static int expm_grid(long long batch, int sms, bool vjp) {
    int occ = 0;
    if (vjp) {
        cudaFuncSetAttribute(k_expm_vjp<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes());
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_expm_vjp<C>, C::NT, Smem<C>::bytes());
    } else {
        cudaFuncSetAttribute(k_expm<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes());
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_expm<C>, C::NT, Smem<C>::bytes());
    }
    occ = std::max(1, std::min(occ, 32));
    return (int)std::min<long long>(batch, (long long)sms * occ);
}

template <class C>
static int expm_batched_impl(int n, long long batch, const double *a, const double *ubar, double *out, double *abar) {
    const size_t GM = C::GMAT;
    int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    DevBuf<double> din, dout, dub, dab, scratch, tape; DevBuf<int> piv;
    std::vector<double> h((size_t)batch * GM);
    qocb_plan *np = nullptr;
    CU_TRY(np, din.alloc((size_t)batch * GM)); CU_TRY(np, dout.alloc((size_t)batch * GM));
    for (long long b = 0; b < batch; ++b) to_planar(a + (size_t)b * 2 * n * n, h.data() + (size_t)b * GM, n, C::NP, false);
    CU_TRY(np, cudaMemcpy(din.p, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice));
    const int grid = expm_grid<C>(batch, sms, ubar != nullptr);
    CU_TRY(np, scratch.alloc((size_t)grid * S_COUNT * GM));
    if (ubar) {
        CU_TRY(np, dub.alloc((size_t)batch * GM)); CU_TRY(np, dab.alloc((size_t)batch * GM));
        CU_TRY(np, tape.alloc((size_t)grid * (8 + kCtaTapeR) * GM)); CU_TRY(np, piv.alloc((size_t)grid * C::NP));
        for (long long b = 0; b < batch; ++b) to_planar(ubar + (size_t)b * 2 * n * n, h.data() + (size_t)b * GM, n, C::NP, false);
        CU_TRY(np, cudaMemcpy(dub.p, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice));
        CU_TRY(np, cudaFuncSetAttribute(k_expm_vjp<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
        k_expm_vjp<C><<<grid, C::NT, Smem<C>::bytes()>>>(din.p, dub.p, dout.p, dab.p, scratch.p, tape.p, piv.p, batch);
    } else {
        CU_TRY(np, cudaFuncSetAttribute(k_expm<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
        k_expm<C><<<grid, C::NT, Smem<C>::bytes()>>>(din.p, dout.p, scratch.p, batch);
    }
    CU_TRY(np, cudaGetLastError());
    CU_TRY(np, cudaDeviceSynchronize());
    CU_TRY(np, cudaMemcpy(h.data(), dout.p, sizeof(double) * h.size(), cudaMemcpyDeviceToHost));
    for (long long b = 0; b < batch; ++b) from_planar(h.data() + (size_t)b * GM, out + (size_t)b * 2 * n * n, n, C::NP);
    if (ubar) {
        CU_TRY(np, cudaMemcpy(h.data(), dab.p, sizeof(double) * h.size(), cudaMemcpyDeviceToHost));
        for (long long b = 0; b < batch; ++b) from_planar(h.data() + (size_t)b * GM, abar + (size_t)b * 2 * n * n, n, C::NP);
    }
    return 0;
}

extern "C" {

int qocb_expm_batched(int32_t n, int64_t batch, const double *a, double *out, int32_t device) {
    if (!a || !out || batch < 1) { set_error((qocb_plan *)nullptr, "bad argument"); return -1; }
    const int NP = pad_dim(n);
    if (NP < 0 || NP > 64) { set_error((qocb_plan *)nullptr, "the standalone batched expm hooks cover n in [1, 64]"); return -1; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error((qocb_plan *)nullptr, "cudaSetDevice failed (no CPU path)"); return -2; }
    { const char *ns = getenv("QOCB_NO_SMALL"); if (n <= kSmallMaxDim && !(ns && ns[0] == '1')) return expm_small_impl(n, batch, a, out); }
    return dispatch(NP, [&] { return expm_batched_impl<C8>(n, batch, a, nullptr, out, nullptr); },
                    [&] { return expm_batched_impl<C16>(n, batch, a, nullptr, out, nullptr); },
                    [&] { return expm_batched_impl<C32>(n, batch, a, nullptr, out, nullptr); },
                    [&] { return expm_batched_impl<C64>(n, batch, a, nullptr, out, nullptr); });
}

int qocb_expm_vjp_batched(int32_t n, int64_t batch, const double *a, const double *ubar, double *out, double *abar,
                          int32_t device) {
    if (!a || !out || !ubar || !abar || batch < 1) { set_error((qocb_plan *)nullptr, "bad argument"); return -1; }
    const int NP = pad_dim(n);
    if (NP < 0 || NP > 64) { set_error((qocb_plan *)nullptr, "the standalone batched expm hooks cover n in [1, 64]"); return -1; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error((qocb_plan *)nullptr, "cudaSetDevice failed (no CPU path)"); return -2; }
    return dispatch(NP, [&] { return expm_batched_impl<C8>(n, batch, a, ubar, out, abar); },
                    [&] { return expm_batched_impl<C16>(n, batch, a, ubar, out, abar); },
                    [&] { return expm_batched_impl<C32>(n, batch, a, ubar, out, abar); },
                    [&] { return expm_batched_impl<C64>(n, batch, a, ubar, out, abar); });
}

}  // extern "C"

// device-resident timing of the small-dimension kernels: `distinct` anti-hermitian matrices -i H of one-norm norm_scale tiled
// over the batch in the caller's interleaved layout; a 256 MiB write between launches evicts the L2
static int expm_small_time(int n, long long batch, double norm_scale, int iters, double *ms_best, int warmup = 2, double *ms_total = nullptr) {
    qocb_plan *np = nullptr;
    DevBuf<double2> din, dout; DevBuf<double> flush;
    const size_t nn = (size_t)n * n, cnt = (size_t)batch * nn;
    CU_TRY(np, din.alloc(cnt)); CU_TRY(np, dout.alloc(cnt));
    const size_t flush_bytes = 256ull << 20;
    CU_TRY(np, flush.alloc(flush_bytes / sizeof(double)));
    const int distinct = 4096;
    std::vector<double> h((size_t)distinct * nn * 2, 0.0);
    unsigned long long st = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { st ^= st << 13; st ^= st >> 7; st ^= st << 17; return ((st >> 11) * (1.0 / 9007199254740992.0)) * 2.0 - 1.0; };
    for (int d = 0; d < distinct; ++d) {
        std::vector<double> hr(nn), hi(nn);
        for (int r = 0; r < n; ++r)
            for (int c = r; c < n; ++c) {
                const double x = rnd(), y = (r == c) ? 0.0 : rnd();
                hr[(size_t)r * n + c] = x; hi[(size_t)r * n + c] = y; hr[(size_t)c * n + r] = x; hi[(size_t)c * n + r] = -y;
            }
        double nrm = 0;
        for (int c = 0; c < n; ++c) { double s_ = 0; for (int r = 0; r < n; ++r) s_ += std::hypot(hr[(size_t)r * n + c], hi[(size_t)r * n + c]); nrm = std::max(nrm, s_); }
        const double f = norm_scale / std::max(nrm, 1e-300);
        for (size_t e = 0; e < nn; ++e) { h[2 * (d * nn + e)] = f * hi[e]; h[2 * (d * nn + e) + 1] = -f * hr[e]; }   // -i H
    }
    for (long long b = 0; b < batch; b += distinct) {
        const long long c_ = std::min<long long>(distinct, batch - b);
        CU_TRY(np, cudaMemcpy(din.p + (size_t)b * nn, h.data(), sizeof(double2) * c_ * nn, cudaMemcpyHostToDevice));
    }
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 1e30;
    double total = 0.;
    for (int i = 0; i < iters + warmup; ++i) {
        CU_TRY(np, cudaMemsetAsync(flush.p, i & 0xff, flush_bytes, 0));
        cudaEventRecord(e0);
        CU_TRY(np, expm_small_launch(n, batch, din.p, dout.p, 0));
        cudaEventRecord(e1);
        CU_TRY(np, cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (i >= warmup) { total += ms; if (ms < best) best = ms; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (ms_best) *ms_best = best;
    if (ms_total) *ms_total = total;
    return 0;
}

template <class C>
static int expm_time_impl(int n, long long batch, double norm_scale, int iters, double *ms_best, int warmup = 2, double *ms_total = nullptr) {
    const size_t GM = C::GMAT;
    qocb_plan *np = nullptr;
    int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    DevBuf<double> din, dout, scratch;
    CU_TRY(np, din.alloc((size_t)batch * GM)); CU_TRY(np, dout.alloc((size_t)batch * GM));
    // a few distinct anti-hermitian matrices -i*H scaled to one-norm `norm_scale`, tiled over the batch
    const int distinct = 16;
    std::vector<double> h((size_t)distinct * GM, 0.0);
    unsigned long long st = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { st ^= st << 13; st ^= st >> 7; st ^= st << 17; return ((st >> 11) * (1.0 / 9007199254740992.0)) * 2.0 - 1.0; };
    for (int d = 0; d < distinct; ++d) {
        std::vector<double> hr((size_t)n * n), hi((size_t)n * n);
        for (int r = 0; r < n; ++r)
            for (int c = r; c < n; ++c) {
                const double x = rnd(), y = (r == c) ? 0.0 : rnd();
                hr[(size_t)r * n + c] = x; hi[(size_t)r * n + c] = y; hr[(size_t)c * n + r] = x; hi[(size_t)c * n + r] = -y;
            }
        double nrm = 0;
        for (int c = 0; c < n; ++c) { double s = 0; for (int r = 0; r < n; ++r) s += std::hypot(hr[(size_t)r * n + c], hi[(size_t)r * n + c]); nrm = std::max(nrm, s); }
        const double f = norm_scale / nrm;
        double *dst = h.data() + (size_t)d * GM;
        for (int r = 0; r < n; ++r)
            for (int c = 0; c < n; ++c) {          // -i * H
                dst[(size_t)r * C::NP + c] = f * hi[(size_t)r * n + c];
                dst[(size_t)C::NP * C::NP + (size_t)r * C::NP + c] = -f * hr[(size_t)r * n + c];
            }
    }
    for (long long b = 0; b < batch; b += distinct) {
        const long long cnt = std::min<long long>(distinct, batch - b);
        CU_TRY(np, cudaMemcpy(din.p + (size_t)b * GM, h.data(), sizeof(double) * cnt * GM, cudaMemcpyHostToDevice));
    }
    const int grid = expm_grid<C>(batch, sms, false);
    CU_TRY(np, scratch.alloc((size_t)grid * 3 * GM));
    CU_TRY(np, cudaFuncSetAttribute(k_expm<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<C>::bytes()));
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 1e30;
    double total = 0.;
    for (int i = 0; i < iters + warmup; ++i) {
        cudaEventRecord(e0);
        k_expm<C><<<grid, C::NT, Smem<C>::bytes()>>>(din.p, dout.p, scratch.p, batch);
        cudaEventRecord(e1);
        CU_TRY(np, cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (i >= warmup) { total += ms; if (ms < best) best = ms; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    CU_TRY(np, cudaGetLastError());
    if (ms_best) *ms_best = best;
    if (ms_total) *ms_total = total;
    return 0;
}

extern "C" {

int qocb_expm_batched_bench(int32_t n, int64_t batch, double norm_scale, int32_t warmup, int32_t iters, double *ms_total, double *ms_best,
                            int32_t device) {
    if (batch < 1 || iters < 1 || warmup < 0) return -1;
    const int NP = pad_dim(n);
    if (NP < 0 || NP > 64) { set_error((qocb_plan *)nullptr, "the standalone batched expm hooks cover n in [1, 64]"); return -1; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error((qocb_plan *)nullptr, "cudaSetDevice failed (no CPU path)"); return -2; }
    { const char *ns = getenv("QOCB_NO_SMALL"); if (n <= kSmallMaxDim && !(ns && ns[0] == '1')) return expm_small_time(n, batch, norm_scale, iters, ms_best, warmup, ms_total); }
    return dispatch(NP, [&] { return expm_time_impl<C8>(n, batch, norm_scale, iters, ms_best, warmup, ms_total); },
                    [&] { return expm_time_impl<C16>(n, batch, norm_scale, iters, ms_best, warmup, ms_total); },
                    [&] { return expm_time_impl<C32>(n, batch, norm_scale, iters, ms_best, warmup, ms_total); },
                    [&] { return expm_time_impl<C64>(n, batch, norm_scale, iters, ms_best, warmup, ms_total); });
}

int qocb_expm_batched_time(int32_t n, int64_t batch, double norm_scale, int32_t iters, double *ms_best, int32_t device) {
    if (!ms_best || batch < 1) return -1;
    const int NP = pad_dim(n);
    if (NP < 0 || NP > 64) { set_error((qocb_plan *)nullptr, "the standalone batched expm hooks cover n in [1, 64]"); return -1; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error((qocb_plan *)nullptr, "cudaSetDevice failed (no CPU path)"); return -2; }
    { const char *ns = getenv("QOCB_NO_SMALL"); if (n <= kSmallMaxDim && !(ns && ns[0] == '1')) return expm_small_time(n, batch, norm_scale, iters, ms_best); }
    return dispatch(NP, [&] { return expm_time_impl<C8>(n, batch, norm_scale, iters, ms_best); },
                    [&] { return expm_time_impl<C16>(n, batch, norm_scale, iters, ms_best); },
                    [&] { return expm_time_impl<C32>(n, batch, norm_scale, iters, ms_best); },
                    [&] { return expm_time_impl<C64>(n, batch, norm_scale, iters, ms_best); });
}

}  // extern "C"
