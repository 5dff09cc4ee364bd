// expm_slice.cuh - per-slice forward and reverse passes of the GRAPE hot path, one CTA per time slice.
//
// forward  : interpolated controls -> generator(s) a_i = G0 + sum_r c_r G_r (G = -1j H pieces)
//            -> Magnus M2/M4/M6 (qoc/core/mathmethods.py:72-164)
//            -> Pade-13 scaling and squaring with a pivoted LU solve (qoc/standard/functions/expm.py:210-252)
// backward : reverse mode over exactly that graph in HIPS-autograd's cotangent convention
//            (what ans_jacobian, qoc/standard/utils/autogradutil.py:10-31, produces on the reference tape),
//            then the Magnus adjoint and the contraction with the control operators.
// The NumPy statement of the same algebra is oracle/adjoint_model.py (tests only).
//
// Shared memory: three padded matrix buffers X0, X1, X2.  Named intermediates that the reverse pass needs
// live on a "tape" in global memory (per slice when stored, per CTA when recomputed).
#pragma once
#include "tile.cuh"
#include "lowrank.cuh"
#include "tma.cuh"

namespace qocb {

__device__ __constant__ double kB[14] = {
    64764752532480000., 32382376266240000., 7771770303897600., 1187353796428800.,
    129060195264000., 10559470521600., 670442572800., 33522128640., 1323241920.,
    40840800., 960960., 16380., 182., 1.};
#define QOCB_THETA13 5.371920351148152
#define QOCB_S3 1.7320508075688772
#define QOCB_S15 3.872983346207417

// tape slots (each GMAT doubles)
enum { T_A = 0, T_A2, T_A4, T_A6, T_W1, T_X1, T_Y, T_LU, T_R = 8 };
// The T_LU slot holds the inverse of the Pade denominator (pivot-free slices, tile.cuh: gj_invert_nopiv) or its LUi factors;
// the slice's permutation row says which: kTapeInverse in every entry for Q^-1, the row permutation of the LU otherwise.
constexpr int kTapeInverse = -1;
__device__ __forceinline__ bool tape_holds_inverse(const int *tpiv) { return tpiv[0] == kTapeInverse; }
// CTA scratch slots
enum { S_A = 0, S_A2, S_A4, S_A6, S_B3, S_C12, S_E, S_P, S_QM, S_T0, S_T1, S_T2, S_T3, S_COUNT };

constexpr int kMaxKR = 16;      // real control channels
constexpr int kMaxQ = 3;        // Magnus nodes

template <class C>
struct Smem {
    double *X0, *X1, *X2;
    double *red;                // 64 + kMaxQ*kMaxKR*NWARP doubles of reduction scratch
    double *coef;               // [kMaxQ][kMaxKR]
    int *piv;                   // [NP] row permutation of the LU, then [8] pivots of the current panel
    uint64_t *bar;              // [2] mbarriers of the TMA feed (k_forward): next Magnus matrix, chunk propagator
    __device__ __forceinline__ Smem(unsigned char *base) {
        double *d = reinterpret_cast<double *>(base);   // base is 128-byte aligned; SMAT * 8 is a multiple of 128 (TMA destinations)
        X0 = d; X1 = d + C::SMAT; X2 = d + 2 * C::SMAT;
        red = d + 3 * C::SMAT;
        coef = red + 64 + kMaxQ * kMaxKR * C::NWARP;
        piv = reinterpret_cast<int *>(coef + kMaxQ * kMaxKR);
        bar = reinterpret_cast<uint64_t *>(piv + C::NP + 8);
    }
    static constexpr size_t bytes() {
        return sizeof(double) * (3 * C::SMAT + 64 + kMaxQ * kMaxKR * C::NWARP + kMaxQ * kMaxKR) + sizeof(int) * (C::NP + 8) + 2 * sizeof(uint64_t);
    }
};

struct GenArgs {
    const double *G0;           // this member's drift generator, planar padded
    const double *G;            // [KR][GMAT] control generators (per member: [E][KR][GMAT], this member's after the offset)
    const double *controls;     // [M][KR]
    const int *itab_idx;        // [N-1][q][2]
    const double *itab_w;       // [N-1][q][2]
    int KR, q, order;
    double dt;
    // Magnus M4 without matrix products: [a2, a1] and the adjoint's [a_i, G_r] are linear in the precomputed commutators
    // C0[r] = [G0, G_r] (per member) and Cs[(s<r)] = [G_s, G_r]; enabled for KR <= kMaxCommKR
    const double *C0, *Cs;
    int comm;
    // member strides (doubles) of G and Cs: KR GMAT and npair GMAT when every member has its own control operators
    // (qocb_set_member_operators), 0 when the members share them
    long long g_stride, cs_stride;
    // member strides (doubles) of the controls and of the drift: a control batch (qocb_set_control_batch) gives every
    // member its own [M][KR] controls (ctl_stride = M KR) and shares G0 / C0 (drift_stride = 0); otherwise ctl_stride = 0
    // and drift_stride = GMAT (C0: KR drift_stride)
    long long ctl_stride, drift_stride;
    // time-dependent operators: channel coefficients of every local node, [slice][q][KR], precomputed by k_node_coefs
    // (KR then counts operator channels); nullptr = interpolate the controls here
    const double *nodecoef;
};
constexpr int kMaxCommKR = 6;
__host__ __device__ inline int comm_pair(int s, int r, int KR) { return s * KR - s * (s + 1) / 2 + (r - s - 1); }   // s < r

// interpolated control coefficients of slice j of member `member` at the Magnus nodes -> sm.coef[i*kMaxKR + r]
template <class C>
__device__ __forceinline__ void load_coefs_to(double *dst, const GenArgs &ga, int j, int member) {
    const double *ctl = ga.controls + member * ga.ctl_stride;
    for (int e = threadIdx.x; e < ga.q * ga.KR; e += C::NT) {
        const int i = e / ga.KR, r = e % ga.KR;
        if (ga.nodecoef) { dst[i * kMaxKR + r] = ga.nodecoef[(size_t)(j * ga.q + i) * ga.KR + r]; continue; }
        const int *id = ga.itab_idx + (j * ga.q + i) * 2;
        const double *w = ga.itab_w + (j * ga.q + i) * 2;
        dst[i * kMaxKR + r] = ctl[id[0] * ga.KR + r] * w[0] + ctl[id[1] * ga.KR + r] * w[1];
    }
    __syncthreads();
}
template <class C>
__device__ __forceinline__ void load_coefs(const Smem<C> &sm, const GenArgs &ga, int j, int member) {
    load_coefs_to<C>(sm.coef, ga, j, member);
}

// owned pair of  alpha0 * G0 + sum_r cf[r] * G_r
template <class C>
__device__ __forceinline__ c2 gen_pair(const GenArgs &ga, int row, int col, double alpha0, const double *cf) {
    c2 v = alpha0 * ldg2<C>(ga.G0, row, col);
    for (int r = 0; r < ga.KR; ++r) v = v + cf[r] * ldg2<C>(ga.G + (size_t)r * C::GMAT, row, col);
    return v;
}

// generators of up to two coefficient sets in ONE pass over the operators: v0 = a0 G0 + sum_r cf[r] G_r,
// v1 = a1 G0 + sum_r cf[kMaxKR + r] G_r, for every element pair the thread owns.  The operator loop is outermost so
// that each step has 2 * TM * TN independent 16-byte loads in flight (the operators live in L2).
template <class C, int NODES>
__device__ __forceinline__ void gen_nodes(const GenArgs &ga, const double *cf, double a0, double a1,
                                          c2 (&v0)[C::TM][C::TN], c2 (&v1)[C::TM][C::TN]) {
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 g = ldg2<C>(ga.G0, row, col);
        v0[i][j] = a0 * g;
        if (NODES > 1) v1[i][j] = a1 * g;
    });
    for (int r = 0; r < ga.KR; ++r) {
        const double c0 = cf[r], c1 = NODES > 1 ? cf[kMaxKR + r] : 0.0;
        const double *g = ga.G + (size_t)r * C::GMAT;
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 x = ldg2<C>(g, row, col);
            v0[i][j] = v0[i][j] + c0 * x;
            if (NODES > 1) v1[i][j] = v1[i][j] + c1 * x;
        });
    }
}

// acc = op(A) op(B) - op(B') op(A') style helpers: load two global matrices into X0/X1 and multiply.
template <class C, bool TA, bool TB, bool NEG>
__device__ __forceinline__ void gmm(const Smem<C> &sm, Acc<C> &acc, const double *gA, const double *gB) {
    __syncthreads();
    g2s<C>(sm.X0, gA);
    if (gB != gA) g2s<C>(sm.X1, gB);
    __syncthreads();
    mma_smem<C, TA, TB, NEG>(acc, sm.X0, gB != gA ? sm.X1 : sm.X0);
}

// ---------------------------------------------------------------------------------------------------------
// Magnus forward: leaves M (unscaled) in X2.  M6 uses CTA scratch slots S_B3, S_C12.
template <class C>
__device__ void magnus_forward(const Smem<C> &sm, const GenArgs &ga, double *scratch) {
    const double dt = ga.dt;
    if (ga.order == 2) {
        c2 v[C::TM][C::TN];
        gen_nodes<C, 1>(ga, sm.coef, 1.0, 1.0, v, v);
        for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(sm.X2, row, col, dt * v[i][j]); });
        __syncthreads();
        return;
    }
    if (ga.order == 4 && ga.comm) {
        // M = dt G0 + sum_r dt/2 (c1_r + c2_r) G_r + f [ sum_r (c1_r - c2_r) C0_r + sum_{s<r} (c2_s c1_r - c2_r c1_s) C_sr ]
        const double f = (QOCB_S3 / 12.0) * dt * dt;
        const double *c1 = sm.coef, *cc2 = sm.coef + kMaxKR;
        c2 v[C::TM][C::TN];
        for_owned<C>([&](int i, int j, int row, int col) { v[i][j] = dt * ldg2<C>(ga.G0, row, col); });
        auto axpy = [&](double w, const double *g) {
            for_owned<C>([&](int i, int j, int row, int col) { v[i][j] = v[i][j] + w * ldg2<C>(g, row, col); });
        };
        for (int r = 0; r < ga.KR; ++r) axpy(0.5 * dt * (c1[r] + cc2[r]), ga.G + (size_t)r * C::GMAT);
        for (int r = 0; r < ga.KR; ++r) axpy(f * (c1[r] - cc2[r]), ga.C0 + (size_t)r * C::GMAT);
        for (int s_ = 0; s_ < ga.KR; ++s_)
            for (int r = s_ + 1; r < ga.KR; ++r)
                axpy(f * (cc2[s_] * c1[r] - cc2[r] * c1[s_]), ga.Cs + (size_t)comm_pair(s_, r, ga.KR) * C::GMAT);
        for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(sm.X2, row, col, v[i][j]); });
        __syncthreads();
        return;
    }
    if (ga.order == 4) {
        {
            c2 v0[C::TM][C::TN], v1[C::TM][C::TN];
            gen_nodes<C, 2>(ga, sm.coef, 1.0, 1.0, v0, v1);
            for_owned<C>([&](int i, int j, int row, int col) {
                sts2<C>(sm.X0, row, col, v0[i][j]);
                sts2<C>(sm.X1, row, col, v1[i][j]);
            });
        }
        __syncthreads();
        Acc<C> acc; acc.zero();
        mma_smem<C, false, false, false>(acc, sm.X1, sm.X0);        // a2 a1
        mma_smem<C, false, false, true>(acc, sm.X0, sm.X1);         // - a1 a2
        const double f = (QOCB_S3 / 12.0) * dt * dt;
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 m = (0.5 * dt) * (lds2<C>(sm.X0, row, col) + lds2<C>(sm.X1, row, col)) + f * accv<C>(acc, i, j);
            sts2<C>(sm.X2, row, col, m);
        });
        __syncthreads();
        return;
    }
    // order 6: b1 = dt a2, b2 = (sqrt15/3) dt (a3 - a1), b3 = (10/3) dt (a3 - 2 a2 + a1); the drift cancels in b2, b3
    double *gB3 = scratch + (size_t)S_B3 * C::GMAT, *gC12 = scratch + (size_t)S_C12 * C::GMAT;
    {
        double c2f[kMaxKR], c3f[kMaxKR];
        for (int r = 0; r < ga.KR; ++r) {
            const double c1 = sm.coef[r], cc2 = sm.coef[kMaxKR + r], c3 = sm.coef[2 * kMaxKR + r];
            c2f[r] = (QOCB_S15 / 3.0) * dt * (c3 - c1);
            c3f[r] = (10.0 / 3.0) * dt * (c3 - 2.0 * cc2 + c1);
        }
        for_owned<C>([&](int, int, int row, int col) {
            sts2<C>(sm.X0, row, col, dt * gen_pair<C>(ga, row, col, 1.0, sm.coef + kMaxKR));    // b1
            sts2<C>(sm.X1, row, col, gen_pair<C>(ga, row, col, 0.0, c2f));                      // b2
            stg2<C>(gB3, row, col, gen_pair<C>(ga, row, col, 0.0, c3f));                        // b3
        });
    }
    __syncthreads();
    Acc<C> acc; acc.zero();
    mma_smem<C, false, false, false>(acc, sm.X0, sm.X1);
    mma_smem<C, false, false, true>(acc, sm.X1, sm.X0);             // c12 = [b1, b2]
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 c12 = accv<C>(acc, i, j);
        stg2<C>(gC12, row, col, c12);
        sts2<C>(sm.X2, row, col, 2.0 * ldg2<C>(gB3, row, col) + c12);                           // e
    });
    __syncthreads();
    acc.zero();
    mma_smem<C, false, false, false>(acc, sm.X0, sm.X2);
    mma_smem<C, false, false, true>(acc, sm.X2, sm.X0);             // d = [b1, e]
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 b1 = lds2<C>(sm.X0, row, col), b2 = lds2<C>(sm.X1, row, col);
        const c2 b3 = ldg2<C>(gB3, row, col), c12 = ldg2<C>(gC12, row, col);
        sts2<C>(sm.X1, row, col, b2 - (1.0 / 60.0) * accv<C>(acc, i, j));                       // qm
        sts2<C>(sm.X2, row, col, (-20.0) * b1 - b3 + c12);                                      // p
    });
    __syncthreads();
    acc.zero();
    mma_smem<C, false, false, false>(acc, sm.X2, sm.X1);
    mma_smem<C, false, false, true>(acc, sm.X1, sm.X2);             // [p, qm]
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 m = lds2<C>(sm.X0, row, col) + 0.5 * ldg2<C>(gB3, row, col) + (1.0 / 240.0) * accv<C>(acc, i, j);
        sts2<C>(sm.X2, row, col, m);
    });
    __syncthreads();
}

// Magnus matrices of TWO consecutive slices in one pass over the operators (orders without products: M2 and the
// product-free M4).  The assembly streams 1 + KR (M2) or 1 + 2 KR + KR (KR - 1) / 2 (M4) operator matrices from L2
// (0.94 MB per n = 64 slice at KR = 4); sharing the operator loads between two slices and parking the second matrix in
// global memory (one 32 n^2-byte store and load) nearly halves that traffic: measured -1.7 us per slice.  (The same
// pairing of the adjoint's inner products was measured to LOSE 8 % of k_backward and is not used.)
// cfa / cfb: node coefficients of the two slices ([q][kMaxKR]).  Out: M_a in X2, M_b in gMb (global).
template <class C>
__device__ __forceinline__ bool magnus_pair_ok(const GenArgs &ga) { return ga.order == 2 || (ga.order == 4 && ga.comm); }

template <class C>
__device__ void magnus_forward_pair(const Smem<C> &sm, const GenArgs &ga, const double *cfa, const double *cfb, double *gMb) {
    const double dt = ga.dt;
    c2 va[C::TM][C::TN], vb[C::TM][C::TN];
    for_owned<C>([&](int i, int j, int row, int col) { va[i][j] = dt * ldg2<C>(ga.G0, row, col); vb[i][j] = va[i][j]; });
    auto axpy = [&](double wa, double wb, const double *g) {
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 x = ldg2<C>(g, row, col);
            va[i][j] = va[i][j] + wa * x;
            vb[i][j] = vb[i][j] + wb * x;
        });
    };
    if (ga.order == 2) {
        for (int r = 0; r < ga.KR; ++r) axpy(dt * cfa[r], dt * cfb[r], ga.G + (size_t)r * C::GMAT);
    } else {
        const double f = (QOCB_S3 / 12.0) * dt * dt;
        const double *a1 = cfa, *a2 = cfa + kMaxKR, *b1 = cfb, *b2 = cfb + kMaxKR;
        for (int r = 0; r < ga.KR; ++r) axpy(0.5 * dt * (a1[r] + a2[r]), 0.5 * dt * (b1[r] + b2[r]), ga.G + (size_t)r * C::GMAT);
        for (int r = 0; r < ga.KR; ++r) axpy(f * (a1[r] - a2[r]), f * (b1[r] - b2[r]), ga.C0 + (size_t)r * C::GMAT);
        for (int s_ = 0; s_ < ga.KR; ++s_)
            for (int r = s_ + 1; r < ga.KR; ++r)
                axpy(f * (a2[s_] * a1[r] - a2[r] * a1[s_]), f * (b2[s_] * b1[r] - b2[r] * b1[s_]),
                     ga.Cs + (size_t)comm_pair(s_, r, ga.KR) * C::GMAT);
    }
    for_owned<C>([&](int i, int j, int row, int col) {
        sts2<C>(sm.X2, row, col, va[i][j]);
        stg2<C>(gMb, row, col, vb[i][j]);
    });
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------
// Pade-13 forward.  In: M in X2.  Out: U = expm(M) in X1 (all threads past a barrier); returns s.
// tape: 8 + s matrices are written when tape != nullptr (T_R + i holds R_i for i < s); piv_out: int[NP].
// Asynchronous feed of k_forward (tma.cuh).  While the end of this slice runs, pade_forward starts
//   * the chunk propagator (matrix idxP of mapP) into X1 as soon as R0 = Q^-1 P no longer reads P (after the product with
//     Q^-1, or after the solve's permuted copy of its right-hand side) - only when the slice needs no squarings, because
//     then U stays in X0 and X1 is free until the chunk product;
//   * the next slice's Magnus matrix (matrix idxM of mapM) into X2 once Q^-1 or the LU factors have gone to the tape.
// Negative indices skip a fetch.  fetchedP reports whether the propagator fetch was issued.
struct Feed {
    const CUtensorMap *mapM, *mapP;
    long long idxM, idxP;
    uint64_t *barM, *barP;
    bool fetchedP;
};

// u_out != nullptr: the caller accepts U in X0 when no squarings are needed (*u_out = X0 or X1); otherwise U is in X1.
// herm != 0: the argument is anti-Hermitian (Hermitian operators): slices with ||A||_1 < QOCB_NOPIV_NORM and no squarings
// invert the Pade denominator without pivoting (tile.cuh: gj_invert_nopiv) and form R0 = Q^-1 P as one product.
#define QOCB_NOPIV_NORM 2.5
template <class C>
__device__ int pade_forward(const Smem<C> &sm, double *tape, int *piv_out, double *tmpY, double *tmpV, int s_cap,
                            Feed *feed = nullptr, const double **u_out = nullptr, int herm = 0, int tape_min = 0) {
    PROF_DECL
    // one-norm: max column sum of |m_ij|   (expm.py:103-116)
    {
        // column c is summed by PARTS threads (rows split mod PARTS), combined in a fixed order, then one max
        constexpr int P = C::PARTS;
        const int c = threadIdx.x % C::NP, part = threadIdx.x / C::NP;
        double s = 0.;
        for (int r = part; r < C::NP; r += P) {
            const double xr = sm.X2[r * C::LD + c], xi = sm.X2[C::PLANE + r * C::LD + c];
            s += sqrt(xr * xr + xi * xi);
        }
        double *cs = sm.red + 64;                                   // [P][NP] <= NT doubles (fits: kMaxQ*kMaxKR*NWARP >= NT/ ...)
        cs[part * C::NP + c] = s;
        __syncthreads();
        if (threadIdx.x < C::NP) {
            double t = 0.;
            for (int q = 0; q < P; ++q) t += cs[q * C::NP + threadIdx.x];
            sm.red[threadIdx.x] = t;
        }
        __syncthreads();
    }
    double norm = 0.;
    {
        const int lane = threadIdx.x & 31;
        for (int c = lane; c < C::NP; c += 32) norm = fmax(norm, sm.red[c]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) norm = fmax(norm, __shfl_xor_sync(0xffffffffu, norm, o));
    }
    int s = 0;
    if (!(norm < QOCB_THETA13)) {                                   // expm.py:238-241
        s = (int)ceil(log2(norm / QOCB_THETA13));
        if (s < 0) s = 0;
    }
    const double scale = ldexp(1.0, -s);
    PROF_MARK(2);
    const bool keep = tape != nullptr;
    // tape_min: slices without squarings are differentiated by the Krylov reverse pass, which reads A, A2 and the LU factors only
    const bool full = keep && !(tape_min && s == 0);
    double *tA = keep ? tape + (size_t)T_A * C::GMAT : tmpV;        // A is always needed once more (for Uo)
    // A = M * 2^-s   -> X2 and tape
    for_owned<C>([&](int, int, int row, int col) {
        const c2 a = scale * lds2<C>(sm.X2, row, col);
        sts2<C>(sm.X2, row, col, a);
        stg2<C>(tA, row, col, a);
    });
    __syncthreads();
    PROF_MARK(32);
    Acc<C> acc;
    double *gYV = keep ? tape + (size_t)T_LU * C::GMAT : tmpV + C::GMAT;
    bool half = false;
    if constexpr (C::NP == 64 && C::NWARP == 8) half = herm != 0;
    if constexpr (C::NP == 64 && C::NWARP == 8) if (half) {
        // anti-Hermitian A: every product below is Hermitian (the last one anti-Hermitian) - upper tiles only (tile.cuh)
        HAcc h;
        h.zero(); mma_herm<C>(h, sm.X2, sm.X2);                          // A2
        PROF_MARK(33);
        herm_store<C, false>(sm.X0, h);
        __syncthreads();
        if (keep) for_owned<C>([&](int, int, int row, int col) {
            stg2<C>(tape + (size_t)T_A2 * C::GMAT, row, col, lds2<C>(sm.X0, row, col));
        });
        PROF_MARK(34);
        h.zero(); mma_herm<C>(h, sm.X0, sm.X0);                          // A4
        PROF_MARK(35);
        herm_store<C, false>(sm.X1, h);
        __syncthreads();
        if (full) for_owned<C>([&](int, int, int row, int col) {
            stg2<C>(tape + (size_t)T_A4 * C::GMAT, row, col, lds2<C>(sm.X1, row, col));
        });
        PROF_MARK(36);
        h.zero(); mma_herm<C>(h, sm.X0, sm.X1);                          // A6
        PROF_MARK(37);
        __syncthreads();                                                 // X0, X1 (operands) are overwritten below
        // the owner of an upper tile evaluates the four polynomials on it and writes the tile and its mirror image; the
        // constant-term polynomials yu, yv stay in registers until the products they are added to are formed
        c2 yu[5], yv[5];
        for_herm_tiles([&](int q, int row, int col, bool diag) {
            const c2 a6 = herm_val(h, q);
            const c2 a2 = lds2<C>(sm.X0, row, col), a4 = lds2<C>(sm.X1, row, col);
            const c2 w1 = kB[13] * a6 + kB[11] * a4 + kB[9] * a2;
            const c2 x1 = kB[12] * a6 + kB[10] * a4 + kB[8] * a2;
            yu[q] = add_diag(kB[7] * a6 + kB[5] * a4 + kB[3] * a2, row, col, kB[1]);
            yv[q] = add_diag(kB[6] * a6 + kB[4] * a4 + kB[2] * a2, row, col, kB[0]);
            sts2<C>(sm.X2, row, col, a6);                                // over A (on the tape; not an operand of A6)
            sts2<C>(sm.X0, row, col, w1);
            sts2<C>(sm.X1, row, col, x1);
            if (!diag) {
                sts2_mirror<C, false>(sm.X2, row, col, a6);
                sts2_mirror<C, false>(sm.X0, row, col, w1);
                sts2_mirror<C, false>(sm.X1, row, col, x1);
            }
        });
        __syncthreads();
        if (full) for_owned<C>([&](int, int, int row, int col) {
            stg2<C>(tape + (size_t)T_A6 * C::GMAT, row, col, lds2<C>(sm.X2, row, col));
            stg2<C>(tape + (size_t)T_W1 * C::GMAT, row, col, lds2<C>(sm.X0, row, col));
            stg2<C>(tape + (size_t)T_X1 * C::GMAT, row, col, lds2<C>(sm.X1, row, col));
        });
        PROF_MARK(38);
        h.zero(); mma_herm<C>(h, sm.X2, sm.X0);                          // A6 W1
        for_herm_tiles([&](int q, int, int, bool) { yu[q] = yu[q] + herm_val(h, q); });       // Y
        h.zero(); mma_herm<C>(h, sm.X2, sm.X1);                          // A6 X1
        for_herm_tiles([&](int q, int, int, bool) { yv[q] = yv[q] + herm_val(h, q); });       // Ve
        PROF_MARK(39);
        __syncthreads();                                                 // operands are overwritten below
        g2s_async<C>(sm.X2, tA);                                         // A back into X2 (A6 is dead), under the stores
        for_herm_tiles([&](int q, int row, int col, bool diag) {
            sts2<C>(sm.X0, row, col, yu[q]);                             // Y over W1
            sts2<C>(sm.X1, row, col, yv[q]);                             // Ve over X1
            if (!diag) { sts2_mirror<C, false>(sm.X0, row, col, yu[q]); sts2_mirror<C, false>(sm.X1, row, col, yv[q]); }
        });
        g2s_async_wait();
        __syncthreads();
        if (full) for_owned<C>([&](int, int, int row, int col) {
            stg2<C>(tape + (size_t)T_Y * C::GMAT, row, col, lds2<C>(sm.X0, row, col));
        });
        PROF_MARK(40);
        h.zero(); mma_herm<C>(h, sm.X2, sm.X0);                          // Uo = A Y, anti-Hermitian
        PROF_MARK(41);
        __syncthreads();                                                 // X2 (operand) is overwritten below
        for_herm_tiles([&](int q, int row, int col, bool diag) {
            const c2 ve = lds2<C>(sm.X1, row, col), uo = herm_val(h, q);
            const c2 pp = ve + uo, qq = ve - uo;                         // P = Ve + Uo, Q = Ve - Uo = P^H
            sts2<C>(sm.X1, row, col, pp);
            sts2<C>(sm.X2, row, col, qq);
            if (!diag) { sts2_mirror<C, false>(sm.X1, row, col, qq); sts2_mirror<C, false>(sm.X2, row, col, pp); }
        });
        __syncthreads();
    }
    if (!half) {
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X2, sm.X2);     // A2
        PROF_MARK(33);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 v = accv<C>(acc, i, j);
            sts2<C>(sm.X0, row, col, v);
            if (keep) stg2<C>(tape + (size_t)T_A2 * C::GMAT, row, col, v);
        });
        __syncthreads();
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X0, sm.X0);     // A4
        PROF_MARK(35);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 v = accv<C>(acc, i, j);
            sts2<C>(sm.X1, row, col, v);
            if (full) stg2<C>(tape + (size_t)T_A4 * C::GMAT, row, col, v);
        });
        __syncthreads();
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X0, sm.X1);     // A6 -> X2 (A is on the tape)
        PROF_MARK(37);
        __syncthreads();                                                    // X0, X1 (operands) are overwritten below
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 a6 = accv<C>(acc, i, j);
            const c2 a2 = lds2<C>(sm.X0, row, col), a4 = lds2<C>(sm.X1, row, col);
            const c2 w1 = kB[13] * a6 + kB[11] * a4 + kB[9] * a2;
            const c2 x1 = kB[12] * a6 + kB[10] * a4 + kB[8] * a2;
            const c2 yu = add_diag(kB[7] * a6 + kB[5] * a4 + kB[3] * a2, row, col, kB[1]);
            const c2 yv = add_diag(kB[6] * a6 + kB[4] * a4 + kB[2] * a2, row, col, kB[0]);
            sts2<C>(sm.X2, row, col, a6);
            sts2<C>(sm.X0, row, col, w1);          // over A2 (own elements only)
            sts2<C>(sm.X1, row, col, x1);          // over A4
            stg2<C>(tmpY, row, col, yu);
            stg2<C>(gYV, row, col, yv);          // parked until Ve is formed
            if (full) {
                stg2<C>(tape + (size_t)T_A6 * C::GMAT, row, col, a6);
                stg2<C>(tape + (size_t)T_W1 * C::GMAT, row, col, w1);
                stg2<C>(tape + (size_t)T_X1 * C::GMAT, row, col, x1);
            }
        });
        __syncthreads();
        PROF_MARK(38);
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X2, sm.X0);     // A6 W1
        PROF_MARK(39);
        __syncthreads();
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 y = accv<C>(acc, i, j) + ldg2<C>(tmpY, row, col);
            sts2<C>(sm.X0, row, col, y);                                    // Y over W1
            if (full) stg2<C>(tape + (size_t)T_Y * C::GMAT, row, col, y);
        });
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X2, sm.X1);     // A6 X1   (X0 not an operand)
        PROF_MARK(42);
        __syncthreads();
        for_owned<C>([&](int i, int j, int row, int col) {
            sts2<C>(sm.X1, row, col, accv<C>(acc, i, j) + ldg2<C>(gYV, row, col));   // Ve over X1
        });
        g2s<C>(sm.X2, tA);                                                  // A back into X2 (A6 is dead)
        __syncthreads();
        PROF_MARK(40);
        acc.zero(); mma_smem<C, false, false, false>(acc, sm.X2, sm.X0);     // Uo = A Y
        PROF_MARK(41);
        __syncthreads();
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 ve = lds2<C>(sm.X1, row, col), uo = accv<C>(acc, i, j);
            sts2<C>(sm.X1, row, col, ve + uo);                              // P
            sts2<C>(sm.X2, row, col, ve - uo);                              // Q
        });
        __syncthreads();
    }
    PROF_MARK(3);
    const bool inverse = herm && s == 0 && norm < QOCB_NOPIV_NORM;
    {
        const bool feedP = feed != nullptr && feed->idxP >= 0 && s == 0;
        if (feed) feed->fetchedP = feedP;
        auto b_free = [&]() {
            if (feedP && threadIdx.x == 0) tma_fetch_matrix<C::NP>(sm.X1, feed->mapP, feed->idxP, feed->barP);
        };
        if (inverse) {
            gj_invert_nopiv<C>(sm.X2, sm.X0);                           // Q^-1 in X2 (X0: scratch, Y is dead)
            PROF_MARK(19);
            acc.zero(); mma_smem<C, false, false, false>(acc, sm.X2, sm.X1);   // R0 = Q^-1 P
            for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(sm.X0, row, col, accv<C>(acc, i, j)); });
            __syncthreads();
            b_free();
            PROF_MARK(25);
        } else {
            lu_factor_blocked<C>(sm.X2, sm.piv, sm.piv + C::NP);
            PROF_MARK(4);
            lu_solve_blocked<C, false>(sm.X2, sm.piv, sm.X1, sm.X0, b_free);   // R0 = Q^-1 P in X0 (Y is dead)
            PROF_MARK(5);
        }
    }
    if (keep) {
        s2g<C>(tape + (size_t)T_LU * C::GMAT, sm.X2);                   // Q^-1, or the LUi factors (tile.cuh) + row permutation
        for (int c = threadIdx.x; c < C::NP; c += C::NT) piv_out[c] = inverse ? kTapeInverse : sm.piv[c];
    }
    if (feed != nullptr && feed->idxM >= 0) {                           // X2 is dead from here on
        __syncthreads();
        if (threadIdx.x == 0) tma_fetch_matrix<C::NP>(sm.X2, feed->mapM, feed->idxM, feed->barM);
    }
    const double *cur = sm.X0;
    for (int i = 0; i < s; ++i) {                                        // expm.py:249-250
        if (keep && i < s_cap) s2g<C>(tape + (size_t)(T_R + i) * C::GMAT, cur);
        acc.zero(); mma_smem<C, false, false, false>(acc, cur, cur);
        __syncthreads();
        for_owned<C>([&](int ii, int jj, int row, int col) { sts2<C>(sm.X1, row, col, accv<C>(acc, ii, jj)); });
        __syncthreads();
        cur = sm.X1;
    }
    if (u_out) *u_out = s == 0 ? sm.X0 : sm.X1;
    if (s == 0 && !u_out) {
        for_owned<C>([&](int, int, int row, int col) { sts2<C>(sm.X1, row, col, lds2<C>(sm.X0, row, col)); });
        __syncthreads();
    }
    PROF_MARK(6);
    return s;
}

// ---------------------------------------------------------------------------------------------------------
// Reverse pass of the Pade graph.  In: ubar (cotangent of U, unconjugated convention) in X0; tape of the
// slice; gU = U_j (== R_s).  Out: mbar (cotangent of the unscaled Magnus matrix) in X0, past a barrier.
template <class C>
__device__ void pade_backward(const Smem<C> &sm, const double *tape, const int *tpiv, int s,
                              const double *gU, double *scratch) {
    PROF_DECL
    Acc<C> acc;
    double *sA = scratch + (size_t)S_A * C::GMAT, *sA2 = scratch + (size_t)S_A2 * C::GMAT;
    double *sA4 = scratch + (size_t)S_A4 * C::GMAT, *sA6 = scratch + (size_t)S_A6 * C::GMAT;
    // squarings: R_i = R_{i-1}^2  =>  rbar_{i-1} = rbar_i R_{i-1}^T + R_{i-1}^T rbar_i
    for (int i = s; i >= 1; --i) {
        g2s<C>(sm.X1, tape + (size_t)(T_R + i - 1) * C::GMAT);
        __syncthreads();
        acc.zero();
        mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);
        mma_smem<C, true, false, false>(acc, sm.X1, sm.X0);
        __syncthreads();
        for_owned<C>([&](int ii, int jj, int row, int col) { sts2<C>(sm.X0, row, col, accv<C>(acc, ii, jj)); });
        __syncthreads();
    }
    // R0 = Q^-1 P:  pbar = Q^-T rbar ; qbar = -pbar R0^T
    g2s<C>(sm.X2, tape + (size_t)T_LU * C::GMAT);
    for (int c = threadIdx.x; c < C::NP; c += C::NT) sm.piv[c] = tpiv[c];
    g2s<C>(sm.X1, s > 0 ? tape + (size_t)T_R * C::GMAT : gU);
    __syncthreads();
    PROF_MARK(10);
    if (tape_holds_inverse(tpiv)) {
        acc.zero(); mma_smem<C, true, false, false>(acc, sm.X2, sm.X0);  // pbar = (Q^-1)^T rbar
        __syncthreads();
        for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(sm.X2, row, col, accv<C>(acc, i, j)); });
        __syncthreads();
    } else {
        lu_solve_blocked<C, true>(sm.X2, sm.piv, sm.X0, sm.X2);         // X2 = pbar = Q^-T rbar (over the dead LU)
    }
    PROF_MARK(11);
    acc.zero(); mma_smem<C, false, true, false>(acc, sm.X2, sm.X1);      // pbar R0^T = -qbar
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 pb = lds2<C>(sm.X2, row, col), t = accv<C>(acc, i, j);
        sts2<C>(sm.X0, row, col, pb + t);                               // uobar = pbar - qbar
        sts2<C>(sm.X2, row, col, pb - t);                               // vebar = pbar + qbar
    });
    g2s<C>(sm.X1, tape + (size_t)T_Y * C::GMAT);
    __syncthreads();
    acc.zero(); mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);      // abar  = uobar Y^T
    for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(sA, row, col, accv<C>(acc, i, j)); });
    __syncthreads();
    g2s<C>(sm.X1, tape + (size_t)T_A * C::GMAT);
    __syncthreads();
    acc.zero(); mma_smem<C, true, false, false>(acc, sm.X1, sm.X0);      // ybar = A^T uobar
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 yb = accv<C>(acc, i, j), vb = lds2<C>(sm.X2, row, col);
        sts2<C>(sm.X0, row, col, yb);                                   // X0 = ybar, X2 = vebar
        stg2<C>(sA6, row, col, kB[7] * yb + kB[6] * vb);
        stg2<C>(sA4, row, col, kB[5] * yb + kB[4] * vb);
        stg2<C>(sA2, row, col, kB[3] * yb + kB[2] * vb);
    });
    g2s<C>(sm.X1, tape + (size_t)T_W1 * C::GMAT);
    __syncthreads();
    acc.zero(); mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);      // ybar W1^T
    __syncthreads();
    g2s<C>(sm.X1, tape + (size_t)T_X1 * C::GMAT);
    __syncthreads();
    mma_smem<C, false, true, false>(acc, sm.X2, sm.X1);                 // + vebar X1^T
    for_owned<C>([&](int i, int j, int row, int col) {
        stg2<C>(sA6, row, col, ldg2<C>(sA6, row, col) + accv<C>(acc, i, j));
    });
    __syncthreads();
    g2s<C>(sm.X1, tape + (size_t)T_A6 * C::GMAT);
    __syncthreads();
    acc.zero(); mma_smem<C, true, false, false>(acc, sm.X1, sm.X0);      // w1bar = A6^T ybar
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 w = accv<C>(acc, i, j);
        stg2<C>(sA6, row, col, ldg2<C>(sA6, row, col) + kB[13] * w);
        stg2<C>(sA4, row, col, ldg2<C>(sA4, row, col) + kB[11] * w);
        stg2<C>(sA2, row, col, ldg2<C>(sA2, row, col) + kB[9] * w);
    });
    acc.zero(); mma_smem<C, true, false, false>(acc, sm.X1, sm.X2);      // x1bar = A6^T vebar
    for_owned<C>([&](int i, int j, int row, int col) {
        const c2 w = accv<C>(acc, i, j);
        stg2<C>(sA6, row, col, ldg2<C>(sA6, row, col) + kB[12] * w);
        stg2<C>(sA4, row, col, ldg2<C>(sA4, row, col) + kB[10] * w);
        stg2<C>(sA2, row, col, ldg2<C>(sA2, row, col) + kB[8] * w);
    });
    __syncthreads();
    // A6 = A2 A4
    g2s<C>(sm.X0, sA6);
    g2s<C>(sm.X1, tape + (size_t)T_A4 * C::GMAT);
    g2s<C>(sm.X2, tape + (size_t)T_A2 * C::GMAT);
    __syncthreads();
    acc.zero(); mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);      // a6bar A4^T
    for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(sA2, row, col, ldg2<C>(sA2, row, col) + accv<C>(acc, i, j)); });
    acc.zero(); mma_smem<C, true, false, false>(acc, sm.X2, sm.X0);      // A2^T a6bar
    for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(sA4, row, col, ldg2<C>(sA4, row, col) + accv<C>(acc, i, j)); });
    __syncthreads();
    // A4 = A2 A2
    g2s<C>(sm.X0, sA4);
    __syncthreads();
    acc.zero();
    mma_smem<C, false, true, false>(acc, sm.X0, sm.X2);
    mma_smem<C, true, false, false>(acc, sm.X2, sm.X0);
    for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(sA2, row, col, ldg2<C>(sA2, row, col) + accv<C>(acc, i, j)); });
    __syncthreads();
    // A2 = A A ; mbar = abar * 2^-s
    g2s<C>(sm.X0, sA2);
    g2s<C>(sm.X1, tape + (size_t)T_A * C::GMAT);
    __syncthreads();
    acc.zero();
    mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);
    mma_smem<C, true, false, false>(acc, sm.X1, sm.X0);
    __syncthreads();
    const double scale = ldexp(1.0, -s);
    for_owned<C>([&](int i, int j, int row, int col) {
        sts2<C>(sm.X0, row, col, scale * (ldg2<C>(sA, row, col) + accv<C>(acc, i, j)));   // X0 = mbar
    });
    __syncthreads();
    PROF_MARK(12);
}

// Reverse pass of the Pade graph for a rank-S cotangent ubar = sum_s lam1_s psi_s^T without squarings (lowrank.cuh).
// In: tape of the slice, psi = psi_j, psi1 = psi_{j+1}, lam1 = lam_{j+1} (planar [s][2][NP]).  Out: mbar in X0.
template <class C>
__device__ void pade_backward_lowrank(const Smem<C> &sm, const double *tape, const int *tperm, const double *psi,
                                      const double *psi1, const double *lam1, int S) {
    static_assert(C::NP == 64 && C::NWARP == 8, "low-rank reverse pass is laid out for NP = 64 with 8 warps");
    PROF_DECL
    constexpr int NP = C::NP, LD = LR_LD, PL = LR_PL, TLD = LR_TLD, TPL = LR_TPL;
    double *X0 = sm.X0, *LEFT = sm.X1, *TMP = sm.X1 + 2 * LR_PL, *RIGHT = sm.X2, *EL = sm.X2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, t = lane & 3;
    const int frow = warp * 8 + (lane >> 2);                       // row of this lane's C-fragment elements
    // register-staged prefetch of the next tape matrix: the loads fly while the current stage computes on X0
    double2 pre[C::GMAT / 2 / C::NT];
    auto pf_load = [&](const double *gm) {
#pragma unroll
        for (int i = 0; i < C::GMAT / 2 / C::NT; ++i) pre[i] = reinterpret_cast<const double2 *>(gm)[threadIdx.x + i * C::NT];
    };
    auto pf_store = [&](double *sdst) {
#pragma unroll
        for (int i = 0; i < C::GMAT / 2 / C::NT; ++i) {
            const int idx = threadIdx.x + i * C::NT;
            const int plane = idx / (C::GPLANE / 2), rem = idx - plane * (C::GPLANE / 2);
            const int row = rem / (NP / 2), cc = rem - row * (NP / 2);
            *reinterpret_cast<double2 *>(sdst + plane * C::PLANE + row * C::LD + cc * 2) = pre[i];
        }
    };
    // ---- stage 0: [0 | lam] -> LEFT[:, 0:8], [p | m] -> TMP[:, 0:8]; LUi -> X0
    for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
        const int row = e >> 2, c = e & 3;
        const bool on = c < S;
        const double lr = on ? lam1[c * 2 * NP + row] : 0., li = on ? lam1[c * 2 * NP + NP + row] : 0.;
        const double pr = on ? psi[c * 2 * NP + row] : 0., pi = on ? psi[c * 2 * NP + NP + row] : 0.;
        const double qr = on ? psi1[c * 2 * NP + row] : 0., qi = on ? psi1[c * 2 * NP + NP + row] : 0.;
        LEFT[row * LD + c] = 0.; LEFT[PL + row * LD + c] = 0.;
        LEFT[row * LD + 4 + c] = lr; LEFT[PL + row * LD + 4 + c] = li;
        TMP[row * TLD + c] = pr + qr; TMP[TPL + row * TLD + c] = pi + qi;
        TMP[row * TLD + 4 + c] = pr - qr; TMP[TPL + row * TLD + 4 + c] = pi - qi;
    }
    g2s<C>(X0, tape + (size_t)T_LU * C::GMAT);
    for (int c = threadIdx.x; c < NP; c += C::NT) sm.piv[c] = tperm[c];
    pf_load(tape + (size_t)T_Y * C::GMAT);
    __syncthreads();
    // ---- stage 1: l = Q^-T lam -> LEFT[:, 4:8]: one thin product with Q^-1, or the thin solve and the row un-permutation
    if (tape_holds_inverse(tperm)) {
        const c2 v = thin_tile<C, true, LD, PL>(X0, LEFT, warp, 0);
        __syncthreads();
        if (t >= 2) {
            *reinterpret_cast<double2 *>(LEFT + frow * LD + 2 * t) = make_double2(v.r0, v.r1);
            *reinterpret_cast<double2 *>(LEFT + PL + frow * LD + 2 * t) = make_double2(v.i0, v.i1);
        }
        pf_store(X0);                                               // Y
        pf_load(tape + (size_t)T_A * C::GMAT);
        __syncthreads();
    } else {
        lu_solve_thin_T<C>(X0, LEFT);
        for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
            const int row = e >> 2, c = e & 3, pr = sm.piv[row];
            RIGHT[pr * LD + c] = LEFT[row * LD + 4 + c]; RIGHT[PL + pr * LD + c] = LEFT[PL + row * LD + 4 + c];
        }
        pf_store(X0);                                               // Y
        pf_load(tape + (size_t)T_A * C::GMAT);
        __syncthreads();
        for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
            const int row = e >> 2, c = e & 3;
            LEFT[row * LD + 4 + c] = RIGHT[row * LD + c]; LEFT[PL + row * LD + 4 + c] = RIGHT[PL + row * LD + c];
        }
    }
    // ---- stage 2: yp = Y p -> TMP[:, 8:12]
    {
        const c2 v = thin_tile<C, false, TLD, TPL>(X0, TMP, warp, 0);
        if (t < 2) {
            *reinterpret_cast<double2 *>(TMP + frow * TLD + 8 + 2 * t) = make_double2(v.r0, v.r1);
            *reinterpret_cast<double2 *>(TMP + TPL + frow * TLD + 8 + 2 * t) = make_double2(v.i0, v.i1);
        }
    }
    __syncthreads();
    pf_store(X0);                                                   // A
    pf_load(tape + (size_t)T_W1 * C::GMAT);
    __syncthreads();
    // ---- stage 3: a = A^T l -> LEFT[:, 0:4]
    {
        const c2 v = thin_tile<C, true, LD, PL>(X0, LEFT, warp, 0);
        __syncthreads();
        if (t >= 2) {
            *reinterpret_cast<double2 *>(LEFT + frow * LD + 2 * (t - 2)) = make_double2(v.r0, v.r1);
            *reinterpret_cast<double2 *>(LEFT + PL + frow * LD + 2 * (t - 2)) = make_double2(v.i0, v.i1);
        }
    }
    pf_store(X0);                                                   // W1
    pf_load(tape + (size_t)T_X1 * C::GMAT);
    // R4, R2 and the polynomial blocks of R6 (elementwise from p, m)
    for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
        const int row = e >> 2, c = e & 3;
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
            const double pv = TMP[pl * TPL + row * TLD + c], mv = TMP[pl * TPL + row * TLD + 4 + c];
            double *R = RIGHT + pl * PL + row * LD;
            R[0 + c] = kB[3] * pv; R[4 + c] = kB[2] * mv; R[8 + c] = kB[9] * pv; R[12 + c] = kB[8] * mv;      // R2 -> X_a
            R[16 + c] = kB[5] * pv; R[20 + c] = kB[4] * mv; R[24 + c] = kB[11] * pv; R[28 + c] = kB[10] * mv;  // R4 -> X_b
            R[40 + c] = kB[13] * pv; R[44 + c] = kB[12] * mv;                                                  // R6 blocks 2, 3
        }
    }
    __syncthreads();
    // ---- stage 4: c1 = b7 p + W1 p -> RIGHT[:, 32:36]
    {
        const c2 v = thin_tile<C, false, TLD, TPL>(X0, TMP, warp, 0);
        if (t < 2) {
            const double2 pr = *reinterpret_cast<const double2 *>(TMP + frow * TLD + 2 * t);
            const double2 pi = *reinterpret_cast<const double2 *>(TMP + TPL + frow * TLD + 2 * t);
            *reinterpret_cast<double2 *>(RIGHT + frow * LD + 32 + 2 * t) = make_double2(v.r0 + kB[7] * pr.x, v.r1 + kB[7] * pr.y);
            *reinterpret_cast<double2 *>(RIGHT + PL + frow * LD + 32 + 2 * t) = make_double2(v.i0 + kB[7] * pi.x, v.i1 + kB[7] * pi.y);
        }
    }
    __syncthreads();
    pf_store(X0);                                                   // X1
    pf_load(tape + (size_t)T_A6 * C::GMAT);
    __syncthreads();
    // ---- stage 5: c2 = b6 m + X1 m -> RIGHT[:, 36:40]
    {
        const c2 v = thin_tile<C, false, TLD, TPL>(X0, TMP, warp, 0);
        if (t >= 2) {
            const double2 mr = *reinterpret_cast<const double2 *>(TMP + frow * TLD + 2 * t);
            const double2 mi = *reinterpret_cast<const double2 *>(TMP + TPL + frow * TLD + 2 * t);
            *reinterpret_cast<double2 *>(RIGHT + frow * LD + 32 + 2 * t) = make_double2(v.r0 + kB[6] * mr.x, v.r1 + kB[6] * mr.y);
            *reinterpret_cast<double2 *>(RIGHT + PL + frow * LD + 32 + 2 * t) = make_double2(v.i0 + kB[6] * mi.x, v.i1 + kB[6] * mi.y);
        }
    }
    __syncthreads();
    pf_store(X0);                                                   // A6
    pf_load(tape + (size_t)T_A4 * C::GMAT);
    __syncthreads();
    // ---- stage 6: [A6^T a | A6^T l] -> LEFT[:, 8:16]
    st_thin<LD, PL>(LEFT, warp * 8, 8, thin_tile<C, true, LD, PL>(X0, LEFT, warp, 0));
    __syncthreads();
    pf_store(X0);                                                   // A4
    pf_load(tape + (size_t)T_A2 * C::GMAT);
    __syncthreads();
    // ---- stage 7: X_a += A4 R6
#pragma unroll
    for (int ct = 0; ct < 2; ++ct) {
        c2 acc = ld_thin<LD, PL>(RIGHT, warp * 8, ct * 8);
        for (int kt = 0; kt < NP / 8; ++kt) tile_mma_thin<C, false, MASK_NONE, false, LD, PL>(acc, X0, warp * 8, kt * 8, RIGHT, kt * 8, 32 + ct * 8);
        st_thin<LD, PL>(RIGHT, warp * 8, ct * 8, acc);
    }
    __syncthreads();
    pf_store(X0);                                                   // A2
    __syncthreads();
    // ---- stage 8a: X_a += A2 R4 (R4 = the untouched X_b block)
#pragma unroll
    for (int ct = 0; ct < 2; ++ct) {
        c2 acc = ld_thin<LD, PL>(RIGHT, warp * 8, ct * 8);
        for (int kt = 0; kt < NP / 8; ++kt) tile_mma_thin<C, false, MASK_NONE, false, LD, PL>(acc, X0, warp * 8, kt * 8, RIGHT, kt * 8, 16 + ct * 8);
        st_thin<LD, PL>(RIGHT, warp * 8, ct * 8, acc);
    }
    __syncthreads();
    // ---- stage 8b: X_b += A2 R6;  Lb2 = A2^T Lb
#pragma unroll
    for (int ct = 0; ct < 2; ++ct) {
        c2 acc = ld_thin<LD, PL>(RIGHT, warp * 8, 16 + ct * 8);
        for (int kt = 0; kt < NP / 8; ++kt) tile_mma_thin<C, false, MASK_NONE, false, LD, PL>(acc, X0, warp * 8, kt * 8, RIGHT, kt * 8, 32 + ct * 8);
        st_thin<LD, PL>(RIGHT, warp * 8, 16 + ct * 8, acc);
        st_thin<LD, PL>(LEFT, warp * 8, 16 + ct * 8, thin_tile<C, true, LD, PL>(X0, LEFT, warp, ct * 8));
    }
    __syncthreads();
    // ---- stage 8c: Lb3 = A2^T Lb2
#pragma unroll
    for (int ct = 0; ct < 2; ++ct) st_thin<LD, PL>(LEFT, warp * 8, 32 + ct * 8, thin_tile<C, true, LD, PL>(X0, LEFT, warp, 16 + ct * 8));
    __syncthreads();
    // ---- stage 9: a2bar = [Lb Lb2 Lb3] [X_a X_b X_c]^T -> X0
    Acc<C> acc;
    acc.zero();
    mma_lowrank<C, LD, PL, LD, PL>(acc, LEFT, 0, RIGHT, 0, 48);
    pf_load(tape + (size_t)T_A * C::GMAT);
    for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(X0, row, col, accv<C>(acc, i, j)); });
    __syncthreads();
    for (int e = threadIdx.x; e < NP * 4; e += C::NT) {             // keep l and yp for the rank-S term
        const int row = e >> 2, c = e & 3;
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
            EL[pl * TPL + row * TLD + c] = LEFT[pl * PL + row * LD + 4 + c];
            EL[pl * TPL + row * TLD + 4 + c] = TMP[pl * TPL + row * TLD + 8 + c];
        }
    }
    __syncthreads();
    pf_store(sm.X1);                                                // A
    __syncthreads();
    // ---- stage 10: mbar = l yp^T + a2bar A^T + A^T a2bar
    acc.zero();
    mma_lowrank<C, TLD, TPL, TLD, TPL>(acc, EL, 0, EL, 4, 4);
    mma_smem<C, false, true, false>(acc, X0, sm.X1);
    mma_smem<C, true, false, false>(acc, sm.X1, X0);
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(X0, row, col, accv<C>(acc, i, j)); });
    __syncthreads();
    PROF_MARK(12);
}

// ---------------------------------------------------------------------------------------------------------
// Rank-S reverse pass on a Krylov basis of A2 (NP = 64, S <= 4, s = 0) - the same graph as pade_backward_lowrank, with
// every product by A4, A6, W1, X1 or Y replaced by repeated application of B = A2 (A4 = B^2, A6 = B^3, W1 / X1 / Y are
// polynomials of B) to the thin blocks.  With Kp[k] = B^k p, Km[k] = B^k m, KL[k] = (B^T)^k [a | l]:
//     X_c = R6            = [ sum_k b(7+2k) Kp[k] | sum_k b(6+2k) Km[k] | b13 Kp[0] | b12 Km[0] ]
//     X_b = R4 + B R6     = [ sum_k b(5+2k) Kp[k] | sum_k b(4+2k) Km[k] | sum_k b(11+2k) Kp[k] | sum_k b(10+2k) Km[k] ]
//     X_a = R2 + B^2 R6 + B R4 = [ sum_k b(3+2k) Kp[k] | sum_k b(2+2k) Km[k] | sum_k b(9+2k) Kp[k] | sum_k b(8+2k) Km[k] ]
//     Y p = sum_k b(1+2k) Kp[k]                          (coefficients beyond b13 / b12 are zero)
//     L_b = [KL[0] | KL[3]],  A2^T L_b = [KL[1] | KL[4]],  A2^T A2^T L_b = [KL[2] | KL[5]]
//     a2bar = L_b X_a^T + (A2^T L_b) X_b^T + (A2^T A2^T L_b) X_c^T,     mbar = l (Y p)^T + a2bar A^T + A^T a2bar.
// Two Krylov chains of six thin (n x 8) DMMA products with ONE resident matrix replace the nine tape matrices of the
// re-associated form: the tape of such a slice is {A, A2, LU} (3 instead of 8 matrices written by the forward pass and
// read here), and the loads are TMA boxes issued one stage ahead into the two matrix buffers.
struct TapeFeed {
    const double *tape;          // tape of the slice (slot s at tape + s * GMAT)
    const CUtensorMap *map;      // tensor map of the buffer holding it, or nullptr: plain loads
    long long idx0;              // matrix index of slot 0 in that buffer
    uint64_t *bar0, *bar1;       // mbarriers of the two matrix buffers (X0, X1)
    uint32_t *ph0, *ph1;
};

template <class C>
__device__ __forceinline__ void tape_fetch(const TapeFeed &tf, double *dst, int slot, uint64_t *bar) {
    if (tf.map) { if (threadIdx.x == 0) tma_fetch_matrix<C::NP>(dst, tf.map, tf.idx0 + slot, bar); }
    else g2s<C>(dst, tf.tape + (size_t)slot * C::GMAT);
}
__device__ __forceinline__ void tape_wait(const TapeFeed &tf, uint64_t *bar, uint32_t *ph) {
    if (tf.map) { mbar_wait(bar, *ph); *ph ^= 1; }
    else __syncthreads();
}

template <class C>
__device__ void pade_backward_krylov(const Smem<C> &sm, const TapeFeed &tf, const int *tperm, const double *psi, const double *psi1,
                                     const double *lam1, int S, int herm = 0) {
    static_assert(C::NP == 64 && C::NWARP == 8, "the Krylov reverse pass is laid out for NP = 64 with 8 warps");
    PROF_DECL
    constexpr int NP = C::NP, LD = LR_LD, PL = LR_PL, TLD = LR_TLD, TPL = LR_TPL, ELD = 8, EPL = NP * ELD;
    double *X0 = sm.X0, *X1 = sm.X1;
    double *LEFT = sm.X1, *RIGHT = sm.X1 + 2 * PL, *PP0 = sm.X1 + 4 * PL, *PP1 = PP0 + 2 * TPL, *EL = PP1 + 2 * TPL;
    static_assert(4 * PL + 4 * TPL + 2 * EPL <= 2 * C::SMAT, "thin buffers exceed the X1 / X2 region");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, t = lane & 3;
    const int frow = warp * 8 + (lane >> 2);
    // ---- stage 0: LU -> X0, A -> X1 (asynchronous); [0 | lam] -> PP1, [p | m] -> PP0
    tape_fetch<C>(tf, X0, T_LU, tf.bar0);
    tape_fetch<C>(tf, X1, T_A, tf.bar1);
    for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
        const int row = e >> 2, c = e & 3;
        const bool on = c < S;
        const double lr = on ? lam1[c * 2 * NP + row] : 0., li = on ? lam1[c * 2 * NP + NP + row] : 0.;
        const double pr = on ? psi[c * 2 * NP + row] : 0., pi = on ? psi[c * 2 * NP + NP + row] : 0.;
        const double qr = on ? psi1[c * 2 * NP + row] : 0., qi = on ? psi1[c * 2 * NP + NP + row] : 0.;
        PP1[row * TLD + c] = 0.; PP1[TPL + row * TLD + c] = 0.;
        PP1[row * TLD + 4 + c] = lr; PP1[TPL + row * TLD + 4 + c] = li;
        PP0[row * TLD + c] = pr + qr; PP0[TPL + row * TLD + c] = pi + qi;
        PP0[row * TLD + 4 + c] = pr - qr; PP0[TPL + row * TLD + 4 + c] = pi - qi;
    }
    for (int c = threadIdx.x; c < NP; c += C::NT) sm.piv[c] = tperm[c];
    __syncthreads();
    tape_wait(tf, tf.bar0, tf.ph0);
    PROF_MARK(43);
    // ---- stage 1: l = Q^-T lam -> PP1[:, 4:8]: one thin product with Q^-1, or the thin solve on PP1[:, 0:8] and the row
    // un-permutation; Q^-1 / the LU factors are dead afterwards: A2 -> X0
    if (tape_holds_inverse(tperm)) {
        const c2 v = thin_tile<C, true, TLD, TPL>(X0, PP1, warp, 0);
        __syncthreads();
        tape_fetch<C>(tf, X0, T_A2, tf.bar0);
        if (t >= 2) {
            *reinterpret_cast<double2 *>(PP1 + frow * TLD + 2 * t) = make_double2(v.r0, v.r1);
            *reinterpret_cast<double2 *>(PP1 + TPL + frow * TLD + 2 * t) = make_double2(v.i0, v.i1);
        }
    } else {
        lu_solve_thin_T<C, TLD, TPL>(X0, PP1);
        tape_fetch<C>(tf, X0, T_A2, tf.bar0);
        for (int e = threadIdx.x; e < NP * 4; e += C::NT) {         // row un-permutation through EL
            const int row = e >> 2, c = e & 3, pr = sm.piv[row];
            EL[pr * ELD + c] = PP1[row * TLD + 4 + c]; EL[EPL + pr * ELD + c] = PP1[TPL + row * TLD + 4 + c];
        }
        __syncthreads();
        for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
            const int row = e >> 2, c = e & 3;
            PP1[row * TLD + 4 + c] = EL[row * ELD + c]; PP1[TPL + row * TLD + 4 + c] = EL[EPL + row * ELD + c];
        }
    }
    __syncthreads();
    tape_wait(tf, tf.bar1, tf.ph1);
    PROF_MARK(44);
    // ---- stage 2: a = A^T l (A in X1) -> PP1[:, 0:4]
    {
        const c2 v = thin_tile<C, true, TLD, TPL>(X1, PP1, warp, 0);
        __syncthreads();
        if (t >= 2) {
            *reinterpret_cast<double2 *>(PP1 + frow * TLD + 2 * (t - 2)) = make_double2(v.r0, v.r1);
            *reinterpret_cast<double2 *>(PP1 + TPL + frow * TLD + 2 * (t - 2)) = make_double2(v.i0, v.i1);
        }
    }
    __syncthreads();                                                // A is dead: the LEFT / RIGHT area (over X1) is free
    // ---- stage 3: KL[0] = [a | l] -> LEFT[:, 0:8]; power-0 terms of RIGHT; EL = [l | b1 p]
    for (int e = threadIdx.x; e < NP * 4; e += C::NT) {
        const int row = e >> 2, c = e & 3;
#pragma unroll
        for (int pl = 0; pl < 2; ++pl) {
            const double av = PP1[pl * TPL + row * TLD + c], lv = PP1[pl * TPL + row * TLD + 4 + c];
            const double pv = PP0[pl * TPL + row * TLD + c], mv = PP0[pl * TPL + row * TLD + 4 + c];
            double *L = LEFT + pl * PL + row * LD, *R = RIGHT + pl * PL + row * LD;
            L[c] = av; L[4 + c] = lv;
            R[0 + c] = kB[3] * pv; R[4 + c] = kB[2] * mv; R[8 + c] = kB[9] * pv; R[12 + c] = kB[8] * mv;       // X_a
            R[16 + c] = kB[5] * pv; R[20 + c] = kB[4] * mv; R[24 + c] = kB[11] * pv; R[28 + c] = kB[10] * mv;   // X_b
            R[32 + c] = kB[7] * pv; R[36 + c] = kB[6] * mv; R[40 + c] = kB[13] * pv; R[44 + c] = kB[12] * mv;   // X_c
            EL[pl * EPL + row * ELD + c] = lv; EL[pl * EPL + row * ELD + 4 + c] = kB[1] * pv;
        }
    }
    __syncthreads();
    tape_wait(tf, tf.bar0, tf.ph0);
    PROF_MARK(45);
    // ---- stage 4: the two Krylov chains with B = A2 in X0
    {
        double *cur = PP0, *nxt = PP1;
        const bool ppart = t < 2;                                   // this lane's tile columns: p block (0:4) or m block (4:8)
        const int cc = 2 * (t & 1);                                 // column pair inside the block
#pragma unroll 1
        for (int k = 0; k < 6; ++k) {
            const int kk = k + 1;                                   // power produced in this step
            const int off0 = (k % 3) * 16 + (k / 3) * 8, off1 = (kk % 3) * 16 + (kk / 3) * 8;   // KL[k], KL[kk] in LEFT
            c2 v, w;
            const bool pair = herm && k < 5;                        // Hermitian A2: both chains from one pass over X0
            if (pair) thin_tile_pair<C, TLD, TPL, LD, PL>(X0, cur, 0, LEFT, off0, warp, v, w);
            else v = thin_tile<C, false, TLD, TPL>(X0, cur, warp, 0);
            st_thin<TLD, TPL>(nxt, warp * 8, 0, v);
            if (pair) st_thin<LD, PL>(LEFT, warp * 8, off1, w);      // KL[kk] = B^T KL[k] (other columns than off0)
            // contributions of B^kk p / B^kk m to X_a, X_b, X_c (sub-blocks 0 / 1 and 2 / 3) and to Y p
            double *Rr = RIGHT + frow * LD, *Ri = RIGHT + PL + frow * LD;
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const int i0 = (ppart ? 3 : 2) + 2 * q + 2 * kk, i1 = (ppart ? 9 : 8) + 2 * q + 2 * kk;
                if (i0 <= (ppart ? 13 : 12)) {
                    const double b = kB[i0];
                    const int col = q * 16 + (ppart ? 0 : 4) + cc;
                    Rr[col] += b * v.r0; Rr[col + 1] += b * v.r1; Ri[col] += b * v.i0; Ri[col + 1] += b * v.i1;
                }
                if (i1 <= (ppart ? 13 : 12)) {
                    const double b = kB[i1];
                    const int col = q * 16 + (ppart ? 8 : 12) + cc;
                    Rr[col] += b * v.r0; Rr[col + 1] += b * v.r1; Ri[col] += b * v.i0; Ri[col + 1] += b * v.i1;
                }
            }
            if (ppart) {
                const double b = kB[1 + 2 * kk];
                double *Er = EL + frow * ELD + 4 + cc, *Ei = EL + EPL + frow * ELD + 4 + cc;
                Er[0] += b * v.r0; Er[1] += b * v.r1; Ei[0] += b * v.i0; Ei[1] += b * v.i1;
            }
            if (k < 5 && !pair)                                     // KL[kk] = B^T KL[k]
                st_thin<LD, PL>(LEFT, warp * 8, off1, thin_tile<C, true, LD, PL>(X0, LEFT, warp, off0));
            __syncthreads();
            double *tmp = cur; cur = nxt; nxt = tmp;
        }
    }
    PROF_MARK(46);
    // ---- stage 5: A2 is dead: A -> X0 (asynchronous) while a2bar = [L_b A2^T L_b A2^T A2^T L_b] [X_a X_b X_c]^T is formed
    tape_fetch<C>(tf, X0, T_A, tf.bar0);
    Acc<C> acc;
    acc.zero();
    mma_lowrank<C, LD, PL, LD, PL>(acc, LEFT, 0, RIGHT, 0, 48);
    __syncthreads();                                                // LEFT / RIGHT are dead
    for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(X1, row, col, accv<C>(acc, i, j)); });
    __syncthreads();
    // anti-Hermitian A (Hermitian operators, real controls): every direction dM is anti-Hermitian, so only the
    // anti-Hermitian part of mbar reaches the gradient, and with A^T = -conj(A)
    //     mbar - mbar^H = Z - Z^H,   Z = l (Y p)^T + (a2bar + a2bar^H) A^T
    // - one dense product instead of two.  sym(+1): X <- X + X^H, sym(-1): X <- (X - X^H) / 2, in place in two phases.
    auto sym = [&](double *X, double sg, double scale) {
        c2 hv[C::TM * C::TN];
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 v = lds2<C>(X, row, col);
            const double tr0 = X[col * C::LD + row], tr1 = X[(col + 1) * C::LD + row];
            const double ti0 = X[C::PLANE + col * C::LD + row], ti1 = X[C::PLANE + (col + 1) * C::LD + row];
            hv[i * C::TN + j] = {scale * (v.r0 + sg * tr0), scale * (v.r1 + sg * tr1), scale * (v.i0 - sg * ti0), scale * (v.i1 - sg * ti1)};
        });
        __syncthreads();
        for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(X, row, col, hv[i * C::TN + j]); });
        __syncthreads();
    };
    if (herm) sym(X1, 1.0, 1.0);
    tape_wait(tf, tf.bar0, tf.ph0);
    PROF_MARK(47);
    // ---- stage 6: mbar = l (Y p)^T + a2bar A^T + A^T a2bar
    acc.zero();
    mma_lowrank<C, ELD, EPL, ELD, EPL>(acc, EL, 0, EL, 4, 4);
    mma_smem<C, false, true, false>(acc, X1, X0);
    if (!herm) mma_smem<C, true, false, false>(acc, X0, X1);
    __syncthreads();
    for_owned<C>([&](int i, int j, int row, int col) { sts2<C>(X0, row, col, accv<C>(acc, i, j)); });
    __syncthreads();
    if (herm) sym(X0, -1.0, 0.5);
    PROF_MARK(12);
}

// Magnus adjoint + contraction  cbar_{i,r} = Re sum_ab abar_i[ab] G_r[ab].  In: mbar in X0, coefficients of
// the slice in sm.coef.  Out: gout[i*KR + r] = dE/dc_{i,r}.
template <class C>
__device__ void magnus_backward(const Smem<C> &sm, const GenArgs &ga, double *scratch, double *gout) {
    Acc<C> acc;
    const double dt = ga.dt;
    // cbar_{node,r} = Re sum_ab abar_node[ab] G_r[ab] for one node: the operator loop is outermost so that every step
    // has 2 * TM * TN independent 16-byte loads in flight; thread partials -> warp shuffle -> per-warp slot in sm.red
    c2 abn[C::TM][C::TN];
    auto contract_node = [&](int node) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        double *red = sm.red + 64;
        for (int r = 0; r < ga.KR; ++r) {
            const double *g = ga.G + (size_t)r * C::GMAT;
            double v = 0.;
            for_owned<C>([&](int i, int j, int row, int col) {
                const c2 x = ldg2<C>(g, row, col);
                const c2 &a = abn[i][j];
                v += a.r0 * x.r0 - a.i0 * x.i0 + a.r1 * x.r1 - a.i1 * x.i1;
            });
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[(node * kMaxKR + r) * C::NWARP + warp] = v;
        }
    };
    if (ga.order == 2) {
        for_owned<C>([&](int i, int j, int row, int col) { abn[i][j] = dt * lds2<C>(sm.X0, row, col); });
        contract_node(0);
    } else if (ga.order == 4 && ga.comm) {
        // cbar_{0,r} = <mbar, dt/2 G_r + f (C0_r + sum_s c2_s C_sr)>,  cbar_{1,r} = <mbar, dt/2 G_r - f (C0_r + sum_s c1_s C_sr)>
        // (<X, Y> = Re sum X.Y): inner products of mbar with the precomputed matrices, no products
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, KR = ga.KR, NPAIR = KR * (KR - 1) / 2;
        double *red = sm.red + 64;
        for_owned<C>([&](int i, int j, int row, int col) { abn[i][j] = lds2<C>(sm.X0, row, col); });
        auto dot = [&](const double *g, int slot) {
            double v = 0.;
            for_owned<C>([&](int i, int j, int row, int col) {
                const c2 x = ldg2<C>(g, row, col);
                const c2 &a = abn[i][j];
                v += a.r0 * x.r0 - a.i0 * x.i0 + a.r1 * x.r1 - a.i1 * x.i1;
            });
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[slot * C::NWARP + warp] = v;
        };
        __syncthreads();
        for (int r = 0; r < KR; ++r) dot(ga.G + (size_t)r * C::GMAT, r);
        for (int r = 0; r < KR; ++r) dot(ga.C0 + (size_t)r * C::GMAT, KR + r);
        for (int pr = 0; pr < NPAIR; ++pr) dot(ga.Cs + (size_t)pr * C::GMAT, 2 * KR + pr);
        __syncthreads();
        const double f = (QOCB_S3 / 12.0) * dt * dt;
        for (int e = threadIdx.x; e < 2 * KR; e += C::NT) {
            const int node = e / KR, r = e % KR;
            auto slot_sum = [&](int slot) { double t = 0.; for (int w = 0; w < C::NWARP; ++w) t += red[slot * C::NWARP + w]; return t; };
            const double *cf = sm.coef + (node == 0 ? kMaxKR : 0);          // node 0 pairs with c2, node 1 with c1
            double acc_k = slot_sum(KR + r);
            for (int s_ = 0; s_ < KR; ++s_) {
                if (s_ == r) continue;
                const double k = s_ < r ? slot_sum(2 * KR + comm_pair(s_, r, KR)) : -slot_sum(2 * KR + comm_pair(r, s_, KR));
                acc_k += cf[s_] * k;
            }
            gout[node * KR + r] = 0.5 * dt * slot_sum(r) + (node == 0 ? f : -f) * acc_k;
        }
        __syncthreads();
        return;
    } else if (ga.order == 4) {
        {
            c2 v0[C::TM][C::TN], v1[C::TM][C::TN];
            gen_nodes<C, 2>(ga, sm.coef, 1.0, 1.0, v0, v1);
            for_owned<C>([&](int i, int j, int row, int col) {
                sts2<C>(sm.X1, row, col, v0[i][j]);                                             // a1
                sts2<C>(sm.X2, row, col, v1[i][j]);                                             // a2
            });
        }
        __syncthreads();
        const double f = (QOCB_S3 / 12.0) * dt * dt;
        acc.zero();
        mma_smem<C, true, false, false>(acc, sm.X2, sm.X0);             // a2^T mbar
        mma_smem<C, false, true, true>(acc, sm.X0, sm.X2);              // - mbar a2^T
        for_owned<C>([&](int i, int j, int row, int col) {
            abn[i][j] = (0.5 * dt) * lds2<C>(sm.X0, row, col) + f * accv<C>(acc, i, j);
        });
        contract_node(0);
        acc.zero();
        mma_smem<C, false, true, false>(acc, sm.X0, sm.X1);             // mbar a1^T
        mma_smem<C, true, false, true>(acc, sm.X1, sm.X0);              // - a1^T mbar
        for_owned<C>([&](int i, int j, int row, int col) {
            abn[i][j] = (0.5 * dt) * lds2<C>(sm.X0, row, col) + f * accv<C>(acc, i, j);
        });
        contract_node(1);
    } else {
        // order 6 (oracle/adjoint_model.py:magnus_bwd), everything staged through CTA scratch
        double *gMB = scratch + (size_t)S_T0 * C::GMAT;      // mbar
        double *gB1 = scratch + (size_t)S_T1 * C::GMAT, *gB2 = scratch + (size_t)S_T2 * C::GMAT;
        double *gB3 = scratch + (size_t)S_B3 * C::GMAT, *gC12 = scratch + (size_t)S_C12 * C::GMAT;
        double *gE = scratch + (size_t)S_E * C::GMAT, *gP = scratch + (size_t)S_P * C::GMAT;
        double *gQM = scratch + (size_t)S_QM * C::GMAT;
        double *gB1b = scratch + (size_t)S_A * C::GMAT, *gB2b = scratch + (size_t)S_A2 * C::GMAT;   // reuse
        double *gB3b = scratch + (size_t)S_A4 * C::GMAT, *gT = scratch + (size_t)S_A6 * C::GMAT;
        double *gX = scratch + (size_t)S_T3 * C::GMAT;
        double c2f[kMaxKR], c3f[kMaxKR];
        for (int r = 0; r < ga.KR; ++r) {
            const double c1 = sm.coef[r], cc2 = sm.coef[kMaxKR + r], c3 = sm.coef[2 * kMaxKR + r];
            c2f[r] = (QOCB_S15 / 3.0) * dt * (c3 - c1);
            c3f[r] = (10.0 / 3.0) * dt * (c3 - 2.0 * cc2 + c1);
        }
        for_owned<C>([&](int, int, int row, int col) {
            stg2<C>(gMB, row, col, lds2<C>(sm.X0, row, col));
            stg2<C>(gB1, row, col, dt * gen_pair<C>(ga, row, col, 1.0, sm.coef + kMaxKR));
            stg2<C>(gB2, row, col, gen_pair<C>(ga, row, col, 0.0, c2f));
            stg2<C>(gB3, row, col, gen_pair<C>(ga, row, col, 0.0, c3f));
        });
        // forward pieces again: c12 = [b1,b2], e = 2 b3 + c12, d = [b1,e], qm = b2 - d/60, p = -20 b1 - b3 + c12
        acc.zero();
        gmm<C, false, false, false>(sm, acc, gB1, gB2);
        mma_smem<C, false, false, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 c12 = accv<C>(acc, i, j);
            stg2<C>(gC12, row, col, c12);
            stg2<C>(gE, row, col, 2.0 * ldg2<C>(gB3, row, col) + c12);
            stg2<C>(gP, row, col, (-20.0) * ldg2<C>(gB1, row, col) - ldg2<C>(gB3, row, col) + c12);
        });
        acc.zero();
        gmm<C, false, false, false>(sm, acc, gB1, gE);
        mma_smem<C, false, false, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            stg2<C>(gQM, row, col, ldg2<C>(gB2, row, col) - (1.0 / 60.0) * accv<C>(acc, i, j));
        });
        // cb = mbar/240: pbar = cb qm^T - qm^T cb ; qbar = p^T cb - cb p^T
        acc.zero();
        gmm<C, false, true, false>(sm, acc, gMB, gQM);                  // X0 = mbar, X1 = qm
        mma_smem<C, true, false, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(gT, row, col, (1.0 / 240.0) * accv<C>(acc, i, j)); });   // pbar
        acc.zero();
        gmm<C, true, false, false>(sm, acc, gP, gMB);                   // X0 = p, X1 = mbar
        mma_smem<C, false, true, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 qb = (1.0 / 240.0) * accv<C>(acc, i, j);
            stg2<C>(gB2b, row, col, qb);                                // b2bar = qbar
            stg2<C>(gX, row, col, (-1.0 / 60.0) * qb);                  // dbar
        });
        // t1 = dbar e^T - e^T dbar ; ebar = b1^T dbar - dbar b1^T
        acc.zero();
        gmm<C, false, true, false>(sm, acc, gX, gE);                    // X0 = dbar, X1 = e
        mma_smem<C, true, false, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 pb = ldg2<C>(gT, row, col);
            stg2<C>(gB1b, row, col, ldg2<C>(gMB, row, col) + accv<C>(acc, i, j) - 20.0 * pb);   // b1bar (so far)
        });
        acc.zero();
        gmm<C, true, false, false>(sm, acc, gB1, gX);                   // X0 = b1, X1 = dbar
        mma_smem<C, false, true, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 eb = accv<C>(acc, i, j), pb = ldg2<C>(gT, row, col);
            stg2<C>(gB3b, row, col, 0.5 * ldg2<C>(gMB, row, col) + 2.0 * eb - pb);              // b3bar
            stg2<C>(gX, row, col, eb + pb);                                                     // c12bar (dbar dead)
        });
        // c12 = [b1, b2]: b1bar += c12bar b2^T - b2^T c12bar ; b2bar += b1^T c12bar - c12bar b1^T
        acc.zero();
        gmm<C, false, true, false>(sm, acc, gX, gB2);                   // X0 = c12bar, X1 = b2
        mma_smem<C, true, false, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) { stg2<C>(gB1b, row, col, ldg2<C>(gB1b, row, col) + accv<C>(acc, i, j)); });
        acc.zero();
        gmm<C, true, false, false>(sm, acc, gB1, gX);                   // X0 = b1, X1 = c12bar
        mma_smem<C, false, true, true>(acc, sm.X1, sm.X0);
        for_owned<C>([&](int i, int j, int row, int col) {
            const c2 b2b = ldg2<C>(gB2b, row, col) + accv<C>(acc, i, j);
            const c2 b1b = ldg2<C>(gB1b, row, col), b3b = ldg2<C>(gB3b, row, col);
            abn[i][j] = (-(QOCB_S15 / 3.0) * dt) * b2b + ((10.0 / 3.0) * dt) * b3b;
            stg2<C>(gT, row, col, dt * b1b - ((20.0 / 3.0) * dt) * b3b);                        // node 1 (pbar is dead)
            stg2<C>(gX, row, col, ((QOCB_S15 / 3.0) * dt) * b2b + ((10.0 / 3.0) * dt) * b3b);   // node 2 (c12bar is dead)
        });
        contract_node(0);
        for_owned<C>([&](int i, int j, int row, int col) { abn[i][j] = ldg2<C>(gT, row, col); });
        contract_node(1);
        for_owned<C>([&](int i, int j, int row, int col) { abn[i][j] = ldg2<C>(gX, row, col); });
        contract_node(2);
    }
    // sum of the per-warp slots
    {
        double *red = sm.red + 64;
        __syncthreads();
        for (int e = threadIdx.x; e < ga.q * ga.KR; e += C::NT) {
            const int i = e / ga.KR, r = e % ga.KR;
            double v = 0.;
            for (int w = 0; w < C::NWARP; ++w) v += red[(i * kMaxKR + r) * C::NWARP + w];
            gout[i * ga.KR + r] = v;
        }
        __syncthreads();
    }
}

}  // namespace qocb
