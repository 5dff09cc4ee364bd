// magnus.cuh - Magnus matrices of ALL slices in one streaming pass (orders without matrix products: M2 and the
// product-free M4; qoc/core/mathmethods.py:72-122).
//
// For those orders the Magnus matrix of a slice is a linear combination of a few fixed operators,
//     M_j = sum_c w_c(j) Op_c,     Op = [G0 | G_r | [G0, G_r] | [G_s, G_r] (s < r)],
// with weights that depend on the interpolated controls only (expm_slice.cuh: magnus_forward).  Assembling it inside the
// expm kernel streams 1 + 2 KR + KR (KR - 1) / 2 operator matrices from L2 per slice - latency-bound with one 8-warp CTA
// per SM (12 - 14 us of a 148 us slice at n = 64, KR = 4).  Here the work is turned around: a CTA keeps a 512-element slab
// of every operator in shared memory and walks over the slices, so each operator element is read once per CTA and the
// kernel is bound by its output stream (32 n^2 bytes per slice, written once, coalesced 16-byte stores).  The matrices go
// into the slice-propagator buffer U - slot j holds M_j until the expm kernel has consumed it (it prefetches it by TMA
// during the previous slice) and overwrites it with U_j - so the pass needs no memory of its own.
#pragma once
#include "expm_slice.cuh"

namespace qocb {

constexpr int kMagThreads = 256, kMagSlab = 2 * kMagThreads, kMagTile = 32, kMagGroup = 8;
constexpr int kMagMaxOps = 1 + 2 * kMaxCommKR + kMaxCommKR * (kMaxCommKR - 1) / 2 > 1 + kMaxKR ? 1 + 2 * kMaxCommKR + kMaxCommKR * (kMaxCommKR - 1) / 2 : 1 + kMaxKR;

__host__ __device__ inline int magnus_op_count(int order, int KR) { return order == 4 ? 1 + 2 * KR + KR * (KR - 1) / 2 : 1 + KR; }
__host__ inline size_t magnus_smem_bytes(int order, int KR) {
    return sizeof(double) * ((size_t)magnus_op_count(order, KR) * (kMagSlab + kMagTile));
}

// out[w][GMAT] = Magnus matrix of work item w = member * Nm1 + slice, for w in the block's range; grid = (slabs, groups)
__global__ void __launch_bounds__(kMagThreads) k_magnus(GenArgs ga, int GMAT, int Nm1, long long W, long long per_block, double *out) {
    extern __shared__ __align__(16) double mg_sm[];
    const int KR = ga.KR, q = ga.q, tid = threadIdx.x;
    const bool m4 = ga.order == 4;
    const int nops = magnus_op_count(ga.order, KR);
    double *ops = mg_sm;                                   // [nops][kMagSlab]
    double *wts = mg_sm + (size_t)nops * kMagSlab;         // [nops][kMagTile]
    const int e0 = blockIdx.x * kMagSlab + 2 * tid;        // first of the two matrix elements (doubles) of this thread
    const bool live = e0 < GMAT;
    const long long wbeg = (long long)blockIdx.y * per_block, wend = min(W, wbeg + per_block);
    const double dt = ga.dt, f = (QOCB_S3 / 12.0) * dt * dt;
    long long member = -1;
    auto load_slab = [&](int c, const double *src) {
        double2 v = make_double2(0., 0.);
        if (live) v = *reinterpret_cast<const double2 *>(src + e0);
        *reinterpret_cast<double2 *>(ops + (size_t)c * kMagSlab + 2 * tid) = v;
    };
    for (long long w0 = wbeg; w0 < wend;) {
        const long long e = w0 / Nm1;
        const int j0 = (int)(w0 - e * Nm1);
        const int cnt = (int)min((long long)kMagTile, min(wend - w0, (long long)(Nm1 - j0)));
        __syncthreads();                                    // the previous tile is done with ops / wts
        if (e != member) {                                  // operator slabs: drift-dependent ones per member, the rest once
            if (member < 0 || ga.drift_stride) {            // a control batch (drift_stride = 0) shares the drift too
                const double *G0 = ga.G0 + e * ga.drift_stride, *C0 = ga.C0 + e * KR * ga.drift_stride;
                load_slab(0, G0);
                if (m4) for (int r = 0; r < KR; ++r) load_slab(1 + KR + r, C0 + (size_t)r * GMAT);
            }
            if (member < 0 || ga.g_stride) {                // per-member control operators (g_stride > 0): also per member
                const double *G = ga.G + e * ga.g_stride, *Cs = ga.Cs + e * ga.cs_stride;
                for (int r = 0; r < KR; ++r) load_slab(1 + r, G + (size_t)r * GMAT);
                if (m4) for (int pr = 0; pr < KR * (KR - 1) / 2; ++pr) load_slab(1 + 2 * KR + pr, Cs + (size_t)pr * GMAT);
            }
            member = e;
        }
        // weights of the tile: wts[c][jj]
        const double *ctl = ga.controls + e * ga.ctl_stride;
        for (int idx = tid; idx < cnt * nops; idx += kMagThreads) {
            const int jj = idx / nops, c = idx - jj * nops, j = j0 + jj;
            auto coef = [&](int node, int r) -> double {
                if (ga.nodecoef) return ga.nodecoef[(size_t)(j * q + node) * KR + r];
                const int *id = ga.itab_idx + (j * q + node) * 2;
                const double *iw = ga.itab_w + (j * q + node) * 2;
                return ctl[id[0] * KR + r] * iw[0] + ctl[id[1] * KR + r] * iw[1];
            };
            double wv;
            if (c == 0) wv = dt;
            else if (!m4) wv = dt * coef(0, c - 1);
            else if (c <= KR) wv = 0.5 * dt * (coef(0, c - 1) + coef(1, c - 1));
            else if (c <= 2 * KR) wv = f * (coef(0, c - 1 - KR) - coef(1, c - 1 - KR));
            else {
                int pr = c - 1 - 2 * KR, s_ = 0;
                while (pr >= KR - 1 - s_) { pr -= KR - 1 - s_; ++s_; }
                const int r = s_ + 1 + pr;                  // comm_pair(s_, r, KR) == c - 1 - 2 KR
                wv = f * (coef(1, s_) * coef(0, r) - coef(1, r) * coef(0, s_));
            }
            wts[c * kMagTile + jj] = wv;
        }
        __syncthreads();
        for (int jj = 0; jj < cnt; jj += kMagGroup) {
            double2 acc[kMagGroup];
#pragma unroll
            for (int u = 0; u < kMagGroup; ++u) acc[u] = make_double2(0., 0.);
            for (int c = 0; c < nops; ++c) {
                const double2 o = *reinterpret_cast<const double2 *>(ops + (size_t)c * kMagSlab + 2 * tid);
                const double *wr = wts + c * kMagTile + jj;
#pragma unroll
                for (int u = 0; u < kMagGroup; u += 2) {
                    const double2 ww = *reinterpret_cast<const double2 *>(wr + u);   // jj and u are even: 16-byte aligned
                    acc[u].x = fma(ww.x, o.x, acc[u].x); acc[u].y = fma(ww.x, o.y, acc[u].y);
                    acc[u + 1].x = fma(ww.y, o.x, acc[u + 1].x); acc[u + 1].y = fma(ww.y, o.y, acc[u + 1].y);
                }
            }
            if (live) {
#pragma unroll
                for (int u = 0; u < kMagGroup; ++u)
                    if (jj + u < cnt) *reinterpret_cast<double2 *>(out + (size_t)(w0 + jj + u) * GMAT + e0) = acc[u];
            }
        }
        w0 += cnt;
    }
}

// ---- the adjoint of the same pass -------------------------------------------------------------------------------------
// The Magnus adjoint of these orders needs the inner products <mbar_j, Op_c> = Re sum_ab mbar_j[ab] Op_c[ab] of the cotangent of
// every slice's Magnus matrix with the control operators and their commutators (expm_slice.cuh: magnus_backward).  Inside
// k_backward that streams 2 KR + KR (KR - 1) / 2 operator matrices from L2 per slice (13 us of a 60 us slice at n = 64).
// Turned around it is one skinny GEMM  D[j][c] = sum_e mbar[j][e] Op'[c][e]  (Op' = Op with the imaginary plane negated):
// k_backward leaves mbar_j in the (dead) A slot of the slice's tape, a CTA of k_magnus_adj keeps a 512-element slab of every
// operator in shared memory and walks over tiles of 8 slices with DMMA (m = slices, n = operators, k = slab elements),
// k_magnus_adj_final sums the slabs in a fixed order and applies the coefficient formulas.  HBM-bound: mbar is read once.
constexpr int kAdjSlab = 512, kAdjLD = kAdjSlab + 8, kAdjMaxOps = 32, kAdjThreads = 256;

__host__ __device__ inline int magnus_adj_op_count(int order, int KR) { return order == 4 ? 2 * KR + KR * (KR - 1) / 2 : KR; }
__host__ inline size_t magnus_adj_smem_bytes(int order, int KR) {
    const int nt = (magnus_adj_op_count(order, KR) + 7) / 8;
    return sizeof(double) * ((size_t)nt * 8 * kAdjLD + (size_t)(kAdjThreads / 32) * nt * 64);
}

// partial[(slab * W + w) * kAdjMaxOps + c] = sum over the slab of mbar_w[e] Op'_c[e];  grid = (slabs, groups of slice tiles)
__global__ void __launch_bounds__(kAdjThreads) k_magnus_adj(GenArgs ga, int GMAT, int GPLANE, long long W, long long tiles_per_block,
                                                            const double *mbar0, long long stride, double *partial) {
    extern __shared__ __align__(16) double ad_sm[];
    const int KR = ga.KR, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const int nops = magnus_adj_op_count(ga.order, KR), NTn = (nops + 7) / 8;
    double *ops = ad_sm;                                    // [NTn * 8][kAdjLD]
    double *red = ad_sm + (size_t)NTn * 8 * kAdjLD;         // [warps][NTn][64]
    const int e_base = blockIdx.x * kAdjSlab;
    // operator slabs: kAdjSlab / kAdjThreads = 2 elements per thread and operator; the loads of eight operators are issued
    // together (a plain strided loop is one L2 round trip per element)
    for (int c0 = 0; c0 < NTn * 8; c0 += 8) {
        double v[8][kAdjSlab / kAdjThreads];
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
            const int c = c0 + cc;
            const double *src = c < KR ? ga.G + (size_t)c * GMAT : (c < 2 * KR ? ga.C0 + (size_t)(c - KR) * GMAT : ga.Cs + (size_t)(c - 2 * KR) * GMAT);
#pragma unroll
            for (int h = 0; h < kAdjSlab / kAdjThreads; ++h) {
                const int e = e_base + tid + h * kAdjThreads;
                v[cc][h] = (c < nops && e < GMAT) ? (e < GPLANE ? __ldg(src + e) : -__ldg(src + e)) : 0.;
            }
        }
#pragma unroll
        for (int cc = 0; cc < 8; ++cc)
#pragma unroll
            for (int h = 0; h < kAdjSlab / kAdjThreads; ++h) ops[(c0 + cc) * kAdjLD + tid + h * kAdjThreads] = v[cc][h];
    }
    __syncthreads();
    const long long tiles = (W + 7) / 8;
    const long long tl0 = (long long)blockIdx.y * tiles_per_block, tl1 = min(tiles, tl0 + tiles_per_block);
    constexpr int KB = kAdjSlab / 32 / 8 * 4;                        // 8 blocks of 8 elements over this warp's 64
    // the contraction index inside a block is permuted (slot t <-> elements 8 kk + 2 t and 8 kk + 2 t + 1 for the block's two
    // DMMAs), so mbar and the operators are 16-byte loads: 64 contiguous bytes per slice row and instruction, all 8 in flight
    // at once, and the fragments of the next tile are requested before the reduction of the current one
    auto load_tile = [&](long long tl, double2 (&a)[KB]) {
        const long long j = tl * 8 + g;
        const double *row = mbar0 + (size_t)min(j, W - 1) * stride + e_base;
#pragma unroll
        for (int kk = 0; kk < KB; ++kk) {
            const int k = warp * 64 + kk * 8 + 2 * t;
            a[kk] = (j < W && e_base + k < GMAT) ? __ldg(reinterpret_cast<const double2 *>(row + k)) : make_double2(0., 0.);
        }
    };
    double2 a[KB], an[KB];
    if (tl0 < tl1) load_tile(tl0, a);
    for (long long tl = tl0; tl < tl1; ++tl) {
        if (tl + 1 < tl1) load_tile(tl + 1, an);
        double acc[4][2];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) { acc[nt][0] = 0.; acc[nt][1] = 0.; }
#pragma unroll
        for (int kk = 0; kk < KB; ++kk) {
            const int k = warp * 64 + kk * 8 + 2 * t;
#pragma unroll
            for (int nt = 0; nt < 4; ++nt)
                if (nt < NTn) {
                    const double2 b = *reinterpret_cast<const double2 *>(ops + (nt * 8 + g) * kAdjLD + k);
                    dmma884(acc[nt][0], acc[nt][1], a[kk].x, b.x);
                    dmma884(acc[nt][0], acc[nt][1], a[kk].y, b.y);
                }
        }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
            if (nt < NTn) { red[(warp * NTn + nt) * 64 + g * 8 + 2 * t] = acc[nt][0]; red[(warp * NTn + nt) * 64 + g * 8 + 2 * t + 1] = acc[nt][1]; }
        __syncthreads();
        for (int o = tid; o < NTn * 64; o += kAdjThreads) {
            const int nt = o >> 6, r = (o >> 3) & 7, c = o & 7;
            double v = 0.;
#pragma unroll
            for (int w_ = 0; w_ < kAdjThreads / 32; ++w_) v += red[(w_ * NTn + nt) * 64 + r * 8 + c];
            const long long jj = tl * 8 + r;
            if (jj < W) partial[((size_t)blockIdx.x * W + jj) * kAdjMaxOps + nt * 8 + c] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < KB; ++kk) a[kk] = an[kk];
    }
}

// node_grad[w][node][r] from the slab sums; only slices whose mbar went through the tape (meta[w] <= s_cap)
__global__ void k_magnus_adj_final(GenArgs ga, const double *partial, int slabs, long long W, const int *meta, int s_cap, double *node_grad) {
    const long long tix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int KR = ga.KR, q = ga.q;
    if (tix >= W * q * KR) return;
    const int r = (int)(tix % KR), node = (int)((tix / KR) % q);
    const long long w = tix / ((long long)KR * q);
    if (meta[w] > s_cap) return;
    auto D = [&](int c) { double v = 0.; for (int sl = 0; sl < slabs; ++sl) v += partial[((size_t)sl * W + w) * kAdjMaxOps + c]; return v; };
    const double dt = ga.dt;
    if (ga.order == 2) { node_grad[tix] = dt * D(r); return; }
    const int j = (int)w;                                   // single member: the slice index
    auto coef = [&](int nd, int rr) -> double {
        if (ga.nodecoef) return ga.nodecoef[(size_t)(j * q + nd) * KR + rr];
        const int *id = ga.itab_idx + (j * q + nd) * 2;
        const double *iw = ga.itab_w + (j * q + nd) * 2;
        return ga.controls[id[0] * KR + rr] * iw[0] + ga.controls[id[1] * KR + rr] * iw[1];
    };
    const double f = (QOCB_S3 / 12.0) * dt * dt;
    double acc = D(KR + r);
    for (int s_ = 0; s_ < KR; ++s_) {
        if (s_ == r) continue;
        const double kk = s_ < r ? D(2 * KR + comm_pair(s_, r, KR)) : -D(2 * KR + comm_pair(r, s_, KR));
        acc += coef(node == 0 ? 1 : 0, s_) * kk;             // node 0 pairs with the coefficients of node 1 and vice versa
    }
    node_grad[tix] = 0.5 * dt * D(r) + (node == 0 ? f : -f) * acc;
}

}  // namespace qocb
