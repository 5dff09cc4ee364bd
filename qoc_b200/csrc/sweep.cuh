// sweep.cuh - state / costate propagation across time slices and the cost reductions.
//
// Reference path: the `for system_eval_step` loop of _evaluate_schroedinger_discrete
// (qoc/core/schroedingerdiscrete.py:393-425) and the state costs (qoc/standard/costs/
// targetstateinfidelity.py:39-63, targetstateinfidelitytime.py:46-73, forbidstates.py:50-81).
//
// The time loop is cut into chunks.  With the chunk propagators P_c = prod U_j (built by the expm kernel)
// the forward recursion psi_{j+1} = U_j psi_j becomes: (1) a short sequential pass over chunk boundaries,
// (2) independent local sweeps of all chunks.  The costate recursion lam_j = U_j^T lam_{j+1} + seed_j is
// affine: (1) local sweeps with zero incoming costate give the particular parts, (2) a sequential pass over
// chunk boundaries, (3) local sweeps with the true incoming costates.  The same three-step scheme is what
// the multi-GPU time-slice sharding uses across ranks.
//
// Vectors are planar (NP reals then NP imaginaries).  psi / lam arrays: [member][step][state][2][NP].
#pragma once
#include <cuda_runtime.h>

namespace qocb {

struct CostTerm {
    int kind;          // 0 coherent target, 1 incoherent target, 2 forbid
    int step;          // 1: evaluated at every cost step, 0: final step only
    int fmax;          // vectors per state (padded)
    int vec_off;       // offset (in vectors) into the plan's vector pool: index (s * fmax + f)
    int cnt_off;       // offset into the counts pool: F_s per state
    int ip_off;        // offset into the shared inner-product scratch
    int coh_off;       // coherent target terms: first slot of this term in the overlap-sum buffer of a state-sharded plan
    double w;          // cost_multiplier / normalisation
};

struct SweepArgs {
    int NP, S, N, E;               // padded dim, states, system_eval_count, ensemble members
    int ces;                       // cost_eval_step
    int nterms, ip_total;
    const CostTerm *terms;
    const double *vecs;            // [..][2][NP]
    const int *counts;
    const double *U;               // [E*(N-1)][2*NP*NP]
    const double *chunkP;          // [nchunks][2*NP*NP]
    const int *chunk_begin;        // [nchunks+1] work-item index w = e*(N-1)+j; chunks never straddle members
    const int *member_chunk0;      // [E+1] first chunk of each member
    double *psi, *lam;             // [E][N][S][2][NP]
    double *part;                  // [nchunks][S][2][NP]
    double *cost_part;             // [nchunks]
    const double *psi_in;          // [S][2][NP] state entering the first local slice (psi0 unless time-sharded)
    int psi_mstride;               // member stride of psi_in in doubles: S*2*NP after qocb_set_member_states, else 0 (shared)
    long long vecs_mstride;        // member stride of vecs in doubles when some term has member vectors (the table then holds
                                   // every member's copy of every term, qocb_add_member_cost), else 0: the kernels that
                                   // evaluate costs offset `vecs` once by e * vecs_mstride
    const double *lam_in;          // [S][2][NP] costate entering the last local state from later shards, or nullptr
    double *b_out;                 // [S][2][NP] k_boundary_bwd also writes the costate at the first local state here
    int j_off, Nglob;              // time sharding: global index of local slice 0; global system_eval_count.
                                   // N above is the LOCAL state count (local slices + 1)
    int add_final_seed;            // this shard owns the final state (seed of the final-step costs)
    // sharding of the initial STATES across ranks (qocb_state_shard_*): S above is the local count, normalisations use the
    // total; the coherent target cost couples all states through T = sum_s <t_s|psi_s>: the forward pass writes the local
    // partial sums (one complex slot per coherent term and cost step) to coh_out and leaves the value to
    // k_coherent_value, the backward pass seeds from the all-reduced totals in coh_in.  Unsharded: S_norm = S, const_on = 1,
    // both pointers null.
    int S_norm, const_on;
    double *coh_out;
    const double *coh_in;
};

// slot of the overlap sum of coherent term `tm` at global state index k (step terms: cost steps k = ces, 2 ces, ...)
__device__ __forceinline__ int coh_slot(const CostTerm &tm, int k, int ces) { return tm.coh_off + (tm.step ? k / ces - 1 : 0); }

constexpr int kSweepThreads = 512;
constexpr int kSwThreads = 256;        // boundary / sweep kernels: a warp holds two 8-row A-fragment sets (128 registers)

// ---- shared-memory staging of one propagator (16-byte cp.async), used only by the short prefix / suffix kernels of the
// time-sharded path; the sweep and boundary kernels feed their mat-vecs from registers (see below) ------------------
// Shared layout: planar, row stride LDS = NP + 2 doubles (rows stay 16-byte aligned).  With two lanes per output
// (k-split) both access patterns are bank-conflict free for 64-bit loads:
//   U   v : lane -> (a = lane / 2,  ks = lane % 2), b = 2 i + ks : bank = (2 a + ks) mod 16
//   U^T v : lane -> (a = lane % 16, ks = lane / 16), b = 2 i + ks : a half-warp reads 16 consecutive doubles
template <int NP> struct SwL {
    static constexpr int LDS = NP + 2, PL = NP * LDS, MAT = 2 * PL;
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int NP>
__device__ __forceinline__ void prefetch_mat(double *sU, const double *gU) {
    constexpr int RCH = NP / 2;                                     // 16-byte chunks per row
    for (int idx = threadIdx.x; idx < NP * NP; idx += kSweepThreads) {   // 2 planes * NP rows * NP/2 chunks
        const int plane = idx / (NP * RCH), rem = idx % (NP * RCH);
        const int row = rem / RCH, cc = rem % RCH;
        cp_async16(sU + plane * SwL<NP>::PL + row * SwL<NP>::LDS + cc * 2, gU + (size_t)idx * 2);
    }
}

// ---- mat-vec of the sweeps ---------------------------------------------------------------------------------------------
// out[s][a] = sum_b U[a][b] in[s][b]   (TRANS: sum_b U[b][a] in[s][b]); vectors planar [s][2][NP] in shared memory.
// The step is a small real GEMM on the FP64 tensor pipe: four states form the eight columns (re, im interleaved) of
//     D = Ur * B1 + Ui * B2,   B1[b][2s + p] = V[2s + p][b],   B2[b][2s + p] = -+ V[2s + (p ^ 1)][b]   (V = rows re_s, im_s)
// so that one m8n8k4 accumulator fragment hands every lane the complex result (re, im) of one state and one row.
// Every element of a propagator is used exactly once per state group, so the matrix is NOT staged through shared memory:
// a warp owns one 8-row tile of the output and loads its A fragments straight from global memory (L2) into registers -
// for the NEXT step while the current one computes (`MatRegs` double buffer in the kernels): 16-byte loads, 8 rows x 64
// bytes per warp instruction (U v), or 4 rows x 64 bytes (U^T v).  The contraction index of the two DMMAs of an 8-wide
// k block is permuted (slot t <-> columns 8 kk + 2 t and 8 kk + 2 t + 1) so that both the A and the B fragments of a block
// are one 16-byte load per lane.  The vectors are copied (32 states at a time) into a scratch with row stride NP + 8, which
// makes the B-fragment loads bank-conflict free; NP / 8 row tiles are spread over the 16 warps, the warps of one tile take
// every GW-th group of four states.
template <int NP> struct MvMap {
    static constexpr int NW = kSwThreads / 32;
    static constexpr int TILES = NP / 8;                 // 8-row tiles of the output
    static constexpr int GW = NW / TILES;                // warps per row tile
    static constexpr int KR = NP / 4;                    // A-fragment elements per lane and plane
    static constexpr int LDV = NP + 8;                   // row stride of the padded vector scratch
    static constexpr int BATCH = 32;                     // states per pass through the scratch
    static_assert(NP % 8 == 0 && NW % TILES == 0, "row tiles must divide the warps");
};

template <int NP> struct MatRegs { double r[MvMap<NP>::KR], i[MvMap<NP>::KR]; };

// 16-byte / 8-byte read-only loads as volatile asm: they keep their place between the (volatile) DMMAs, which is how the
// prefetch of the next matrix is interleaved with the products of the current one - a warp that issues all its loads at
// once sits in the load/store queue for as long as the matrix takes to arrive (64 KB at ~64 B/clk)
__device__ __forceinline__ void ldg_nc2(double &x, double &y, const double *p) {
    asm volatile("ld.global.nc.v2.f64 {%0, %1}, [%2];\n" : "=d"(x), "=d"(y) : "l"(p));
}
__device__ __forceinline__ void ldg_nc1(double &x, const double *p) {
    asm volatile("ld.global.nc.f64 %0, [%1];\n" : "=d"(x) : "l"(p));
}
// the A-fragment elements of k block kk (columns 8 kk + 2 t, 8 kk + 2 t + 1) of row a = tile * 8 + g
template <int NP, bool TRANS>
__device__ __forceinline__ void load_mat_block(MatRegs<NP> &m, const double *__restrict__ g, int a, int t, int kk) {
    if (TRANS) {
        const int b = 8 * kk + 2 * t;
        ldg_nc1(m.r[2 * kk], g + b * NP + a); ldg_nc1(m.r[2 * kk + 1], g + (b + 1) * NP + a);
        ldg_nc1(m.i[2 * kk], g + NP * NP + b * NP + a); ldg_nc1(m.i[2 * kk + 1], g + NP * NP + (b + 1) * NP + a);
    } else {
        ldg_nc2(m.r[2 * kk], m.r[2 * kk + 1], g + a * NP + 8 * kk + 2 * t);
        ldg_nc2(m.i[2 * kk], m.i[2 * kk + 1], g + NP * NP + a * NP + 8 * kk + 2 * t);
    }
}

// S: the states of the mat-vecs this matrix will be used for (warps without a state group load nothing)
template <int NP, bool TRANS>
__device__ __forceinline__ void load_mat_regs(MatRegs<NP> &m, const double *__restrict__ g, int S) {
    using M = MvMap<NP>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int tile = warp % M::TILES, gsel = warp / M::TILES;
    if (gsel * 4 >= S) return;
#pragma unroll
    for (int kk = 0; kk < NP / 8; ++kk) load_mat_block<NP, TRANS>(m, g, tile * 8 + (lane >> 2), lane & 3, kk);
}

// all threads call (contains barriers); `in` must be complete and `out` free before the call; `out` is complete after the
// caller's next barrier.  vpad: 2 * BATCH * LDV doubles of scratch.  gnext != nullptr: the matrix at gnext is loaded into
// `nxt` along the way (the loads of k block kk between the DMMAs of k block kk of the warp's first state group).
template <int NP, bool TRANS>
__device__ __forceinline__ void matvec_regs(double *out, const double *in, const MatRegs<NP> &m, int S, double *vpad,
                                            MatRegs<NP> &nxt, const double *__restrict__ gnext) {
    using M = MvMap<NP>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gi = lane >> 2, t = lane & 3;
    const int tile = warp % M::TILES, gsel = warp / M::TILES;
    for (int sb = 0; sb < S; sb += M::BATCH) {
        const int sc = min(M::BATCH, S - sb);
        if (sb > 0) __syncthreads();                                 // the fragment loads of the previous batch are done
        for (int i = threadIdx.x; i < sc * 2 * NP; i += kSwThreads) {
            const int row = i / NP, col = i - row * NP;
            vpad[row * M::LDV + col] = in[(size_t)sb * 2 * NP + i];
        }
        __syncthreads();
        for (int gq = gsel; gq * 4 < sc; gq += M::GW) {
            const int row1 = min(8 * gq + gi, 2 * sc - 1), row2 = row1 ^ 1;      // columns past the last state: never stored
            const double *p1 = vpad + row1 * M::LDV + 2 * t, *p2 = vpad + row2 * M::LDV + 2 * t;
            const bool pf = gnext != nullptr && sb == 0 && gq == gsel;
            double c0 = 0., c1 = 0., d0 = 0., d1 = 0.;
#pragma unroll
            for (int kk = 0; kk < NP / 8; ++kk) {
                if (pf) load_mat_block<NP, TRANS>(nxt, gnext, tile * 8 + gi, t, kk);
                const double2 b1 = *reinterpret_cast<const double2 *>(p1 + 8 * kk);
                const double2 b2 = *reinterpret_cast<const double2 *>(p2 + 8 * kk);
                dmma884(c0, c1, m.r[2 * kk], b1.x);
                dmma884(d0, d1, m.i[2 * kk], b2.x);
                dmma884(c0, c1, m.r[2 * kk + 1], b1.y);
                dmma884(d0, d1, m.i[2 * kk + 1], b2.y);
            }
            // column 2 t = re (B2 carries -Vi there), column 2 t + 1 = im (+Vr)
            const int s = sb + 4 * gq + t;
            if (s < S) {
                out[(size_t)s * 2 * NP + tile * 8 + gi] = c0 - d0;
                out[(size_t)s * 2 * NP + NP + tile * 8 + gi] = c1 + d1;
            }
        }
    }
}

// shared-memory variant (matrix staged by prefetch_mat, row stride NP + 2): used by the short prefix / suffix kernels of
// the time-sharded path.  Two lanes per output split the dot product.
template <int NP, bool TRANS>
__device__ __forceinline__ void matvec_smem(double *out, const double *in, const double *sU, int S) {
    constexpr int LDS = SwL<NP>::LDS, PL = SwL<NP>::PL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ks = TRANS ? (lane >> 4) : (lane & 1);
    const int sub = TRANS ? (lane & 15) : (lane >> 1);
    for (int base = warp * 16; base < S * NP; base += (kSweepThreads / 32) * 16) {      // warp-uniform trip count
        const int o = base + sub;
        const bool live = o < S * NP;
        const int oo = live ? o : 0;
        const int s = oo / NP, a = oo % NP;
        const double *vr = in + s * 2 * NP, *vi = vr + NP;
        double xr = 0., xi = 0., yr = 0., yi = 0.;
#pragma unroll 8
        for (int i = 0; i < NP / 2; ++i) {
            const int b = 2 * i + ks;
            const int idx = TRANS ? (b * LDS + a) : (a * LDS + b);
            const double ur = sU[idx], ui = sU[PL + idx];
            const double br = vr[b], bi = vi[b];
            xr = fma(ur, br, xr); yr = fma(ui, bi, yr);
            xi = fma(ur, bi, xi); yi = fma(ui, br, yi);
        }
        double re = xr - yr, im = xi + yi;
        re += __shfl_xor_sync(0xffffffffu, re, TRANS ? 16 : 1);
        im += __shfl_xor_sync(0xffffffffu, im, TRANS ? 16 : 1);
        if (live && ks == 0) { out[s * 2 * NP + a] = re; out[s * 2 * NP + NP + a] = im; }
    }
}

__device__ __forceinline__ bool is_step_cost_state(int k, int ces) { return k != 0 && (k % ces) == 0; }

// inner products <v_{t,s,f} | psi_s> for every active term -> ip[2*(ip_off + s*fmax + f)]; one warp per vector
__device__ void cost_inner_products(const SweepArgs &a, const double *psi, double *ip, bool step_state, bool final_state) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int t = 0; t < a.nterms; ++t) {
        const CostTerm tm = a.terms[t];
        if (!((tm.step && step_state) || (!tm.step && final_state))) continue;
        for (int e = warp; e < a.S * tm.fmax; e += nw) {
            const int s = e / tm.fmax, f = e % tm.fmax;
            double pr = 0., pi = 0.;
            if (f < a.counts[tm.cnt_off + s]) {
                const double *v = a.vecs + (size_t)(tm.vec_off + e) * 2 * a.NP;
                const double *p = psi + s * 2 * a.NP;
                for (int b = lane; b < a.NP; b += 32) {       // conj(v) * psi
                    const double vr = v[b], vi = v[a.NP + b], xr = p[b], xi = p[a.NP + b];
                    pr += vr * xr + vi * xi;
                    pi += vr * xi - vi * xr;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { pr += __shfl_xor_sync(0xffffffffu, pr, o); pi += __shfl_xor_sync(0xffffffffu, pi, o); }
            if (lane == 0) { ip[2 * (tm.ip_off + e)] = pr; ip[2 * (tm.ip_off + e) + 1] = pi; }
        }
    }
    __syncthreads();
}

// value of the active cost terms at one state set (thread 0 returns it; other threads return 0)
__device__ double cost_value(const SweepArgs &a, const double *ip, bool step_state, bool final_state, int kglob) {
    double val = 0.;
    if (threadIdx.x == 0) {
        for (int t = 0; t < a.nterms; ++t) {
            const CostTerm tm = a.terms[t];
            if (!((tm.step && step_state) || (!tm.step && final_state))) continue;
            if (tm.kind == 0) {
                double tr = 0., ti = 0.;
                for (int s = 0; s < a.S; ++s) { tr += ip[2 * (tm.ip_off + s * tm.fmax)]; ti += ip[2 * (tm.ip_off + s * tm.fmax) + 1]; }
                if (a.coh_out) {                                   // states sharded: the value needs the sum over ALL ranks
                    const int sl = coh_slot(tm, kglob, a.ces);
                    a.coh_out[2 * sl] = tr; a.coh_out[2 * sl + 1] = ti;
                } else {
                    val += tm.w * (1.0 - (tr * tr + ti * ti) / ((double)a.S_norm * a.S_norm));
                }
            } else if (tm.kind == 1) {
                double acc = 0.;
                for (int s = 0; s < a.S; ++s) {
                    const double r = ip[2 * (tm.ip_off + s * tm.fmax)], i = ip[2 * (tm.ip_off + s * tm.fmax) + 1];
                    acc += r * r + i * i;
                }
                val += tm.w * ((a.const_on ? 1.0 : 0.0) - acc / a.S_norm);
            } else {
                double acc = 0.;
                for (int s = 0; s < a.S; ++s) {
                    const int F = a.counts[tm.cnt_off + s];
                    double sub = 0.;
                    for (int f = 0; f < F; ++f) {
                        const double r = ip[2 * (tm.ip_off + s * tm.fmax + f)], i = ip[2 * (tm.ip_off + s * tm.fmax + f) + 1];
                        sub += r * r + i * i;
                    }
                    acc += sub / F;
                }
                val += tm.w * acc;
            }
        }
    }
    return val;
}

// lam[s][a] += d cost / d psi_s[a] in autograd's convention (d/dx - i d/dy):  sum coef * conj(v[a])
__device__ void cost_add_seed(const SweepArgs &a, const double *ip, double *lam, bool step_state, bool final_state, int kglob,
                              int sb = 0, int sc = -1) {
    if (sc < 0) sc = a.S;                                  // lam holds states [sb, sb + sc) only
    for (int t = 0; t < a.nterms; ++t) {
        const CostTerm tm = a.terms[t];
        if (!((tm.step && step_state) || (!tm.step && final_state))) continue;
        double tr = 0., ti = 0.;
        if (tm.kind == 0) {
            if (a.coh_in) { const int sl = coh_slot(tm, kglob, a.ces); tr = a.coh_in[2 * sl]; ti = a.coh_in[2 * sl + 1]; }
            else for (int s = 0; s < a.S; ++s) { tr += ip[2 * (tm.ip_off + s * tm.fmax)]; ti += ip[2 * (tm.ip_off + s * tm.fmax) + 1]; }
        }
        for (int o = threadIdx.x; o < sc * a.NP; o += blockDim.x) {
            const int sl = o / a.NP, s = sb + sl, b = o % a.NP;
            const int F = a.counts[tm.cnt_off + s];
            double sr = 0., si = 0.;
            for (int f = 0; f < F; ++f) {
                const double *v = a.vecs + (size_t)(tm.vec_off + s * tm.fmax + f) * 2 * a.NP;
                double cr, ci;         // coefficient = scale * conj(ip or total)
                if (tm.kind == 0) { const double k = -2.0 * tm.w / ((double)a.S_norm * a.S_norm); cr = k * tr; ci = -k * ti; }
                else if (tm.kind == 1) { const double k = -2.0 * tm.w / a.S_norm; cr = k * ip[2 * (tm.ip_off + s * tm.fmax)]; ci = -k * ip[2 * (tm.ip_off + s * tm.fmax) + 1]; }
                else { const double k = 2.0 * tm.w / F; cr = k * ip[2 * (tm.ip_off + s * tm.fmax + f)]; ci = -k * ip[2 * (tm.ip_off + s * tm.fmax + f) + 1]; }
                const double vr = v[b], vi = -v[a.NP + b];              // conj(v)
                sr += cr * vr - ci * vi;
                si += cr * vi + ci * vr;
            }
            lam[sl * 2 * a.NP + b] += sr;
            lam[sl * 2 * a.NP + a.NP + b] += si;
        }
    }
    __syncthreads();
}

// state-sharded plans: value of the coherent target terms from the all-reduced overlap sums, added to *cost by the one
// rank that counts constants.  nslots[t] slots per term (cost steps of a step term, 1 otherwise).
__global__ void k_coherent_value(const CostTerm *terms, int nterms, const double *coh, int ces, int Nglob, int S_norm, int E, double *cost) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double val = 0.;
    for (int t = 0; t < nterms; ++t) {
        const CostTerm tm = terms[t];
        if (tm.kind != 0) continue;
        const int cnt = tm.step ? (Nglob - 1) / ces : 1;
        for (int q = 0; q < cnt; ++q) {
            const double tr = coh[2 * (tm.coh_off + q)], ti = coh[2 * (tm.coh_off + q) + 1];
            val += tm.w * (1.0 - (tr * tr + ti * ti) / ((double)S_norm * S_norm));
        }
    }
    *cost += val / E;
}

// dynamic smem layout of the sweep kernels: vpad (padded vector scratch of the mat-vec) | v0 (S*2*NP) | v1 (S*2*NP) | ip (2*ip_total)
__host__ __device__ inline size_t sweep_pad_doubles(int NP) { return (size_t)2 * 32 * (NP + 8); }   // 2 BATCH rows of LDV
__host__ __device__ inline size_t sweep_smem_bytes(int NP, int S, int ip_total) {
    return sizeof(double) * (sweep_pad_doubles(NP) + (size_t)4 * S * NP + (size_t)2 * (ip_total > 0 ? ip_total : 1));
}
// prefix / suffix kernels of the time-sharded path: U (padded) | v0 | v1
__host__ __device__ inline size_t prefix_smem_bytes(int NP, int S) {
    return sizeof(double) * ((size_t)2 * NP * (NP + 2) + (size_t)4 * S * NP);
}

template <int NP> struct SweepSmem {
    double *vpad, *v0, *v1, *ip;
    // S: states held by this CTA
    __device__ __forceinline__ SweepSmem(double *sm, int S) {
        vpad = sm;
        v0 = sm + 2 * MvMap<NP>::BATCH * MvMap<NP>::LDV; v1 = v0 + S * 2 * NP; ip = v1 + S * 2 * NP;
    }
    __device__ __forceinline__ void swap() { double *t = v0; v0 = v1; v1 = t; }
};

// (1) boundary states: psi[b_{c+1}] = P_c psi[b_c], sequential over the chunks of one member; grid = (E, state groups):
// the pass is a chain of dependent mat-vecs (per step: the next propagator's register prefetch, one k-split mat-vec, a
// barrier, the store of the boundary state), so the states are spread over CTAs (no coupling between states in this pass)
#ifdef QOCB_PROFILE
#define BPROF_DECL long long bpt__ = clock64();
#define BPROF(id) do { if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) { const long long t__ = clock64(); g_prof[id] += t__ - bpt__; bpt__ = t__; } } while (0)
#else
#define BPROF_DECL
#define BPROF(id) do { } while (0)
#endif

template <int NP>
__global__ void __launch_bounds__(kSwThreads) k_boundary_fwd(SweepArgs a) {
    extern __shared__ __align__(16) double sm_raw[];
    const int spg = (a.S + gridDim.y - 1) / gridDim.y, sb = blockIdx.y * spg;
    const int S = min(spg, a.S - sb), VS = S * 2 * NP, VSA = a.S * 2 * NP, off = sb * 2 * NP;
    if (S <= 0) return;
    SweepSmem<NP> sm(sm_raw, S);
    const int e = blockIdx.x;
    const int c0 = a.member_chunk0[e], c1 = a.member_chunk0[e + 1];
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, false>(cur, a.chunkP + (size_t)c0 * 2 * NP * NP, S);
    const double *psi_in = a.psi_in + (size_t)e * a.psi_mstride + off;
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = psi_in[i];
    double *psi_e = a.psi + (size_t)e * a.N * VSA + off;
    for (int i = threadIdx.x; i < VS; i += kSwThreads) psi_e[i] = psi_in[i];
    BPROF_DECL
    for (int c = c0; c < c1; ++c) {
        const double *gn = c + 1 < c1 ? a.chunkP + (size_t)(c + 1) * 2 * NP * NP : nullptr;   // prefetched inside the mat-vec
        const int kend = a.chunk_begin[c + 1] - e * (a.N - 1);      // state index at the end of chunk c
        BPROF(20);
        __syncthreads();                                            // v0 is complete
        BPROF(21);
        matvec_regs<NP, false>(sm.v1, sm.v0, cur, S, sm.vpad, nxt, gn);
        __syncthreads();
        BPROF(22);
        for (int i = threadIdx.x; i < VS; i += kSwThreads) psi_e[(size_t)kend * VSA + i] = sm.v1[i];
        sm.swap();
        cur = nxt;
        BPROF(23);
#ifdef QOCB_PROFILE
        if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) g_prof[24] += 1;
#endif
    }
}

// (2) local forward sweeps + cost values; grid = nchunks
template <int NP>
__global__ void __launch_bounds__(kSwThreads) k_sweep_fwd(SweepArgs a) {
    extern __shared__ __align__(16) double sm_raw[];
    const int S = a.S, VS = S * 2 * NP;
    SweepSmem<NP> sm(sm_raw, S);
    const int c = blockIdx.x;
    const int wb = a.chunk_begin[c], we = a.chunk_begin[c + 1];
    const int e = wb / (a.N - 1), jb = wb - e * (a.N - 1), je = we - e * (a.N - 1);
    const double *gU = a.U + (size_t)(e * (a.N - 1)) * 2 * NP * NP;
    a.vecs += (size_t)e * a.vecs_mstride;                            // member e's cost vectors (0: shared)
    double *psi_e = a.psi + (size_t)e * a.N * VS;
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, false>(cur, gU + (size_t)jb * 2 * NP * NP, S);
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = psi_e[(size_t)jb * VS + i];
    __syncthreads();
    double cost = 0.;
    for (int j = jb; j < je; ++j) {
        const int k = j + 1;                                          // state produced by slice j
        if (k < je) {
            matvec_regs<NP, false>(sm.v1, sm.v0, cur, S, sm.vpad, nxt, k + 1 < je ? gU + (size_t)k * 2 * NP * NP : nullptr);
            __syncthreads();
            for (int i = threadIdx.x; i < VS; i += kSwThreads) psi_e[(size_t)k * VS + i] = sm.v1[i];
        } else {
            for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v1[i] = psi_e[(size_t)k * VS + i];   // boundary state
            __syncthreads();
        }
        const bool st = is_step_cost_state(k + a.j_off, a.ces), fin = (k + a.j_off == a.Nglob - 1);
        if (a.nterms > 0 && (st || fin)) {
            cost_inner_products(a, sm.v1, sm.ip, st, fin);
            cost += cost_value(a, sm.ip, st, fin, k + a.j_off);
        }
        sm.swap();
        cur = nxt;
        __syncthreads();
    }
    if (threadIdx.x == 0) a.cost_part[c] = cost;
}

// (3a/3c) local backward sweeps.  PARTICULAR: zero incoming costate, result -> part[c], nothing stored.
// otherwise: incoming lam[je] read from the lam array (written by k_boundary_bwd), lam[j] stored for j in (jb, je).
template <int NP, bool PARTICULAR>
__global__ void __launch_bounds__(kSwThreads) k_sweep_bwd(SweepArgs a) {
    extern __shared__ __align__(16) double sm_raw[];
    const int S = a.S, VS = S * 2 * NP;
    SweepSmem<NP> sm(sm_raw, S);
    const int c = blockIdx.x;
    const int wb = a.chunk_begin[c], we = a.chunk_begin[c + 1];
    const int e = wb / (a.N - 1), jb = wb - e * (a.N - 1), je = we - e * (a.N - 1);
    const double *gU = a.U + (size_t)(e * (a.N - 1)) * 2 * NP * NP;
    a.vecs += (size_t)e * a.vecs_mstride;
    const double *psi_e = a.psi + (size_t)e * a.N * VS;
    double *lam_e = a.lam + (size_t)e * a.N * VS;
    const int jstop = PARTICULAR ? jb : jb + 1;
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, true>(cur, gU + (size_t)(je - 1) * 2 * NP * NP, S);
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = PARTICULAR ? 0. : lam_e[(size_t)je * VS + i];
    __syncthreads();
    for (int j = je - 1; j >= jstop; --j) {
        matvec_regs<NP, true>(sm.v1, sm.v0, cur, S, sm.vpad, nxt,      // lam_j = U_j^T lam_{j+1}
                              j - 1 >= jstop ? gU + (size_t)(j - 1) * 2 * NP * NP : nullptr);
        __syncthreads();
        const bool st = is_step_cost_state(j + a.j_off, a.ces);
        if (a.nterms > 0 && st) {                                     // + seed_j (state j < N-1: step costs only)
            cost_inner_products(a, psi_e + (size_t)j * VS, sm.ip, true, false);
            cost_add_seed(a, sm.ip, sm.v1, true, false, j + a.j_off);
        }
        if (!PARTICULAR)
            for (int i = threadIdx.x; i < VS; i += kSwThreads) lam_e[(size_t)j * VS + i] = sm.v1[i];
        sm.swap();
        cur = nxt;
        __syncthreads();
    }
    if (PARTICULAR)
        for (int i = threadIdx.x; i < VS; i += kSwThreads) a.part[(size_t)c * VS + i] = sm.v0[i];
}

// (3b) boundary costates, sequential over the chunks of one member (last to first); grid = (E, state groups).
// lam[N-1] = lam_in + seed_{N-1};  lam[b_c] = P_c^T lam[b_{c+1}] + part_c
template <int NP>
__global__ void __launch_bounds__(kSwThreads) k_boundary_bwd(SweepArgs a, int have_part) {
    extern __shared__ __align__(16) double sm_raw[];
    const int spg = (a.S + gridDim.y - 1) / gridDim.y, sb = blockIdx.y * spg;
    const int S = min(spg, a.S - sb), VS = S * 2 * NP, VSA = a.S * 2 * NP, off = sb * 2 * NP;
    if (S <= 0) return;
    SweepSmem<NP> sm(sm_raw, S);
    const int e = blockIdx.x;
    const int c0 = a.member_chunk0[e], c1 = a.member_chunk0[e + 1];
    a.vecs += (size_t)e * a.vecs_mstride;
    const double *psi_e = a.psi + (size_t)e * a.N * VSA;
    double *lam_e = a.lam + (size_t)e * a.N * VSA + off;
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, true>(cur, a.chunkP + (size_t)(c1 - 1) * 2 * NP * NP, S);
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = a.lam_in ? a.lam_in[off + i] : 0.;
    __syncthreads();
    if (a.nterms > 0 && a.add_final_seed) {                         // inner products of ALL states (coherent sums)
        const bool st = is_step_cost_state(a.N - 1 + a.j_off, a.ces);
        cost_inner_products(a, psi_e + (size_t)(a.N - 1) * VSA, sm.ip, st, true);
        cost_add_seed(a, sm.ip, sm.v0, st, true, a.N - 1 + a.j_off, sb, S);
    }
    for (int i = threadIdx.x; i < VS; i += kSwThreads) lam_e[(size_t)(a.N - 1) * VSA + i] = sm.v0[i];
    for (int c = c1 - 1; c >= c0; --c) {
        const int kbeg = a.chunk_begin[c] - e * (a.N - 1);
        __syncthreads();
        matvec_regs<NP, true>(sm.v1, sm.v0, cur, S, sm.vpad, nxt, c - 1 >= c0 ? a.chunkP + (size_t)(c - 1) * 2 * NP * NP : nullptr);
        __syncthreads();
        if (have_part) {
            for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v1[i] += a.part[(size_t)c * VSA + off + i];
            __syncthreads();
        }
        for (int i = threadIdx.x; i < VS; i += kSwThreads) lam_e[(size_t)kbeg * VSA + i] = sm.v1[i];
        sm.swap();
        cur = nxt;
    }
    __syncthreads();
    if (a.b_out && e == 0)
        for (int i = threadIdx.x; i < VS; i += kSwThreads) a.b_out[off + i] = sm.v0[i];
}

// ---- three-level scheme (single member, no step costs): the sequential boundary passes run on COARSE chunks (2^d sweep
// chunks each); these kernels fill in the states / costates at the sweep-chunk boundaries inside every coarse chunk, all
// coarse chunks at once.  grid = (coarse chunks, state groups); a.chunkP / a.chunk_begin: sweep level; span = 2^d.
template <int NP>
__global__ void __launch_bounds__(kSwThreads) k_mid_fwd(SweepArgs a, int nfine, int span) {
    extern __shared__ __align__(16) double sm_raw[];
    const int spg = (a.S + gridDim.y - 1) / gridDim.y, sb = blockIdx.y * spg;
    const int S = min(spg, a.S - sb), VS = S * 2 * NP, VSA = a.S * 2 * NP, off = sb * 2 * NP;
    const int c0 = blockIdx.x * span, c1 = min(c0 + span, nfine);
    if (S <= 0 || c1 - c0 < 2) return;               // the end state of the last sweep chunk is the coarse pass's
    SweepSmem<NP> sm(sm_raw, S);
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, false>(cur, a.chunkP + (size_t)c0 * 2 * NP * NP, S);
    double *psi_e = a.psi + off;
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = psi_e[(size_t)a.chunk_begin[c0] * VSA + i];
    for (int c = c0; c < c1 - 1; ++c) {
        const double *gn = c + 2 < c1 ? a.chunkP + (size_t)(c + 1) * 2 * NP * NP : nullptr;
        const int kend = a.chunk_begin[c + 1];
        __syncthreads();
        matvec_regs<NP, false>(sm.v1, sm.v0, cur, S, sm.vpad, nxt, gn);
        __syncthreads();
        for (int i = threadIdx.x; i < VS; i += kSwThreads) psi_e[(size_t)kend * VSA + i] = sm.v1[i];
        sm.swap();
        cur = nxt;
    }
}

// PARTICULAR (step costs): zero incoming costate, the particular parts of the sweep chunks (a.part) combine into the
// particular part of the coarse chunk -> part_out[coarse chunk]; nothing else stored.  Otherwise: incoming costate = the
// coarse pass's value at the end of the coarse chunk, costates at the sweep-chunk beginnings stored (have_part: + part[c]).
template <int NP, bool PARTICULAR>
__global__ void __launch_bounds__(kSwThreads) k_mid_bwd(SweepArgs a, int nfine, int span, int have_part, double *part_out) {
    extern __shared__ __align__(16) double sm_raw[];
    const int spg = (a.S + gridDim.y - 1) / gridDim.y, sb = blockIdx.y * spg;
    const int S = min(spg, a.S - sb), VS = S * 2 * NP, VSA = a.S * 2 * NP, off = sb * 2 * NP;
    const int c0 = blockIdx.x * span, c1 = min(c0 + span, nfine);
    if (S <= 0 || c1 <= c0 || (!PARTICULAR && c1 - c0 < 2)) return;
    SweepSmem<NP> sm(sm_raw, S);
    MatRegs<NP> cur = {}, nxt = {};
    load_mat_regs<NP, true>(cur, a.chunkP + (size_t)(c1 - 1) * 2 * NP * NP, S);
    double *lam_e = a.lam + off;
    for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v0[i] = PARTICULAR ? 0. : lam_e[(size_t)a.chunk_begin[c1] * VSA + i];
    const int clast = PARTICULAR ? c0 : c0 + 1;
    for (int c = c1 - 1; c >= clast; --c) {                          // costate at the beginning of sweep chunk c
        const double *gn = c - 1 >= clast ? a.chunkP + (size_t)(c - 1) * 2 * NP * NP : nullptr;
        const int kbeg = a.chunk_begin[c];
        __syncthreads();
        matvec_regs<NP, true>(sm.v1, sm.v0, cur, S, sm.vpad, nxt, gn);
        __syncthreads();
        if (have_part) {
            for (int i = threadIdx.x; i < VS; i += kSwThreads) sm.v1[i] += a.part[(size_t)c * VSA + off + i];
            __syncthreads();
        }
        if (!PARTICULAR)
            for (int i = threadIdx.x; i < VS; i += kSwThreads) lam_e[(size_t)kbeg * VSA + i] = sm.v1[i];
        sm.swap();
        cur = nxt;
    }
    __syncthreads();
    if (PARTICULAR)
        for (int i = threadIdx.x; i < VS; i += kSwThreads) part_out[(size_t)blockIdx.x * VSA + off + i] = sm.v0[i];
}

template <int NP> struct PrefixSmem {
    double *U[1], *v0, *v1;
    __device__ __forceinline__ PrefixSmem(double *sm, int S) { U[0] = sm; v0 = sm + SwL<NP>::MAT; v1 = v0 + S * 2 * NP; }
    __device__ __forceinline__ void swap() { double *t = v0; v0 = v1; v1 = t; }
};

// time sharding: state entering shard `rank` = P_{rank-1} ... P_0 psi0 (allP: [world][2*NP*NP]); grid = 1
template <int NP>
__global__ void __launch_bounds__(kSweepThreads) k_prefix_states(const double *allP, const double *psi0, double *psi_in,
                                                                 int rank, int S) {
    extern __shared__ __align__(16) double sm_raw[];
    const int VS = S * 2 * NP;
    PrefixSmem<NP> sm(sm_raw, S);
    for (int i = threadIdx.x; i < VS; i += kSweepThreads) sm.v0[i] = psi0[i];
    __syncthreads();
    for (int r = 0; r < rank; ++r) {
        prefetch_mat<NP>(sm.U[0], allP + (size_t)r * 2 * NP * NP);
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        matvec_smem<NP, false>(sm.v1, sm.v0, sm.U[0], S);
        __syncthreads();
        sm.swap();
    }
    for (int i = threadIdx.x; i < VS; i += kSweepThreads) psi_in[i] = sm.v0[i];
}

// time sharding: costate entering shard `rank` from the later shards: lam_in(world-1) = 0,
// lam_in(g) = P_{g+1}^T lam_in(g+1) + b_{g+1}   (allb: [world][S][2][NP]); grid = 1
template <int NP>
__global__ void __launch_bounds__(kSweepThreads) k_suffix_costates(const double *allP, const double *allb, double *lam_in,
                                                                   int rank, int world, int S) {
    extern __shared__ __align__(16) double sm_raw[];
    const int VS = S * 2 * NP;
    PrefixSmem<NP> sm(sm_raw, S);
    for (int i = threadIdx.x; i < VS; i += kSweepThreads) sm.v0[i] = 0.;
    __syncthreads();
    for (int r = world - 1; r > rank; --r) {
        prefetch_mat<NP>(sm.U[0], allP + (size_t)r * 2 * NP * NP);
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        matvec_smem<NP, true>(sm.v1, sm.v0, sm.U[0], S);
        __syncthreads();
        for (int i = threadIdx.x; i < VS; i += kSweepThreads) sm.v1[i] += allb[(size_t)r * VS + i];
        __syncthreads();
        sm.swap();
    }
    for (int i = threadIdx.x; i < VS; i += kSweepThreads) lam_in[i] = sm.v0[i];
}

}  // namespace qocb
