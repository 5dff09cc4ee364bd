// tile.cuh - CTA-cooperative complex128 matrix primitives for sm_100a.
//
// One CTA owns one n x n complex matrix problem (n padded to NP).  Matrices are PLANAR (a real plane
// followed by an imaginary plane), row-major: dense NP x NP in global memory, row stride LD = NP + 4 in
// shared memory.  With LD = 4 (mod 8) every 64-bit fragment load of the FP64 tensor-core instruction
// (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4, the native FP64 MMA on sm_100a; tcgen05 has no f64 kind) is
// bank-conflict free for A, B, A^T and B^T operands alike.
//
// Element ownership: in every accumulator / epilogue / elementwise step a thread touches the SAME set of
// (row, col) pairs (the DMMA accumulator layout of its warp tile).  Dependent elementwise chains on
// global scratch matrices therefore need no barrier: a thread only ever re-reads what it wrote itself.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace qocb {

// optional phase profiler (-DQOCB_PROFILE): thread 0 of CTA 0 accumulates clock64() deltas per phase id
#ifdef QOCB_PROFILE
__device__ long long g_prof[48];
#define PROF_DECL long long prof_t0__ = clock64();
#define PROF_MARK(id) do { __syncthreads(); if (blockIdx.x == 0 && threadIdx.x == 0) { const long long t__ = clock64(); g_prof[id] += t__ - prof_t0__; prof_t0__ = t__; } else { prof_t0__ = 0; } } while (0)
#else
#define PROF_DECL
#define PROF_MARK(id) do { } while (0)
#endif

template <int NP_, int WM_, int WN_>
struct Cfg {
    static constexpr int NP = NP_, WM = WM_, WN = WN_;
    static constexpr int NWARP = WM * WN, NT = 32 * NWARP;
    static constexpr int TM = NP / 8 / WM, TN = NP / 8 / WN;   // 8x8 tiles per warp
    static constexpr int LD = NP + 4;
    static constexpr int PLANE = NP * LD;                      // doubles per smem plane
    static constexpr int SMAT = 2 * PLANE;                     // doubles per smem matrix
    static constexpr int GPLANE = NP * NP;
    static constexpr int GMAT = 2 * NP * NP;                   // doubles per global matrix
    static constexpr int PARTS = NT / NP;                      // threads per column in triangular solves
    static_assert(NP % (8 * WM) == 0 && NP % (8 * WN) == 0, "warp tiling must divide NP");
    static_assert(NT % NP == 0 && PARTS >= 1 && PARTS <= 32 && (32 % PARTS) == 0, "bad PARTS");
};

// Complex products use the 3M scheme: with A = Ar + i Ai, B = Br + i Bi,
//     P1 = Ar Br,  P2 = Ai Bi,  P3 = (Ar + Ai)(Br + Bi)   =>   Re(AB) = P1 - P2,  Im(AB) = P3 - P1 - P2,
// three real DMMA products per k-step instead of four (the operand sums are one DADD per fragment element and k-step).
// The accumulator keeps the three partial products apart - they are independent chains for the tensor pipe - and they are
// combined once, when the result is read (accv).  Normwise the rounding error is that of the four-product form (both are
// sums of products of the same magnitudes); everything downstream is tested against the oracle at 1e-10 / 1e-12.
template <class C>
struct Acc {
    double v[C::TM][C::TN][6];   // [0..1] P1 (col, col+1), [2..3] P2, [4..5] P3
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < C::TM; ++i)
#pragma unroll
            for (int j = 0; j < C::TN; ++j)
#pragma unroll
                for (int e = 0; e < 6; ++e) v[i][j][e] = 0.0;
    }
};

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// acc += (+/-) op(A) * op(B), A and B resident in shared memory (planar, stride LD).
template <class C, bool TA, bool TB, bool NEG>
__device__ __forceinline__ void mma_smem(Acc<C> &acc, const double *__restrict__ A, const double *__restrict__ B) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int row0 = (warp / C::WN) * C::TM * 8 + g;
    const int col0 = (warp % C::WN) * C::TN * 8 + g;
#pragma unroll 2
    for (int kk = 0; kk < C::NP / 4; ++kk) {
        const int k = kk * 4 + t;
        double ar[C::TM], ai[C::TM], sa[C::TM], br[C::TN], bi[C::TN], sb[C::TN];
#pragma unroll
        for (int i = 0; i < C::TM; ++i) {
            const int r = row0 + i * 8;
            const int idx = TA ? (k * C::LD + r) : (r * C::LD + k);
            double xr = A[idx], xi = A[C::PLANE + idx];
            if (NEG) { xr = -xr; xi = -xi; }
            ar[i] = xr; ai[i] = xi; sa[i] = xr + xi;
        }
#pragma unroll
        for (int j = 0; j < C::TN; ++j) {
            const int c = col0 + j * 8;
            const int idx = TB ? (c * C::LD + k) : (k * C::LD + c);
            br[j] = B[idx]; bi[j] = B[C::PLANE + idx]; sb[j] = br[j] + bi[j];
        }
#pragma unroll
        for (int i = 0; i < C::TM; ++i)
#pragma unroll
            for (int j = 0; j < C::TN; ++j) dmma884(acc.v[i][j][0], acc.v[i][j][1], ar[i], br[j]);
#pragma unroll
        for (int i = 0; i < C::TM; ++i)
#pragma unroll
            for (int j = 0; j < C::TN; ++j) dmma884(acc.v[i][j][2], acc.v[i][j][3], ai[i], bi[j]);
#pragma unroll
        for (int i = 0; i < C::TM; ++i)
#pragma unroll
            for (int j = 0; j < C::TN; ++j) dmma884(acc.v[i][j][4], acc.v[i][j][5], sa[i], sb[j]);
    }
}

// Visit the element pairs this thread owns: f(tm, tn, row, col) owns (row, col) and (row, col + 1).
template <class C, class F>
__device__ __forceinline__ void for_owned(F &&f) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row0 = (warp / C::WN) * C::TM * 8 + (lane >> 2);
    const int col0 = (warp % C::WN) * C::TN * 8 + (lane & 3) * 2;
#pragma unroll
    for (int i = 0; i < C::TM; ++i)
#pragma unroll
        for (int j = 0; j < C::TN; ++j) f(i, j, row0 + i * 8, col0 + j * 8);
}

struct c2 { double r0, r1, i0, i1; };   // a complex element pair

template <class C> __device__ __forceinline__ c2 ldg2(const double *__restrict__ g, int row, int col) {
    const double2 r = *reinterpret_cast<const double2 *>(g + row * C::NP + col);
    const double2 i = *reinterpret_cast<const double2 *>(g + C::GPLANE + row * C::NP + col);
    return {r.x, r.y, i.x, i.y};
}
template <class C> __device__ __forceinline__ void stg2(double *__restrict__ g, int row, int col, const c2 &v) {
    *reinterpret_cast<double2 *>(g + row * C::NP + col) = make_double2(v.r0, v.r1);
    *reinterpret_cast<double2 *>(g + C::GPLANE + row * C::NP + col) = make_double2(v.i0, v.i1);
}
template <class C> __device__ __forceinline__ c2 lds2(const double *s, int row, int col) {
    const double2 r = *reinterpret_cast<const double2 *>(s + row * C::LD + col);
    const double2 i = *reinterpret_cast<const double2 *>(s + C::PLANE + row * C::LD + col);
    return {r.x, r.y, i.x, i.y};
}
template <class C> __device__ __forceinline__ void sts2(double *s, int row, int col, const c2 &v) {
    *reinterpret_cast<double2 *>(s + row * C::LD + col) = make_double2(v.r0, v.r1);
    *reinterpret_cast<double2 *>(s + C::PLANE + row * C::LD + col) = make_double2(v.i0, v.i1);
}
template <class C> __device__ __forceinline__ c2 accv(const Acc<C> &a, int i, int j) {
    const double *p = a.v[i][j];                                   // 3M recombination
    return {p[0] - p[2], p[1] - p[3], p[4] - p[0] - p[2], p[5] - p[1] - p[3]};
}
__device__ __forceinline__ c2 operator+(const c2 &a, const c2 &b) { return {a.r0 + b.r0, a.r1 + b.r1, a.i0 + b.i0, a.i1 + b.i1}; }
__device__ __forceinline__ c2 operator-(const c2 &a, const c2 &b) { return {a.r0 - b.r0, a.r1 - b.r1, a.i0 - b.i0, a.i1 - b.i1}; }
__device__ __forceinline__ c2 operator*(double s, const c2 &a) { return {s * a.r0, s * a.r1, s * a.i0, s * a.i1}; }
__device__ __forceinline__ c2 czero() { return {0., 0., 0., 0.}; }
// ---- (anti-)Hermitian products at NP = 64, 8 warps -----------------------------------------------------------------------
// Every product of the Pade polynomial of an ANTI-Hermitian argument A has a Hermitian result (A2 = A A and the polynomials in
// it: A4, A6, A6 W1, A6 X1) or an anti-Hermitian one (A Y).  Only the 36 of the 64 8x8 tiles on and above the diagonal are
// computed; herm_store writes each of them and its (+/-) conjugate transpose.  Tile assignment: rows p and 7 - p hold
// 8 - p and p + 1 upper tiles, nine together; warp p takes the first five of row p, warp p + 4 the other 3 - p and the
// p + 1 of row 7 - p.  Warps p and p + 4 share a scheduler, so every tensor pipe runs 9 tile-products per k-step instead of
// the 16 of the full product.
struct HAcc {
    double v[5][6];              // per tile: P1 (col, col + 1), P2, P3 of the 3M scheme (Acc)
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int q = 0; q < 5; ++q)
#pragma unroll
            for (int e = 0; e < 6; ++e) v[q][e] = 0.0;
    }
};
// tile q of this warp -> (row tile, column tile); false for the fifth tile of a four-tile warp
__device__ __forceinline__ bool herm_tile(int warp, int q, int &rt, int &ct) {
    const int p = warp & 3;
    if (warp < 4) { rt = p; ct = p + q; return true; }
    const int n0 = 3 - p;
    if (q < n0) { rt = p; ct = p + 5 + q; } else { rt = 7 - p; ct = 7 - p + (q - n0); }
    if (q >= 4) { rt = 7 - p; ct = 7; return false; }
    return true;
}
// NT tiles of one warp; ONE_ROW: all of them in the same row tile (one A fragment per k-step).  The fragments of k-step
// kk + 1 are loaded while the DMMAs of kk-step kk issue (two warps per scheduler leave little else to hide the latency).
template <class C, int NT, bool ONE_ROW>
__device__ __forceinline__ void herm_loop(HAcc &acc, const double *__restrict__ A, const double *__restrict__ B,
                                          const int (&ra)[5], const int (&cb)[5]) {
    constexpr int NA = ONE_ROW ? 1 : NT;
    double ar[NA], ai[NA], br[NT], bi[NT];
#pragma unroll
    for (int q = 0; q < NA; ++q) { ar[q] = A[ra[q]]; ai[q] = A[C::PLANE + ra[q]]; }
#pragma unroll
    for (int q = 0; q < NT; ++q) { br[q] = B[cb[q]]; bi[q] = B[C::PLANE + cb[q]]; }
#pragma unroll 4
    for (int kk = 0; kk < C::NP / 4; ++kk) {
        const int kn = (kk + 1 < C::NP / 4) ? kk + 1 : kk;
        double nar[NA], nai[NA], nbr[NT], nbi[NT], sa[NA], sb[NT];
#pragma unroll
        for (int q = 0; q < NA; ++q) { nar[q] = A[ra[q] + kn * 4]; nai[q] = A[C::PLANE + ra[q] + kn * 4]; sa[q] = ar[q] + ai[q]; }
#pragma unroll
        for (int q = 0; q < NT; ++q) {
            nbr[q] = B[cb[q] + kn * 4 * C::LD]; nbi[q] = B[C::PLANE + cb[q] + kn * 4 * C::LD]; sb[q] = br[q] + bi[q];
        }
#pragma unroll
        for (int q = 0; q < NT; ++q) dmma884(acc.v[q][0], acc.v[q][1], ar[ONE_ROW ? 0 : q], br[q]);
#pragma unroll
        for (int q = 0; q < NT; ++q) dmma884(acc.v[q][2], acc.v[q][3], ai[ONE_ROW ? 0 : q], bi[q]);
#pragma unroll
        for (int q = 0; q < NT; ++q) dmma884(acc.v[q][4], acc.v[q][5], sa[ONE_ROW ? 0 : q], sb[q]);
#pragma unroll
        for (int q = 0; q < NA; ++q) { ar[q] = nar[q]; ai[q] = nai[q]; }
#pragma unroll
        for (int q = 0; q < NT; ++q) { br[q] = nbr[q]; bi[q] = nbi[q]; }
    }
}
template <class C>
__device__ __forceinline__ void mma_herm(HAcc &acc, const double *__restrict__ A, const double *__restrict__ B) {
    static_assert(C::NP == 64 && C::NWARP == 8, "tile assignment of the Hermitian product is for 64 x 64 and 8 warps");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    int ra[5], cb[5];                                      // fragment offsets of k-step 0: A[row][t], B[t][col]
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        int rt, ct;
        herm_tile(warp, q, rt, ct);
        ra[q] = (rt * 8 + g) * C::LD + t;
        cb[q] = t * C::LD + ct * 8 + g;
    }
    if (warp < 4) herm_loop<C, 5, true>(acc, A, B, ra, cb);
    else herm_loop<C, 4, false>(acc, A, B, ra, cb);
}
// D = the product held in acc: upper tiles as computed, lower tiles as their conjugate transposes (ANTI: negated ones)
template <class C, bool ANTI>
__device__ __forceinline__ void herm_store(double *D, const HAcc &acc) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        int rt, ct;
        if (!herm_tile(warp, q, rt, ct)) continue;
        const double *a = acc.v[q];
        const c2 v = {a[0] - a[2], a[1] - a[3], a[4] - a[0] - a[2], a[5] - a[1] - a[3]};
        const int row = rt * 8 + g, col = ct * 8 + 2 * t;
        sts2<C>(D, row, col, v);
        if (rt != ct) {
            const double sr = ANTI ? -1.0 : 1.0, si = ANTI ? 1.0 : -1.0;
            D[col * C::LD + row] = sr * v.r0;
            D[(col + 1) * C::LD + row] = sr * v.r1;
            D[C::PLANE + col * C::LD + row] = si * v.i0;
            D[C::PLANE + (col + 1) * C::LD + row] = si * v.i1;
        }
    }
}

// the 3M recombination of tile q of a Hermitian product
__device__ __forceinline__ c2 herm_val(const HAcc &acc, int q) {
    const double *a = acc.v[q];
    return {a[0] - a[2], a[1] - a[3], a[4] - a[0] - a[2], a[5] - a[1] - a[3]};
}
// D[col][row], D[col + 1][row] = conj(v) (ANTI: -conj(v)): the mirror image of the pair (row, col), (row, col + 1)
template <class C, bool ANTI>
__device__ __forceinline__ void sts2_mirror(double *D, int row, int col, const c2 &v) {
    const double sr = ANTI ? -1.0 : 1.0, si = ANTI ? 1.0 : -1.0;
    D[col * C::LD + row] = sr * v.r0;
    D[(col + 1) * C::LD + row] = sr * v.r1;
    D[C::PLANE + col * C::LD + row] = si * v.i0;
    D[C::PLANE + (col + 1) * C::LD + row] = si * v.i1;
}
// visit the upper tiles of this warp: f(q, row, col, diagonal_tile) owns (row, col), (row, col + 1) of tile q
template <class F>
__device__ __forceinline__ void for_herm_tiles(F &&f) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 5; ++q) {
        int rt, ct;
        if (!herm_tile(warp, q, rt, ct)) continue;
        f(q, rt * 8 + (lane >> 2), ct * 8 + (lane & 3) * 2, rt == ct);
    }
}
// asynchronous global -> shared copy of one planar matrix (16-byte cp.async); complete after g2s_async_wait + a barrier
template <class C> __device__ __forceinline__ void g2s_async(double *__restrict__ s, const double *__restrict__ g) {
    constexpr int CH = C::GMAT / 2, RCH = C::NP / 2;
    for (int idx = threadIdx.x; idx < CH; idx += C::NT) {
        const int plane = idx / (C::GPLANE / 2);
        const int rem = idx - plane * (C::GPLANE / 2);
        const int row = rem / RCH, cc = rem - row * RCH;
        const unsigned sa = (unsigned)__cvta_generic_to_shared(s + plane * C::PLANE + row * C::LD + cc * 2);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(g + (size_t)idx * 2) : "memory");
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void g2s_async_wait() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// real identity contribution on the diagonal of an owned pair
__device__ __forceinline__ c2 add_diag(c2 v, int row, int col, double d) {
    if (row == col) v.r0 += d;
    if (row == col + 1) v.r1 += d;
    return v;
}

// cooperative copy global (dense planar) -> shared (padded planar); caller provides the barriers
// global -> shared copy of one planar matrix.  cp.async keeps all of a thread's 16-byte chunks in flight at once (a loop of
// load / store pairs whose trip count the compiler cannot see is one L2 round trip per chunk: 16 of them at NP = 64);
// the data is visible to the other threads after the caller's next barrier, as with plain stores.
template <class C> __device__ __forceinline__ void g2s(double *__restrict__ s, const double *__restrict__ g) {
    g2s_async<C>(s, g);
    g2s_async_wait();
}
template <class C> __device__ __forceinline__ void s2g(double *__restrict__ g, const double *__restrict__ s) {
    constexpr int CH = C::GMAT / 2;
    constexpr int RCH = C::NP / 2;
    for (int idx = threadIdx.x; idx < CH; idx += C::NT) {
        const int plane = idx / (C::GPLANE / 2);
        const int rem = idx - plane * (C::GPLANE / 2);
        const int row = rem / RCH, cc = rem - row * RCH;
        reinterpret_cast<double2 *>(g)[idx] = *reinterpret_cast<const double2 *>(s + plane * C::PLANE + row * C::LD + cc * 2);
    }
}

// ---- small complex helpers -------------------------------------------------------------------------
struct cplx { double r, i; };
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.r * b.r - a.i * b.i, a.r * b.i + a.i * b.r}; }
__device__ __forceinline__ cplx crecip(cplx a) {
    // Smith's algorithm (robust against overflow), as LAPACK's zladiv does for zgesv pivots
    if (fabs(a.r) >= fabs(a.i)) { const double q = a.i / a.r, d = a.r + a.i * q; return {1.0 / d, -q / d}; }
    const double q = a.r / a.i, d = a.r * q + a.i; return {q / d, -1.0 / d};
}

// ---- blocked LU with partial pivoting on a shared-memory matrix, FP64 tensor cores for everything but the panels --
// Semantics of zgesv (qoc/standard/functions/expm.py:246 -> numpy.linalg.solve -> LAPACK zgetrf/zgetrs): row
// pivoting with pivot = first row maximising |re| + |im| (izamax).  Block size 8 = one DMMA tile.
//
// Storage after lu_factor_blocked ("LUi" format, also what the reverse-pass tape holds for pivoted slices):
//   * off-diagonal blocks: L (below) and U (above) as usual;
//   * every 8 x 8 diagonal block holds the INVERSES of its triangular factors: strictly lower part = strictly lower
//     part of inv(L_kk) (unit diagonal implied), upper part incl. diagonal = inv(U_kk).  Triangular solves then are
//     tile products only (trsm via inverted diagonal blocks), issued as DMMA like every other product;
//   * perm[i] = source row of row i of the permuted matrix:  (Pi Q)[i] = Q[perm[i]],  Pi Q = L U.
// Work split: warp 0 factors the 8-column panel (warp-synchronous, no block barrier inside); afterwards every warp
// owns whole column tiles (row swaps, U12 = inv(L11) A12 and the trailing update of that column tile need only
// __syncwarp), so one LU costs 2 block barriers per panel.  The solves are barrier-free: each warp carries its own
// 8 right-hand-side columns through the whole forward and backward substitution.
enum { MASK_NONE = 0, MASK_LINV = 1, MASK_UINV = 2 };

// DMMA A-fragment element (row r0+g, k k0+t) of op(M); T: op = transpose.  Masks act on the STORED coordinates.
template <class C, bool T, int MASK>
__device__ __forceinline__ void ld_afrag(const double *M, int r0, int k0, int g, int t, double &re, double &im) {
    const int r = r0 + g, k = k0 + t;
    const int mr = T ? k : r, mc = T ? r : k;
    re = M[mr * C::LD + mc]; im = M[C::PLANE + mr * C::LD + mc];
    if (MASK == MASK_LINV) { if (mr == mc) { re = 1.0; im = 0.0; } else if (mr < mc) { re = 0.0; im = 0.0; } }
    if (MASK == MASK_UINV) { if (mr > mc) { re = 0.0; im = 0.0; } }
}

// acc (8 x 8 complex tile at rows ar0, cols bc0) += sign * op(A)[ar0:+8, ak0:+8] * B[bk0:+8, bc0:+8]
template <class C, bool T, int MASK, bool NEG>
__device__ __forceinline__ void tile_mma(c2 &acc, const double *A, int ar0, int ak0, const double *B, int bk0, int bc0) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    double p1a = 0., p1b = 0., p2a = 0., p2b = 0., p3a = 0., p3b = 0.;   // 3M partial products (see Acc)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
        double ar, ai;
        ld_afrag<C, T, MASK>(A, ar0, ak0 + 4 * ks, g, t, ar, ai);
        if (NEG) { ar = -ar; ai = -ai; }
        const int bidx = (bk0 + 4 * ks + t) * C::LD + bc0 + g;
        const double br = B[bidx], bi = B[C::PLANE + bidx];
        dmma884(p1a, p1b, ar, br);
        dmma884(p2a, p2b, ai, bi);
        dmma884(p3a, p3b, ar + ai, br + bi);
    }
    acc.r0 += p1a - p2a; acc.r1 += p1b - p2b;
    acc.i0 += p3a - p1a - p2a; acc.i1 += p3b - p1b - p2b;
}
template <class C> __device__ __forceinline__ c2 ld_ctile(const double *M, int r0, int c0) {
    const int lane = threadIdx.x & 31;
    return lds2<C>(M, r0 + (lane >> 2), c0 + (lane & 3) * 2);
}
template <class C> __device__ __forceinline__ void st_ctile(double *M, int r0, int c0, const c2 &v) {
    const int lane = threadIdx.x & 31;
    sts2<C>(M, r0 + (lane >> 2), c0 + (lane & 3) * 2, v);
}

// W[rt] -= op(LU)[rt, kb] * W[kb] for the row tiles rt = r_begin, r_begin + r_step, ... < r_end of one column tile; two
// row tiles per trip give the DMMA pipe independent accumulator chains
template <class C, bool T>
__device__ __forceinline__ void tile_update_rows(const double *LU, double *W, int kb, int c0, int r_begin, int r_end, int r_step) {
    int rt = r_begin;
    for (; rt + r_step < r_end; rt += 2 * r_step) {
        c2 a = ld_ctile<C>(W, rt * 8, c0), b = ld_ctile<C>(W, (rt + r_step) * 8, c0);
        tile_mma<C, T, MASK_NONE, true>(a, LU, rt * 8, kb * 8, W, kb * 8, c0);
        tile_mma<C, T, MASK_NONE, true>(b, LU, (rt + r_step) * 8, kb * 8, W, kb * 8, c0);
        st_ctile<C>(W, rt * 8, c0, a);
        st_ctile<C>(W, (rt + r_step) * 8, c0, b);
    }
    if (rt < r_end) {
        c2 a = ld_ctile<C>(W, rt * 8, c0);
        tile_mma<C, T, MASK_NONE, true>(a, LU, rt * 8, kb * 8, W, kb * 8, c0);
        st_ctile<C>(W, rt * 8, c0, a);
    }
}

// warp 0: unblocked LU with partial pivoting of the panel (rows j0.., columns j0..j0+7), then the in-place inversion
// of the diagonal block's triangular factors.  piv8: shared int[8]; perm: shared int[NP].
template <class C>
__device__ void lu_panel_warp(double *Q, int *perm, int *piv8, int j0) {
    // Register-resident panel: lane owns panel rows j0 + lane (a) and j0 + lane + 32 (b).  Rows are not moved
    // while the panel is factored; each row tracks the POSITION it would occupy under LAPACK's sequential swaps
    // (pos), the pivot is found with one integer REDUX on the high word of |re| + |im| (ties inside 2^-20 are
    // resolved towards the smaller row - any of them is an admissible pivot), and the pivot row is broadcast
    // with shuffles.  Rows are written back to their final positions at the end.
    constexpr bool TWO = C::NP > 32;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    double *Qr = Q, *Qi = Q + C::PLANE;
    const int ra = j0 + lane, rb = j0 + lane + 32;
    const bool va = ra < C::NP, vb = TWO && rb < C::NP;
    cplx pa[8], pb[8];
#pragma unroll
    for (int c = 0; c < 8; c += 2) {                                // 16-byte accesses: a row's 8 panel entries are contiguous
        double2 r = make_double2(0., 0.), i = r;
        if (va) { r = *reinterpret_cast<const double2 *>(Qr + ra * C::LD + j0 + c); i = *reinterpret_cast<const double2 *>(Qi + ra * C::LD + j0 + c); }
        pa[c] = {r.x, i.x}; pa[c + 1] = {r.y, i.y};
        r = make_double2(0., 0.); i = r;
        if (vb) { r = *reinterpret_cast<const double2 *>(Qr + rb * C::LD + j0 + c); i = *reinterpret_cast<const double2 *>(Qi + rb * C::LD + j0 + c); }
        pb[c] = {r.x, i.x}; pb[c + 1] = {r.y, i.y};
    }
    int posa = ra, posb = rb;
    bool useda = !va, usedb = !vb;
    cplx dinv[8];                                                   // reciprocals of the U diagonal
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        // one REDUX finds the pivot and its owner: key = high word of |re| + |im| with its low 6 bits replaced by
        // 63 - (32 * half + lane).  Magnitudes within 2^-14 of the maximum count as ties (any of them is an admissible
        // pivot) and go to the smallest row id.
        const int ka = useda ? -1 : ((__double2hiint(fabs(pa[j].r) + fabs(pa[j].i)) & ~63) | (63 - lane));
        const int kb = usedb ? -1 : ((__double2hiint(fabs(pb[j].r) + fabs(pb[j].i)) & ~63) | (31 - lane));
        const int kmax = __reduce_max_sync(FULL, max(ka, kb));
        const int id = 63 - (kmax & 63);
        const bool from_a = id < 32;
        const int owner = id & 31;
        const bool mine_a = from_a && lane == owner, mine_b = !from_a && lane == owner;
        const int q = __shfl_sync(FULL, from_a ? posa : posb, owner);          // position of the pivot row
        cplx u[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            if (c >= j) {
                const double sr = from_a ? pa[c].r : pb[c].r, si = from_a ? pa[c].i : pb[c].i;
                u[c].r = __shfl_sync(FULL, sr, owner); u[c].i = __shfl_sync(FULL, si, owner);
            }
        }
        // LAPACK swap of positions j0 + j and q
        const int tgt = j0 + j;
        if (posa == tgt && !mine_a) posa = q;
        if (posb == tgt && !mine_b) posb = q;
        if (mine_a) { posa = tgt; useda = true; }
        if (mine_b) { posb = tgt; usedb = true; }
        if (lane == 0) { piv8[j] = q; const int tp = perm[tgt]; perm[tgt] = perm[q]; perm[q] = tp; }
        // 1 / u_jj: hardware reciprocal seed + two Newton steps (the IEEE division sequence is ~3x as many instructions,
        // and the panel is bound by the instruction issue of this one warp)
        const double nn = u[j].r * u[j].r + u[j].i * u[j].i;
        double dn;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(dn) : "d"(nn));
        dn = fma(dn, fma(-nn, dn, 1.0), dn);
        dn = fma(dn, fma(-nn, dn, 1.0), dn);
        const cplx inv = {u[j].r * dn, -u[j].i * dn};
        dinv[j] = inv;
        if (!useda) {
            const cplx l = cmul(pa[j], inv);
            pa[j] = l;
#pragma unroll
            for (int c = 0; c < 8; ++c) if (c > j) { pa[c].r -= l.r * u[c].r - l.i * u[c].i; pa[c].i -= l.r * u[c].i + l.i * u[c].r; }
        }
        if (TWO && !usedb) {
            const cplx l = cmul(pb[j], inv);
            pb[j] = l;
#pragma unroll
            for (int c = 0; c < 8; ++c) if (c > j) { pb[c].r -= l.r * u[c].r - l.i * u[c].i; pb[c].i -= l.r * u[c].i + l.i * u[c].r; }
        }
    }
#ifdef QOCB_PROFILE
    long long pt0__ = clock64();
#endif
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 8; c += 2) {
        if (va) {
            *reinterpret_cast<double2 *>(Qr + posa * C::LD + j0 + c) = make_double2(pa[c].r, pa[c + 1].r);
            *reinterpret_cast<double2 *>(Qi + posa * C::LD + j0 + c) = make_double2(pa[c].i, pa[c + 1].i);
        }
        if (vb) {
            *reinterpret_cast<double2 *>(Qr + posb * C::LD + j0 + c) = make_double2(pb[c].r, pb[c + 1].r);
            *reinterpret_cast<double2 *>(Qi + posb * C::LD + j0 + c) = make_double2(pb[c].i, pb[c + 1].i);
        }
    }
    __syncwarp();
    // invert the diagonal block's factors: lanes 0-7 one column of inv(L_kk), lanes 8-15 one column of inv(U_kk).
    // Column c of the inverse = substitution applied to e_c, fully unrolled with x in registers; block entries are
    // shared-memory broadcasts.  Right-looking form: as soon as x[r] is known every later partial sum is updated with it,
    // so the dependent chain is one complex multiply-add per row.
    cplx x[8];
    const int c = lane & 7;
    const double *Br = Qr + j0 * C::LD + j0, *Bi = Qi + j0 * C::LD + j0;
    // One instruction stream for both triangles (separate branches would run one after the other in this warp): lanes
    // 8-15 walk U backwards by mirroring the indices, rr = 7 - r, and scale by the reciprocal diagonal; lanes 0-7 walk L
    // forwards with a unit diagonal.
    const bool isU = lane >= 8;
    if (lane < 16) {
#pragma unroll
        for (int r = 0; r < 8; ++r) x[r] = {((isU ? 7 - r : r) == c) ? 1.0 : 0.0, 0.0};
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const cplx d = dinv[7 - r];
            if (isU) x[r] = cmul(x[r], d);
#pragma unroll
            for (int r2 = 0; r2 < 8; ++r2)
                if (r2 > r) {
                    const int off = isU ? (7 - r2) * C::LD + (7 - r) : r2 * C::LD + r;
                    const double er = Br[off], ei = Bi[off];
                    x[r2].r -= er * x[r].r - ei * x[r].i; x[r2].i -= er * x[r].i + ei * x[r].r;
                }
        }
    }
    __syncwarp();
    if (lane < 16) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int rr = isU ? 7 - r : r;
            if (isU ? rr <= c : rr > c) { Qr[(j0 + rr) * C::LD + j0 + c] = x[r].r; Qi[(j0 + rr) * C::LD + j0 + c] = x[r].i; }
        }
    }
    __syncwarp();
#ifdef QOCB_PROFILE
    if (blockIdx.x == 0 && threadIdx.x == 0) g_prof[16] += clock64() - pt0__;
#endif
}

// In-place blocked LU of Q (LUi format).  perm: shared int[NP]; piv8: shared int[8].  Ends with a barrier.
template <class C>
__device__ void lu_factor_blocked(double *Q, int *perm, int *piv8) {
    constexpr int NB = C::NP / 8;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < C::NP; i += C::NT) perm[i] = i;
    __syncthreads();
    PROF_DECL
    for (int kb = 0; kb < NB; ++kb) {
        const int j0 = kb * 8;
        if (warp == 0) lu_panel_warp<C>(Q, perm, piv8, j0);
        __syncthreads();
        PROF_MARK(14);
        for (int ct = warp; ct < NB; ct += C::NWARP) {
            if (ct == kb) continue;
            if (lane < 16) {                                       // the panel's row swaps on this column tile
                double *pl = Q + (lane >> 3) * C::PLANE;
                const int c = ct * 8 + (lane & 7);
                for (int j = 0; j < 8; ++j) {
                    const int p = piv8[j], r = j0 + j;
                    if (p != r) { const double t0 = pl[r * C::LD + c]; pl[r * C::LD + c] = pl[p * C::LD + c]; pl[p * C::LD + c] = t0; }
                }
            }
            __syncwarp();
            if (ct > kb) {
                c2 u = czero();                                    // U12 = inv(L11) A12
                tile_mma<C, false, MASK_LINV, false>(u, Q, j0, j0, Q, j0, ct * 8);
                __syncwarp();
                st_ctile<C>(Q, j0, ct * 8, u);
                __syncwarp();
                tile_update_rows<C, false>(Q, Q, kb, ct * 8, kb + 1, NB, 1);   // A22 -= L21 U12
            }
        }
        __syncthreads();
        PROF_MARK(15);
    }
}

// ---- inverse of the Pade denominator WITHOUT pivoting ----------------------------------------------------------------
// For an anti-Hermitian argument A = -i H dt (every physical GRAPE problem: H0 and the control operators are Hermitian)
// the Pade denominator Q = V - U is a polynomial of A with real coefficients: it is a normal matrix with eigenvalues
// q(i lam) = b0 e^{-i lam / 2} (1 + O(1e-10)) for the eigenvalues i lam of A, so its Hermitian part is b0 cos(lam / 2) > 0
// as long as |lam| <= ||A||_1 < pi.  A matrix with a positive definite Hermitian part can be eliminated without pivoting
// with bounded growth (Golub & Van Loan, sec. 4.2.2: every Schur complement keeps a positive definite Hermitian part), and
// over the range pade_forward admits here (Hermitian operators, ||A||_1 < 2.5, no squarings) the Pade-13 coefficients give
// 1 <= |q(i lam)| / b0 <= 1.032, i.e. cond_2(Q) <= 1.032.  An explicit inverse is then as accurate as a solve, and
// R0 = Q^-1 P is one dense product instead of two dependent block substitutions; the reverse passes apply Q^-T as a product
// too.  Everything else goes through the pivoted factorisation above.

// One warp: Gauss-Jordan inverse of an 8 x 8 tile held in the DMMA accumulator layout (lane (g, t): row g, columns 2t, 2t + 1),
// no pivoting.  Step j scales row j by 1 / a_jj and eliminates column j from every other row of [A | Z], Z = I at the start;
// the dependent chain per step is one pivot broadcast, the reciprocal (hardware seed + two Newton steps) and one complex
// multiply-add.  Columns of A that have been eliminated are not read again and are left as they come out.
__device__ __forceinline__ c2 shfl_c2(const c2 &v, int src) {
    constexpr unsigned FULL = 0xffffffffu;
    return {__shfl_sync(FULL, v.r0, src), __shfl_sync(FULL, v.r1, src), __shfl_sync(FULL, v.i0, src), __shfl_sync(FULL, v.i1, src)};
}
__device__ __forceinline__ c2 gj_tile_inverse(c2 a) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    c2 z = {g == 2 * t ? 1.0 : 0.0, g == 2 * t + 1 ? 1.0 : 0.0, 0., 0.};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int tj = j >> 1;
        const bool odd = (j & 1) != 0;
        const double sr = odd ? a.r1 : a.r0, si = odd ? a.i1 : a.i0;     // this lane's entry of column j
        const double pr = __shfl_sync(FULL, sr, 4 * j + tj), pi = __shfl_sync(FULL, si, 4 * j + tj);      // a_jj
        const double er = __shfl_sync(FULL, sr, 4 * g + tj), ei = __shfl_sync(FULL, si, 4 * g + tj);      // a_gj
        const c2 u = shfl_c2(a, 4 * j + t), w = shfl_c2(z, 4 * j + t);                                      // row j of A and Z
        const double nn = pr * pr + pi * pi;
        double dn;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(dn) : "d"(nn));
        dn = fma(dn, fma(-nn, dn, 1.0), dn);
        dn = fma(dn, fma(-nn, dn, 1.0), dn);
        const cplx inv = {pr * dn, -pi * dn};
        // row j: x <- x / a_jj; other rows: x <- x - (a_gj / a_jj) row_j
        const cplx l = g == j ? cplx{0., 0.} : cmul({er, ei}, inv);
        const double fr = g == j ? inv.r : -l.r, fi = g == j ? inv.i : -l.i;
        const c2 base_a = g == j ? czero() : a, base_z = g == j ? czero() : z;
        a = {base_a.r0 + fr * u.r0 - fi * u.i0, base_a.r1 + fr * u.r1 - fi * u.i1, base_a.i0 + fr * u.i0 + fi * u.r0, base_a.i1 + fr * u.i1 + fi * u.r1};
        z = {base_z.r0 + fr * w.r0 - fi * w.i0, base_z.r1 + fr * w.r1 - fi * w.i1, base_z.i0 + fr * w.i0 + fi * w.r0, base_z.i1 + fr * w.i1 + fi * w.r1};
    }
    return z;
}

// Q <- Q^-1 in place (W: scratch matrix of the same shape), block Gauss-Jordan on 8 x 8 tiles without pivoting.  Ends with
// a barrier.  Step kb, with D^-1 = inv(Q[kb, kb]) already in the diagonal slot of the source:
//     Q[kb, j] <- D^-1 Q[kb, j],   Q[i, j] <- Q[i, j] - Q[i, kb] Q[kb, j]  (new row kb),   Q[i, kb] <- -Q[i, kb] D^-1,
//     Q[kb, kb] <- D^-1                                                                      (i, j != kb).
// Warp j owns column tile j and writes it to the other buffer (source and destination alternate between Q and W), so a
// step reads the old column kb while its owner writes the new one and needs one block barrier.  Look-ahead: the owner of
// column kb + 1 updates its diagonal tile first and inverts it in registers, in the shadow of the other columns' updates.
// Every step has NB (NB - 1) independent tile products of the update and NB - 1 of the row and column panels.
template <class C>
__device__ void gj_invert_nopiv(double *Q, double *W) {
    constexpr int NB = C::NP / 8;
    static_assert(NB == 1 || NB <= C::NWARP, "one warp per column tile");
    static_assert(NB == 1 || NB % 2 == 0, "the inverse ends in Q after an even number of steps");
    const int warp = threadIdx.x >> 5;
    PROF_DECL
    if (warp == 0) st_ctile<C>(Q, 0, 0, gj_tile_inverse(ld_ctile<C>(Q, 0, 0)));
    __syncthreads();
    PROF_MARK(17);
    if constexpr (NB > 1) {
        const int j = warp, c0 = warp * 8;
        for (int kb = 0; kb < NB; ++kb) {
            const double *S = (kb & 1) ? W : Q;
            double *D = (kb & 1) ? Q : W;
            const int k0 = kb * 8;
            if (j < NB && j != kb) {
                c2 r = czero();                                    // new row kb: D^-1 Q[kb, j]
                tile_mma<C, false, MASK_NONE, false>(r, S, k0, k0, S, k0, c0);
                st_ctile<C>(D, k0, c0, r);
                __syncwarp();
                const bool ahead = j == kb + 1;
                if (ahead) {                                       // the next diagonal tile first, then its inverse
                    c2 v = ld_ctile<C>(S, c0, c0);
                    tile_mma<C, false, MASK_NONE, true>(v, S, c0, k0, D, k0, c0);
                    st_ctile<C>(D, c0, c0, gj_tile_inverse(v));
                }
                c2 v[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i) v[i] = ld_ctile<C>(S, i * 8, c0);
#pragma unroll
                for (int i = 0; i < NB; ++i)
                    if (i != kb && !(ahead && i == j)) tile_mma<C, false, MASK_NONE, true>(v[i], S, i * 8, k0, D, k0, c0);
#pragma unroll
                for (int i = 0; i < NB; ++i)
                    if (i != kb && !(ahead && i == j)) st_ctile<C>(D, i * 8, c0, v[i]);
            } else if (j == kb) {                                  // new column kb: -Q[i, kb] D^-1, and D^-1 itself
                c2 v[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    v[i] = czero();
                    if (i != kb) tile_mma<C, false, MASK_NONE, true>(v[i], S, i * 8, k0, S, k0, k0);
                    else v[i] = ld_ctile<C>(S, k0, k0);
                }
#pragma unroll
                for (int i = 0; i < NB; ++i) st_ctile<C>(D, i * 8, c0, v[i]);
            }
            __syncthreads();
            PROF_MARK(18);
        }
    }
}

// X <- Q^{-1} B (TRANS = false) or Q^{-T} B (TRANS = true); LU in LUi format.  B is read from `B`, the result is
// written to `X` (B != X: the row permutation is applied out of place).  Both end with a barrier.
struct NoHook { __device__ __forceinline__ void operator()() const {} };

// `b_free` is called by every thread once B is no longer read (TRANS = false: right after the row permutation has been
// applied out of place) - k_forward uses it to start an asynchronous fetch into that buffer
template <class C, bool TRANS, class Hook = NoHook>
__device__ void lu_solve_blocked(const double *LU, const int *perm, double *B, double *X, Hook b_free = Hook()) {
    constexpr int NB = C::NP / 8;
    const int warp = threadIdx.x >> 5;
    double *W = TRANS ? B : X;                                     // the substitutions run in place on W
    if (!TRANS) {                                                  // X[i] = B[perm[i]]
        for (int idx = threadIdx.x; idx < 2 * C::NP * (C::NP / 2); idx += C::NT) {
            const int plane = idx / (C::NP * (C::NP / 2)), rem = idx % (C::NP * (C::NP / 2));
            const int row = rem / (C::NP / 2), cc = rem % (C::NP / 2);
            *reinterpret_cast<double2 *>(X + plane * C::PLANE + row * C::LD + 2 * cc) =
                *reinterpret_cast<const double2 *>(B + plane * C::PLANE + perm[row] * C::LD + 2 * cc);
        }
        __syncthreads();
        b_free();
    }
    for (int ct = warp; ct < NB; ct += C::NWARP) {
        const int c0 = ct * 8;
        if (!TRANS) {
            for (int kb = 0; kb < NB; ++kb) {                      // L z = b
                c2 z = czero();
                tile_mma<C, false, MASK_LINV, false>(z, LU, kb * 8, kb * 8, W, kb * 8, c0);
                __syncwarp();
                st_ctile<C>(W, kb * 8, c0, z);
                __syncwarp();
                tile_update_rows<C, false>(LU, W, kb, c0, kb + 1, NB, 1);
                __syncwarp();
            }
            for (int kb = NB - 1; kb >= 0; --kb) {                 // U x = z
                c2 z = czero();
                tile_mma<C, false, MASK_UINV, false>(z, LU, kb * 8, kb * 8, W, kb * 8, c0);
                __syncwarp();
                st_ctile<C>(W, kb * 8, c0, z);
                __syncwarp();
                tile_update_rows<C, false>(LU, W, kb, c0, 0, kb, 1);
                __syncwarp();
            }
        } else {
            for (int kb = 0; kb < NB; ++kb) {                      // U^T y = b
                c2 z = czero();
                tile_mma<C, true, MASK_UINV, false>(z, LU, kb * 8, kb * 8, W, kb * 8, c0);
                __syncwarp();
                st_ctile<C>(W, kb * 8, c0, z);
                __syncwarp();
                tile_update_rows<C, true>(LU, W, kb, c0, kb + 1, NB, 1);
                __syncwarp();
            }
            for (int kb = NB - 1; kb >= 0; --kb) {                 // L^T z = y
                c2 z = czero();
                tile_mma<C, true, MASK_LINV, false>(z, LU, kb * 8, kb * 8, W, kb * 8, c0);
                __syncwarp();
                st_ctile<C>(W, kb * 8, c0, z);
                __syncwarp();
                tile_update_rows<C, true>(LU, W, kb, c0, 0, kb, 1);
                __syncwarp();
            }
        }
    }
    __syncthreads();
    if (TRANS) {                                                   // X[perm[i]] = W[i]
        for (int idx = threadIdx.x; idx < 2 * C::NP * (C::NP / 2); idx += C::NT) {
            const int plane = idx / (C::NP * (C::NP / 2)), rem = idx % (C::NP * (C::NP / 2));
            const int row = rem / (C::NP / 2), cc = rem % (C::NP / 2);
            *reinterpret_cast<double2 *>(X + plane * C::PLANE + perm[row] * C::LD + 2 * cc) =
                *reinterpret_cast<const double2 *>(W + plane * C::PLANE + row * C::LD + 2 * cc);
        }
        __syncthreads();
    }
}

// block-wide sum of NV doubles per thread -> result valid in all threads; red needs NV * NWARP doubles
template <class C, int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double *__restrict__ red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    }
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int q = 0; q < NV; ++q) red[q * C::NWARP + warp] = v[q];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        double s = 0.;
        for (int w = 0; w < C::NWARP; ++w) s += red[q * C::NWARP + w];
        v[q] = s;
    }
}

}  // namespace qocb
