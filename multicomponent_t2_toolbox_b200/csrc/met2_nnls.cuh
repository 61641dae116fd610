// met2_nnls.cuh — warp-per-voxel Lawson-Hanson NNLS in the Gram domain (FP64, sm_100a).
//
// Takes over scipy's Lawson-Hanson routine reached from intravoxel_algorithms/algorithms.py:55-82 (nnls) and, with the
// Tikhonov term, algorithms.py:262-269 (A = [D; sqrt(lambda) L]).  Same pivot rule and control flow as nnls.f:
//   outer: w = A^T(b - A x); j = argmax_{j in Z} w_j (first max), stop if w_j <= 0; accept j unless the column is
//          numerically dependent on the positive set or its new coefficient is <= 0 (then w_j := 0 and re-pick);
//   inner: iter++ (stop at itmax = 3n, current x kept); if all z_P > 0 leave; alpha = min_{z_i<=0} x_i/(x_i - z_i)
//          (first min); x += alpha (z - x); move the blocking index and every x_i <= 0 out of P; re-solve.
// What differs is the arithmetic: instead of Householder/Givens on the m x n matrix we keep, per warp, the inverse
// Cholesky factor T (upper triangular, packed) of the positive-set Gram matrix, (G + lambda K)_PP^-1 = T T^T:
//   append column j :  r = T^T g_Pj ; rho^2 = G_jj - r.r ; new column of T = [-T r ; 1] / rho ; y_new = (c_j - r.y)/rho
//   remove position k: Givens rotations on column pairs of T that empty row k (parameters from a prefix sum of squares)
//   solve            : z = T y   with y = T^T c_P
// Every step is a (triangular) matrix-vector product spread over the 32 lanes; no serial substitution chains.
// Measured against SciPy on the design prototype (tools/proto_gram_nnls2.py): identical supports, <= 1e-9 relative.
//
// Memory: all per-warp state lives in the kernel's dynamic shared memory and is addressed as S[offset] (32-bit
// shared-window addressing, LDS/STS); round-1 profiling of a pointer-based version showed generic LD.E + R2UR and
// local-memory reloads dominating the issue slots (profiles/r01_t2_fit_v1_ncu_summary.txt).
#pragma once
#ifdef MET2_HOST_EMU
#include "simt_emu.h"   // tests/emu: CPU emulation of the device code for the "not gpu" tests; never part of libmet2.so
#else
#include <cuda_runtime.h>
#endif
#include <stdint.h>

namespace met2 {

#ifdef MET2_HOST_EMU
static simt::Shared& S = simt::g_shared;
// decision trace of the active-set solver for the CPU emulation build (MET2_EMU_TRACE=1); compiles to nothing in CUDA
#define MET2_TRACE(lane, ...)                                              \
    do {                                                                   \
        if ((lane) == 0 && getenv("MET2_EMU_TRACE")) fprintf(stderr, __VA_ARGS__); \
    } while (0)
#else
#define MET2_TRACE(lane, ...) \
    do {                      \
    } while (0)
extern __shared__ __align__(16) double S[];   // the dynamic shared memory of every met2 kernel
#endif

constexpr unsigned FULL_MASK = 0xffffffffu;

// Unroll factor of the runtime-trip mat-vec loops.  The kernels with ten or more resident warps per SM (nT2 <= 64) and
// the 16-warp FA search are bound by instruction fetch — compact loops measured faster
// (profiles/r01_t2_fit_v8_ncu_summary.txt).  A translation unit whose kernels run with three or four warps per SM
// (T2SPARC's 96 T2 bins) has nothing to hide latency with but instruction-level parallelism and may ask for unrolled
// loops from NS = MET2_UNROLL_WIDE_NS on (measured: T2SPARC 319 -> 281 ms per volume; the same switch slowed the FA
// search down, 138 -> 250 ms, which is why it is per translation unit).
#ifndef MET2_UNROLL_WIDE_NS
#define MET2_UNROLL_WIDE_NS 99
#endif
template <int NS>
struct Unroll {
    static constexpr int v = (NS >= MET2_UNROLL_WIDE_NS) ? 4 : 1;
};

__host__ __device__ constexpr __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }

__host__ __device__ __forceinline__ size_t align_up256(size_t x) { return (x + 255) & ~(size_t)255; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

__device__ __forceinline__ void warp_sum2(double& a, double& b) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ta = __shfl_xor_sync(FULL_MASK, a, o);
        double tb = __shfl_xor_sync(FULL_MASK, b, o);
        a += ta;
        b += tb;
    }
}

// Index of the largest strictly positive value over the warp (lowest index on ties); -1 if no lane has v > 0.
// Positive doubles order like their bit patterns, so two 32-bit REDUX max passes find the maximum.
__device__ __forceinline__ int warp_argmax_pos(double v, int index) {
    unsigned long long key = (v > 0.0) ? (unsigned long long)__double_as_longlong(v) : 0ull;
    unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
    unsigned mhi = __reduce_max_sync(FULL_MASK, hi);
    unsigned mlo = __reduce_max_sync(FULL_MASK, (hi == mhi) ? lo : 0u);
    if ((mhi | mlo) == 0u) return -1;
    bool win = (key != 0ull) && (hi == mhi) && (lo == mlo);
    return (int)__reduce_min_sync(FULL_MASK, win ? (unsigned)index : 0xffffffffu);
}

// Index of the smallest value among lanes with index >= 0 and v >= 0 (lowest index on ties); -1 if none.
__device__ __forceinline__ int warp_argmin_nonneg(double v, int index, double& vmin) {
    bool valid = (index >= 0) && (v >= 0.0) && (v < 1.0e308);
    unsigned long long key = valid ? (unsigned long long)__double_as_longlong(v + 0.0) : ~0ull;
    unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
    unsigned mhi = __reduce_min_sync(FULL_MASK, hi);
    unsigned mlo = __reduce_min_sync(FULL_MASK, (hi == mhi) ? lo : 0xffffffffu);
    if (mhi == 0xffffffffu && mlo == 0xffffffffu) return -1;
    bool win = valid && (hi == mhi) && (lo == mlo);
    unsigned best = __reduce_min_sync(FULL_MASK, win ? (unsigned)index : 0xffffffffu);
    vmin = __longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo));
    return (int)best;
}

// Per-warp workspace as offsets (in doubles) into S.  NS = slots per lane; vectors have LEN = 32*NS entries.
//   T  : packed upper triangular, column-major: T(k, i) at S[T + tri(i) + k], k <= i < pmax
//   gs : position-space scratch (gathered Gram column / c_P / rotation cosines)
//   rs : position-space scratch (r, y / rotation sines)
//   xs : current feasible x in position space
//   cc : c = A^T b in column space
//   xc : x in column space (zeros outside P)
//   ix : position -> column (ints, stored in the space of LEN/2 doubles)
//   aux: two doubles after ix — [0] the pointer to the transposed dictionary [n][m] of the solve in flight (global
//        memory), [1] (as int) the offset of its right-hand side in S; read only by the rare D-space evaluation of a
//        nearly dependent candidate (dspace_candidate), kept here rather than in registers (see set_dspace)
// The two entries of the augmented 8 x 16 block [S | I] that lane `lane` owns in ldl_8x8 (entry e = lane + 32 sl:
// e < 36 -> (r, c) of the upper triangle of S, row-major; e >= 36 -> (r, 8 + c') with c' < r, the strictly-lower part
// of the inverse factor), packed as bytes r0 | c0 << 8 | r1 << 16 | c1 << 24.  Depends on the lane only: computed once
// per kernel (Slots::carve) — recomputed inside every elimination it was 9 % of the 96-register X2 kernel.
__device__ __forceinline__ unsigned ldl_lane_code(int lane) {
    unsigned code = 0u;
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
        const int e = lane + 32 * sl;
        int rr, cc;
        if (e < 36) {
            rr = 0;
            int rem = e;
#pragma unroll
            for (int t = 0; t < 7; ++t)
                if (rem >= 8 - rr) {
                    rem -= 8 - rr;
                    ++rr;
                }
            cc = rr + rem;
        } else {
            const int f = e - 36;
            rr = 1;
#pragma unroll
            for (int t = 0; t < 6; ++t)
                if (f >= (rr * (rr + 1)) / 2) ++rr;
            cc = 8 + f - (rr * (rr - 1)) / 2;
        }
        code |= ((unsigned)rr | ((unsigned)cc << 8)) << (16 * sl);
    }
    return code;
}

template <int NS>
struct Slots {
    int T, gs, rs, xs, cc, xc, ix;
    unsigned code;   // ldl_lane_code of this lane
    static constexpr int LEN = 32 * NS;
    __host__ __device__ static int doubles(int pmax) { return tri(pmax) + 5 * LEN + LEN / 2 + 2; }
    __device__ __forceinline__ void carve(int base, int pmax) {
        T = base;
        gs = T + tri(pmax);
        rs = gs + LEN;
        xs = rs + LEN;
        cc = xs + LEN;
        xc = cc + LEN;
        ix = xc + LEN;
        code = ldl_lane_code((int)(threadIdx.x & 31));
    }
    __device__ __forceinline__ int aux() const { return ix + LEN / 2; }
};

__device__ __forceinline__ int& SI(int off, int k) { return reinterpret_cast<int*>(S + off)[k]; }

// Tell the plain solves of this warp where the transposed dictionary [n][m] (global memory) and the right-hand side
// (offset in S) are, for the D-space evaluation of nearly dependent candidates.  Dt = nullptr switches it off.
// Two shared-memory words per warp instead of three kernel-lifetime registers per thread: with the pointer as an
// argument of nnls_gram the 80-register FA select kernel spilled (FA stage +6 %).
template <int NS>
__device__ __forceinline__ void set_dspace(const Slots<NS>& W, const double* Dt, int oM, int lane) {
    if (lane == 0) {
        *reinterpret_cast<const double**>(S + W.aux()) = Dt;
        SI(W.aux() + 1, 0) = oM;
    }
    __syncwarp();
}

// Column space: lane owns columns NS*lane + s (s < NS) so that its NS values are contiguous (128-bit LDS for NS = 2, 4).
// Position space: lane owns positions lane + 32 t, so that sets with p <= 32 only touch slot 0.
template <int NS>
__device__ __forceinline__ int colof(int lane, int s) { return NS * lane + s; }

// NS contiguous doubles from shared memory at S[off .. off+NS); off must be even when NS is even.
template <int NS>
__device__ __forceinline__ void lds_vec(int off, double (&v)[NS]) {
    if constexpr (NS == 2) {
        double2 t = *reinterpret_cast<const double2*>(S + off);
        v[0] = t.x; v[1] = t.y;
    } else if constexpr (NS == 4) {
        double2 t = *reinterpret_cast<const double2*>(S + off);
        double2 u = *reinterpret_cast<const double2*>(S + off + 2);
        v[0] = t.x; v[1] = t.y; v[2] = u.x; v[3] = u.y;
    } else {
#pragma unroll
        for (int s = 0; s < NS; ++s) v[s] = S[off + s];
    }
}

// NS contiguous doubles from global memory (read-only path); p must be 16-byte aligned when `vec` is set.
template <int NS>
__device__ __forceinline__ void ldg_vec(const double* __restrict__ p, bool vec, int nvalid, double (&v)[NS]) {
    if ((NS == 2 || NS == 4) && vec && nvalid >= NS) {
#pragma unroll
        for (int s = 0; s < NS; s += 2) {
            double2 t = __ldg(reinterpret_cast<const double2*>(p + s));
            v[s] = t.x;
            v[s + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int s = 0; s < NS; ++s) v[s] = (s < nvalid) ? __ldg(p + s) : 0.0;
    }
}

// out[t] (position i = lane + 32 t) = sum_{k <= i, k < p} T(k, i) * v[k]   — column dot products, T^T v.
// Two accumulators per slot for ILP; the triangle predicate is a single compare against kmax[t] (= i for live
// positions, -1 otherwise) so it compiles to predication.  Kept deliberately compact: this kernel is bound by
// instruction fetch (6 KB L0 / 32 KB L1.5 instruction caches), smaller code measured faster than more unrolling.
template <int NS>
__device__ __forceinline__ void tmul_transposed(int oT, int oV, int p, int lane, double (&out)[NS]) {
    double a0[NS], a1[NS];
    int base[NS], kmax[NS];
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        a0[t] = a1[t] = 0.0;
        base[t] = oT + tri(i);
        kmax[t] = (i < p) ? i : -1;
    }
    int k = 0;
#pragma unroll (Unroll<NS>::v)
    for (; k + 1 < p; k += 2) {
        const double v0 = S[oV + k], v1 = S[oV + k + 1];
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            if (32 * t + 31 >= k) {   // uniform: slot t only holds positions <= 32 t + 31
                const double t0 = (k <= kmax[t]) ? S[base[t] + k] : 0.0;
                const double t1 = (k + 1 <= kmax[t]) ? S[base[t] + k + 1] : 0.0;
                a0[t] = fma(t0, v0, a0[t]);
                a1[t] = fma(t1, v1, a1[t]);
            }
        }
    }
    if (k < p) {
        const double v0 = S[oV + k];
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            const double t0 = (k <= kmax[t]) ? S[base[t] + k] : 0.0;
            a0[t] = fma(t0, v0, a0[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < NS; ++t) out[t] = a0[t] + a1[t];
}

// out[t] (position k = lane + 32 t) = sum_{i >= k, i < p} T(k, i) * v[i]   — row dot products, T v.
template <int NS>
__device__ __forceinline__ void tmul(int oT, int oV, int p, int lane, double (&out)[NS]) {
    double a0[NS], a1[NS];
#pragma unroll
    for (int t = 0; t < NS; ++t) a0[t] = a1[t] = 0.0;
    int i = 0;
    int t0 = oT;
#pragma unroll (Unroll<NS>::v)
    for (; i + 1 < p; i += 2) {
        const double v0 = S[oV + i], v1 = S[oV + i + 1];
        const int t1 = t0 + i + 1;
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            if (32 * t <= i + 1) {   // uniform: slot t only holds rows >= 32 t
                const int k = lane + 32 * t;
                const double e0 = (k <= i) ? S[t0 + k] : 0.0;
                const double e1 = (k <= i + 1) ? S[t1 + k] : 0.0;
                a0[t] = fma(e0, v0, a0[t]);
                a1[t] = fma(e1, v1, a1[t]);
            }
        }
        t0 = t1 + i + 2;
    }
    if (i < p) {
        const double v0 = S[oV + i];
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            const int k = lane + 32 * t;
            const double e0 = (k <= i) ? S[t0 + k] : 0.0;
            a0[t] = fma(e0, v0, a0[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < NS; ++t) out[t] = a0[t] + a1[t];
}

// 1/sqrt(d) from the single-precision hardware estimate plus two Newton steps in double (relative error ~1e-16); the
// library rsqrt() costs ~3x the instructions and sits on the serial pivot chain of every factorisation step.
__device__ __forceinline__ double rsqrt_fast(double d) {
    if (!(d > 1e-30 && d < 1e30)) return rsqrt(d);
    double r = (double)rsqrtf((float)d);
    double e = fma(-d * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    e = fma(-d * r, r, 1.0);
    r = fma(0.5 * r, e, r);
    return r;
}

// 1/d from the single-precision hardware reciprocal plus two Newton steps in double (relative error ~1e-16).
__device__ __forceinline__ double rcp_fast(double d) {
    if (!(d > 1e-30 && d < 1e30)) return 1.0 / d;
    double r = (double)__frcp_rn((float)d);
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// FP64 tensor-core MMA m8n8k4 (DMMA.8x8x4 on sm_100a): D(8x8) += A(8x4) B(4x8).  Fragments: A[lane/4][lane%4],
// B[lane%4][lane/4], C/D[lane/4][2*(lane%4) + {0,1}] (verified on B200 by tools/dmma_probe.cu; 16 cycles issue interval,
// 26 cycles dependent latency).
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
#ifdef MET2_HOST_EMU
    emu_dmma884(d0, d1, a, b);
#else
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
#endif
}

// Symmetric Gaussian elimination on the augmented 8 x 8 block [S | I] held as accumulator fragments (s0, s1) =
// S[g][2q], S[g][2q + 1] (g = lane / 4, q = lane % 4): afterwards the 8 x 16 array FR = S[W.gs .. W.gs + 128) (row stride
// 16; spans gs and, for NS = 2, rs) holds D L1^T in its left half (S = L1 D L1^T, pivots d_r = FR[17 r]) and M = L1^-1 in
// its right half, so that chol(S) = R = D^1/2 L1^T (R[r][c] = FR[16 r + c] / sqrt(d_r), c >= r) and
// R^-1[r][c] = M[c][r] / sqrt(d_c) = FR[16 c + 8 + r] / sqrt(d_c) for r < c, 1 / sqrt(d_c) on the diagonal.
// The 36 upper-triangular entries of the left half and the 28 strictly-lower entries of M are exactly two per lane and
// stay in REGISTERS; a row is published to FR once, when it becomes the pivot row.  One __syncwarp and one fast
// reciprocal per step on the dependency chain.  nv = live rows (the rest are virtual identity rows of a partial block).
// (First version: an 8-step Cholesky with three barriers per step plus a serial triangular inverse on 8 lanes, ~20 % of
// the kernel's stall samples in profiles/r01_t2_fit_v8_ncu_summary.txt; second: the same elimination with every entry
// updated in shared memory, 16 % of the executed instructions in the v11 capture.)
template <int NS>
__device__ __forceinline__ void ldl_8x8(const Slots<NS>& W, double s0, double s1, int nv, int lane, bool& ok) {
    const int g = lane >> 2, q = lane & 3;
    const int oFR = W.gs;
    S[oFR + g * 16 + 2 * q] = s0;
    S[oFR + g * 16 + 2 * q + 1] = s1;
    S[oFR + g * 16 + 8 + 2 * q] = (2 * q == g) ? 1.0 : 0.0;
    S[oFR + g * 16 + 8 + 2 * q + 1] = (2 * q + 1 == g) ? 1.0 : 0.0;
    __syncwarp();
    // entry e = lane + 32 s: e < 36 -> (r, c) of the upper triangle, row-major; e >= 36 -> (r, 8 + c') with c' < r
    int er[2], ec[2];
    double ev[2];
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
        er[sl] = (int)((W.code >> (16 * sl)) & 0xffu);
        ec[sl] = (int)((W.code >> (16 * sl + 8)) & 0xffu);
        ev[sl] = S[oFR + er[sl] * 16 + ec[sl]];
    }
#pragma unroll 1
    for (int k = 0; k < nv - 1; ++k) {
        const double d = S[oFR + k * 17];
        if (!(d > 0.0)) ok = false;
        const double inv = rcp_fast(d);
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
            if (er[sl] > k && (ec[sl] < 8 || ec[sl] - 8 <= k)) {
                const double m = S[oFR + k * 16 + er[sl]] * inv;
                ev[sl] = fma(-m, S[oFR + k * 16 + ec[sl]], ev[sl]);
            }
        }
        // row k+1 is final now: publish it (this step only read row k, so one barrier per step is enough)
#pragma unroll
        for (int sl = 0; sl < 2; ++sl)
            if (er[sl] == k + 1) S[oFR + er[sl] * 16 + ec[sl]] = ev[sl];
        __syncwarp();
    }
    if (!(S[oFR + (nv - 1) * 17] > 0.0)) ok = false;
}

// Blocked rebuild of the inverse Cholesky factor T for a GIVEN positive set (warm start): A = (G + lam K)_PP = R^T R,
// T = R^-1, processed in column blocks J of 8 with the 8x8x4 FP64 MMA:
//     R_top = T_old^T A[P_old, J]           (tiles of 8 rows; staged where the new columns of T will live)
//     S     = A[J, J] - R_top^T R_top       (8 x 8)
//     T_JJ  = chol(S)^-1                    (8 x 8, unblocked in a 64-double scratch)
//     T[:, J] = [ -(T_old R_top) T_JJ ; T_JJ ]
// Same arithmetic class as the column-by-column append (blocked Cholesky + triangular inverse) at ~1/6 of the issued
// instructions: one DMMA replaces 8 DFMA plus the shared-memory loads that feed them.
// Aent(kpos, jpos) returns the matrix entry for positions (kpos, jpos) < p.  Returns false if a pivot is not positive.
template <int NS, class AENT>
__device__ __forceinline__ bool rebuild_T_blocked(const Slots<NS>& W, AENT&& Aent, int p, int lane) {
    const int oT = W.T;
    const int g = lane >> 2, q = lane & 3;
    const int nb = (p + 7) >> 3;
    bool ok = true;
#pragma unroll 1
    for (int b = 0; b < nb; ++b) {
        const int c0 = 8 * b;                       // first column of the block = size of the set already factored
        const int jg = c0 + g;                      // this lane's B-fragment column
        const int colg = oT + tri(jg);              // ... and where that column of T lives (staging area)
        const bool jlive = jg < p;
        const int ca = c0 + 2 * q, cb = ca + 1;     // this lane's accumulator columns
        const int cola = oT + tri(ca), colb = oT + tri(cb);
        if (b > 0) {
            // ---- stage A[P_old, J] where the new columns of T will live: entry (k, j) at tri(c0 + j) + k
#pragma unroll 1
            for (int e = lane; e < 8 * c0; e += 32) {
                const int kk = e >> 3, j = c0 + (e & 7);
                if (j < p) S[oT + tri(j) + kk] = Aent(kk, j);
            }
            __syncwarp();
            // ---- R_top = T_old^T A[P_old, J], 8-row tiles in DESCENDING order so that a tile may overwrite its rows
#pragma unroll 1
            for (int it = b - 1; it >= 0; --it) {
                const int ii = 8 * it + g;
                const int coli = oT + tri(ii);
                double d0 = 0.0, d1 = 0.0;
#pragma unroll 1
                for (int ks = 0; ks < 2 * it + 2; ++ks) {
                    const int kk = 4 * ks + q;
                    const double af = (kk <= ii) ? S[coli + kk] : 0.0;
                    const double bf = jlive ? S[colg + kk] : 0.0;
                    dmma884(d0, d1, af, bf);
                }
                __syncwarp();
                if (ca < p) S[cola + ii] = d0;
                if (cb < p) S[colb + ii] = d1;
            }
            __syncwarp();
        }
        // ---- S = A_JJ - R_top^T R_top (virtual rows/columns beyond p are the identity)
        double s0, s1;
        {
            const int r = c0 + g;
            s0 = (r < p && ca < p) ? Aent(r, ca) : ((r == ca) ? 1.0 : 0.0);
            s1 = (r < p && cb < p) ? Aent(r, cb) : ((r == cb) ? 1.0 : 0.0);
        }
#pragma unroll 1
        for (int is = 0; is < 2 * b; ++is) {
            const double v = jlive ? S[colg + 4 * is + q] : 0.0;
            dmma884(s0, s1, -v, v);
        }
        // ---- T_JJ = chol(S)^-1 by symmetric Gaussian elimination on the augmented block [S | I]: after the steps the
        //      left half holds D L1^T (S = L1 D L1^T) and the right half M = L1^-1, so R = D^1/2 L1^T and
        //      T_JJ[r][c] = M[c][r] / sqrt(d_c) for r <= c.  The 36 upper-triangular entries of the left half and the 28
        //      strictly-lower entries of M are exactly two per lane and stay in REGISTERS; a row is published to the
        //      8 x 16 array FR (S[W.gs .. W.gs + 128), spanning gs and rs) once, when it becomes the pivot row.  One
        //      __syncwarp and one fast reciprocal per step on the dependency chain.  (First version: an 8-step Cholesky
        //      with three barriers per step plus a serial triangular inverse on 8 lanes, ~20 % of the kernel's stall
        //      samples in profiles/r01_t2_fit_v8_ncu_summary.txt; second: the same elimination with every entry updated
        //      in shared memory, 16 % of the executed instructions in the v11 capture.)
        {
            const int oFR = W.gs;
            // rows beyond the set (virtual identity rows of a partial last block) need no elimination
            const int nv = (p - c0 < 8) ? (p - c0) : 8;
            ldl_8x8<NS>(W, s0, s1, nv, lane, ok);
            // T_JJ (row-major 8 x 8) -> S[W.rs ..]; FR overlaps rs, so gather into registers first
            const int c = lane & 7;
            const double ric = rsqrt_fast(S[oFR + c * 17]);
            double tv[2];
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {
                const int rr = pass * 4 + (lane >> 3);
                tv[pass] = (rr < c) ? S[oFR + c * 16 + 8 + rr] * ric : ((rr == c) ? ric : 0.0);
            }
            __syncwarp();
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) S[W.rs + (pass * 4 + (lane >> 3)) * 8 + c] = tv[pass];
        }
        __syncwarp();
        if (b > 0) {
            // ---- U = T_old R_top, tiles in ASCENDING order (tile kt only needs rows >= 8 kt of R_top), then
            //      new columns = -(U T_JJ) for the same tile
            const double tj0 = S[W.rs + q * 8 + g], tj1 = S[W.rs + (4 + q) * 8 + g];   // T_JJ B-fragments
#pragma unroll 1
            for (int kt = 0; kt < b; ++kt) {
                const int kk = 8 * kt + g;
                double d0 = 0.0, d1 = 0.0;
#pragma unroll 1
                for (int is = 2 * kt; is < 2 * b; ++is) {
                    const int i2 = 4 * is + q;
                    const double af = (kk <= i2) ? S[oT + tri(i2) + kk] : 0.0;
                    const double bf = jlive ? S[colg + i2] : 0.0;
                    dmma884(d0, d1, af, bf);
                }
                __syncwarp();   // rows 8kt..8kt+7 of R_top are no longer needed by anyone
                if (ca < p) S[cola + kk] = d0;
                if (cb < p) S[colb + kk] = d1;
                __syncwarp();
                double e0 = 0.0, e1 = 0.0;
                {
                    const int jp0 = c0 + q, jp1 = c0 + 4 + q;
                    const double a0 = (jp0 < p) ? S[oT + tri(jp0) + kk] : 0.0;
                    const double a1 = (jp1 < p) ? S[oT + tri(jp1) + kk] : 0.0;
                    dmma884(e0, e1, a0, tj0);
                    dmma884(e0, e1, a1, tj1);
                }
                __syncwarp();
                if (ca < p) S[cola + kk] = -e0;
                if (cb < p) S[colb + kk] = -e1;
            }
        }
        // ---- diagonal block: T[c0 + r][c0 + c] = T_JJ[r][c] for r <= c (two entries per lane)
#pragma unroll
        for (int pass = 0; pass < 2; ++pass) {
            const int rr = pass * 4 + (lane >> 3), c = lane & 7;
            if (rr <= c && c0 + c < p) S[oT + tri(c0 + c) + c0 + rr] = S[W.rs + rr * 8 + c];
        }
        __syncwarp();
    }
    return ok;
}

// Blocked Cholesky factorisation A = U^T U of the n x n matrix Aent(r, c) (natural order, all n columns): U upper
// triangular, packed column-major in the T region (U(k, j) at S[W.T + tri(j) + k], k <= j), by block rows of 8 on the
// FP64 tensor cores (up-looking):
//     W_IJ = A_IJ - sum_{K < I} U_KI^T U_KJ        (J >= I; DMMA 8x8x4, two block columns in flight)
//     U_II = chol(W_II), Tinv = U_II^-1             (ldl_8x8: elimination on [W_II | I])
//     U_IJ = Tinv^T W_IJ                            (J > I; W_IJ staged at U_IJ's own place)
// This is the factor the BayesReg evidence needs (bayesian_interpolation.py:113-119: U = cholesky(A), log prod diag U,
// U f): round 1 took it from the INVERSE factor (U f = T^T (A f), log det = -sum log T_kk), which costs 1.5x the
// flops and loses sqrt(cond A) ~ 1e4 ulps in the small entries of U f — enough, on the flat evidence curve of
// BayesReg + InvT2, to move Brent's lambda by more than the reference moves under a 1e-13 perturbation of its input
// (DESIGN.md §5).  Rows / columns >= n of the last block are virtual identity rows.  Returns false if a pivot is not
// positive.  Uses S[W.gs .. W.gs + 128) and S[W.rs .. W.rs + 64) as scratch.
template <int NS, class AENT>
__device__ __forceinline__ bool chol_upper_blocked(const Slots<NS>& W, AENT&& Aent, int n, int lane) {
    const int oT = W.T;
    const int g = lane >> 2, q = lane & 3;
    const int nb = (n + 7) >> 3;
    bool ok = true;
#pragma unroll 1
    for (int I = 0; I < nb; ++I) {
        const int r0 = 8 * I;
        const int rg = r0 + g;                      // accumulator row / column of U^T read as the A fragment
        const bool rlive = rg < n;
        const int colrg = oT + tri(rg);
        // ---- diagonal block: W_II = A_II - sum_K U_KI^T U_KI, then U_II and Tinv = U_II^-1
        {
            const int ca = r0 + 2 * q, cb = ca + 1;
            double s0 = (rlive && ca < n) ? Aent(rg, ca) : ((rg == ca) ? 1.0 : 0.0);
            double s1 = (rlive && cb < n) ? Aent(rg, cb) : ((rg == cb) ? 1.0 : 0.0);
#pragma unroll 1
            for (int ks = 0; ks < 2 * I; ++ks) {
                const double v = rlive ? S[colrg + 4 * ks + q] : 0.0;
                dmma884(s0, s1, -v, v);
            }
            const int nv = (n - r0 < 8) ? (n - r0) : 8;
            ldl_8x8<NS>(W, s0, s1, nv, lane, ok);
            const int oFR = W.gs;
            const int c = lane & 7;
            const double ric = rsqrt_fast(S[oFR + c * 17]);
            double tv[2], uv[2];
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {
                const int rr = pass * 4 + (lane >> 3);
                tv[pass] = (rr < c) ? S[oFR + c * 16 + 8 + rr] * ric : ((rr == c) ? ric : 0.0);      // Tinv[rr][c]
                uv[pass] = (rr <= c) ? S[oFR + rr * 16 + c] * rsqrt_fast(S[oFR + rr * 17]) : 0.0;     // U_II[rr][c]
            }
            __syncwarp();
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {
                const int rr = pass * 4 + (lane >> 3);
                S[W.rs + rr * 8 + c] = tv[pass];
                if (rr <= c && r0 + c < n) S[oT + tri(r0 + c) + r0 + rr] = uv[pass];
            }
            __syncwarp();
        }
        // ---- block row: U_IJ for J > I, two block columns at a time (independent accumulators hide the DMMA latency)
        const double ti0 = S[W.rs + q * 8 + g], ti1 = S[W.rs + (4 + q) * 8 + g];   // A fragments of Tinv^T: Tinv[k][g]
#pragma unroll 1
        for (int J = I + 1; J < nb; J += 2) {
            double d0[2], d1[2];
            int colg[2], cola[2], colb[2];
            bool glive[2], alive[2], blive[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int c0 = 8 * (J + h);
                const bool on = (J + h) < nb;
                glive[h] = on && (c0 + g < n);
                alive[h] = on && (c0 + 2 * q < n);
                blive[h] = on && (c0 + 2 * q + 1 < n);
                colg[h] = oT + tri(c0 + g);
                cola[h] = oT + tri(c0 + 2 * q);
                colb[h] = oT + tri(c0 + 2 * q + 1);
                d0[h] = (rlive && alive[h]) ? Aent(rg, c0 + 2 * q) : 0.0;
                d1[h] = (rlive && blive[h]) ? Aent(rg, c0 + 2 * q + 1) : 0.0;
            }
#pragma unroll 1
            for (int ks = 0; ks < 2 * I; ++ks) {
                const int kk = 4 * ks + q;
                const double a = rlive ? -S[colrg + kk] : 0.0;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double bf = glive[h] ? S[colg[h] + kk] : 0.0;
                    dmma884(d0[h], d1[h], a, bf);
                }
            }
            // stage W_IJ at U_IJ's own place (rows r0 .. r0 + 7 of the block's columns)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (rlive && alive[h]) S[cola[h] + rg] = d0[h];
                if (rlive && blive[h]) S[colb[h] + rg] = d1[h];
            }
            __syncwarp();
            double e0[2] = {0.0, 0.0}, e1[2] = {0.0, 0.0};
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const double b0 = (glive[h] && r0 + q < n) ? S[colg[h] + r0 + q] : 0.0;
                const double b1 = (glive[h] && r0 + 4 + q < n) ? S[colg[h] + r0 + 4 + q] : 0.0;
                dmma884(e0[h], e1[h], ti0, b0);
                dmma884(e0[h], e1[h], ti1, b1);
            }
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (rlive && alive[h]) S[cola[h] + rg] = e0[h];
                if (rlive && blive[h]) S[colb[h] + rg] = e1[h];
            }
        }
        __syncwarp();
    }
    return ok;
}

// Inclusive prefix sum over positions (lane + 32 t ordering).
template <int NS>
__device__ __forceinline__ void warp_scan_positions(double (&v)[NS], int lane) {
    double carry = 0.0;
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        double s = v[t];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            double u = __shfl_up_sync(FULL_MASK, s, o);
            if (lane >= o) s += u;
        }
        s += carry;
        v[t] = s;
        carry = __shfl_sync(FULL_MASK, s, 31);
    }
}

// Delete position k of the positive set (p -> p-1): re-triangularise T, shift idx and x.
// PS = position slots per lane (positions lane + 32 t, t < PS): ceil(pmax / 32), which can be smaller than the column
// slots NS of the Slots layout (FA stage: 60 columns, at most 32 positions) — the loops then run half as long.
template <int NS, int PS = NS>
__device__ __forceinline__ void remove_position(const Slots<NS>& W, int k, int& p, int lane, double (&x)[PS]) {
    const int oT = W.T;
    // rotation parameters from the prefix sums of squares of row k
    double tau[PS], Sq[PS];
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int q = lane + 32 * t;
        tau[t] = (q >= k && q < p) ? S[oT + tri(q) + k] : 0.0;
        Sq[t] = tau[t] * tau[t];
    }
    warp_scan_positions<PS>(Sq, lane);
    // nu_q = sqrt(S_q); step q (k <= q <= p-2) needs c_q = tau_{q+1}/nu_{q+1}, s_q = nu_q/nu_{q+1}
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int q = lane + 32 * t;
        if (q >= k && q < p) {
            S[W.rs + q] = sqrt(Sq[t]);   // nu_q
            S[W.gs + q] = tau[t];        // tau_q
        }
    }
    __syncwarp();
    double cq[PS], sq[PS];
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int q = lane + 32 * t;
        cq[t] = 0.0;
        sq[t] = 1.0;
        if (q >= k && q + 1 < p) {
            double inv = 1.0 / S[W.rs + q + 1];
            cq[t] = S[W.gs + q + 1] * inv;
            sq[t] = S[W.rs + q] * inv;
        }
    }
    __syncwarp();
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int q = lane + 32 * t;
        if (q >= k && q + 1 < p) {
            S[W.gs + q] = cq[t];
            S[W.rs + q] = sq[t];
        }
        if (q < p) S[W.xs + q] = x[t];   // x is shifted through xs below
    }
    __syncwarp();
    int idx_next[PS];
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int i = lane + 32 * t;
        idx_next[t] = (i >= k && i + 1 < p) ? SI(W.ix, i + 1) : -1;
        if (i >= k) x[t] = (i + 1 < p) ? S[W.xs + i + 1] : 0.0;
    }
    // row sweep: lane-slot owns old row rr (rr != k); carry starts as T(rr, k)
    double carry[PS];
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int rr = lane + 32 * t;
        carry[t] = (rr < k) ? S[oT + tri(k) + rr] : 0.0;
    }
#pragma unroll (Unroll<NS>::v)
    for (int q = k; q + 1 < p; ++q) {
        const double c = S[W.gs + q], s = S[W.rs + q];
        const int tq1 = oT + tri(q + 1), tq = oT + tri(q);
        double nv[PS];
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int rr = lane + 32 * t;
            double b = (rr <= q + 1 && rr != k) ? S[tq1 + rr] : 0.0;
            nv[t] = s * b - c * carry[t];
            carry[t] = fma(s, carry[t], c * b);
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int rr = lane + 32 * t;
            if (rr != k && rr <= q + 1) S[tq + rr - (rr > k ? 1 : 0)] = nv[t];
        }
    }
    __syncwarp();
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int i = lane + 32 * t;
        if (idx_next[t] >= 0) SI(W.ix, i) = idx_next[t];
    }
    --p;
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int i = lane + 32 * t;
        if (i < p) S[W.xs + i] = x[t];
    }
    __syncwarp();
}

// D-space evaluation of a candidate column j that the Gram-domain test finds (nearly) dependent on the positive set:
// the candidate's orthogonal residual q = d_j - D_P a with a = T r (r = T^T g_Pj is in S[W.rs..]), rho^2 = q.q and the
// numerator of its entering coefficient q.b — m p FMAs, errors of `a` enter quadratically.  Plain NNLS only (lam = 0).
// DESIGN.md §5: without it Lawson-Hanson stopped one exchange short in 1 of 1 500 voxels on the 96-bin grid
// (rho^2 = G_jj - r.r = -1.2e-13 for a column SciPy's QR-based test accepts).  Leaves a in S[W.gs..].
// Everything is passed and returned BY VALUE: a reference argument would force the caller's Slots / rho^2 / y_new into
// local memory on the hot path (measured with the first, by-reference version: T2 stage +3.3 %, FA stage +3 %).
template <int PS>
__device__ __noinline__ double2 dspace_candidate(int oT, int oGs, int oRs, int oIx, const double* __restrict__ DtR,
                                                 int oMR, int mrows, int j, int p, int lane) {
    double a[PS];
    tmul<PS>(oT, oRs, p, lane, a);
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int k = lane + 32 * t;
        if (k < p) S[oGs + k] = a[t];
    }
    __syncwarp();
    double qq = 0.0, qb = 0.0;
    for (int e = lane; e < mrows; e += 32) {
        double qe = __ldg(DtR + j * mrows + e);
        for (int k = 0; k < p; ++k) qe = fma(-S[oGs + k], __ldg(DtR + SI(oIx, k) * mrows + e), qe);
        qq = fma(qe, qe, qq);
        qb = fma(qe, S[oMR + e], qb);
    }
    warp_sum2(qq, qb);
    MET2_TRACE(lane, "  rescue j=%d: D-space rho2=%.17g, y_new numerator %.17g\n", j, qq, qb);
    __syncwarp();
    return make_double2(qq, qb);
}

// Gram-domain Lawson-Hanson.  On entry S[W.cc + 0..n) holds c = A^T b (visible to the whole warp).
// G: n x n row-major Gram matrix of the unregularised dictionary — in shared memory at offset oG (GSH) or in global
// memory at Gg.  reg: add lam * K, K given in 5-band form at S[oKb + d*n + c] = K[c+d-2][c].
// On exit S[W.ix..] / S[W.xs..] hold the positive set and its coefficients, S[W.xc..] the solution in column space;
// returns p.  status gets bit 0 on itmax.
// ldg: row stride of G (shared: n rounded up to even so that rows stay 16-byte aligned; global: n).
// p0 > 0: WARM START — positions 0..p0-1 of S[W.ix..]/S[W.xs..] hold a feasible point (support and coefficients, e.g.
// the solution for the previous lambda of a Brent/L-curve search).  T, y, z are rebuilt for the new Gram matrix by p0
// appends, then the secondary loop runs first (interpolating from that x if the new least-squares solution on the old
// support has non-positive entries) and the main loop continues as usual.  The minimiser of the (strictly convex)
// Tikhonov problem does not depend on the starting point; tools/proto_warm_start.py measured identical supports and
// lambda/k_est within 1e-11 against SciPy's cold-started path, with 13x fewer main-loop iterations.
template <int NS, bool GSH, int PS = NS>
__device__ __forceinline__ int nnls_gram(const Slots<NS>& W, int oG, const double* __restrict__ Gg, int ldg, int oKb,
                                         bool reg, double lam, int n, int mrows, int lane, int& status, int p0 = 0,
                                         bool t_ready = false) {
    const int itmax = 3 * n;
    auto Gat = [&](int r, int c) -> double { return GSH ? S[oG + r * ldg + c] : __ldg(Gg + r * ldg + c); };
    const int col0 = NS * lane;
    double creg[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        int col = col0 + s;
        creg[s] = (col < n) ? S[W.cc + col] : 0.0;
        if (col < n) S[W.xc + col] = 0.0;
    }
    unsigned inP = 0u;
    double x[PS], y[PS], z[PS];
#pragma unroll
    for (int t = 0; t < PS; ++t) x[t] = y[t] = z[t] = 0.0;
    int p = 0, iter = 0;
    __syncwarp();

    // Append column j at position p: returns false (nothing changed) if it is numerically dependent on the set or,
    // when `need_positive`, if its new coefficient is not positive (the two acceptance tests of nnls.f).
    auto append = [&](int j, bool need_positive, bool zero_x) -> bool {
        double gjj = Gat(j, j);
        if (reg) gjj = fma(lam, S[oKb + 2 * n + j], gjj);
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p) {
                int r = SI(W.ix, i);
                double gv = Gat(j, r);   // G is symmetric: column j == row j
                if (reg) {
                    int d = r - j + 2;
                    if (d >= 0 && d <= 4) gv = fma(lam, S[oKb + d * n + j], gv);
                }
                S[W.gs + i] = gv;
            }
        }
        __syncwarp();
        double r[PS];
        tmul_transposed<PS>(W.T, W.gs, p, lane, r);
        double s1 = 0.0, s2 = 0.0;
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p) {
                s1 = fma(r[t], r[t], s1);
                s2 = fma(r[t], y[t], s2);
                S[W.rs + i] = r[t];
            }
        }
        warp_sum2(s1, s2);
        double rho2 = gjj - s1;
        const double cj = S[W.cc + j];
        double rinv = rsqrt_fast(rho2);
        double ynew = (cj - s2) * rinv;
        if (!reg && p > 0 && rho2 < 1e-10 * gjj) {
            // rho^2 = G_jj - r.r is below the rounding of its terms (nearly collinear long-T2 columns of the 96/100-bin
            // grids): the Gram form resolves rho^2/G_jj to ~1e-16, nnls.f accepts down to ~5e-27.  Rare, so out of line.
            __syncwarp();
            const double* DtR = *reinterpret_cast<const double* const*>(S + W.aux());
            if (DtR) {
                const double2 qd = dspace_candidate<PS>(W.T, W.gs, W.rs, W.ix, DtR, SI(W.aux() + 1, 0), mrows, j, p, lane);
                rho2 = qd.x;
                rinv = rsqrt_fast(rho2);
                ynew = qd.y * rinv;
            }
        }
        // nnls.f: reject if the column is numerically dependent on P (unorm + |a_new|*0.01 == unorm, i.e.
        // rho < ~1e-14 unorm) or if its new coefficient ("ztest") is not positive
        const bool ok = (rho2 > 0.0) && (rho2 > 1.2e-28 * s1) && (!need_positive || ynew > 0.0);
        MET2_TRACE(lane, "  append j=%d p=%d gjj=%.17g rho2=%.17g ynew=%.17g -> %s\n", j, p, gjj, rho2, ynew,
                   ok ? "accepted" : "rejected");
        __syncwarp();
        if (!ok) return false;
        double acc[PS];
        tmul<PS>(W.T, W.rs, p, lane, acc);
        const int tp = W.T + tri(p);
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int k = lane + 32 * t;
            if (k < p) {
                double tk = -acc[t] * rinv;
                S[tp + k] = tk;
                z[t] = fma(ynew, tk, z[t]);
            } else if (k == p) {
                S[tp + p] = rinv;
                z[t] = ynew * rinv;
                y[t] = ynew;
                SI(W.ix, p) = j;
                if (zero_x) S[W.xs + p] = 0.0;   // x of an entering column is 0 until the solve is accepted
            }
        }
        if (j / NS == lane) inP |= 1u << (j % NS);
        ++p;
        __syncwarp();
        return true;
    };

    bool secondary_first = false;
    if (p0 > 0 && p0 <= mrows && p0 <= n) {
        auto Aent = [&](int kpos, int jpos) -> double {
            const int r = SI(W.ix, kpos), c = SI(W.ix, jpos);
            double a = Gat(r, c);
            if (reg) {
                const int d = r - c + 2;
                if (d >= 0 && d <= 4) a = fma(lam, S[oKb + d * n + c], a);
            }
            return a;
        };
        // t_ready: the caller already placed the factor of this set and lambda in the T region (shared full-set
        // factor tables of the X2 driver)
        const bool good = t_ready ? true : rebuild_T_blocked<NS>(W, Aent, p0, lane);
        if (good) {
            p = p0;
#pragma unroll 1
            for (int i = 0; i < p; ++i) {
                const int col = SI(W.ix, i);
                if (col / NS == lane) inP |= 1u << (col % NS);
            }
            // x = the carried-over coefficients; y = T^T c_P and z = T y are computed at the top of the secondary loop
#pragma unroll
            for (int t = 0; t < PS; ++t) {
                int i = lane + 32 * t;
                x[t] = (i < p) ? S[W.xs + i] : 0.0;
            }
            secondary_first = true;
        }
        // not positive definite in floating point: fall through to a cold start (p = 0, x = y = z = 0)
    }

    bool have_yz = false;
    if (secondary_first && t_ready) {
        // Start from the FULL set with a shared factor: drop every column whose unconstrained coefficient is not positive
        // in one go (highest position first, so the positions still to be examined do not move) instead of letting the
        // secondary loop take them out one re-solve at a time.  x stays a feasible point on the reduced set, so the
        // loop below continues as for any warm start; the minimiser does not depend on how the set was reached.
        // (Measured: T2 stage 426 -> 398 ms.  The same one-step drop for EVERY warm start did not pay — X2 unchanged,
        // L-curve 598 -> 621 ms — because a carried-over support rarely loses more than one or two columns.)
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p) S[W.gs + i] = S[W.cc + SI(W.ix, i)];
        }
        __syncwarp();
        tmul_transposed<PS>(W.T, W.gs, p, lane, y);
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p) S[W.rs + i] = y[t];
        }
        __syncwarp();
        tmul<PS>(W.T, W.rs, p, lane, z);
        __syncwarp();
        unsigned negm = 0u;
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p && z[t] <= 0.0) negm |= 1u << t;
        }
        int cur = p;
        have_yz = (__ballot_sync(FULL_MASK, negm != 0u) == 0u);   // nothing to drop: y and z are the loop's first solve
        while (true) {
            int k = -1;
#pragma unroll
            for (int t = 0; t < PS; ++t) {
                int i = lane + 32 * t;
                if (((negm >> t) & 1u) && i < cur && i > k) k = i;
            }
            k = (int)__reduce_max_sync(FULL_MASK, (unsigned)(k + 1)) - 1;
            if (k < 0 || p <= 1) break;
            const int colk = SI(W.ix, k);
            if (colk / NS == lane) inP &= ~(1u << (colk % NS));
            if (lane == 0) S[W.xc + colk] = 0.0;
            __syncwarp();
            remove_position<NS, PS>(W, k, p, lane, x);
            cur = k;
        }
        if (!have_yz) {
#pragma unroll
            for (int t = 0; t < PS; ++t) y[t] = z[t] = 0.0;
        }
    }

    while (true) {
      if (!secondary_first) {
        if (p >= n || p >= mrows) break;
        // ---- dual vector w = c - (G + lam K) x on the zero set
        double w[NS];
        if (p > 0) {
            double w1[NS];
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                w[s] = creg[s];
                w1[s] = 0.0;
            }
            int k = 0;
            if (GSH) {
                // rows of G in shared memory: one vector LDS per row and lane (columns NS*lane .. NS*lane+NS-1)
                const bool live = col0 < n;
#pragma unroll (Unroll<NS>::v)
                for (; k + 1 < p; k += 2) {
                    const int r0 = oG + SI(W.ix, k) * ldg + col0, r1 = oG + SI(W.ix, k + 1) * ldg + col0;
                    const double x0 = S[W.xs + k], x1 = S[W.xs + k + 1];
                    if (live) {
                        double g0[NS], g1[NS];
                        lds_vec<NS>(r0, g0);
                        lds_vec<NS>(r1, g1);
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            w[s] = fma(-x0, g0[s], w[s]);
                            w1[s] = fma(-x1, g1[s], w1[s]);
                        }
                    }
                }
                if (k < p) {
                    const int r0 = oG + SI(W.ix, k) * ldg + col0;
                    const double x0 = S[W.xs + k];
                    if (live) {
                        double g0[NS];
                        lds_vec<NS>(r0, g0);
#pragma unroll
                        for (int s = 0; s < NS; ++s) w[s] = fma(-x0, g0[s], w[s]);
                    }
                }
            } else {
                const bool vec = ((ldg & 1) == 0);
                const int nvalid = n - col0;   // columns this lane really owns (<= 0: none)
#pragma unroll (Unroll<NS>::v)
                for (; k + 1 < p; k += 2) {
                    const double* g0 = Gg + SI(W.ix, k) * ldg + col0;
                    const double* g1 = Gg + SI(W.ix, k + 1) * ldg + col0;
                    const double x0 = S[W.xs + k], x1 = S[W.xs + k + 1];
                    if (nvalid > 0) {
                        double v0[NS], v1[NS];
                        ldg_vec<NS>(g0, vec, nvalid, v0);
                        ldg_vec<NS>(g1, vec, nvalid, v1);
#pragma unroll
                        for (int s = 0; s < NS; ++s) {
                            w[s] = fma(-x0, v0[s], w[s]);
                            w1[s] = fma(-x1, v1[s], w1[s]);
                        }
                    }
                }
                if (k < p) {
                    const double* g0 = Gg + SI(W.ix, k) * ldg + col0;
                    const double x0 = S[W.xs + k];
                    if (nvalid > 0) {
                        double v0[NS];
                        ldg_vec<NS>(g0, vec, nvalid, v0);
#pragma unroll
                        for (int s = 0; s < NS; ++s) w[s] = fma(-x0, v0[s], w[s]);
                    }
                }
            }
#pragma unroll
            for (int s = 0; s < NS; ++s) w[s] += w1[s];
            if (reg) {
#pragma unroll
                for (int s = 0; s < NS; ++s) {
                    int col = col0 + s;
                    if (col < n) {
                        double acc = 0.0;
#pragma unroll
                        for (int d = 0; d < 5; ++d) {
                            int c2 = col + d - 2;
                            if (c2 >= 0 && c2 < n) acc = fma(S[oKb + d * n + col], S[W.xc + c2], acc);
                        }
                        w[s] = fma(-lam, acc, w[s]);
                    }
                }
            }
        } else {
#pragma unroll
            for (int s = 0; s < NS; ++s) w[s] = creg[s];
        }
        // ---- pick the entering column
        unsigned rejected = 0u;
        bool accepted = false;
        while (true) {
            double bv = 0.0;
            int bj = -1;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                int col = col0 + s;
                if (col < n && !((inP >> s) & 1u) && !((rejected >> s) & 1u) && w[s] > bv) {
                    bv = w[s];
                    bj = col;
                }
            }
            const int j = warp_argmax_pos(bv, bj);
            if (j < 0) break;
            if (!append(j, true, true)) {
                if (j / NS == lane) rejected |= 1u << (j % NS);
                continue;
            }
            accepted = true;
            break;
        }
        if (!accepted) break;
      }
        bool fresh = secondary_first;   // after an append z was updated incrementally
        secondary_first = false;
        // ---- secondary loop
        bool stop = false;
        while (true) {
            if (fresh && have_yz) {
                have_yz = false;   // computed by the block-drop step above
            } else if (fresh) {
                // y = T^T c_P and z = T y from scratch (after a warm-start rebuild or a removal)
#pragma unroll
                for (int t = 0; t < PS; ++t) {
                    int i = lane + 32 * t;
                    if (i < p) S[W.gs + i] = S[W.cc + SI(W.ix, i)];
                }
                __syncwarp();
                tmul_transposed<PS>(W.T, W.gs, p, lane, y);
#pragma unroll
                for (int t = 0; t < PS; ++t) {
                    int i = lane + 32 * t;
                    if (i < p) S[W.rs + i] = y[t];
                    else y[t] = 0.0;
                }
                __syncwarp();
                tmul<PS>(W.T, W.rs, p, lane, z);
                __syncwarp();
            }
            fresh = true;
            ++iter;
            if (iter > itmax) {
                status |= 1;
                stop = true;
                break;
            }
            bool neg = false;
#pragma unroll
            for (int t = 0; t < PS; ++t) {
                int i = lane + 32 * t;
                if (i < p && z[t] <= 0.0) neg = true;
            }
            if (!__any_sync(FULL_MASK, neg)) break;
            double bt = 2.0;
            int bi = -1;
#pragma unroll
            for (int t = 0; t < PS; ++t) {
                int i = lane + 32 * t;
                if (i < p && z[t] <= 0.0) {
                    double tt = x[t] / (x[t] - z[t]);
                    if (tt < bt) {
                        bt = tt;
                        bi = i;
                    }
                }
            }
            double alpha;
            int jb = warp_argmin_nonneg(bt, bi, alpha);
            if (jb < 0) break;
#pragma unroll
            for (int t = 0; t < PS; ++t) {
                int i = lane + 32 * t;
                if (i < p) x[t] = x[t] + alpha * (z[t] - x[t]);
            }
            int k = jb;
            while (true) {
                int colk = SI(W.ix, k);
                MET2_TRACE(lane, "  remove col=%d (position %d of %d) alpha=%.17g\n", colk, k, p, alpha);
                if (colk / NS == lane) inP &= ~(1u << (colk % NS));
                if (lane == 0) S[W.xc + colk] = 0.0;
                __syncwarp();
                remove_position<NS, PS>(W, k, p, lane, x);
                int q = 0x7fffffff;
#pragma unroll
                for (int t = PS - 1; t >= 0; --t) {
                    int i = lane + 32 * t;
                    if (i < p && x[t] <= 0.0) q = i;
                }
                q = (int)__reduce_min_sync(FULL_MASK, (unsigned)q);
                if (q == 0x7fffffff) break;
                k = q;
            }
        }
        if (stop) break;
#pragma unroll
        for (int t = 0; t < PS; ++t) {
            int i = lane + 32 * t;
            if (i < p) {
                x[t] = z[t];
                S[W.xs + i] = z[t];
                if (reg) S[W.xc + SI(W.ix, i)] = z[t];
            }
        }
        __syncwarp();
    }
    // xs mirrors x on every path; make the column-space copy current for the caller
#pragma unroll
    for (int t = 0; t < PS; ++t) {
        int i = lane + 32 * t;
        if (i < p) S[W.xc + SI(W.ix, i)] = x[t];
    }
    __syncwarp();
    return p;
}

}  // namespace met2
