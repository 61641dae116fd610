// met2_degibbs.cu — Gibbs-ringing removal by local subvoxel shifts (Kellner et al., MRM 76:1574, 2016; the method of
// MRtrix3's mrdegibbs in its basic 2-D mode), applied to every in-plane slice of a multi-echo volume.  No counterpart in
// the reference: an optional preprocessing step after Step 1.  Partial-Fourier acquisitions are out of scope, as they are
// in mrdegibbs's basic mode.
//
// Definition (tests/degibbs_oracle.py restates it in NumPy operation for operation; the kernels are bitwise equal to it):
//  Input vol [nx][ny][nz][nt] C-order float64, read as [n0 = nx][n1 = ny][S = nz nt]: slice s = z nt + t is the n0 x n1
//  image u[x][y] = vol[x][y][z][t].  Parameters nsh >= 1 (shifts per half pixel), 0 <= minW <= maxW, 2 maxW < n0, n1.
//  Tables (met2_degibbs_tables, one per in-plane size n; every entry is cos(2 pi P / Q) for integers P, Q, see dg_cos2pi):
//    cos[r] = cos(2 pi r / n), sin[r] = sin(2 pi r / n)   (r = 0..n-1),
//    c[k]   = 1 + cos(2 pi f(k)), f = numpy.fft.fftfreq(n)  (= 1 + cos[k]),
//    h[q][d] = Re((1/n) sum_k exp(i 2 pi f(k) (d + s_q)))   (q = 0..2 nsh, d = 0..n-1), the band-limited interpolation
//      kernel for a shift s_q = m_q / (2 nsh), with m_q = 0, +1, .., +nsh, -1, .., -nsh for q = 0, 1, .., 2 nsh.
//      h[0] is the exact delta (h[0][0] = 1, else 0); for m != 0 the closed form (the Dirichlet kernel), x = d + s_q:
//      odd n: sin(pi x) / (n sin(pi x / n));  even n: (sin(pi x (n-1)/n) / sin(pi x / n) + cos(pi x)) / n.
//  1. Split.  G0[k0][k1] = c1[k1] / (c0[k0] + c1[k1]), or 1/2 where c0[k0] + c1[k1] == 0 (both at Nyquist).
//     Products: real a by a twiddle (c, w) is (a c, a w); complex (a, b) by (c, w) is (a c - b w, a w + b c).
//     Forward twiddle of index (k x) mod n: (cos, -sin); inverse: (cos, sin).  Every sum starts from 0.0 and runs over
//     its index ascending.  The 2-D transforms run rows (axis 1, over y) then columns (axis 0, over x):
//       A[x][k1]  = sum_y u[x][y] (cos, -sin)[k1 y]                        (real input)
//       U[k0][k1] = sum_x A[x][k1] (cos, -sin)[k0 x];  P = (U_re G0, U_im G0)
//       B[k0][y]  = sum_k1 P[k0][k1] (cos, sin)[k1 y]
//       v0[x][y]  = (sum_k0 (B_re[k0][y] cos[k0 x] - B_im[k0][y] sin[k0 x])) / (n0 n1)  (the real part only)
//       v1 = u - v0.
//  2. Unring each periodic line of v0 along axis 0 and of v1 along axis 1 (length n):
//     y_q[j] = sum_{d=0}^{n-1} h[q][d] x[(j - d) mod n];
//     TV_L(q, j) = sum_{w=minW}^{maxW} |y_q[j-w] - y_q[j-w-1]|,  TV_R(q, j) = sum_{w=minW}^{maxW} |y_q[j+w] - y_q[j+w+1]|
//     (indices mod n, every sum direct — no sliding update, so its rounding does not depend on j);
//     best = +inf, sel = 0; for q = 0..2 nsh: if TV_L < best: best = TV_L, sel = q; then the same with TV_R (strict <:
//     the first minimum wins, q = 0 wins ties; a line whose TVs are all NaN keeps q = 0);
//     s = m_sel / (2 nsh);  out[j] = (1 - s) y[j] + s y[j-1] for s > 0, else (1 - |s|) y[j] + |s| y[j+1], y = y_sel.
//  3. out = unring0(v0) + unring1(v1).
//  Only IEEE +, -, *, / and |.| (the library is built with -fmad=false), so NumPy reproduces every bit given the tables.
//  dg_cos2pi uses only IEEE operations and exact integer reduction, so the tables the kernels build on the device are
//  the bits met2_degibbs_tables returns on the host.
//
// Layout: the slice index is the fastest axis of the volume, so every kernel gives the DG_TS lanes of a thread row DG_TS
// consecutive slices (coalesced loads and stores) and no relayout is needed.  A CTA owns one line position and DG_TS
// slices: the DFT kernel stages its DG_TS lines and the twiddles in shared memory and each thread row computes outputs k;
// the unringing kernel stages h (31 KB at n = 96, 84 KB at n = 256 for nsh = 20), its DG_TS lines and one y_q tile in
// shared memory, each thread convolves DG_R consecutive positions with a sliding register window (two shared loads per
// DG_R multiply-adds), and the same thread then keeps the running TV minimum of those positions.  y at the chosen shift
// is recomputed at the end by the same sum (same bits) instead of being kept for all q.  Limits: n0, n1 <= DG_MAX_N = 256
// (DG_TS ceil(n / DG_R) threads per CTA), and (2 nsh + 1 + 2 DG_TS) n doubles of shared memory <= 227 KB, i.e.
// nsh <= 40 at n = 256.
#include <math.h>

#include "met2_host.h"

namespace met2 {

#ifdef MET2_HOST_EMU
static simt::Shared& S = simt::g_shared;
#else
extern __shared__ __align__(16) double S[];
#endif

constexpr int DG_TS = 16;          // slices per CTA: the lanes of a thread row
constexpr int DG_R = 4;            // positions per thread of the unringing convolution
constexpr int DG_KY = 16;          // thread rows of a DFT CTA
constexpr int DG_MAX_N = 256;
constexpr size_t DG_SMEM_MAX = 227 * 1024;
enum { DG_FWD_ROWS = 0, DG_FWD_COLS_G0 = 1, DG_INV_ROWS = 2, DG_INV_COLS_RE = 3 };

// ------------------------------------------------------------------------------------------------ tables
// Taylor polynomials of cos and sin on |phi| <= pi/4 (terms to phi^20 / phi^21: truncation < 1e-23), Horner in phi^2
__host__ __device__ inline double dg_cos_poly(double phi) {
    const double x2 = phi * phi;
    double p = 4.110317623312165e-19;
    p = p * x2 + -1.5619206968586225e-16;
    p = p * x2 + 4.779477332387385e-14;
    p = p * x2 + -1.1470745597729725e-11;
    p = p * x2 + 2.08767569878681e-09;
    p = p * x2 + -2.755731922398589e-07;
    p = p * x2 + 2.48015873015873e-05;
    p = p * x2 + -0.001388888888888889;
    p = p * x2 + 0.041666666666666664;
    p = p * x2 + -0.5;
    return p * x2 + 1.0;
}

__host__ __device__ inline double dg_sin_poly(double phi) {
    const double x2 = phi * phi;
    double p = 1.9572941063391263e-20;
    p = p * x2 + -8.22063524662433e-18;
    p = p * x2 + 2.8114572543455206e-15;
    p = p * x2 + -7.647163731819816e-13;
    p = p * x2 + 1.6059043836821613e-10;
    p = p * x2 + -2.505210838544172e-08;
    p = p * x2 + 2.7557319223985893e-06;
    p = p * x2 + -0.0001984126984126984;
    p = p * x2 + 0.008333333333333333;
    p = p * x2 + -0.16666666666666666;
    return (p * x2 + 1.0) * phi;
}

// cos(2 pi P / Q), Q > 0: P mod Q and the octant exactly in integers, then a polynomial on |phi| <= pi/4
__host__ __device__ inline double dg_cos2pi(long long P, long long Q) {
    long long r = P % Q;
    if (r < 0) r += Q;
    const int o = (int)((8 * r) / Q);                  // octant of the angle 2 pi r / Q
    const long long rem = 8 * r - (long long)o * Q;    // (angle - o pi/4) = (pi/4) rem / Q
    const double pi4 = 0.7853981633974483;
    double cp, sp;                                      // cos and sin of the angle minus its quadrant's start
    if ((o & 1) == 0) {
        const double phi = pi4 * (double)rem / (double)Q;
        cp = dg_cos_poly(phi), sp = dg_sin_poly(phi);
    } else {
        const double phi = pi4 * (double)(Q - rem) / (double)Q;
        cp = dg_sin_poly(phi), sp = dg_cos_poly(phi);
    }
    switch (o >> 1) {
        case 0: return cp;
        case 1: return -sp;
        case 2: return -cp;
        default: return sp;
    }
}

__host__ __device__ inline double dg_sin2pi(long long P, long long Q) { return dg_cos2pi(4 * P - Q, 4 * Q); }

__host__ __device__ inline long long dg_table_len(int n, int nsh) { return (long long)n * (2 * nsh + 4); }

// shift m of position q in the search order 0, +1, .., +nsh, -1, .., -nsh
__host__ __device__ inline int dg_shift(int q, int nsh) { return q <= nsh ? q : nsh - q; }

// entry i of the table of size n: cos[n], sin[n], c[n], h[2 nsh + 1][n]
__host__ __device__ inline double dg_table_entry(int n, int nsh, long long i) {
    if (i < n) return dg_cos2pi(i, n);
    if (i < 2 * n) return dg_sin2pi(i - n, n);
    if (i < 3 * n) return 1.0 + dg_cos2pi(i - 2 * n, n);
    const long long qd = i - 3 * n;
    const int q = (int)(qd / n), d = (int)(qd - (long long)q * n);
    const int m = dg_shift(q, nsh);
    if (m == 0) return d == 0 ? 1.0 : 0.0;              // no shift: an exact delta, so y_0 = x
    const long long D = 2LL * nsh;
    const long long X = D * d + m;                      // x = d + s_q = X / D, never 0
    const double den = dg_sin2pi(X, 2 * D * n);         // sin(pi x / n)
    if (n & 1) return dg_sin2pi(X, 2 * D) / ((double)n * den);
    return (dg_sin2pi(X * (n - 1), 2 * D * n) / den + dg_cos2pi(X, 2 * D)) / (double)n;
}

__global__ void degibbs_tables_kernel(int n0, int n1, int nsh, double* __restrict__ t0, double* __restrict__ t1) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long l0 = dg_table_len(n0, nsh), l1 = dg_table_len(n1, nsh);
    if (i < l0)
        t0[i] = dg_table_entry(n0, nsh, i);
    else if (i < l0 + l1)
        t1[i - l0] = dg_table_entry(n1, nsh, i - l0);
}

// ------------------------------------------------------------------------------------------------ lines
// A line along axis 1 (a row: fixed x) has stride S; along axis 0 (a column: fixed y) stride n1 S.  p is the fixed index.
struct DgLine {
    long long base, stride;
    int n, p;
    long long s;                                        // this lane's slice
};

__device__ __forceinline__ DgLine dg_line(int axis, int n0, int n1, long long nS) {
    const long long nst = (nS + DG_TS - 1) / DG_TS;
    DgLine L;
    L.p = (int)(blockIdx.x / nst);
    L.s = (long long)(blockIdx.x - (long long)L.p * nst) * DG_TS + threadIdx.x;
    L.n = axis == 0 ? n0 : n1;
    L.stride = axis == 0 ? (long long)n1 * nS : nS;
    L.base = axis == 0 ? (long long)L.p * nS : (long long)L.p * n1 * nS;
    return L;
}

// One pass of the split (step 1).  DG_FWD_ROWS: u -> A (real input); DG_FWD_COLS_G0: A -> P; DG_INV_ROWS: P -> B;
// DG_INV_COLS_RE: B -> (v0, v1).  Shared: the CTA's lines (re, im) [n][DG_TS] and the twiddles cos[n], sin[n].
__global__ void __launch_bounds__(DG_TS * DG_KY) degibbs_dft_kernel(int mode, const double* __restrict__ in_re,
                                                                     const double* __restrict__ in_im,
                                                                     const double* __restrict__ u, int n0, int n1,
                                                                     long long nS, const double* __restrict__ t0,
                                                                     const double* __restrict__ t1,
                                                                     double* __restrict__ out_re,
                                                                     double* __restrict__ out_im) {
    const int axis = (mode == DG_FWD_ROWS || mode == DG_INV_ROWS) ? 1 : 0;
    const DgLine L = dg_line(axis, n0, n1, nS);
    const int n = L.n, tx = threadIdx.x, ty = threadIdx.y;
    const bool lane_ok = L.s < nS;
    const double* tab = axis == 0 ? t0 : t1;
    const long long oRe = 0, oIm = (long long)n * DG_TS, oCos = 2LL * n * DG_TS, oSin = oCos + n;
    for (int i = ty; i < n; i += DG_KY) {
        const long long g = L.base + i * L.stride + L.s;
        S[oRe + i * DG_TS + tx] = lane_ok ? in_re[g] : 0.0;
        S[oIm + i * DG_TS + tx] = (lane_ok && mode != DG_FWD_ROWS) ? in_im[g] : 0.0;
    }
    for (int i = ty * DG_TS + tx; i < n; i += DG_TS * DG_KY) {
        S[oCos + i] = tab[i];
        S[oSin + i] = tab[n + i];
    }
    __syncthreads();
    const bool fwd = mode == DG_FWD_ROWS || mode == DG_FWD_COLS_G0;
    for (int k = ty; k < n; k += DG_KY) {
        double acc_re = 0.0, acc_im = 0.0;
        int idx = 0;                                    // (k x) mod n
        for (int x = 0; x < n; ++x) {
            const double c = S[oCos + idx], w = fwd ? -S[oSin + idx] : S[oSin + idx];
            const double ar = S[oRe + x * DG_TS + tx];
            if (mode == DG_FWD_ROWS) {
                acc_re = acc_re + ar * c;
                acc_im = acc_im + ar * w;
            } else {
                const double ai = S[oIm + x * DG_TS + tx];
                acc_re = acc_re + (ar * c - ai * w);
                if (mode != DG_INV_COLS_RE) acc_im = acc_im + (ar * w + ai * c);
            }
            idx += k;
            if (idx >= n) idx -= n;
        }
        if (!lane_ok) continue;
        const long long g = L.base + k * L.stride + L.s;
        if (mode == DG_FWD_COLS_G0) {                   // line p = k1, output k = k0
            const double c1 = t1[2 * n1 + L.p], den = t0[2 * n0 + k] + c1;
            const double g0 = den == 0.0 ? 0.5 : c1 / den;
            out_re[g] = acc_re * g0;
            out_im[g] = acc_im * g0;
        } else if (mode == DG_INV_COLS_RE) {
            const double v0 = acc_re / (double)((long long)n0 * n1);
            out_re[g] = v0;
            out_im[g] = u[g] - v0;
        } else {
            out_re[g] = acc_re;
            out_im[g] = acc_im;
        }
    }
}

// ------------------------------------------------------------------------------------------------ unringing
// y_q[j] of one lane's line in shared memory (the sum of the main loop, term by term: the same bits)
__device__ __forceinline__ double dg_conv(const long long oH, const long long oX, int n, int j, int tx) {
    double acc = 0.0;
    int e = j;
    for (int d = 0; d < n; ++d) {
        acc = acc + S[oH + d] * S[oX + e * DG_TS + tx];
        e = e == 0 ? n - 1 : e - 1;
    }
    return acc;
}

// i mod n for -n <= i < 2n: the TV and interpolation neighbours (2 maxW < n keeps them in that range)
__device__ __forceinline__ int dg_wrap(int i, int n) { return i < 0 ? i + n : (i >= n ? i - n : i); }

// Step 2 on the lines along `axis` of src; out = result (accumulate = 0) or out + result (accumulate = 1).
// Block (DG_TS, gb): thread row ty owns positions j0 = DG_R ty .. j0 + DG_R - 1.  Shared: h [2 nsh + 1][n], the lines
// [n][DG_TS], the current y_q [n][DG_TS].
__global__ void __launch_bounds__(1024) degibbs_unring_kernel(const double* __restrict__ src, int axis, int n0, int n1,
                                                              long long nS, const double* __restrict__ tab, int nsh,
                                                              int minW, int maxW, int accumulate,
                                                              double* __restrict__ out) {
    const DgLine L = dg_line(axis, n0, n1, nS);
    const int n = L.n, tx = threadIdx.x, ty = threadIdx.y;
    const int nq = 2 * nsh + 1;
    const bool lane_ok = L.s < nS;
    const long long oH = 0, oX = (long long)nq * n, oY = oX + (long long)n * DG_TS;
    const int nthr = DG_TS * blockDim.y, t = ty * DG_TS + tx;
    for (int i = t; i < nq * n; i += nthr) S[oH + i] = tab[3 * n + i];
    for (int i = ty; i < n; i += blockDim.y) S[oX + i * DG_TS + tx] = lane_ok ? src[L.base + i * L.stride + L.s] : 0.0;
    __syncthreads();
    const int j0 = DG_R * ty;
    const bool active = j0 < n;
    double best[DG_R];
    int sel[DG_R];
#pragma unroll
    for (int r = 0; r < DG_R; ++r) best[r] = INFINITY, sel[r] = 0;
    for (int q = 0; q < nq; ++q) {
        if (active) {
            const long long oHq = oH + (long long)q * n;
            double w[DG_R], acc[DG_R];
#pragma unroll
            for (int r = 0; r < DG_R; ++r) {
                // x[(j0 + r - d) mod n] at d = 0; the padded positions reach j0 + r = n + 2, two wraps at n = 1
                w[r] = S[oX + ((j0 + r) % n) * DG_TS + tx];
                acc[r] = 0.0;
            }
            int e = j0;                                             // (j0 - d) mod n
            for (int d = 0; d < n; ++d) {
                const double hd = S[oHq + d];
#pragma unroll
                for (int r = 0; r < DG_R; ++r) acc[r] = acc[r] + hd * w[r];
#pragma unroll
                for (int r = DG_R - 1; r > 0; --r) w[r] = w[r - 1];
                e = e == 0 ? n - 1 : e - 1;
                w[0] = S[oX + e * DG_TS + tx];
            }
#pragma unroll
            for (int r = 0; r < DG_R; ++r)
                if (j0 + r < n) S[oY + (j0 + r) * DG_TS + tx] = acc[r];
        }
        __syncthreads();
        if (active) {
#pragma unroll
            for (int r = 0; r < DG_R; ++r) {
                const int j = j0 + r;
                if (j >= n) break;
                double tvl = 0.0, tvr = 0.0;
                for (int wv = minW; wv <= maxW; ++wv)
                    tvl = tvl + fabs(S[oY + dg_wrap(j - wv, n) * DG_TS + tx] - S[oY + dg_wrap(j - wv - 1, n) * DG_TS + tx]);
                for (int wv = minW; wv <= maxW; ++wv)
                    tvr = tvr + fabs(S[oY + dg_wrap(j + wv, n) * DG_TS + tx] - S[oY + dg_wrap(j + wv + 1, n) * DG_TS + tx]);
                if (tvl < best[r]) best[r] = tvl, sel[r] = q;
                if (tvr < best[r]) best[r] = tvr, sel[r] = q;
            }
        }
        __syncthreads();                                           // before the next q overwrites y
    }
    if (!active) return;
#pragma unroll
    for (int r = 0; r < DG_R; ++r) {
        const int j = j0 + r;
        if (j >= n) break;
        const long long oHq = oH + (long long)sel[r] * n;
        const double s = (double)dg_shift(sel[r], nsh) / (double)(2 * nsh);
        const double y0 = dg_conv(oHq, oX, n, j, tx);
        double o;
        if (s > 0.0) {
            const double y1 = dg_conv(oHq, oX, n, dg_wrap(j - 1, n), tx);
            o = (1.0 - s) * y0 + s * y1;
        } else {
            const double as = fabs(s);
            const double y1 = dg_conv(oHq, oX, n, dg_wrap(j + 1, n), tx);
            o = (1.0 - as) * y0 + as * y1;
        }
        if (lane_ok) {
            const long long g = L.base + j * L.stride + L.s;
            out[g] = accumulate ? out[g] + o : o;
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
static size_t dg_unring_smem(int n, int nsh) { return sizeof(double) * ((size_t)(2 * nsh + 1) * n + 2 * (size_t)n * DG_TS); }
static size_t dg_dft_smem(int n) { return sizeof(double) * (2 * (size_t)n * DG_TS + 2 * (size_t)n); }

struct DgWs {
    double *t0, *t1, *a_re, *a_im, *b_re, *b_im;
};

static size_t dg_carve(int nx, int ny, long long nS, int nsh, void* ws, DgWs* W) {
    const size_t l0 = align256(sizeof(double) * (size_t)dg_table_len(nx, nsh)),
                 l1 = align256(sizeof(double) * (size_t)dg_table_len(ny, nsh)),
                 v = align256(sizeof(double) * (size_t)nx * ny * nS);
    if (W) {
        char* p = (char*)ws;
        W->t0 = (double*)p;
        W->t1 = (double*)(p + l0);
        W->a_re = (double*)(p + l0 + l1);
        W->a_im = (double*)(p + l0 + l1 + v);
        W->b_re = (double*)(p + l0 + l1 + 2 * v);
        W->b_im = (double*)(p + l0 + l1 + 3 * v);
    }
    return l0 + l1 + 4 * v;
}

static int dg_check(const char* what, int nx, int ny, int nz, int nt, int nsh, int minW, int maxW) {
    if (nx < 1 || ny < 1 || nz < 1 || nt < 1 || nx > DG_MAX_N || ny > DG_MAX_N)
        return set_error(MET2_ERR_ARG, "%s: bad sizes nx=%d ny=%d nz=%d nt=%d (in-plane sizes 1..%d)", what, nx, ny, nz, nt,
                         DG_MAX_N);
    const long long nS = (long long)nz * nt;
    if ((long long)max(nx, ny) * ((nS + DG_TS - 1) / DG_TS) > 0x7fffffffLL)
        return set_error(MET2_ERR_ARG, "%s: too many slices (nz * nt = %lld)", what, nS);
    if (nsh < 1 || minW < 0 || minW > maxW || 2 * (long long)maxW >= nx || 2 * (long long)maxW >= ny)
        return set_error(MET2_ERR_ARG, "%s: need nsh >= 1, 0 <= minW <= maxW < n/2 (nsh=%d minW=%d maxW=%d, n=%d x %d)",
                         what, nsh, minW, maxW, nx, ny);
    if (nsh > 1024 || dg_unring_smem(max(nx, ny), nsh) > DG_SMEM_MAX)
        return set_error(MET2_ERR_ARG, "%s: nsh=%d at n=%d needs %zu B of shared memory per CTA, over %zu", what, nsh,
                         max(nx, ny), dg_unring_smem(max(nx, ny), nsh), DG_SMEM_MAX);
    return MET2_OK;
}

}  // namespace met2

using namespace met2;

extern "C" int64_t met2_degibbs_tables(int n, int nsh, double* host_out) {
    if (n < 1 || n > DG_MAX_N || nsh < 1 || nsh > 1024)
        return set_error(MET2_ERR_ARG, "met2_degibbs_tables: need 1 <= n <= %d and 1 <= nsh <= 1024 (n=%d nsh=%d)",
                         DG_MAX_N, n, nsh);
    const long long len = dg_table_len(n, nsh);
    if (host_out)
        for (long long i = 0; i < len; ++i) host_out[i] = dg_table_entry(n, nsh, i);
    return (int64_t)len;
}

extern "C" int64_t met2_degibbs_workspace_bytes(int nx, int ny, int nz, int nt, int nsh, int minW, int maxW) {
    if (dg_check("met2_degibbs_workspace_bytes", nx, ny, nz, nt, nsh, minW, maxW)) return MET2_ERR_ARG;
    return (int64_t)dg_carve(nx, ny, (long long)nz * nt, nsh, nullptr, nullptr);
}

extern "C" int met2_degibbs(const double* vol, int nx, int ny, int nz, int nt, int nsh, int minW, int maxW, double* out,
                            void* workspace, void* stream) {
    int rc = dg_check("met2_degibbs", nx, ny, nz, nt, nsh, minW, maxW);
    if (rc) return rc;
    if (!vol || !out || !workspace) return set_error(MET2_ERR_ARG, "met2_degibbs: NULL argument");
    if ((const void*)out == (const void*)vol) return set_error(MET2_ERR_ARG, "met2_degibbs: out must not alias vol");
    cudaStream_t st = (cudaStream_t)stream;
    const long long nS = (long long)nz * nt, nst = (nS + DG_TS - 1) / DG_TS;
    DgWs W;
    dg_carve(nx, ny, nS, nsh, workspace, &W);
    const int nmax = max(nx, ny);
    const size_t dsm = dg_dft_smem(nmax), usm = dg_unring_smem(nmax, nsh);
    cudaError_t e = cudaFuncSetAttribute(degibbs_dft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(degibbs_unring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usm);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "degibbs kernel attr: %s", cudaGetErrorString(e));
    const long long ltab = dg_table_len(nx, nsh) + dg_table_len(ny, nsh);
    MET2_LAUNCH((unsigned)((ltab + 255) / 256), 256, 0, st, degibbs_tables_kernel)(nx, ny, nsh, W.t0, W.t1);
    const dim3 dblk(DG_TS, DG_KY);
    const unsigned rows = (unsigned)(nx * nst), cols = (unsigned)(ny * nst);
    MET2_LAUNCH(rows, dblk, dsm, st, degibbs_dft_kernel)(DG_FWD_ROWS, vol, nullptr, nullptr, nx, ny, nS, W.t0, W.t1,
                                                          W.a_re, W.a_im);
    MET2_LAUNCH(cols, dblk, dsm, st, degibbs_dft_kernel)(DG_FWD_COLS_G0, W.a_re, W.a_im, nullptr, nx, ny, nS, W.t0, W.t1,
                                                          W.b_re, W.b_im);
    MET2_LAUNCH(rows, dblk, dsm, st, degibbs_dft_kernel)(DG_INV_ROWS, W.b_re, W.b_im, nullptr, nx, ny, nS, W.t0, W.t1,
                                                          W.a_re, W.a_im);
    MET2_LAUNCH(cols, dblk, dsm, st, degibbs_dft_kernel)(DG_INV_COLS_RE, W.a_re, W.a_im, vol, nx, ny, nS, W.t0, W.t1,
                                                          W.b_re, W.b_im);
    // thread rows: ceil(n / DG_R), rounded up to even so that a CTA is whole warps
    auto rows_of = [](int n) { const int g = (n + DG_R - 1) / DG_R; return (unsigned)(g + (g & 1)); };
    MET2_LAUNCH(cols, dim3(DG_TS, rows_of(nx)), usm, st, degibbs_unring_kernel)(W.b_re, 0, nx, ny, nS, W.t0, nsh, minW,
                                                                                 maxW, 0, out);
    MET2_LAUNCH(rows, dim3(DG_TS, rows_of(ny)), usm, st, degibbs_unring_kernel)(W.b_im, 1, nx, ny, nS, W.t1, nsh, minW,
                                                                                 maxW, 1, out);
    count_launch(7);
    return check_launch("met2_degibbs");
}
