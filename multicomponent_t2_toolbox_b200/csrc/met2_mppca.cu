// met2_mppca.cu — Marchenko-Pastur PCA denoising of a multi-echo volume (Veraart et al. 2016, the method of MRtrix3's
// dwidenoise), with a per-voxel noise sigma map.  No counterpart in the reference: an optional Step 1 beside NESMA and TV.
//
// Definition (tests/mppca_oracle.py restates it in NumPy operation for operation; the kernel is bitwise equal to it):
//  Inputs: vol [nx][ny][nz][N] C-order float64 (Step 1's input: data * mask, negatives clipped to 0), mask [nx][ny][nz]
//  int32, patch radius r >= 1, N <= MET2_MAX_NTE.  For every voxel c = (i, j, k) with mask == 1:
//  1. Window.  On each axis a of size n_a: w_a = min(2r + 1, n_a), s_a = min(max(c_a - r, 0), n_a - w_a) — near an edge
//     the window shifts to stay inside the volume instead of shrinking.  Samples are all voxels of the box, whatever
//     their mask, in C order (i slowest, k fastest).  Every voxel has the same M = w_x w_y w_z (125 at r = 2); M < 2 is
//     an argument error.
//  2. mu_e = (sum_s X_se, from 0.0 in sample order) / M;  Xc = X - mu.
//  3. C = Xc^T Xc (N x N, unnormalised), every entry summed from 0.0 in sample order.  The kernel forms every entry
//     (e, f) as the sum of xc_e * xc_f; IEEE products commute, so this is the e <= f triangle mirrored.
//  4. Eigendecomposition of C by cyclic Jacobi with the parallel round-robin pair order:
//     - Np = N rounded up to even (index N is a dummy that is never rotated), m = Np - 1.  A sweep is the rounds
//       rr = 0..m-1; in round rr index j is paired with mate(j) = m if j == rr, rr if j == m, else (2 rr - j) mod m.
//       All Np / 2 pairs of a round are disjoint, and every pair (p, q), p < q, occurs once per sweep.
//     - Rotation parameters of pair (p, q), all from the matrix at the start of the round: skip the pair when
//       |a_pq| <= 2^-53 tr, tr = sum_e C_ee (from 0.0, echo order, once before the first sweep) — scale invariant, and
//       it lets windows of rank < N (a single slice at r = 2: M - 1 = 24 < 32) converge, whose null-space entries sit
//       at rounding level forever.  Otherwise theta = (a_qq - a_pp) / (2 a_pq), t = 1 / (|theta| + sqrt(theta^2 + 1)),
//       negated when theta < 0, c = 1 / sqrt(t^2 + 1), s = t c.  A skipped pair (and the dummy) has c = 1, s = t = 0.
//     - The round is A <- J^T A J and V <- V J, J holding every pair's rotation (J_pp = J_qq = c, J_pq = s,
//       J_qp = -s).  With rot(c, s, own is p, u_own, w_mate) = own is p ? c u - s w : s w + c u:
//         same pair {i, j}:  a'_pp = a_pp - t a_pq, a'_qq = a_qq + t a_pq, a'_pq = a'_qp = 0 (a_pq kept if skipped);
//         key(i) < key(j) (key = smaller index of the pair):  a'_ij = rot(c_i, s_i, i is p, T_i, T_i')  with
//           T_x = rot(c_j, s_j, j is p, a_xj, a_xj')  (columns first, then rows);
//         key(i) > key(j):  a'_ij = rot(c_j, s_j, j is p, U_j, U_j')  with  U_y = rot(c_i, s_i, i is p, a_iy, a_i'y),
//           the mirror of the entry computed the other way, so A stays exactly symmetric;
//         v'_ej = rot(c_j, s_j, j is p, v_ej, v_ej').
//       (i' = mate(i); rows and columns of the dummy are zero.)
//     - Stop after a sweep that rotates no pair, or after MPPCA_MAX_SWEEPS sweeps.
//     - ell = diag(A) sorted ascending, ties by the lower index; w_j the matching columns of V.
//  5. MP classification.  R = min(N, M - 1), Q = max(N, M - 1), lambda_p = max(ell_{N-R+p}, 0) / Q (p = 0..R-1, the R
//     largest).  S = 0, sigma^2 = 0, cut = 0; for p = 0..R-1: S += lambda_p, gamma = (p + 1) / Q, s1 = S / (p + 1),
//     s2 = (lambda_p - lambda_0) / (4 sqrt(gamma)); if s2 < s1 then sigma^2 = s1, cut = p + 1.  The noise components are
//     the first n_noise = cut + (N - R) in ascending order; n_signal = N - n_noise.
//  6. Reconstruction of the centre voxel only (no aggregation of overlapping patches: each voxel depends only on its
//     own window).  d = x_c - mu; t_j = w_j^T d (from 0.0, echo order) for every signal component j;
//     x_hat_e = max(mu_e + sum_j w_je t_j, 0), the sum from 0.0 over j in ascending eigenvalue order.
//  7. out[c] = x_hat, sigma[c] = sqrt(sigma^2), n_signal[c] (int32).
//  Voxels with mask != 1: out = 0, sigma = 0, n_signal = 0 (as NESMA).  A window holding a non-finite sample: out[c] =
//  the voxel's input, sigma = NaN, n_signal = -1; the eigensolver never sees it.
//  Only IEEE +, -, *, / and sqrt (the library is built with -fmad=false), so NumPy reproduces every bit.
//
// Layout: a compacted list of the masked voxels (three small kernels: per-chunk counts, a serial scan of the chunk
// counts, the ordered list; they also write the zeros of the unmasked voxels), then one warp per listed voxel.  Lane l
// owns echoes / columns l and l + 32.  A and V live in shared memory (Np^2 doubles each: 16 KB per warp at N = 32, 64 KB
// at N = 64): in registers a lane would need a whole column of both, 128 doubles per slot at N = 64.  A round is one
// pass over its Np / 2 row pairs: each lane loads the four entries of A and of V it needs for its column(s), the warp
// synchronises, and each lane stores its two new entries of A and of V.
#include <math.h>

#include "met2_host.h"

namespace met2 {

#ifdef MET2_HOST_EMU
static simt::Shared& S = simt::g_shared;
#else
extern __shared__ __align__(16) double S[];
#endif

constexpr unsigned MP_FULL = 0xffffffffu;
constexpr int MPPCA_MAX_SWEEPS = 32;
constexpr int MPPCA_MAX_WARPS = 4;          // voxels per block of the main kernel
constexpr int MPPCA_CHUNK = 1024;           // voxels per block of the list kernels
constexpr double MPPCA_TINY = 1.1102230246251565e-16;   // 2^-53

__host__ __device__ inline long long mppca_warp_doubles(int N) {
    const int Np = N + (N & 1);
    return 2LL * Np * Np + 6LL * Np;          // A, V, c, s, mu, xs (centred row, then d), ev, tt
}

// ------------------------------------------------------------------------------------------------ masked-voxel list
// Per chunk of MPPCA_CHUNK voxels: the number of voxels with mask == 1 (and the zero outputs of the others).
__global__ void __launch_bounds__(MPPCA_CHUNK) mppca_count_kernel(const int* __restrict__ mask, long long V3, int N,
                                                                  double* __restrict__ out, double* __restrict__ sigma,
                                                                  int* __restrict__ nsig, int* __restrict__ chunk_count) {
    __shared__ int wc[MPPCA_CHUNK / 32];
    const long long v = (long long)blockIdx.x * MPPCA_CHUNK + threadIdx.x;
    const bool in = v < V3 && mask[v] == 1;
    if (v < V3 && !in) {
        for (int e = 0; e < N; ++e) out[v * N + e] = 0.0;
        sigma[v] = 0.0;
        nsig[v] = 0;
    }
    const unsigned b = __ballot_sync(MP_FULL, in);
    if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int w = 0; w < MPPCA_CHUNK / 32; ++w) n += wc[w];
        chunk_count[blockIdx.x] = n;
    }
}

// chunk_off = exclusive prefix sum of chunk_count; total = the list length (one thread: a few hundred chunks)
__global__ void mppca_scan_kernel(const int* __restrict__ chunk_count, int nch, int* __restrict__ chunk_off,
                                  int* __restrict__ total) {
    if (threadIdx.x != 0) return;
    int acc = 0;
    for (int b = 0; b < nch; ++b) {
        chunk_off[b] = acc;
        acc += chunk_count[b];
    }
    *total = acc;
}

// list[chunk_off[b] + rank within the chunk] = v for the voxels with mask == 1, in voxel order
__global__ void __launch_bounds__(MPPCA_CHUNK) mppca_list_kernel(const int* __restrict__ mask, long long V3,
                                                                 const int* __restrict__ chunk_off, int* __restrict__ list) {
    __shared__ int wc[MPPCA_CHUNK / 32];
    const long long v = (long long)blockIdx.x * MPPCA_CHUNK + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const bool in = v < V3 && mask[v] == 1;
    const unsigned b = __ballot_sync(MP_FULL, in);
    if (lane == 0) wc[w] = __popc(b);
    __syncthreads();
    if (in) {
        int pos = chunk_off[blockIdx.x];
        for (int k = 0; k < w; ++k) pos += wc[k];
        pos += __popc(b & ((1u << lane) - 1u));
        list[pos] = (int)v;
    }
}

// ------------------------------------------------------------------------------------------------ the voxel kernel
// rot(c, s, own is p, u_own, w_mate): the new own entry of a (column or row) rotation of the pair
__device__ __forceinline__ double mp_rot(double c, double s, bool own_p, double u, double w) {
    return own_p ? c * u - s * w : s * w + c * u;
}

__device__ __forceinline__ int mp_mate(int j, int rr, int m) {
    if (j == m) return rr;
    if (j == rr) return m;
    int k = (2 * rr - j) % m;
    return k < 0 ? k + m : k;
}

template <int NSL>
__global__ void __launch_bounds__(MPPCA_MAX_WARPS * 32) mppca_kernel(const double* __restrict__ vol,
                                                                    const int* __restrict__ list,
                                                                    const int* __restrict__ total, int nx, int ny,
                                                                    int nz, int N, int r, int wpb,
                                                                    double* __restrict__ out, double* __restrict__ sigma,
                                                                    int* __restrict__ nsig) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long li = (long long)blockIdx.x * wpb + w;
    if (li >= *total) return;                               // warp-uniform
    const long long v = list[li];
    const int cz = (int)(v % nz), cy = (int)((v / nz) % ny), cx = (int)(v / ((long long)nz * ny));
    const int wx = min(2 * r + 1, nx), wy = min(2 * r + 1, ny), wz = min(2 * r + 1, nz);
    const int sx = min(max(cx - r, 0), nx - wx), sy = min(max(cy - r, 0), ny - wy), sz = min(max(cz - r, 0), nz - wz);
    const int M = wx * wy * wz;
    const int Np = N + (N & 1), m = Np - 1;
    const long long base = (long long)w * mppca_warp_doubles(N);
    const long long oA = base, oV = oA + (long long)Np * Np, oC = oV + (long long)Np * Np, oS = oC + Np, oMu = oS + Np,
                    oX = oMu + Np, oE = oX + Np, oT = oE + Np;
    // 2. mean, and the non-finite check
    double mu[NSL];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int e = lane + 32 * k;
        double acc = 0.0;
        if (e < N) {
            for (int ix = sx; ix < sx + wx; ++ix)
                for (int iy = sy; iy < sy + wy; ++iy)
                    for (int iz = sz; iz < sz + wz; ++iz) {
                        const double x = vol[(((long long)ix * ny + iy) * nz + iz) * N + e];
                        bad |= !isfinite(x);
                        acc = acc + x;
                    }
        }
        mu[k] = acc / (double)M;
    }
    if (__any_sync(MP_FULL, bad)) {
#pragma unroll
        for (int k = 0; k < NSL; ++k) {
            const int e = lane + 32 * k;
            if (e < N) out[v * N + e] = vol[v * N + e];
        }
        if (lane == 0) {
            sigma[v] = NAN;
            nsig[v] = -1;
        }
        return;
    }
    // A = 0, V = I (dummy row and column zero)
    for (int i = lane; i < Np * Np; i += 32) {
        const int a = i / Np, b = i - a * Np;
        S[oA + i] = 0.0;
        S[oV + i] = (a == b && a < N) ? 1.0 : 0.0;
    }
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int e = lane + 32 * k;
        if (e < N) S[oMu + e] = mu[k];
    }
    __syncwarp();
    // 3. covariance: per sample, the centred row in shared memory, then each lane adds its column(s)
    for (int ix = sx; ix < sx + wx; ++ix)
        for (int iy = sy; iy < sy + wy; ++iy)
            for (int iz = sz; iz < sz + wz; ++iz) {
                const double* row = vol + (((long long)ix * ny + iy) * nz + iz) * N;
#pragma unroll
                for (int k = 0; k < NSL; ++k) {
                    const int e = lane + 32 * k;
                    if (e < N) S[oX + e] = row[e] - mu[k];
                }
                __syncwarp();
#pragma unroll
                for (int k = 0; k < NSL; ++k) {
                    const int f = lane + 32 * k;
                    if (f < N) {
                        const double xf = S[oX + f];
                        for (int e = 0; e < N; ++e) S[oA + e * Np + f] = S[oA + e * Np + f] + S[oX + e] * xf;
                    }
                }
                __syncwarp();
            }
    double tr = 0.0;
    for (int e = 0; e < N; ++e) tr = tr + S[oA + e * Np + e];
    const double thr = MPPCA_TINY * tr;
    // 4. cyclic Jacobi, round-robin pairs
    for (int sweep = 0; sweep < MPPCA_MAX_SWEEPS; ++sweep) {
        bool any = false;
        for (int rr = 0; rr < m; ++rr) {
            double cj[NSL], sj[NSL], tj[NSL], app[NSL], aqq[NSL], apq[NSL];
            bool rot[NSL];
#pragma unroll
            for (int k = 0; k < NSL; ++k) {
                const int j = lane + 32 * k;
                cj[k] = 1.0, sj[k] = 0.0, tj[k] = 0.0, app[k] = aqq[k] = apq[k] = 0.0, rot[k] = false;
                if (j < N) {
                    const int j2 = mp_mate(j, rr, m);
                    const int p = min(j, j2), q = max(j, j2);
                    app[k] = S[oA + p * Np + p];
                    aqq[k] = S[oA + q * Np + q];            // the dummy's row and column are zero
                    apq[k] = S[oA + p * Np + q];
                    if (q < N) {
                        if (!(fabs(apq[k]) <= thr)) {
                            const double theta = (aqq[k] - app[k]) / (2.0 * apq[k]);
                            double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
                            if (theta < 0.0) t = -t;
                            const double c = 1.0 / sqrt(t * t + 1.0);
                            cj[k] = c, sj[k] = t * c, tj[k] = t, rot[k] = true;
                        }
                    }
                    S[oC + j] = cj[k];
                    S[oS + j] = sj[k];
                    any |= rot[k];
                }
            }
            __syncwarp();
            for (int pk = 0; pk < Np / 2; ++pk) {
                const int a0 = pk == 0 ? rr : (rr + pk) % m;
                const int a1 = pk == 0 ? m : (rr - pk + m) % m;
                const int pi = min(a0, a1), qi = max(a0, a1);
                const double ci = S[oC + pi], si = S[oS + pi];
                double nap[NSL], naq[NSL], nvp[NSL], nvq[NSL];
#pragma unroll
                for (int k = 0; k < NSL; ++k) {
                    const int j = lane + 32 * k;
                    nap[k] = naq[k] = nvp[k] = nvq[k] = 0.0;
                    if (j < N) {
                        const int j2 = mp_mate(j, rr, m);
                        const bool jp = j < j2;
                        const double xpj = S[oA + pi * Np + j], xpj2 = S[oA + pi * Np + j2];
                        const double xqj = S[oA + qi * Np + j], xqj2 = S[oA + qi * Np + j2];
                        if (j == pi) {
                            nap[k] = app[k] - tj[k] * apq[k];
                            naq[k] = rot[k] ? 0.0 : apq[k];
                        } else if (j == qi) {
                            nap[k] = rot[k] ? 0.0 : apq[k];
                            naq[k] = aqq[k] + tj[k] * apq[k];
                        } else if (pi < min(j, j2)) {            // columns first (pair of j), then rows (pair of i)
                            const double Tp = mp_rot(cj[k], sj[k], jp, xpj, xpj2);
                            const double Tq = mp_rot(cj[k], sj[k], jp, xqj, xqj2);
                            nap[k] = mp_rot(ci, si, true, Tp, Tq);
                            naq[k] = mp_rot(ci, si, false, Tq, Tp);
                        } else {                                  // the mirror: columns by the pair of i, rows by j's
                            const double Up = mp_rot(ci, si, true, xpj, xqj), Up2 = mp_rot(ci, si, true, xpj2, xqj2);
                            const double Uq = mp_rot(ci, si, false, xqj, xpj), Uq2 = mp_rot(ci, si, false, xqj2, xpj2);
                            nap[k] = mp_rot(cj[k], sj[k], jp, Up, Up2);
                            naq[k] = mp_rot(cj[k], sj[k], jp, Uq, Uq2);
                        }
                        nvp[k] = mp_rot(cj[k], sj[k], jp, S[oV + pi * Np + j], S[oV + pi * Np + j2]);
                        nvq[k] = mp_rot(cj[k], sj[k], jp, S[oV + qi * Np + j], S[oV + qi * Np + j2]);
                    }
                }
                __syncwarp();
#pragma unroll
                for (int k = 0; k < NSL; ++k) {
                    const int j = lane + 32 * k;
                    if (j < N) {
                        S[oA + pi * Np + j] = nap[k];
                        S[oV + pi * Np + j] = nvp[k];
                        if (qi < N) {
                            S[oA + qi * Np + j] = naq[k];
                            S[oV + qi * Np + j] = nvq[k];
                        }
                    }
                }
            }
            __syncwarp();
        }
        if (!__any_sync(MP_FULL, any)) break;
    }
    // ascending eigenvalues (ties: lower index first) and their column indices
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int j = lane + 32 * k;
        if (j < N) {
            const double d = S[oA + j * Np + j];
            int rank = 0;
            for (int i = 0; i < N; ++i) {
                const double di = S[oA + i * Np + i];
                rank += (di < d || (di == d && i < j));
            }
            S[oE + rank] = d;
            S[oT + rank] = (double)j;           // column index, read back before tt overwrites it
        }
    }
    __syncwarp();
    // 5. MP classification (every lane, the same sequence)
    const int R = min(N, M - 1);
    const double Q = (double)max(N, M - 1);
    const int off = N - R;
    double Ssum = 0.0, sigma2 = 0.0;
    int cut = 0;
    const double e0 = S[oE + off];
    const double l0 = (e0 > 0.0 ? e0 : 0.0) / Q;
    for (int p = 0; p < R; ++p) {
        const double ep = S[oE + off + p];
        const double lp = (ep > 0.0 ? ep : 0.0) / Q;
        Ssum = Ssum + lp;
        const double gamma = (double)(p + 1) / Q;
        const double s1 = Ssum / (double)(p + 1);
        const double s2 = (lp - l0) / (4.0 * sqrt(gamma));
        if (s2 < s1) {
            sigma2 = s1;
            cut = p + 1;
        }
    }
    const int n_noise = cut + off;
    // 6. reconstruction of the centre voxel
    int col[NSL];
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int j = lane + 32 * k;
        col[k] = j < N ? (int)S[oT + j] : 0;
        if (j < N) S[oX + j] = vol[v * N + j] - mu[k];
    }
    __syncwarp();
    double tt[NSL];
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int pos = lane + 32 * k;
        tt[k] = 0.0;
        if (pos >= n_noise && pos < N) {
            double acc = 0.0;
            for (int e = 0; e < N; ++e) acc = acc + S[oV + e * Np + col[k]] * S[oX + e];
            tt[k] = acc;
        }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int pos = lane + 32 * k;
        if (pos < N) S[oT + pos] = tt[k];
        if (pos < N) S[oX + pos] = (double)col[k];   // the column of sorted position pos
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NSL; ++k) {
        const int e = lane + 32 * k;
        if (e < N) {
            double acc = 0.0;
            for (int pos = n_noise; pos < N; ++pos) acc = acc + S[oV + e * Np + (int)S[oX + pos]] * S[oT + pos];
            const double x = mu[k] + acc;
            out[v * N + e] = x > 0.0 ? x : 0.0;
        }
    }
    if (lane == 0) {
        sigma[v] = sqrt(sigma2);
        nsig[v] = N - n_noise;
    }
}

struct MppcaWs {
    int* chunk_count;
    int* chunk_off;
    int* total;
    int* list;
};

static size_t mppca_carve(long long V3, void* ws, MppcaWs* W) {
    const long long nch = (V3 + MPPCA_CHUNK - 1) / MPPCA_CHUNK;
    const size_t a = align256((size_t)nch * sizeof(int)), t = align256(sizeof(int)),
                 l = align256((size_t)V3 * sizeof(int));
    if (W) {
        char* p = (char*)ws;
        W->chunk_count = (int*)p;
        W->chunk_off = (int*)(p + a);
        W->total = (int*)(p + 2 * a);
        W->list = (int*)(p + 2 * a + t);
    }
    return 2 * a + t + l;
}

static int mppca_check(const char* what, int nx, int ny, int nz, int nt, int r) {
    if (nx < 1 || ny < 1 || nz < 1 || nt < 1 || nt > MET2_MAX_NTE || r < 1 || (long long)nx * ny * nz > 0x7fffffffLL)
        return set_error(MET2_ERR_ARG, "%s: bad sizes nx=%d ny=%d nz=%d nt=%d r=%d", what, nx, ny, nz, nt, r);
    const long long M = (long long)min(2 * r + 1, nx) * min(2 * r + 1, ny) * min(2 * r + 1, nz);
    if (M < 2) return set_error(MET2_ERR_ARG, "%s: the window holds %lld sample(s), at least 2 needed", what, M);
    return MET2_OK;
}

}  // namespace met2

using namespace met2;

extern "C" int64_t met2_mppca_workspace_bytes(int nx, int ny, int nz, int nt, int r) {
    if (mppca_check("met2_mppca_workspace_bytes", nx, ny, nz, nt, r)) return MET2_ERR_ARG;
    return (int64_t)mppca_carve((long long)nx * ny * nz, nullptr, nullptr);
}

extern "C" int met2_mppca(const double* vol, const int32_t* mask, int nx, int ny, int nz, int nt, int r, double* out,
                          double* sigma, int32_t* n_signal, void* workspace, void* stream) {
    int rc = mppca_check("met2_mppca", nx, ny, nz, nt, r);
    if (rc) return rc;
    if (!vol || !mask || !out || !sigma || !n_signal || !workspace)
        return set_error(MET2_ERR_ARG, "met2_mppca: NULL argument");
    if ((const void*)out == (const void*)vol) return set_error(MET2_ERR_ARG, "met2_mppca: out must not alias vol");
    cudaStream_t st = (cudaStream_t)stream;
    const long long V3 = (long long)nx * ny * nz;
    const unsigned nch = (unsigned)((V3 + MPPCA_CHUNK - 1) / MPPCA_CHUNK);
    MppcaWs W;
    mppca_carve(V3, workspace, &W);
    const size_t per_warp = sizeof(double) * (size_t)mppca_warp_doubles(nt);
    int wpb = (int)((227 * 1024 - 1024) / per_warp);
    if (wpb > MPPCA_MAX_WARPS) wpb = MPPCA_MAX_WARPS;
    const size_t smem = per_warp * wpb;
    cudaError_t e = nt <= 32 ? cudaFuncSetAttribute(mppca_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                             : cudaFuncSetAttribute(mppca_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "mppca_kernel attr (%zu B): %s", smem, cudaGetErrorString(e));
    MET2_LAUNCH(nch, MPPCA_CHUNK, 0, st, mppca_count_kernel)(mask, V3, nt, out, sigma, n_signal, W.chunk_count);
    MET2_LAUNCH(1, 32, 0, st, mppca_scan_kernel)(W.chunk_count, (int)nch, W.chunk_off, W.total);
    MET2_LAUNCH(nch, MPPCA_CHUNK, 0, st, mppca_list_kernel)(mask, V3, W.chunk_off, W.list);
    // one warp per listed voxel; the list length stays on the device, so blocks past it return at once
    const unsigned blocks = (unsigned)((V3 + wpb - 1) / wpb);
    if (nt <= 32)
        MET2_LAUNCH(blocks, wpb * 32, smem, st, mppca_kernel<1>)(vol, W.list, W.total, nx, ny, nz, nt, r, wpb, out, sigma,
                                                                 n_signal);
    else
        MET2_LAUNCH(blocks, wpb * 32, smem, st, mppca_kernel<2>)(vol, W.list, W.total, nx, ny, nz, nt, r, wpb, out, sigma,
                                                                 n_signal);
    count_launch(4);
    return check_launch("met2_mppca");
}
