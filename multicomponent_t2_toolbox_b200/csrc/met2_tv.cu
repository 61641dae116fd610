// met2_tv.cu — Step 1 with --denoise TV (motor/motor_recon_met2_real_data.py:293-303 of the reference): per echo volume,
// scikit-image's wavelet noise estimate (estimate_sigma -> _sigma_est_dwt on PyWavelets' single-level db2 transform) and
// its Chambolle total-variation filter (_denoise_tv_chambolle_nd) with weight 2 sigma, eps 2e-4, at most 200 iterations.
//
// Both follow the NumPy restatement of tests/tv_oracle.py operation for operation (built with -fmad=false), so every
// field, the iteration count and sigma are bitwise equal to it:
//  * met2_noise_sigma: one launch per db2 high-pass pass (axis 0, 1, 2 of the squeezed volume), then one block per echo
//    takes the exact median of |c| over the nonzero coefficients by radix selection on the 64-bit patterns of |c|
//    (monotone for non-negative doubles).
//  * met2_tv_chambolle: the fields live echo-major in the workspace; every iteration is four launches over the echoes that
//    are still running — (a) out = image + d(p) and d^2, (b) g, |g| and the in-place p update, (c) the pairwise partial
//    sums of d^2 and |g|, (d) one block that finishes both sums, applies the stop test and rebuilds the list of running
//    echoes.  No grid-wide barrier and no block waits on another, so the SIMT emulator (tests/emu) runs the same code.
//
// The energy sums reproduce NumPy's whole-array `.sum()` (DOUBLE_pairwise_sum over the flattened C-order array): the
// recursion halves n at n / 2 rounded down to a multiple of 8 until n <= 128, where a leaf sums with eight interleaved
// accumulators.  The recursion depth K at which the smallest node first has n <= 128 splits the array into 2^K nodes of
// at most 2 leaves each; above them the tree is perfect, so it is combined pairwise (2i, 2i + 1) level by level.
#include <math.h>

#include "met2_host.h"

namespace met2 {

constexpr unsigned TV_FULL = 0xffffffffu;
constexpr int TV_LEAF = 128;         // NumPy's PW_BLOCKSIZE
constexpr int TV_THREADS = 256;      // threads of the per-voxel kernels and of the partial-sum kernel
constexpr int TV_NODES_PER_BLOCK = TV_THREADS / 8;   // partial-sum kernel: 8 lanes per depth-K node
constexpr int TV_FIN_THREADS = 256;

// the squeezed volume: its axes of size > 1, in order, with their flat (C-order) strides
struct TvGeom {
    long long n;          // voxels per echo
    int nd;               // number of axes of size > 1 (1..3)
    int size[3];
    long long stride[3];
    int depth;            // K
    int nodes;            // 2^K
    int parts;            // partial sums per echo and field written by the partial-sum kernel: max(1, nodes / 32)
};

__host__ __device__ inline long long pairwise_left(long long n) {
    const long long h = n / 2;
    return h - h % 8;
}

// ------------------------------------------------------------------------------------------------ layout
// in [rows][cols] -> out [cols][rows] through a 32 x 32 tile; 1-D grid of ceil(rows/32) * ceil(cols/32) blocks of 32 x 8
__global__ void tv_transpose_kernel(const double* __restrict__ in, double* __restrict__ out, long long rows, int cols) {
    __shared__ double tile[32][33];
    const long long nrb = (rows + 31) / 32;
    const long long rb = ((long long)blockIdx.x % nrb) * 32;
    const int cb = (int)((long long)blockIdx.x / nrb) * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const long long row = rb + r;
        const int col = cb + (int)threadIdx.x;
        tile[r][threadIdx.x] = (row < rows && col < cols) ? in[row * cols + col] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int col = cb + r;
        const long long row = rb + threadIdx.x;
        if (row < rows && col < cols) out[(size_t)col * rows + row] = tile[threadIdx.x][r];
    }
}

// ------------------------------------------------------------------------------------------------ noise sigma
// One db2 high-pass pass along `axis` of the [nt][n0][n1][n2] view (element strides s_t, s[0..2]):
// out[o] = sum_j dec_hi[j] * ext(2o + 1 - j), summed from 0.0 with j ascending, ext = PyWavelets' 'symmetric' mode.
// out is [nt][m0][m1][m2] contiguous with m_axis = (n_axis + 3) / 2.
__global__ void tv_dwt_hi_kernel(const double* __restrict__ in, long long s_t, long long s0, long long s1, long long s2,
                                 int n0, int n1, int n2, int nt, int axis, double* __restrict__ out) {
    const double h[4] = {-0.48296291314469025, 0.836516303737469, -0.22414386804185735, -0.12940952255092145};
    const int m0 = axis == 0 ? (n0 + 3) / 2 : n0;
    const int m1 = axis == 1 ? (n1 + 3) / 2 : n1;
    const int m2 = axis == 2 ? (n2 + 3) / 2 : n2;
    const long long per = (long long)m0 * m1 * m2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= per * nt) return;
    const int t = (int)(idx / per);
    long long r = idx - (long long)t * per;
    const int o2 = (int)(r % m2);
    r /= m2;
    const int o1 = (int)(r % m1);
    const int o0 = (int)(r / m1);
    const int o = axis == 0 ? o0 : (axis == 1 ? o1 : o2);
    const int n = axis == 0 ? n0 : (axis == 1 ? n1 : n2);
    const long long sa = axis == 0 ? s0 : (axis == 1 ? s1 : s2);
    const long long base = (long long)t * s_t + (axis == 0 ? 0 : (long long)o0 * s0) + (axis == 1 ? 0 : (long long)o1 * s1) +
                           (axis == 2 ? 0 : (long long)o2 * s2);
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int k = (2 * o + 1 - j) % (2 * n);
        if (k < 0) k += 2 * n;
        const int src = k < n ? k : 2 * n - 1 - k;
        acc = acc + h[j] * in[base + (long long)src * sa];
    }
    out[idx] = acc;
}

// One block per echo: sigma = median(|c| over c != 0) / norm.ppf(0.75), NumPy's median (mean of the two middle values
// for an even count); NaN if a coefficient is NaN or none is nonzero.
__global__ void __launch_bounds__(256) tv_sigma_median_kernel(const double* __restrict__ band, long long B,
                                                              double* __restrict__ sigma) {
    __shared__ unsigned long long hist[256];
    __shared__ unsigned long long s_cnt[2];
    __shared__ unsigned long long s_prefix, s_k;
    const double* c = band + (size_t)blockIdx.x * B;
    const int tid = threadIdx.x;
    if (tid == 0) s_cnt[0] = s_cnt[1] = 0;
    __syncthreads();
    unsigned long long nz = 0, nn = 0;
    for (long long i = tid; i < B; i += blockDim.x) {
        const double x = c[i];
        nz += (x != 0.0);
        nn += (x != x);
    }
    atomicAdd(&s_cnt[0], nz);
    atomicAdd(&s_cnt[1], nn);
    __syncthreads();
    const unsigned long long count = s_cnt[0];
    if (s_cnt[1] != 0 || count == 0) {
        if (tid == 0) sigma[blockIdx.x] = NAN;
        return;
    }
    double mid[2];
    const int nsel = (count % 2) ? 1 : 2;
    for (int q = 0; q < nsel; ++q) {
        unsigned long long k = (count % 2) ? (count - 1) / 2 : count / 2 - 1 + q;   // rank among the nonzero |c|
        unsigned long long prefix = 0, known = 0;
        for (int shift = 56; shift >= 0; shift -= 8) {
            for (int b = tid; b < 256; b += blockDim.x) hist[b] = 0;
            __syncthreads();
            for (long long i = tid; i < B; i += blockDim.x) {
                const double x = c[i];
                if (x != 0.0) {
                    const unsigned long long u = (unsigned long long)__double_as_longlong(fabs(x));
                    if ((u & known) == prefix) atomicAdd(&hist[(u >> shift) & 255], 1ull);
                }
            }
            __syncthreads();
            if (tid == 0) {
                unsigned long long cum = 0;
                int b = 0;
                while (b < 255 && cum + hist[b] <= k) cum += hist[b++];
                s_k = k - cum;
                s_prefix = prefix | ((unsigned long long)b << shift);
            }
            __syncthreads();
            k = s_k;
            prefix = s_prefix;
            known |= 255ull << shift;
        }
        mid[q] = __longlong_as_double((long long)prefix);
    }
    if (tid == 0) {
        const double med = nsel == 1 ? mid[0] : (mid[0] + mid[1]) / 2.0;
        sigma[blockIdx.x] = med / 0.6744897501960817;
    }
}

// ------------------------------------------------------------------------------------------------ TV (Chambolle)
__global__ void tv_init_kernel(int nt, int* __restrict__ active, int32_t* __restrict__ iterations) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nt) return;
    active[1 + t] = t;
    iterations[t] = 0;
    if (t == 0) active[0] = nt;
}

// (a) out = image + d with d = -p.sum(0), then d[1:] += p[ax][:-1] per axis; sq = d**2.  At the first iteration
// out = image and d = 0.  One thread per voxel; blocks stride over (running echo, voxel block).
__global__ void __launch_bounds__(TV_THREADS) tv_out_kernel(const double* __restrict__ img, const double* __restrict__ p,
                                                            const int* __restrict__ active, TvGeom g, int first,
                                                            double* __restrict__ out, double* __restrict__ sq) {
    const long long N = g.n;
    const long long bpe = (N + TV_THREADS - 1) / TV_THREADS;
    const long long items = (long long)active[0] * bpe;
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int e = active[1 + item / bpe];
        const long long v = (item % bpe) * TV_THREADS + threadIdx.x;
        if (v >= N) continue;
        const size_t ev = (size_t)e * N + v;
        if (first) {
            out[ev] = img[ev];
            sq[ev] = 0.0;
            continue;
        }
        const double* pe = p + (size_t)e * g.nd * N;
        double s = 0.0;   // NumPy's reduction starts from the identity
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a < g.nd) s = s + pe[(size_t)a * N + v];
        double d = -s;
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a < g.nd && (v / g.stride[a]) % g.size[a] > 0) d = d + pe[(size_t)a * N + v - g.stride[a]];
        out[ev] = img[ev] + d;
        sq[ev] = d * d;
    }
}

// (b) g[ax] = diff(out, ax) (0 on the last slice), nrm = sqrt(sum g^2) -> sq; nrm = nrm * (tau / w) + 1;
// p = (p - tau g) / nrm.  Thread v alone reads and writes p(v).
__global__ void __launch_bounds__(TV_THREADS) tv_p_kernel(const double* __restrict__ out, double* __restrict__ p,
                                                          const int* __restrict__ active, TvGeom g,
                                                          const double* __restrict__ weight, double* __restrict__ sq) {
    const long long N = g.n;
    const long long bpe = (N + TV_THREADS - 1) / TV_THREADS;
    const long long items = (long long)active[0] * bpe;
    const double tau = 1.0 / (2.0 * g.nd);
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int e = active[1 + item / bpe];
        const long long v = (item % bpe) * TV_THREADS + threadIdx.x;
        if (v >= N) continue;
        const double* oe = out + (size_t)e * N;
        double* pe = p + (size_t)e * g.nd * N;
        const double o = oe[v];
        double gr[3];
        double n2 = 0.0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            gr[a] = 0.0;
            if (a < g.nd) {
                if ((v / g.stride[a]) % g.size[a] < g.size[a] - 1) gr[a] = oe[v + g.stride[a]] - o;
                n2 = n2 + gr[a] * gr[a];
            }
        }
        double nrm = sqrt(n2);
        sq[(size_t)e * N + v] = nrm;
        nrm = nrm * (tau / weight[e]);
        nrm = nrm + 1.0;
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a < g.nd) pe[(size_t)a * N + v] = (pe[(size_t)a * N + v] - tau * gr[a]) / nrm;
    }
}

// NumPy's pairwise leaf (n <= 128) of a[0..n) by the 8 lanes of a group (j = lane within the group): accumulator j on
// lane j, combined ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)) by xor shuffles, then the tail.  Every lane of the
// warp must call it (shuffles); all 8 lanes of a group return the same value.
__device__ __forceinline__ double tv_leaf8(const double* __restrict__ a, int n, int j) {
    const int nb = n - n % 8;
    double r = 0.0;
    if (n >= 8) {
        r = a[j];
        for (int i = 8 + j; i < nb; i += 8) r += a[i];
    }
    r += __shfl_xor_sync(TV_FULL, r, 1);
    r += __shfl_xor_sync(TV_FULL, r, 2);
    r += __shfl_xor_sync(TV_FULL, r, 4);
    double res;
    if (n < 8) {
        res = 0.0;
        for (int i = 0; i < n; ++i) res += a[i];
    } else {
        res = r;
        for (int i = nb; i < n; ++i) res += a[i];
    }
    return res;
}

// (c) per running echo, the sums of sq_d and sq_n over the depth-K nodes [32 b, 32 b + 32), combined as the perfect tree
// they form -> part[e][0][b], part[e][1][b].  8 lanes per node.
__global__ void __launch_bounds__(TV_THREADS) tv_partials_kernel(const double* __restrict__ sq_d,
                                                                 const double* __restrict__ sq_n,
                                                                 const int* __restrict__ active, TvGeom g,
                                                                 double* __restrict__ part) {
    __shared__ double vals[2][TV_NODES_PER_BLOCK];
    const long long N = g.n;
    const int bpe = g.parts;
    const long long items = (long long)active[0] * bpe;
    const int grp = threadIdx.x >> 3, j = threadIdx.x & 7;
    const int cnt = g.nodes < TV_NODES_PER_BLOCK ? g.nodes : TV_NODES_PER_BLOCK;
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int e = active[1 + item / bpe];
        const int blk = (int)(item % bpe);
        const int node = blk * TV_NODES_PER_BLOCK + grp;
        long long start = 0, n = 0;
        if (node < g.nodes) {            // descend from the root along the bits of the node index
            n = N;
            for (int bit = g.depth - 1; bit >= 0; --bit) {
                const long long l = pairwise_left(n);
                if ((node >> bit) & 1) {
                    start += l;
                    n -= l;
                } else {
                    n = l;
                }
            }
        }
        const long long na = n > TV_LEAF ? pairwise_left(n) : n, nb = n - na;   // nb > 0: two leaves, each <= 128
        const double* d = sq_d + (size_t)e * N + start;
        const double* q = sq_n + (size_t)e * N + start;
        double vd = tv_leaf8(d, (int)na, j), vn = tv_leaf8(q, (int)na, j);
        const double vd2 = tv_leaf8(d + na, (int)nb, j), vn2 = tv_leaf8(q + na, (int)nb, j);
        if (nb > 0) {
            vd = vd + vd2;
            vn = vn + vn2;
        }
        if (j == 0) {
            vals[0][grp] = vd;
            vals[1][grp] = vn;
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            double x = vals[0][threadIdx.x], y = vals[1][threadIdx.x];
            for (int o = 1; o < cnt; o <<= 1) {
                x += __shfl_xor_sync(TV_FULL, x, o);
                y += __shfl_xor_sync(TV_FULL, y, o);
            }
            if (threadIdx.x == 0) {
                part[((size_t)e * 2 + 0) * bpe + blk] = x;
                part[((size_t)e * 2 + 1) * bpe + blk] = y;
            }
        }
        __syncthreads();
    }
}

// perfect pairwise tree over v[0..P) (P a power of two) by one warp; lane 0's result is the sum
__device__ double tv_warp_tree(const double* __restrict__ v, int P, int lane) {
    double x;
    if (P >= 32) {
        const int per = P / 32;
        double st[32];
        int lv[32], sp = 0;
        for (int k = 0; k < per; ++k) {
            double cur = v[lane * per + k];
            int l = 0;
            while (sp > 0 && lv[sp - 1] == l) {
                cur = st[sp - 1] + cur;
                --sp;
                ++l;
            }
            st[sp] = cur;
            lv[sp] = l;
            ++sp;
        }
        x = st[0];
    } else {
        x = lane < P ? v[lane] : 0.0;
    }
    const int cnt = P < 32 ? P : 32;
    for (int o = 1; o < cnt; o <<= 1) x += __shfl_xor_sync(TV_FULL, x, o);
    return x;
}

// (d) one block: per running echo E = (sum d^2 + w * sum |g|) / N and the stop test of _denoise_tv_chambolle_nd; a finished
// echo gets its iteration count (i + 1 at the break, max_iter at the cap) and leaves the list of running echoes.
__global__ void __launch_bounds__(TV_FIN_THREADS) tv_energy_kernel(const double* __restrict__ part, TvGeom g,
                                                                   const double* __restrict__ weight, double eps, int it,
                                                                   int max_iter, int* __restrict__ active,
                                                                   double* __restrict__ e_init, double* __restrict__ e_prev,
                                                                   int32_t* __restrict__ iterations) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int n_active = active[0];
    const int P = g.parts;
    for (int k = warp; k < n_active; k += nwarps) {
        const int e = active[1 + k];
        const double sd = tv_warp_tree(part + (size_t)e * 2 * P, P, lane);
        const double sn = tv_warp_tree(part + ((size_t)e * 2 + 1) * P, P, lane);
        if (lane == 0) {
            double E = sd;
            E += weight[e] * sn;
            E /= (double)g.n;
            int done = 0;
            if (it == 0) {
                e_init[e] = E;
                e_prev[e] = E;
            } else if (fabs(e_prev[e] - E) < eps * e_init[e]) {
                done = it + 1;
            } else {
                e_prev[e] = E;
            }
            if (!done && it + 1 == max_iter) done = max_iter;
            if (done) iterations[e] = done;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int m = 0;
        for (int k = 0; k < n_active; ++k) {
            const int e = active[1 + k];
            if (iterations[e] == 0) active[1 + m++] = e;
        }
        active[0] = m;
    }
}

struct TvPlan {
    TvGeom g;
    size_t off_img, off_out, off_p, off_sqd, off_sqn, off_part, off_einit, off_eprev, off_active, bytes;
};

static bool tv_sizes_ok(int nx, int ny, int nz, int nt) {
    return nx > 0 && ny > 0 && nz > 0 && nt > 0 && (nx > 1 || ny > 1 || nz > 1);
}

static TvGeom tv_geometry(int nx, int ny, int nz) {
    TvGeom g = {};
    g.n = (long long)nx * ny * nz;
    const int dims[3] = {nx, ny, nz};
    const long long strides[3] = {(long long)ny * nz, nz, 1};
    for (int a = 0; a < 3; ++a)
        if (dims[a] > 1) {
            g.size[g.nd] = dims[a];
            g.stride[g.nd] = strides[a];
            ++g.nd;
        }
    for (int a = g.nd; a < 3; ++a) {
        g.size[a] = 1;
        g.stride[a] = 1;
    }
    long long m = g.n;
    while (m > TV_LEAF) {   // the smallest node at each depth is the left child of the smallest node above it
        m = pairwise_left(m);
        ++g.depth;
    }
    g.nodes = 1 << g.depth;
    g.parts = g.nodes > TV_NODES_PER_BLOCK ? g.nodes / TV_NODES_PER_BLOCK : 1;
    return g;
}

static TvPlan tv_plan(int nx, int ny, int nz, int nt) {
    TvPlan pl;
    pl.g = tv_geometry(nx, ny, nz);
    const size_t field = (size_t)nt * pl.g.n * sizeof(double);
    size_t o = 0;
    pl.off_img = o;
    o += align256(field);
    pl.off_out = o;
    o += align256(field);
    pl.off_p = o;
    o += align256(field * pl.g.nd);
    pl.off_sqd = o;
    o += align256(field);
    pl.off_sqn = o;
    o += align256(field);
    pl.off_part = o;
    o += align256((size_t)nt * 2 * pl.g.parts * sizeof(double));
    pl.off_einit = o;
    o += align256((size_t)nt * sizeof(double));
    pl.off_eprev = o;
    o += align256((size_t)nt * sizeof(double));
    pl.off_active = o;
    o += align256((size_t)(nt + 1) * sizeof(int));
    pl.bytes = o;
    return pl;
}

// sizes of the band after each db2 pass; returns the largest intermediate (doubles per echo)
static long long sigma_band(int nx, int ny, int nz, int dims_out[3]) {
    int d[3] = {nx, ny, nz};
    long long largest = 1;
    for (int a = 0; a < 3; ++a) {
        if (d[a] > 1) d[a] = (d[a] + 3) / 2;
        const long long s = (long long)d[0] * d[1] * d[2];
        if (s > largest) largest = s;
    }
    for (int a = 0; a < 3; ++a) dims_out[a] = d[a];
    return largest;
}

}  // namespace met2

using namespace met2;

extern "C" int64_t met2_noise_sigma_workspace_bytes(int nx, int ny, int nz, int nt) {
    if (!tv_sizes_ok(nx, ny, nz, nt)) return set_error(MET2_ERR_ARG, "met2_noise_sigma_workspace_bytes: bad size");
    int dims[3];
    const long long largest = sigma_band(nx, ny, nz, dims);
    return (int64_t)(2 * align256((size_t)nt * largest * sizeof(double)));
}

extern "C" int met2_noise_sigma(const double* vol, int nx, int ny, int nz, int nt, double* sigma, void* workspace,
                                void* stream) {
    if (!vol || !sigma || !workspace || !tv_sizes_ok(nx, ny, nz, nt))
        return set_error(MET2_ERR_ARG, "met2_noise_sigma: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    int dims_out[3];
    const long long largest = sigma_band(nx, ny, nz, dims_out);
    double* buf[2] = {(double*)workspace, (double*)((char*)workspace + align256((size_t)nt * largest * sizeof(double)))};
    // pass 1 reads the caller's [nx][ny][nz][nt] volume; later passes read the previous [nt][m0][m1][m2] band
    const double* in = vol;
    long long s_t = 1, s[3] = {(long long)ny * nz * nt, (long long)nz * nt, nt};
    int n[3] = {nx, ny, nz};
    int launches = 0;
    for (int a = 0; a < 3; ++a) {
        if (n[a] == 1) continue;   // np.squeeze: an axis of size 1 is not transformed
        double* o = buf[launches % 2];
        const long long total = (long long)nt * n[0] * n[1] * n[2] / n[a] * ((n[a] + 3) / 2);
        MET2_LAUNCH((unsigned)((total + 255) / 256), 256, 0, st, tv_dwt_hi_kernel)(in, s_t, s[0], s[1], s[2], n[0], n[1],
                                                                                   n[2], nt, a, o);
        ++launches;
        n[a] = (n[a] + 3) / 2;
        s[2] = 1;
        s[1] = n[2];
        s[0] = (long long)n[1] * n[2];
        s_t = (long long)n[0] * n[1] * n[2];
        in = o;
    }
    MET2_LAUNCH((unsigned)nt, 256, 0, st, tv_sigma_median_kernel)(in, (long long)n[0] * n[1] * n[2], sigma);
    count_launch(launches + 1);
    return check_launch("met2_noise_sigma");
}

extern "C" int64_t met2_tv_workspace_bytes(int nx, int ny, int nz, int nt) {
    if (!tv_sizes_ok(nx, ny, nz, nt)) return set_error(MET2_ERR_ARG, "met2_tv_workspace_bytes: bad size");
    return (int64_t)tv_plan(nx, ny, nz, nt).bytes;
}

extern "C" int met2_tv_chambolle(const double* vol, int nx, int ny, int nz, int nt, const double* weight, double eps,
                                 int max_iter, double* out, int32_t* iterations, void* workspace, void* stream) {
    if (!vol || !weight || !out || !iterations || !workspace || out == vol || !tv_sizes_ok(nx, ny, nz, nt) ||
        max_iter < 1)
        return set_error(MET2_ERR_ARG, "met2_tv_chambolle: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const TvPlan pl = tv_plan(nx, ny, nz, nt);
    const TvGeom& g = pl.g;
    char* ws = (char*)workspace;
    double* img = (double*)(ws + pl.off_img);
    double* outE = (double*)(ws + pl.off_out);
    double* p = (double*)(ws + pl.off_p);
    double* sqd = (double*)(ws + pl.off_sqd);
    double* sqn = (double*)(ws + pl.off_sqn);
    double* part = (double*)(ws + pl.off_part);
    double* e_init = (double*)(ws + pl.off_einit);
    double* e_prev = (double*)(ws + pl.off_eprev);
    int* active = (int*)(ws + pl.off_active);
    const long long N = g.n;
    const unsigned tgrid = (unsigned)(((N + 31) / 32) * ((nt + 31) / 32));
    MET2_LAUNCH(tgrid, dim3(32, 8), 0, st, tv_transpose_kernel)(vol, img, N, nt);
    cudaMemsetAsync(p, 0, (size_t)nt * g.nd * N * sizeof(double), st);
    MET2_LAUNCH((unsigned)((nt + 127) / 128), 128, 0, st, tv_init_kernel)(nt, active, iterations);
    // blocks stride over (running echo, voxel block): once every echo has stopped, the remaining launches exit at once
    const long long vox_items = (long long)nt * ((N + TV_THREADS - 1) / TV_THREADS);
    const long long cap = (long long)sm_count() * 8;
    const unsigned vgrid = (unsigned)(vox_items < cap ? vox_items : cap);
    const long long part_items = (long long)nt * g.parts;
    const unsigned pgrid = (unsigned)(part_items < cap ? part_items : cap);
    for (int it = 0; it < max_iter; ++it) {
        MET2_LAUNCH(vgrid, TV_THREADS, 0, st, tv_out_kernel)(img, p, active, g, it == 0 ? 1 : 0, outE, sqd);
        MET2_LAUNCH(vgrid, TV_THREADS, 0, st, tv_p_kernel)(outE, p, active, g, weight, sqn);
        MET2_LAUNCH(pgrid, TV_THREADS, 0, st, tv_partials_kernel)(sqd, sqn, active, g, part);
        MET2_LAUNCH(1, TV_FIN_THREADS, 0, st, tv_energy_kernel)(part, g, weight, eps, it, max_iter, active, e_init, e_prev,
                                                                iterations);
    }
    MET2_LAUNCH(tgrid, dim3(32, 8), 0, st, tv_transpose_kernel)(outE, out, (long long)nt, (int)N);
    count_launch(3 + 4 * max_iter);
    return check_launch("met2_tv_chambolle");
}
