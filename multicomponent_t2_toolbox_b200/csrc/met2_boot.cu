// met2_boot.cu — per-voxel bootstrap uncertainty of the six maps: replicate synthesis (met2_boot_resample) and the
// per-voxel summary of the refitted replicates (met2_boot_summary).  The refit in between is the caller's own
// met2_t2_fit(_echo) with the point fit's configuration; nothing here knows about the fit.
//
// Definition (tests/boot_oracle.py restates it in NumPy; both kernels are bitwise equal to that restatement):
//  * Replicates: wild bootstrap with Rademacher signs.  For voxel v with the signal sig[v] the point fit used and its
//    fitted signal est[v] (D f * km, raw units, as met2_t2_fit returns it), replicate b (0 <= b < B) is
//        r_e = sig_e - est_e,   s*_e = est_e + r_e if bit e of h is 0,  est_e - r_e if it is 1,
//    with h = splitmix64(seed, g * B + b) and g = voxel_offset + v, the voxel's position in the WHOLE voxel list:
//        x = seed + (g * B + b + 1) * 0x9E3779B97F4A7C15, x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9,
//        x = (x ^ (x >> 27)) * 0x94D049BB133111EB, h = x ^ (x >> 31)           (all mod 2^64)
//    One 64-bit word covers MET2_MAX_NTE = 64 echoes.  Keying on g makes a voxel's replicates independent of chunking,
//    slabs and the number of GPUs.  Every replicate keeps the point fit's flip-angle index: the FA is not searched
//    again (with FA smoothing the search ran on the smoothed volume, not on sig), so the intervals are conditional on
//    the estimated flip angle.  The refit re-selects lambda in every replicate.
//  * Validity: a replicate counts when its status lacks MET2_ST_SKIPPED (the bit after which the T2 kernels write
//    zeros); n_valid[v] is their number.
//  * Summary per voxel and map (MWF, IEWF, FWF, T2_M, T2_IE, TWC, the column order of `maps`), over the valid
//    replicates in replicate order: mean = sequential sum / n; sd = two-pass, sequential, ddof 1 (0 for n = 1);
//    p2.5 / p97.5 = NumPy's default 'linear' percentile: idx = (n - 1) * (q / 100), gamma = idx - floor(idx) and
//    numpy's _lerp (a + (b - a) gamma, or b - (b - a)(1 - gamma) for gamma >= 0.5), with numpy's clamp of an index at
//    or past the last element.  n = 0 gives four zeros (the reference's convention for unfitted voxels); a NaN among a
//    map's valid values makes that map's four numbers NaN.
//
// met2_boot_resample: one warp per replicate row, lane l writing echoes l and l + 32 (coalesced rows; the hash is
// integer work done once per row).  met2_boot_summary: one warp per voxel.  Lanes 0..5 form the sums of one map each
// (the order is sequential, so the parallelism is across maps and voxels); then, map by map, the warp compacts the
// valid values into shared memory in replicate order (ballot + prefix popcount), pads them to a power of two with
// +inf and sorts them with a bitonic network, from which lane 0 takes the two order statistics of each percentile.
#include <math.h>

#include "met2_host.h"

namespace met2 {

constexpr unsigned BOOT_FULL = 0xffffffffu;
constexpr int BOOT_MAX_B = 1024;
constexpr int BOOT_RES_THREADS = 256;
constexpr int BOOT_SUM_WARPS = 4;      // voxels per block of the summary kernel

__host__ __device__ inline uint64_t boot_splitmix64(uint64_t seed, uint64_t k) {
    uint64_t x = seed + (k + 1ull) * 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// rows r = v * B + b of rep_sig [V * B][nTE]; the warps stride over the rows
__global__ void __launch_bounds__(BOOT_RES_THREADS)
    boot_resample_kernel(const double* __restrict__ sig, const double* __restrict__ est,
                         const int32_t* __restrict__ fa_index, long long V, int nTE, int B, uint64_t seed,
                         long long voxel_offset, double* __restrict__ rep_sig, int32_t* __restrict__ rep_fa) {
    const int lane = threadIdx.x & 31;
    const long long rows = V * B;
    const long long nwarps = (long long)gridDim.x * (BOOT_RES_THREADS / 32);
    for (long long r = (long long)blockIdx.x * (BOOT_RES_THREADS / 32) + (threadIdx.x >> 5); r < rows; r += nwarps) {
        const long long v = r / B;
        const int b = (int)(r - v * B);
        const uint64_t h = boot_splitmix64(seed, (uint64_t)(voxel_offset + v) * (uint64_t)B + (uint64_t)b);
        const double* s = sig + v * nTE;
        const double* m = est + v * nTE;
        double* o = rep_sig + r * nTE;
        for (int e = lane; e < nTE; e += 32) {
            const double res = s[e] - m[e];
            o[e] = ((h >> e) & 1ull) ? m[e] - res : m[e] + res;
        }
        if (lane == 0) rep_fa[r] = fa_index[v];
    }
}

// numpy.percentile(a[:n], q, method="linear") of the ascending values a[0..n-1], n >= 1
template <class A>
__device__ inline double boot_percentile(A& a, long base, int n, double q) {
    const double vi = (double)(n - 1) * (q / 100.0);
    double prev = floor(vi);
    long ip = (long)prev, in = ip + 1;
    if (vi >= (double)(n - 1)) {   // numpy: index -1 for both, and gamma is taken against that -1
        ip = in = n - 1;
        prev = -1.0;
    }
    const double gamma = vi - prev;
    const double lo = a[base + ip], hi = a[base + in];
    const double diff = hi - lo;
    return gamma >= 0.5 ? hi - diff * (1.0 - gamma) : lo + diff * gamma;
}

// one warp per voxel; dynamic shared memory: BOOT_SUM_WARPS * P doubles, P = the power of two >= max(B, 32)
__global__ void __launch_bounds__(BOOT_SUM_WARPS * 32)
    boot_summary_kernel(const double* __restrict__ rep_maps, const uint32_t* __restrict__ rep_status, long long V,
                        int B, int P, double* __restrict__ stats, int32_t* __restrict__ n_valid) {
#ifdef MET2_HOST_EMU
    simt::Shared& sh = simt::g_shared;
#else
    extern __shared__ double boot_smem[];
    double* sh = boot_smem;
#endif
    const int lane = threadIdx.x & 31;
    const int w = threadIdx.x >> 5;
    const long long v = (long long)blockIdx.x * BOOT_SUM_WARPS + w;
    if (v >= V) return;   // whole warps only; the kernel has no block-wide barrier
    const double* M = rep_maps + (size_t)v * B * 6;
    const uint32_t* st = rep_status + (size_t)v * B;
    int n = 0;
    for (int b0 = 0; b0 < B; b0 += 32) {
        const int b = b0 + lane;
        n += __popc(__ballot_sync(BOOT_FULL, b < B && !(st[b] & MET2_ST_SKIPPED)));
    }
    // lane m < 6: mean, sd and the NaN test of map m, sequential in replicate order
    double mean = 0.0, sd = 0.0;
    int has_nan = 0;
    if (lane < 6 && n > 0) {
        double s = 0.0;
        for (int b = 0; b < B; ++b)
            if (!(st[b] & MET2_ST_SKIPPED)) {
                const double x = M[(size_t)b * 6 + lane];
                s = s + x;
                has_nan |= (x != x);
            }
        mean = s / (double)n;
        if (n > 1) {
            double ss = 0.0;
            for (int b = 0; b < B; ++b)
                if (!(st[b] & MET2_ST_SKIPPED)) {
                    const double d = M[(size_t)b * 6 + lane] - mean;
                    ss = ss + d * d;
                }
            sd = sqrt(ss / (double)(n - 1));
        }
    }
    double* out = stats + (size_t)v * 24;
    if (lane == 0) n_valid[v] = n;
    const long base = (long)w * P;
    for (int m = 0; m < 6; ++m) {
        const double mean_m = __shfl_sync(BOOT_FULL, mean, m);
        const double sd_m = __shfl_sync(BOOT_FULL, sd, m);
        const int nan_m = __shfl_sync(BOOT_FULL, has_nan, m);
        if (n == 0 || nan_m) {
            if (lane < 4) out[m * 4 + lane] = n == 0 ? 0.0 : NAN;
            continue;
        }
        int k = 0;   // compaction of the valid values in replicate order
        for (int b0 = 0; b0 < B; b0 += 32) {
            const int b = b0 + lane;
            const bool ok = b < B && !(st[b] & MET2_ST_SKIPPED);
            const unsigned bal = __ballot_sync(BOOT_FULL, ok);
            if (ok) sh[base + k + __popc(bal & ((1u << lane) - 1u))] = M[(size_t)b * 6 + m];
            k += __popc(bal);
        }
        for (int i = n + lane; i < P; i += 32) sh[base + i] = INFINITY;
        __syncwarp();
        for (int kk = 2; kk <= P; kk <<= 1)          // bitonic sort, ascending
            for (int j = kk >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < P / 2; t += 32) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i + j;
                    const double x = sh[base + i], y = sh[base + l];
                    if (((i & kk) == 0) ? (x > y) : (x < y)) {
                        sh[base + i] = y;
                        sh[base + l] = x;
                    }
                }
                __syncwarp();
            }
        if (lane == 0) {
            out[m * 4 + 0] = mean_m;
            out[m * 4 + 1] = sd_m;
            out[m * 4 + 2] = boot_percentile(sh, base, n, 2.5);
            out[m * 4 + 3] = boot_percentile(sh, base, n, 97.5);
        }
        __syncwarp();   // lane 0 reads the sorted values before the next map overwrites them
    }
}

static int boot_pow2(int B) {
    int P = 32;
    while (P < B) P <<= 1;
    return P;
}

}  // namespace met2

using namespace met2;

extern "C" int met2_boot_resample(const double* sig, const double* est_signal, const int32_t* fa_index, int64_t V,
                                  int nTE, int B, uint64_t seed, int64_t voxel_offset, double* rep_sig,
                                  int32_t* rep_fa_index, void* stream) {
    if (B < 1 || B > BOOT_MAX_B || nTE < 1 || nTE > MET2_MAX_NTE || V < 0 || voxel_offset < 0 ||
        (V > 0 && (!sig || !est_signal || !fa_index || !rep_sig || !rep_fa_index)))
        return set_error(MET2_ERR_ARG, "met2_boot_resample: bad argument");
    if (V == 0) return MET2_OK;
    const long long rows = (long long)V * B;
    const long long blocks = (rows + BOOT_RES_THREADS / 32 - 1) / (BOOT_RES_THREADS / 32);
    const long long cap = (long long)sm_count() * 16;
    MET2_LAUNCH((unsigned)(blocks < cap ? blocks : cap), BOOT_RES_THREADS, 0, (cudaStream_t)stream,
                boot_resample_kernel)(sig, est_signal, fa_index, (long long)V, nTE, B, (uint64_t)seed,
                                      (long long)voxel_offset, rep_sig, rep_fa_index);
    count_launch(1);
    return check_launch("met2_boot_resample");
}

extern "C" int met2_boot_summary(const double* rep_maps, const uint32_t* rep_status, int64_t V, int B, double* stats,
                                 int32_t* n_valid, void* stream) {
    if (B < 1 || B > BOOT_MAX_B || V < 0 || (V > 0 && (!rep_maps || !rep_status || !stats || !n_valid)))
        return set_error(MET2_ERR_ARG, "met2_boot_summary: bad argument");
    if (V == 0) return MET2_OK;
    const int P = boot_pow2(B);
    const long long blocks = (V + BOOT_SUM_WARPS - 1) / BOOT_SUM_WARPS;
    MET2_LAUNCH((unsigned)blocks, BOOT_SUM_WARPS * 32, (size_t)BOOT_SUM_WARPS * P * sizeof(double),
                (cudaStream_t)stream, boot_summary_kernel)(rep_maps, rep_status, (long long)V, B, P, stats, n_valid);
    count_launch(1);
    return check_launch("met2_boot_summary");
}
