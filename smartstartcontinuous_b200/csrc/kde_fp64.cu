// kde_fp64.cu -- SmartStart stage 1 in float64, following scipy.stats.gaussian_kde (1.18) operation for operation
// (SS_PRECISION_FP64, ss_kde_set_precision).  With N points and w = 1/N scipy computes
//   w_sum = sum(w), neff = 1/sum(w*w), factor = neff**(-1/(d+4))
//   mean  = sum(x*w)/w_sum,  C = (X-mean) @ ((X-mean)*w).T * (1/fact),  fact = w_sum - sum(w*w)/w_sum
//   L     = cholesky(C, lower) * factor
//   P, Z  = L^-1 x_i, L^-1 q_j (triangular solves);  norm = (2 pi)^(-d/2) / prod diag(L)
//   dens_j = sum_i w * (exp(-|P_i - Z_j|^2 / 2) * norm)         (a sequential loop over i)
// and the reference's UCB is alpha * values + sqrt(beta * log(n) / (n * (dens * volume))) with `values` float32, so
// alpha * values is a float32 product.  The sums of equal terms (w_sum, sum(w*w)) are numpy's pairwise sums,
// restated on the host; scipy takes neff from a BLAS dot product instead, whose order depends on the BLAS build
// and the CPU, and which differs from the pairwise sum by a few ulps (a ~1e-15 relative change of the density).
//
// Kernels (all on the context stream):
//   1. kde64_mean_partial_kernel / kde64_mean_kernel   sum(x*w) per block, reduced in a fixed order, / w_sum
//   2. kde64_cov_partial_kernel / kde64_fit_kernel     centred cross products per block, reduced in a fixed order,
//                                                      * 1/fact; Cholesky on one thread; * factor; norm
//   3. kde64_whiten_kernel                             forward substitution into [rows][D] doubles (D = pad_dim(d);
//                                                      zero coordinates add exactly 0 to |P - Z|^2)
//   4. kde_pairs_fp64_kernel<D, Q>                     the pair sums, every product and sum rounded on its own
//   5. kde_finish_fp64_kernel                          slices in order, density, UCB, np.argmax-ordered pick
// What is not bit-exact: the summation orders of OpenBLAS's dgemm (inside np.cov) and dtrsm against the fixed
// orders here, the slice partial sums against scipy's single running sum, and CUDA's exp against glibc's (both
// within 1 ulp): densities agree with scipy to ~1e-13 relative (tests/test_gpu_kde_fp64.py).
//
// A query's density depends on N (and d) alone: the point slices are cut from N, never from m, the grid or the
// GPU, so the same query gives the same bits in any batch, at any position, on any query shard.
#include <cmath>
#include <unordered_map>

#include "kde_shared.cuh"

namespace {

constexpr int K64_FIT_THREADS = 256;
constexpr int K64_FIT_ROWS = 2048;          // rows per block of the fit passes (a block count from N alone) ...
constexpr int K64_FIT_MAX_BLOCKS = 256;     // ... up to this many blocks
constexpr int K64_THREADS = 128;            // pair kernel
constexpr int K64_MAX_SLICES = 256;         // point slices per query (partial sums the finish kernel adds)
constexpr int K64_FIN_THREADS = 256;
constexpr double K64_PAD_POINT = 1e300;     // padding points: |P - Z|^2 overflows to inf, exp(-inf) = 0 exactly

struct KdeFit64 {
    double mean[SS_MAX_D];
    double l[SS_MAX_D * SS_MAX_D];   // scipy's cho_cov = cholesky(C) * factor, row-major d x d, lower
    double norm;                     // (2 pi)^(-d/2) / prod diag(cho_cov)
    int status;                      // 0 ok, 1 C is not positive definite
};

__host__ __device__ constexpr int k64_tile_pts(int D) { return (2048 / D) / 32 * 32; }   // 16 KB of shared memory
__host__ __device__ constexpr int k64_queries_per_thread(int D) { return D <= 4 ? 4 : (D <= 8 ? 2 : 1); }

// numpy's pairwise summation (np.add.reduce over a contiguous float64 array) of n copies of t; the recursion
// only meets O(log n) distinct lengths
double pairwise_sum_equal(double t, long long n, std::unordered_map<long long, double>& memo) {
    if (n < 8) {
        double r = 0.0;
        for (long long i = 0; i < n; ++i) r += t;
        return r;
    }
    if (n <= 128) {
        double r[8];
        for (int j = 0; j < 8; ++j) r[j] = t;
        long long i = 8;
        for (; i < n - n % 8; i += 8)
            for (int j = 0; j < 8; ++j) r[j] += t;
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res += t;
        return res;
    }
    auto it = memo.find(n);
    if (it != memo.end()) return it->second;
    long long n2 = n / 2;
    n2 -= n2 % 8;
    const double s = pairwise_sum_equal(t, n2, memo) + pairwise_sum_equal(t, n - n2, memo);
    memo[n] = s;
    return s;
}

// sum over the block's threads, in a fixed order (shuffle tree, then the warps in order); valid in thread 0
__device__ double k64_block_sum(double v, double* red) {
    for (int off = 16; off > 0; off >>= 1) v = __dadd_rn(v, __shfl_down_sync(0xffffffffu, v, off));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0) {
        t = red[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) t = __dadd_rn(t, red[w]);
    }
    __syncthreads();
    return t;
}

// ---- 1. means ------------------------------------------------------------------------------------------------
// partial[b][k] = sum over the block's rows of x[i][k] * w
__global__ void __launch_bounds__(K64_FIT_THREADS)
kde64_mean_partial_kernel(const double* __restrict__ data, long long n, int d, double w, double* __restrict__ partial) {
    __shared__ double red[K64_FIT_THREADS / 32];
    for (int k = 0; k < d; ++k) {
        double s = 0.0;
        for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
            s = __dadd_rn(s, __dmul_rn(data[i * d + k], w));
        s = k64_block_sum(s, red);
        if (threadIdx.x == 0) partial[(size_t)blockIdx.x * d + k] = s;
    }
}

// one warp per coordinate: mean[k] = (sum over the blocks' partials, fixed order) / w_sum
__global__ void __launch_bounds__(K64_FIT_THREADS)
kde64_mean_kernel(const double* __restrict__ partial, int nblocks, int d, double w_sum, KdeFit64* __restrict__ fit) {
    const int lane = threadIdx.x & 31;
    for (int k = threadIdx.x >> 5; k < d; k += blockDim.x >> 5) {
        double s = 0.0;
        for (int b = lane; b < nblocks; b += 32) s = __dadd_rn(s, partial[(size_t)b * d + k]);
        for (int off = 16; off > 0; off >>= 1) s = __dadd_rn(s, __shfl_down_sync(0xffffffffu, s, off));
        if (lane == 0) fit->mean[k] = __ddiv_rn(s, w_sum);
    }
}

// ---- 2. covariance and fit --------------------------------------------------------------------------------------
// grid (blocks, d): row j = blockIdx.y; partial[b][j][k] = sum_i (x_ij - mean_j) * ((x_ik - mean_k) * w), k <= j --
// np.cov's X @ (X * w).T with the lower triangle's left factor unweighted
template <int DM>
__global__ void __launch_bounds__(K64_FIT_THREADS)
kde64_cov_partial_kernel(const double* __restrict__ data, long long n, int d, double w, const KdeFit64* __restrict__ fit,
                         double* __restrict__ partial) {
    __shared__ double red[K64_FIT_THREADS / 32];
    const int j = blockIdx.y;
    double mean[DM], loc[DM];
#pragma unroll
    for (int k = 0; k < DM; ++k) {
        mean[k] = k <= j && k < d ? fit->mean[k] : 0.0;
        loc[k] = 0.0;
    }
    const double mean_j = fit->mean[j];
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double a = __dsub_rn(data[i * d + j], mean_j);
#pragma unroll
        for (int k = 0; k < DM; ++k)
            if (k <= j) loc[k] = __dadd_rn(loc[k], __dmul_rn(a, __dmul_rn(__dsub_rn(data[i * d + k], mean[k]), w)));
    }
#pragma unroll
    for (int k = 0; k < DM; ++k) {
        if (k > j) break;
        const double s = k64_block_sum(loc[k], red);
        if (threadIdx.x == 0) partial[((size_t)blockIdx.x * d + j) * d + k] = s;
    }
}

// one block: C[j][k] = (sum of the partials, fixed order) * inv_fact; Cholesky of C on thread 0; L * factor; norm
__global__ void __launch_bounds__(K64_FIT_THREADS)
kde64_fit_kernel(const double* __restrict__ partial, int nblocks, int d, double inv_fact, double factor, double norm0,
                 KdeFit64* __restrict__ fit) {
    __shared__ double cov[SS_MAX_D * SS_MAX_D];
    const int lane = threadIdx.x & 31;
    for (int q = threadIdx.x >> 5; q < d * d; q += blockDim.x >> 5) {
        const int j = q / d, k = q % d;
        if (k > j) continue;
        double s = 0.0;
        for (int b = lane; b < nblocks; b += 32) s = __dadd_rn(s, partial[(size_t)b * d * d + q]);
        for (int off = 16; off > 0; off >>= 1) s = __dadd_rn(s, __shfl_down_sync(0xffffffffu, s, off));
        if (lane == 0) cov[q] = __dmul_rn(s, inv_fact);
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double* l = fit->l;
    int status = 0;
    for (int j = 0; j < d; ++j) {
        for (int i = j; i < d; ++i) {
            double s = cov[i * d + j];
            for (int k = 0; k < j; ++k) s = __dsub_rn(s, __dmul_rn(l[i * d + k], l[j * d + k]));
            if (i == j) {
                if (!(s > 0.0)) { status = 1; s = 1.0; }
                l[j * d + j] = __dsqrt_rn(s);
            } else {
                l[i * d + j] = __ddiv_rn(s, l[j * d + j]);
            }
        }
        for (int i = 0; i < j; ++i) l[i * d + j] = 0.0;
    }
    double norm = norm0;
    for (int q = 0; q < d * d; ++q) l[q] = __dmul_rn(l[q], factor);
    for (int k = 0; k < d; ++k) norm = __ddiv_rn(norm, l[k * d + k]);
    fit->norm = norm;
    fit->status = status;
}

// ---- 3. whitening -----------------------------------------------------------------------------------------------
// out[i][k] = y_k = (x_ik - sum_{j<k} L_kj y_j) / L_kk, k < d (dtrsm's order), 0 for d <= k < D; rows n..n_pad get
// `pad` in coordinate 0
__global__ void __launch_bounds__(256)
kde64_whiten_kernel(const double* __restrict__ x, long long n, long long n_pad, int d, int D,
                    const KdeFit64* __restrict__ fit, double pad, double* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    double* o = out + (size_t)i * D;
    if (i >= n) {
        for (int k = 0; k < D; ++k) o[k] = k == 0 ? pad : 0.0;
        return;
    }
    double y[SS_MAX_D];
    for (int k = 0; k < d; ++k) {
        double s = x[i * d + k];
        for (int j = 0; j < k; ++j) s = __dsub_rn(s, __dmul_rn(y[j], fit->l[k * d + j]));
        y[k] = __ddiv_rn(s, fit->l[k * d + k]);
        o[k] = y[k];
    }
    for (int k = d; k < D; ++k) o[k] = 0.0;
}

// ---- 4. the pair kernel -----------------------------------------------------------------------------------------
// grid (query tiles, point slices); partial[slice][j] = sum over the slice's points, in index order, of
// w * (exp(-|P_i - Z_j|^2 / 2) * norm).  Each thread keeps Q whitened queries in registers; point tiles stream
// through shared memory and every lane reads the same point (broadcast).
template <int D, int Q>
__global__ void __launch_bounds__(K64_THREADS)
kde_pairs_fp64_kernel(const double* __restrict__ pts, long long n_tiles, int slice_tiles, const double* __restrict__ qw,
                      long long m_pad, double w, const KdeFit64* __restrict__ fit, double* __restrict__ partial) {
    constexpr int TILE = k64_tile_pts(D);
    __shared__ double tile[TILE * D];
    const long long t0 = (long long)blockIdx.y * slice_tiles;
    const long long t1 = t0 + slice_tiles < n_tiles ? t0 + slice_tiles : n_tiles;
    const long long qbase = ((long long)blockIdx.x * K64_THREADS + threadIdx.x) * Q;
    const double norm = fit->norm;
    double z[Q][D], acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        acc[q] = 0.0;
#pragma unroll
        for (int k = 0; k < D; ++k) z[q][k] = qw[(qbase + q) * D + k];
    }
    for (long long t = t0; t < t1; ++t) {
        const double* src = pts + (size_t)t * TILE * D;
        for (int e = threadIdx.x; e < TILE * D; e += K64_THREADS) tile[e] = src[e];
        __syncthreads();
#pragma unroll 2
        for (int i = 0; i < TILE; ++i) {
            double p[D];
#pragma unroll
            for (int k = 0; k < D; ++k) p[k] = tile[i * D + k];
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                double r = __dsub_rn(p[0], z[q][0]);
                double arg = __dmul_rn(r, r);
#pragma unroll
                for (int k = 1; k < D; ++k) {
                    r = __dsub_rn(p[k], z[q][k]);
                    arg = __dadd_rn(arg, __dmul_rn(r, r));
                }
                const double e = exp(-__dmul_rn(arg, 0.5));
                acc[q] = __dadd_rn(acc[q], __dmul_rn(w, __dmul_rn(e, norm)));
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) partial[(size_t)blockIdx.y * m_pad + qbase + q] = acc[q];
}

// ---- 5. finish --------------------------------------------------------------------------------------------------
// one thread per query: the slices in order, density, UCB (alpha * V rounded in float32, as numpy does with the
// float32 values), then the np.argmax pick (NaN first, then the larger value, then the lower index) per block and,
// in the last block, over the blocks; the result goes to the host slots
__global__ void __launch_bounds__(K64_FIN_THREADS)
kde_finish_fp64_kernel(const double* __restrict__ partial, int n_slices, long long m, long long m_pad,
                       const float* __restrict__ values, const KdeFit64* __restrict__ fit, double n_transitions,
                       double volume, float alpha32, double beta_log_n, double* __restrict__ density,
                       double* __restrict__ ucb_out, double* __restrict__ block_v, long long* __restrict__ block_i,
                       KdeResult* __restrict__ result, unsigned long long* __restrict__ host_out,
                       unsigned long long seq) {
    __shared__ double s_v[32];
    __shared__ long long s_i[32];
    __shared__ bool s_last;
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    double u = 0.0;
    long long idx = -1;
    if (j < m) {
        double dens = partial[j];
        for (int s = 1; s < n_slices; ++s) dens = __dadd_rn(dens, partial[(size_t)s * m_pad + j]);
        const double c_hat = __dmul_rn(n_transitions, __dmul_rn(dens, volume));
        u = __dadd_rn((double)__fmul_rn(alpha32, values[j]), __dsqrt_rn(__ddiv_rn(beta_log_n, c_hat)));
        idx = j;
        if (density) density[j] = dens;
        if (ucb_out) ucb_out[j] = u;
    }
    block_argmax(u, idx, s_v, s_i);
    if (threadIdx.x == 0) {
        block_v[blockIdx.x] = u;
        block_i[blockIdx.x] = idx;
        __threadfence();
        const unsigned int done = atomicAdd(&result->blocks_done, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double v = 0.0;
    long long bi = -1;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
        const double ov = block_v[b];
        const long long oi = block_i[b];
        if (argmax_better(ov, oi, v, bi)) { v = ov; bi = oi; }
    }
    block_argmax(v, bi, s_v, s_i);
    if (threadIdx.x == 0) {
        result->best_ucb = v;
        result->best_j = bi;
        result->blocks_done = 0;
        if (host_out) {
            const unsigned int tag = (unsigned int)seq | 0x80000000u;          // host_slot_tag
            host_slot_put(host_out, 0, v, tag);
            host_slot_put(host_out, 1, __longlong_as_double(bi), tag);
            host_slot_put(host_out, 2, __hiloint2double(0, fit->status), tag);
        }
    }
}

template <int D>
cudaError_t launch_pairs_fp64(ss_ctx* c, const double* pts, long long n_tiles, int slice_tiles, int n_slices,
                              const double* qw, long long m_pad, double w, const KdeFit64* fit, double* partial) {
    constexpr int Q = k64_queries_per_thread(D);
    const dim3 grid((unsigned)(m_pad / ((long long)K64_THREADS * Q)), (unsigned)n_slices);
    kde_pairs_fp64_kernel<D, Q><<<grid, K64_THREADS, 0, c->stream>>>(pts, n_tiles, slice_tiles, qw, m_pad, w, fit, partial);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace

extern "C" int ss_kde_set_precision(ss_ctx* c, int precision) {
    if (!c) return SS_EINVAL;
    if (precision != SS_PRECISION_FP32 && precision != SS_PRECISION_FP64)
        SS_FAIL(c, SS_EINVAL, "kde: the selection's precision is SS_PRECISION_FP32 or SS_PRECISION_FP64");
    c->kde_fp64 = precision == SS_PRECISION_FP64;
    return SS_OK;
}

int kde_run_fp64(ss_ctx* c, const double* data_dev, long long n, int d, const double* queries_dev, long long m,
                 const float* values_dev, long long n_transitions, double volume, double alpha, double beta,
                 double* density_dev, double* ucb_dev, int64_t* out_best_j, double* out_best_ucb) {
    const int D = pad_dim(d);
    if (D < 0) SS_FAIL(c, SS_EUNSUPPORTED, "kde: state dimension > 32 is not supported");
    // scipy's scalars, with numpy's sums of the N equal weights
    const double w = 1.0 / (double)n;
    std::unordered_map<long long, double> memo;
    const double w_sum = pairwise_sum_equal(w, n, memo);
    memo.clear();
    const double sum_ww = pairwise_sum_equal(w * w, n, memo);
    const double neff = 1.0 / sum_ww;
    const double factor = std::pow(neff, -1.0 / (d + 4));
    const double fact = w_sum - sum_ww / w_sum;                          // ddof = 1
    const double inv_fact = 1.0 / fact;
    const double norm0 = std::pow(2.0 * 3.14159265358979323846, -d / 2.0);
    const double beta_log_n = beta * std::log((double)n_transitions);

    const int fit_blocks = (int)std::min<long long>((n + K64_FIT_ROWS - 1) / K64_FIT_ROWS, K64_FIT_MAX_BLOCKS);
    const int TILE = k64_tile_pts(D), Q = k64_queries_per_thread(D);
    const long long n_tiles = (n + TILE - 1) / TILE, n_pad = n_tiles * TILE;
    const int slice_tiles = (int)((n_tiles + K64_MAX_SLICES - 1) / K64_MAX_SLICES);
    const int n_slices = (int)((n_tiles + slice_tiles - 1) / slice_tiles);
    const long long qtile = (long long)K64_THREADS * Q;
    const long long m_pad = (m + qtile - 1) / qtile * qtile;
    const int fin_blocks = (int)((m + K64_FIN_THREADS - 1) / K64_FIN_THREADS);
    SS_CUDA_CHECK(c, c->kde_moments.ensure((size_t)fit_blocks * d * d * 8));
    SS_CUDA_CHECK(c, c->kde_fit.ensure(sizeof(KdeFit64)));
    SS_CUDA_CHECK(c, c->kde_pts.ensure((size_t)n_pad * D * 8));
    SS_CUDA_CHECK(c, c->kde_qw.ensure((size_t)m_pad * D * 8));
    SS_CUDA_CHECK(c, c->kde_partial.ensure((size_t)n_slices * m_pad * 8));
    SS_CUDA_CHECK(c, c->kde_block_best.ensure((size_t)fin_blocks * 16));
    SS_CUDA_CHECK(c, c->kde_result.ensure(sizeof(KdeResult)));
    KdeFit64* fit = c->kde_fit.as<KdeFit64>();
    KdeResult* res = c->kde_result.as<KdeResult>();
    double* partial = c->kde_moments.as<double>();
    if (!c->kde_result_clean) SS_CUDA_CHECK(c, cudaMemsetAsync(res, 0, sizeof(KdeResult), c->stream));
    c->kde_result_clean = false;

    kde64_mean_partial_kernel<<<fit_blocks, K64_FIT_THREADS, 0, c->stream>>>(data_dev, n, d, w, partial);
    kde64_mean_kernel<<<1, K64_FIT_THREADS, 0, c->stream>>>(partial, fit_blocks, d, w_sum, fit);
    const dim3 cov_grid(fit_blocks, d);
    if (d <= 4)
        kde64_cov_partial_kernel<4><<<cov_grid, K64_FIT_THREADS, 0, c->stream>>>(data_dev, n, d, w, fit, partial);
    else if (d <= 8)
        kde64_cov_partial_kernel<8><<<cov_grid, K64_FIT_THREADS, 0, c->stream>>>(data_dev, n, d, w, fit, partial);
    else
        kde64_cov_partial_kernel<SS_MAX_D><<<cov_grid, K64_FIT_THREADS, 0, c->stream>>>(data_dev, n, d, w, fit, partial);
    kde64_fit_kernel<<<1, K64_FIT_THREADS, 0, c->stream>>>(partial, fit_blocks, d, inv_fact, factor, norm0, fit);
    kde64_whiten_kernel<<<(unsigned)((n_pad + 255) / 256), 256, 0, c->stream>>>(data_dev, n, n_pad, d, D, fit,
                                                                                K64_PAD_POINT, c->kde_pts.as<double>());
    kde64_whiten_kernel<<<(unsigned)((m_pad + 255) / 256), 256, 0, c->stream>>>(queries_dev, m, m_pad, d, D, fit, 0.0,
                                                                                c->kde_qw.as<double>());
    c->launches += 6;
    SS_CUDA_CHECK(c, cudaGetLastError());
    timer_mark(c, "kde_fit_whiten");

    cudaError_t e = cudaSuccess;
    const double* pts = c->kde_pts.as<double>();
    const double* qw = c->kde_qw.as<double>();
    double* pair_partial = c->kde_partial.as<double>();
    switch (D) {
#define KDE64_CASE(DD) \
    case DD: e = launch_pairs_fp64<DD>(c, pts, n_tiles, slice_tiles, n_slices, qw, m_pad, w, fit, pair_partial); break;
        KDE64_CASE(1) KDE64_CASE(2) KDE64_CASE(3) KDE64_CASE(4) KDE64_CASE(6) KDE64_CASE(8)
        KDE64_CASE(12) KDE64_CASE(16) KDE64_CASE(24) KDE64_CASE(32)
#undef KDE64_CASE
    }
    SS_CUDA_CHECK(c, e);
    timer_mark(c, "kde_pairs");

    double* bv = c->kde_block_best.as<double>();
    long long* bi = reinterpret_cast<long long*>(bv + fin_blocks);
    if (!c->host_kde) {
        SS_CUDA_CHECK(c, cudaHostAlloc(&c->host_kde, 4096, cudaHostAllocMapped));
        std::memset(c->host_kde, 0, 4096);
        SS_CUDA_CHECK(c, cudaHostGetDevicePointer(&c->host_kde_dev, c->host_kde, 0));
    }
    const unsigned long long seq = ++c->host_kde_seq;
    kde_finish_fp64_kernel<<<fin_blocks, K64_FIN_THREADS, 0, c->stream>>>(
        pair_partial, n_slices, m, m_pad, values_dev, fit, (double)n_transitions, volume, (float)alpha, beta_log_n,
        density_dev, ucb_dev, bv, bi, res, reinterpret_cast<unsigned long long*>(c->host_kde_dev), seq);
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    timer_mark(c, "kde_finish");

    double slots[KDE_HOST_SLOTS];
    const int rc_wait = host_slots_wait(c, c->host_kde, KDE_HOST_SLOTS, host_slot_tag(seq), slots, "kde");
    if (rc_wait) return rc_wait;
    int hstat[2];                                     // status (low word)
    std::memcpy(hstat, &slots[2], 8);
    if (hstat[0] != 0) SS_FAIL(c, SS_ESINGULAR, "kde: data covariance is not positive definite (singular matrix)");
    *out_best_ucb = slots[0];
    std::memcpy(out_best_j, &slots[1], 8);
    c->kde_result_clean = true;
    return SS_OK;
}
