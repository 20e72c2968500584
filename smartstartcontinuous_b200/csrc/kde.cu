// kde.cu -- SmartStart stage 1 on sm_100a: Gaussian KDE (Scott bandwidth) over the replay
// buffer, UCB score and arg-max, replacing scipy.stats.gaussian_kde + numpy at
// smartexplorationcontinuous.py:260-280.
//
// Pipeline (all on the context stream):
//   1. kde_moments_kernel    fp64 shifted first/second moments of the data set (per-block partials);
//   2.  + kde_fit_block      the last block fits: mean, covariance (ddof=1), Scott factor, Cholesky,
//                            whitening matrix  Wm = sqrt(log2(e)/2) * L^-1, normalisation constant
//   3. kde_whiten_kernel     fp64 -> fp32: y = Wm (x - mean); points stored as
//                            [2y0,2y0, 2y1,2y1, ..., -|y|^2,-|y|^2] (duplicated for packed f32x2
//                            math), queries as [y0, .., y_{D-1}, -|y|^2]; the largest |y|^2 is kept
//   4. kde_pairs_kernel      the hot loop: sum_i exp2(-|y_q - y_i|^2) for a tile of queries x a
//                            slice of points; points streamed through shared memory with bulk
//                            async copies (TMA, UBLKCP) + mbarriers, two queries per packed
//                            f32x2 instruction.
//                            EXPANDED variant (default): the exponent is built as
//                            -|q|^2 - |x|^2 + 2 q.x  (1 FADD2 + D FFMA2 per query pair instead of
//                            D FADD2 + D FMUL2/FFMA2); optionally (SS_KDE_POLY_ON) every
//                            KDE_POLY_EVERY-th point evaluates exp2 with a degree-4 polynomial on
//                            the FMA pipe instead of MUFU.EX2.  The expansion
//                            cancels in FP32, so it is only used while max|y|^2 <= KDE_EXPAND_LIMIT
//                            (density error <~ 4e-8 * max|y|^2 relative, measured); otherwise the
//                            DIFFERENCE variant (exact differences, MUFU only) runs instead.  The
//                            choice is made on the device (no host round trip): both variants are
//                            launched, one of them returns immediately.
//   5. kde_finish_kernel     fp64: reduce point-slices, rescue underflowed queries in fp64, density,
//                            UCB and the np.argmax-ordered arg-max (single pass, last block reduces)
//
// Roofline: SFU (MUFU.EX2, 16 / clk / SM) and FP32 pipes, co-limited; see DESIGN.md.
#include <cuda_bf16.h>

#include <atomic>
#include <cstdlib>
#include <cstring>

#include "kde_shared.cuh"

namespace {

constexpr int KDE_THREADS = 128;      // threads per CTA in the pair kernel
constexpr int KDE_TILE_FLOATS = 4096;  // 16 KB of points per shared-memory stage
constexpr int KDE_STAGES = 2;
constexpr double KDE_RESCUE_BELOW = 7.8886090522101181e-31;  // 2^-100
constexpr int KDE_FIN_Q = 32;              // queries per block of the finish kernel (one per lane; the warps split the slices)
#ifndef SS_KDE_POLY_EVERY
#define SS_KDE_POLY_EVERY 5
#endif
// Measured on B200 (config 2): the polynomial path does not pay on the CUDA cores -- packed f32x2
// instructions hold the dispatch port for two cycles, so the kernel is dispatch- and XU-bound at
// the same ~13.4 evaluations/clk/SM with or without it (419 us without, 425-441 us with 1/10..1/5
// of the points on the polynomial).  Kept behind a switch (validated: 3e-6 relative density error).
#ifndef SS_KDE_POLY_ON
#define SS_KDE_POLY_ON 0
#endif
constexpr int KDE_POLY_EVERY = SS_KDE_POLY_EVERY;   // one point in KDE_POLY_EVERY takes the polynomial exp2
constexpr float KDE_EXPAND_LIMIT = 1000.f; // max |y|^2 for the expanded-exponent CUDA-core variant
                                           // (density error ~4e-8 * max|y|^2 relative, measured)
constexpr float KDE_TC_LIMIT = 700.f;      // same for the tcgen05 variant (~7e-8 * max|y|^2, measured)

struct KdeFit {
    double mean[SS_MAX_D];
    double wm[SS_MAX_D * SS_MAX_D];   // whitening matrix (lower triangular), row-major d x d
    double norm;                      // N * (2 pi)^(d/2) * prod diag(L)
    int status;                       // 0 ok, 1 not positive definite
    int max_norm2_bits;               // float bits of max |y|^2 over points and queries
};

__host__ __device__ constexpr int kde_point_stride(int D) { return ((2 * D + 2 + 3) / 4) * 4; }
__host__ __device__ constexpr int kde_tile_pts(int D) {
    return (KDE_TILE_FLOATS / kde_point_stride(D)) / (4 * KDE_POLY_EVERY) * (4 * KDE_POLY_EVERY);
}
__host__ __device__ constexpr int kde_queries_per_thread(int D) {
    return D <= 4 ? 8 : (D <= 8 ? 4 : 2);
}

// ---- 1. moments ------------------------------------------------------------------------
// partial[b] = { sum (x - x0) [d], sum (x - x0)(x - x0)^T lower-tri [d(d+1)/2] }, x0 = data[0]
// (shifted by the first data point so the fp64 one-pass covariance does not cancel)
template <int DF>
__device__ void kde_fit_block(const double* __restrict__ data, long long n, int d, const double* __restrict__ partial,
                              int nblocks, KdeFit* __restrict__ fit);

// The last block to finish (atomic ticket) reduces the per-block partials and fits the estimator
// (kde_fit_block), so moments + fit are one launch.
template <int DM>
__global__ void __launch_bounds__(256)
kde_moments_kernel(const double* __restrict__ data, long long n, int d, double* __restrict__ partial,
                   unsigned int* __restrict__ ticket, KdeFit* __restrict__ fit, double* __restrict__ sums_out) {
    __shared__ double sm[8];
    __shared__ bool s_last;
    pdl_trigger();       // the whitening kernel may be scheduled (it waits for the fit)
    constexpr int NM = DM + DM * (DM + 1) / 2;
    const int nm = d + d * (d + 1) / 2;
    double loc[NM];
#pragma unroll
    for (int i = 0; i < NM; ++i) loc[i] = 0.0;
    double x0[DM], v[DM];
#pragma unroll
    for (int j = 0; j < DM; ++j) x0[j] = j < d ? data[j] : 0.0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
#pragma unroll
        for (int j = 0; j < DM; ++j) v[j] = j < d ? data[i * d + j] - x0[j] : 0.0;
        // moments laid out for the *runtime* d: index p advances only over j,k < d
        int p = d;
#pragma unroll
        for (int j = 0; j < DM; ++j) {
            if (j < d) {
                loc[j] += v[j];
#pragma unroll
                for (int k = 0; k <= j; ++k) loc[p + k] += v[j] * v[k];
                p += j + 1;
            }
        }
    }
    for (int q = 0; q < nm; ++q) {
        double s = loc[q];
        for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
        if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
            partial[(size_t)blockIdx.x * nm + q] = t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && sums_out) {
        // running-moments mode (device mirror): leave the reduced sums and the shift x0 = data[0], no fit
        __threadfence();
        for (int q = threadIdx.x >> 5; q < nm; q += blockDim.x >> 5) {
            double s = 0.0;
            for (int b = threadIdx.x & 31; b < (int)gridDim.x; b += 32) s += partial[(size_t)b * nm + q];
            for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
            if ((threadIdx.x & 31) == 0) sums_out[q] = s;
        }
        if ((int)threadIdx.x < d) sums_out[nm + threadIdx.x] = data[threadIdx.x];
        if (threadIdx.x == 0) *ticket = 0;
        return;
    }
    if (s_last) {
        __threadfence();
        // (matrix scratch sized for the dimension at hand: with d <= 4 the serial fit runs out of registers
        // instead of a 24 KB local-memory frame -- ~8 us of the call at d = 3)
        if (d <= 4) kde_fit_block<4>(data, n, d, partial, (int)gridDim.x, fit);
        else if (d <= 8) kde_fit_block<8>(data, n, d, partial, (int)gridDim.x, fit);
        else kde_fit_block<SS_MAX_D>(data, n, d, partial, (int)gridDim.x, fit);
        if (threadIdx.x == 0) *ticket = 0;
    }
}

// ---- 2. fit ----------------------------------------------------------------------------
template <int DF>
__device__ void kde_fit_block(const double* __restrict__ data, long long n, int d, const double* __restrict__ partial,
                              int nblocks, KdeFit* __restrict__ fit) {
    __shared__ double mom[SS_MAX_D + SS_MAX_D * (SS_MAX_D + 1) / 2];
    const int nm = d + d * (d + 1) / 2;
    // one warp per moment: lanes stride over the per-block partials, fixed-order shuffle reduction
    for (int q = threadIdx.x >> 5; q < nm; q += blockDim.x >> 5) {
        double s = 0.0;
        for (int b = threadIdx.x & 31; b < nblocks; b += 32) s += partial[(size_t)b * nm + q];
        for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
        if ((threadIdx.x & 31) == 0) mom[q] = s;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const double N = (double)n;
    const double factor = pow(N, -1.0 / (d + 4));          // scotts_factor
    // DF x DF scratch with compile-time strides; for DF <= 4 the loops unroll and the matrices stay in registers
    constexpr bool UNROLL = DF <= 4;
    double cov[DF * DF], l[DF * DF], inv[DF * DF];
    {
        int p = d;
#pragma unroll(DF <= 4 ? DF * DF : 1)
        for (int j = 0; j < DF; ++j) {
            if (j < d) {
                fit->mean[j] = data[j] + mom[j] / N;
#pragma unroll(DF <= 4 ? DF * DF : 1)
                for (int k = 0; k < DF; ++k) {
                    if (k <= j) {
                        const double c = (mom[p + k] - mom[j] * mom[k] / N) / (N - 1.0);   // ddof = 1
                        cov[j * DF + k] = c * factor * factor;
                        cov[k * DF + j] = cov[j * DF + k];
                    }
                }
                p += j + 1;
            }
        }
    }
    // Cholesky (lower)
    int status = 0;
#pragma unroll(DF <= 4 ? DF * DF : 1)
    for (int j = 0; j < DF; ++j) {
        if (!UNROLL && j >= d) break;
#pragma unroll(DF <= 4 ? DF * DF : 1)
        for (int k = 0; k < DF; ++k) {
            if (!UNROLL && k >= d) break;
            if (j < d && k < d) {
                if (k <= j) {
                    double s = cov[j * DF + k];
#pragma unroll(DF <= 4 ? DF * DF : 1)
                    for (int q = 0; q < DF; ++q)
                        if (q < k) s -= l[j * DF + q] * l[k * DF + q];
                    if (j == k) {
                        if (!(s > 0.0)) { status = 1; s = 1.0; }
                        l[j * DF + j] = sqrt(s);
                    } else {
                        l[j * DF + k] = s / l[k * DF + k];
                    }
                } else {
                    l[j * DF + k] = 0.0;
                }
            }
        }
    }
    // inverse of the lower-triangular factor
#pragma unroll(DF <= 4 ? DF * DF : 1)
    for (int j = 0; j < DF * DF; ++j) inv[j] = 0.0;
#pragma unroll(DF <= 4 ? DF * DF : 1)
    for (int c = 0; c < DF; ++c) {
        if (!UNROLL && c >= d) break;
        if (c < d) {
            inv[c * DF + c] = 1.0 / l[c * DF + c];
#pragma unroll(DF <= 4 ? DF * DF : 1)
            for (int r = 0; r < DF; ++r) {
                if (!UNROLL && r >= d) break;
                if (r > c && r < d) {
                    double s = 0.0;
#pragma unroll(DF <= 4 ? DF * DF : 1)
                    for (int q = 0; q < DF; ++q)
                        if (q >= c && q < r) s -= l[r * DF + q] * inv[q * DF + c];
                    inv[r * DF + c] = s / l[r * DF + r];
                }
            }
        }
    }
    // exp(-e/2) = exp2(-(sqrt(log2(e)/2) |L^-1 (q-x)|)^2)
    const double scale = sqrt(0.5 * 1.4426950408889634074);
    double det = 1.0;
#pragma unroll(DF <= 4 ? DF * DF : 1)
    for (int j = 0; j < DF; ++j)
        if (j < d) det *= l[j * DF + j];
#pragma unroll(DF <= 4 ? DF * DF : 1)
    for (int j = 0; j < DF; ++j) {
        if (!UNROLL && j >= d) break;
#pragma unroll(DF <= 4 ? DF * DF : 1)
        for (int k = 0; k < DF; ++k) {
            if (!UNROLL && k >= d) break;
            if (j < d && k < d) fit->wm[j * d + k] = inv[j * DF + k] * scale;
        }
    }
    fit->norm = N * pow(2.0 * 3.14159265358979323846, 0.5 * d) * det;
    fit->status = status;
    fit->max_norm2_bits = 0;
}

// fit from running sums (device mirror): sums[0 .. nm) over the n - 1 buffer rows, shifted by x0 = sums[nm ..),
// plus the one extra data row `last` (the newest s2) -> the same estimator the moments kernel fits
__global__ void __launch_bounds__(32)
kde_fit_from_sums_kernel(const double* __restrict__ sums, const double* __restrict__ last, long long n, int d,
                         double* __restrict__ scratch, KdeFit* __restrict__ fit) {
    pdl_trigger();
    const int nm = d + d * (d + 1) / 2;
    const double* x0 = sums + nm;
    if (threadIdx.x == 0) {
        int p = d;
        for (int j = 0; j < d; ++j) {
            const double vj = last[j] - x0[j];
            scratch[j] = sums[j] + vj;
            for (int k = 0; k <= j; ++k) scratch[p + k] = sums[p + k] + vj * (last[k] - x0[k]);
            p += j + 1;
        }
    }
    __syncwarp();
    if (d <= 4) kde_fit_block<4>(x0, n, d, scratch, 1, fit);
    else if (d <= 8) kde_fit_block<8>(x0, n, d, scratch, 1, fit);
    else kde_fit_block<SS_MAX_D>(x0, n, d, scratch, 1, fit);
}

// ---- 3. whitening ----------------------------------------------------------------------
// points:  out[i] = [2y0,2y0, .., 2y_{D-1},2y_{D-1}, -|y|^2,-|y|^2, 0..]; padding rows are far away
//          (exp2 -> 0 in either pair-kernel variant)
// queries: out[i] = [y0, .., y_{D-1}, -|y|^2]
// |y|^2 is taken from the FP32-rounded coordinates, so the expanded exponent equals the squared
// distance between the rounded points (what the difference variant computes).
template <bool POINTS>
__global__ void kde_whiten_kernel(const double* __restrict__ x, long long n, long long n_pad, int d,
                                  int D, KdeFit* __restrict__ fit, float* __restrict__ out) {
    const int stride = POINTS ? kde_point_stride(D) : D + 1;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    float norm2 = 0.f;
    if (i < n_pad) {
        float* o = out + (size_t)i * stride;
        if (i >= n) {
            for (int j = 0; j < stride; ++j) o[j] = 0.f;
            // far away for both variants: 2y0 = 1e18 (difference form) and -|y|^2 = -1e30 (expanded form)
            if (POINTS) { o[0] = 1e18f; o[1] = 1e18f; o[2 * D] = -1e30f; o[2 * D + 1] = -1e30f; }
        } else {
            double c[SS_MAX_D];
            for (int j = 0; j < d; ++j) c[j] = x[i * d + j] - fit->mean[j];
            double nn = 0.0;
            for (int j = 0; j < D; ++j) {
                double y = 0.0;
                if (j < d)
                    for (int k = 0; k <= j; ++k) y += fit->wm[j * d + k] * c[k];
                const float yf = (float)y;
                nn += (double)yf * (double)yf;
                if (POINTS) {
                    o[2 * j] = 2.f * yf;
                    o[2 * j + 1] = 2.f * yf;
                } else {
                    o[j] = yf;
                }
            }
            norm2 = (float)nn;
            if (POINTS) {
                o[2 * D] = -norm2;
                o[2 * D + 1] = -norm2;
                for (int j = 2 * D + 2; j < stride; ++j) o[j] = 0.f;
            } else {
                o[D] = -norm2;
            }
        }
    }
    // largest |y|^2 (non-negative floats order like their bit patterns)
    for (int off = 16; off > 0; off >>= 1) norm2 = fmaxf(norm2, __shfl_xor_sync(0xffffffffu, norm2, off));
    if ((threadIdx.x & 31) == 0 && norm2 > 0.f) atomicMax(&fit->max_norm2_bits, __float_as_int(norm2));
}

// ---- 4. the pair kernel ----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine; SASS: UBLKCP), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// exp2 of a packed pair on the FMA pipe: Cody-Waite split + degree-4 minimax polynomial on
// [-0.5, 0.5] (max relative error 2.7e-6 in FP32), exponent inserted with an integer add.
__device__ __forceinline__ float2 exp2_poly2(float2 e) {
    const float MAGIC = 12582912.f;     // 1.5 * 2^23: e + MAGIC rounds e to an integer in the low mantissa bits
    const float2 ec = make_float2(fmaxf(e.x, -126.f), fmaxf(e.y, -126.f));
    const float2 t = __fadd2_rn(ec, make_float2(MAGIC, MAGIC));
    const float2 nf = __fadd2_rn(t, make_float2(-MAGIC, -MAGIC));
    const float2 f = __ffma2_rn(nf, make_float2(-1.f, -1.f), ec);
    float2 p = __ffma2_rn(f, make_float2(0.009570102207362652f, 0.009570102207362652f),
                          make_float2(0.05591785907745361f, 0.05591785907745361f));
    p = __ffma2_rn(p, f, make_float2(0.240247443318367f, 0.240247443318367f));
    p = __ffma2_rn(p, f, make_float2(0.6931217908859253f, 0.6931217908859253f));
    p = __ffma2_rn(p, f, make_float2(0.9999992847442627f, 0.9999992847442627f));
    // bits(MAGIC) << 23 == 0 (mod 2^32): shifting t's bits leaves exactly n << 23
    return make_float2(__int_as_float(__float_as_int(p.x) + (__float_as_int(t.x) << 23)),
                       __int_as_float(__float_as_int(p.y) + (__float_as_int(t.y) << 23)));
}

// grid: (query tiles, point slices).  partial[slice][q] = sum over the slice's points.
// EXPANDED: exponent = -|q|^2 - |x|^2 + 2 q.x (optionally every KDE_POLY_EVERY-th point on the
// FMA-pipe exp2); !EXPANDED: exponent = -|q - x|^2 from exact differences, MUFU.EX2 only.
template <int D, bool EXPANDED>
__global__ void __launch_bounds__(KDE_THREADS)
kde_pairs_kernel(const float* __restrict__ pts, long long n_tiles, const float* __restrict__ qw,
                 long long m_pad, const KdeFit* __restrict__ fit, float* __restrict__ partial) {
    constexpr int PS = kde_point_stride(D);           // floats per point in smem/global
    constexpr int Q = kde_queries_per_thread(D);      // queries per thread (Q/2 packed pairs)
    constexpr int TILE_PTS = kde_tile_pts(D);
    constexpr int TILE_FLOATS = TILE_PTS * PS;
    constexpr uint32_t TILE_BYTES = TILE_FLOATS * 4;
    constexpr int PE = KDE_POLY_EVERY;
    static_assert(TILE_PTS % PE == 0, "tiles hold whole groups of PE points");

    (void)fit;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tiles = reinterpret_cast<float*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)KDE_STAGES * TILE_BYTES);

    const int tid = threadIdx.x;
    // this CTA's slice of point tiles
    const long long per = (n_tiles + gridDim.y - 1) / gridDim.y;
    const long long t0 = blockIdx.y * per;
    const long long t1 = t0 + per < n_tiles ? t0 + per : n_tiles;
    const long long nt = t1 > t0 ? t1 - t0 : 0;

    if (tid == 0) {
        for (int s = 0; s < KDE_STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < KDE_STAGES && s < nt; ++s) {
            mbar_expect_tx(&full[s], TILE_BYTES);
            bulk_g2s(tiles + (size_t)s * TILE_FLOATS, pts + (size_t)(t0 + s) * TILE_FLOATS, TILE_BYTES,
                     &full[s]);
        }
    }

    // queries of this thread: q = (blockIdx.x * KDE_THREADS + tid) * Q + [0, Q); slot D holds -|q|^2
    const long long qbase = ((long long)blockIdx.x * KDE_THREADS + tid) * Q;
    float2 qv[Q / 2][D + 1];
#pragma unroll
    for (int p = 0; p < Q / 2; ++p)
#pragma unroll
        for (int j = 0; j <= D; ++j)
            qv[p][j] = make_float2(qw[(qbase + 2 * p) * (D + 1) + j], qw[(qbase + 2 * p + 1) * (D + 1) + j]);

    float2 total[Q / 2];
#pragma unroll
    for (int p = 0; p < Q / 2; ++p) total[p] = make_float2(0.f, 0.f);

    for (long long it = 0; it < nt; ++it) {
        const int s = (int)(it % KDE_STAGES);
        mbar_wait(&full[s], (uint32_t)((it / KDE_STAGES) & 1));
        const float* tp = tiles + (size_t)s * TILE_FLOATS;
        float2 acc[Q / 2];
#pragma unroll
        for (int p = 0; p < Q / 2; ++p) acc[p] = make_float2(0.f, 0.f);
#pragma unroll 1
        for (int i0 = 0; i0 < TILE_PTS; i0 += PE) {
#pragma unroll
            for (int u = 0; u < PE; ++u) {
                // broadcast loads: every lane reads the same point
                float xs[PS];
#pragma unroll
                for (int v = 0; v < PS / 4; ++v) {
                    float4 f = *reinterpret_cast<const float4*>(tp + (i0 + u) * PS + 4 * v);
                    xs[4 * v] = f.x; xs[4 * v + 1] = f.y; xs[4 * v + 2] = f.z; xs[4 * v + 3] = f.w;
                }
#pragma unroll
                for (int p = 0; p < Q / 2; ++p) {
                    float2 e;
                    if (EXPANDED) {
                        e = __fadd2_rn(make_float2(xs[2 * D], xs[2 * D + 1]), qv[p][D]);
#pragma unroll
                        for (int j = 0; j < D; ++j) e = __ffma2_rn(qv[p][j], make_float2(xs[2 * j], xs[2 * j + 1]), e);
                        if (SS_KDE_POLY_ON && u == PE - 1)
                            acc[p] = __fadd2_rn(acc[p], exp2_poly2(e));
                        else
                            acc[p] = __fadd2_rn(acc[p], make_float2(ex2_approx(e.x), ex2_approx(e.y)));
                    } else {
                        // q - x from the stored 2x: dlt = q - 0.5 * (2x), one FFMA2 per dimension
                        float2 dlt = __ffma2_rn(make_float2(xs[0], xs[1]), make_float2(-.5f, -.5f), qv[p][0]);
                        e = __fmul2_rn(dlt, dlt);
#pragma unroll
                        for (int j = 1; j < D; ++j) {
                            dlt = __ffma2_rn(make_float2(xs[2 * j], xs[2 * j + 1]), make_float2(-.5f, -.5f), qv[p][j]);
                            e = __ffma2_rn(dlt, dlt, e);
                        }
                        acc[p] = __fadd2_rn(acc[p], make_float2(ex2_approx(-e.x), ex2_approx(-e.y)));
                    }
                }
            }
        }
#pragma unroll
        for (int p = 0; p < Q / 2; ++p) total[p] = __fadd2_rn(total[p], acc[p]);
        __syncthreads();                                   // everyone is done with stage s
        if (tid == 0 && it + KDE_STAGES < nt) {
            mbar_expect_tx(&full[s], TILE_BYTES);
            bulk_g2s(tiles + (size_t)s * TILE_FLOATS,
                     pts + (size_t)(t0 + it + KDE_STAGES) * TILE_FLOATS, TILE_BYTES, &full[s]);
        }
    }
    float* out = partial + (size_t)blockIdx.y * m_pad + qbase;
#pragma unroll
    for (int p = 0; p < Q / 2; ++p) {
        out[2 * p] = total[p].x;
        out[2 * p + 1] = total[p].y;
    }
}

#include "kde_tc.cuh"

// ---- 5. finish: slice reduction, fp64 rescue, density, UCB, arg-max --------------------
__global__ void __launch_bounds__(256)
kde_finish_kernel(const float* __restrict__ partial, int n_slices, long long m, long long m_pad,
                  const double* __restrict__ data, long long n, int d,
                  const double* __restrict__ queries, const float* __restrict__ values,
                  const KdeFit* __restrict__ fit, double n_transitions, double volume, double alpha,
                  double beta, double* __restrict__ density, double* __restrict__ ucb_out,
                  double* __restrict__ block_v, long long* __restrict__ block_i,
                  KdeResult* __restrict__ result, unsigned long long* __restrict__ host_out, unsigned long long seq) {
    __shared__ double s_v[32];
    __shared__ long long s_i[32];
    __shared__ int s_list[256];
    __shared__ int s_nlist;
    __shared__ double s_red[8];
    __shared__ double s_part[8][KDE_FIN_Q];
    __shared__ bool s_last;
    pdl_wait();          // programmatic dependent of the pair kernel
    if (threadIdx.x == 0) s_nlist = 0;
    __syncthreads();

    // slice reduction: lane = query (32 consecutive floats per load), the 8 warps take the slices warp, warp + 8, ...
    // with 8 loads in flight each, then warp 0 adds the 8 partial sums in warp order (a fixed order) and owns
    // the queries from here on.  [4 threads per query with 4 loads in flight each: 20 us for 148 slices, all of it
    // load latency -- ncu r02n.]
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const long long jq0 = blockIdx.x * (long long)KDE_FIN_Q + lane;
    const long long j = wrp == 0 ? jq0 : m;          // non-owners behave like out-of-range threads
    double sum = 0.0;
    if (jq0 < m) {
#pragma unroll 8
        for (int s = wrp; s < n_slices; s += 8) sum += (double)partial[(size_t)s * m_pad + jq0];
    }
    s_part[wrp][lane] = sum;
    __syncthreads();
    if (wrp == 0) {
        sum = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) sum += s_part[w][lane];
    }
    if (j < m && !(sum >= KDE_RESCUE_BELOW)) s_list[atomicAdd(&s_nlist, 1)] = threadIdx.x;
    __syncthreads();
    // fp64 rescue of queries whose fp32 sum underflowed (far from every data point):
    // the whole block recomputes sum_i exp(-|L^-1 (q - x_i)|^2 / 2) exactly as scipy does.
    const int nres = s_nlist;
    for (int r = 0; r < nres; ++r) {
        const int owner = s_list[r];
        const long long jq = blockIdx.x * (long long)KDE_FIN_Q + owner;
        double yq[SS_MAX_D];
        for (int a = 0; a < d; ++a) {
            double y = 0.0;
            for (int k = 0; k <= a; ++k) y += fit->wm[a * d + k] * (queries[jq * d + k] - fit->mean[k]);
            yq[a] = y;
        }
        double part = 0.0;
        for (long long i = threadIdx.x; i < n; i += blockDim.x) {
            double e = 0.0;
            for (int a = 0; a < d; ++a) {
                double y = 0.0;
                for (int k = 0; k <= a; ++k) y += fit->wm[a * d + k] * (data[i * d + k] - fit->mean[k]);
                double df = yq[a] - y;
                e += df * df;
            }
            part += exp2(-e);
        }
        for (int off = 16; off > 0; off >>= 1) part += __shfl_down_sync(0xffffffffu, part, off);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = part;
        __syncthreads();
        if (threadIdx.x == owner) {
            double t = 0.0;
            for (int w = 0; w < 8; ++w) t += s_red[w];
            sum = t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && nres) atomicAdd(&result->n_rescued, nres);

    double u = 0.0;
    long long idx = -1;
    if (j < m) {
        const double dens = sum / fit->norm;
        const double c_hat = n_transitions * (dens * volume);
        u = alpha * (double)values[j] + sqrt((beta * log(n_transitions)) / c_hat);
        idx = j;
        if (density) density[j] = dens;
        if (ucb_out) ucb_out[j] = u;
    }
    block_argmax(u, idx, s_v, s_i);
    if (threadIdx.x == 0) {
        block_v[blockIdx.x] = u;
        block_i[blockIdx.x] = idx;
        __threadfence();
        unsigned int done = atomicAdd(&result->blocks_done, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        double v = 0.0;
        long long bi = -1;
        for (int b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
            double ov = block_v[b];
            long long oi = block_i[b];
            if (argmax_better(ov, oi, v, bi)) { v = ov; bi = oi; }
        }
        block_argmax(v, bi, s_v, s_i);
        if (threadIdx.x == 0) {
            result->best_ucb = v;
            result->best_j = bi;
            result->blocks_done = 0;
            result->n_rescued = 0;
            if (host_out) {
                const unsigned int tag = (unsigned int)seq | 0x80000000u;          // host_slot_tag
                host_slot_put(host_out, 0, v, tag);
                host_slot_put(host_out, 1, __longlong_as_double(bi), tag);
                host_slot_put(host_out, 2, __hiloint2double(fit->max_norm2_bits, fit->status), tag);
            }
        }
    }
}

template <int D>
cudaError_t launch_pairs(ss_ctx* c, bool expanded, const float* pts, long long n_tiles, const float* qw,
                         long long m_pad, int slices, const KdeFit* fit, float* partial) {
    constexpr int Q = kde_queries_per_thread(D);
    const size_t smem = (size_t)KDE_STAGES * kde_tile_pts(D) * kde_point_stride(D) * 4 + KDE_STAGES * 8;
    cudaError_t e = cudaFuncSetAttribute(kde_pairs_kernel<D, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(kde_pairs_kernel<D, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid((unsigned)(m_pad / (KDE_THREADS * Q)), (unsigned)slices);
    if (expanded)
        kde_pairs_kernel<D, true><<<grid, KDE_THREADS, smem, c->stream>>>(pts, n_tiles, qw, m_pad, fit, partial);
    else
        kde_pairs_kernel<D, false><<<grid, KDE_THREADS, smem, c->stream>>>(pts, n_tiles, qw, m_pad, fit, partial);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace

// pair-stage variants, fastest first; a call starts optimistically with the fastest one its shape
// allows and repeats the pair stage with KDE_DIFFERENCE when the precision guard (max |y|^2, known
// only after whitening) rejects the expanded exponent.
enum KdeVariant { KDE_TC = 0, KDE_EXPANDED = 1, KDE_DIFFERENCE = 2 };

// exact running sums of the first n rows of data_dev (device mirror: after a bulk upload / periodically)
int kde_exact_sums(ss_ctx* c, const double* data_dev, long long n, int d, double* sums_dev) {
    const int mom_blocks = (int)std::min<long long>(c->sm_count * 2, (n + 255) / 256);
    const int nm = d + d * (d + 1) / 2;
    SS_CUDA_CHECK(c, c->kde_moments.ensure((size_t)mom_blocks * nm * 8));
    SS_CUDA_CHECK(c, c->kde_fit.ensure(sizeof(KdeFit)));
    SS_CUDA_CHECK(c, c->kde_result.ensure(sizeof(KdeResult)));
    KdeResult* res = c->kde_result.as<KdeResult>();
    if (!c->kde_result_clean) {
        SS_CUDA_CHECK(c, cudaMemsetAsync(res, 0, sizeof(KdeResult), c->stream));
        c->kde_result_clean = true;
    }
    if (d <= 8)
        kde_moments_kernel<8><<<mom_blocks, 256, 0, c->stream>>>(data_dev, n, d, c->kde_moments.as<double>(),
                                                                 &res->moments_ticket, c->kde_fit.as<KdeFit>(), sums_dev);
    else
        kde_moments_kernel<SS_MAX_D><<<mom_blocks, 256, 0, c->stream>>>(data_dev, n, d, c->kde_moments.as<double>(),
                                                                        &res->moments_ticket, c->kde_fit.as<KdeFit>(),
                                                                        sums_dev);
    c->launches += 1;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}

int kde_run_fp64(ss_ctx* c, const double* data_dev, long long n, int d, const double* queries_dev, long long m,
                 const float* values_dev, long long n_transitions, double volume, double alpha, double beta,
                 double* density_dev, double* ucb_dev, int64_t* out_best_j, double* out_best_ucb);

int kde_run(ss_ctx* c, const double* data_dev, long long n, int d, const double* queries_dev,
            long long m, const float* values_dev, long long n_transitions, double volume,
            double alpha, double beta, double* density_dev, double* ucb_dev, int64_t* out_best_j,
            double* out_best_ucb, const double* running_sums) {
    if (c->kde_fp64)     // SS_PRECISION_FP64 (kde_fp64.cu): fits from the data rows, never from running sums
        return kde_run_fp64(c, data_dev, n, d, queries_dev, m, values_dev, n_transitions, volume, alpha, beta,
                            density_dev, ucb_dev, out_best_j, out_best_ucb);
    const int D = pad_dim(d);
    if (D < 0) SS_FAIL(c, SS_EUNSUPPORTED, "kde: state dimension > 32 is not supported");
    const int mom_blocks = (int)std::min<long long>(c->sm_count * 2, (n + 255) / 256);
    const int nm = d + d * (d + 1) / 2;
    const int fin_blocks = (int)((m + KDE_FIN_Q - 1) / KDE_FIN_Q);
    SS_CUDA_CHECK(c, c->kde_moments.ensure((size_t)mom_blocks * nm * 8));
    SS_CUDA_CHECK(c, c->kde_fit.ensure(sizeof(KdeFit)));
    SS_CUDA_CHECK(c, c->kde_block_best.ensure((size_t)fin_blocks * 16));
    SS_CUDA_CHECK(c, c->kde_result.ensure(sizeof(KdeResult)));
    KdeFit* fit = c->kde_fit.as<KdeFit>();
    KdeResult* res = c->kde_result.as<KdeResult>();

    // the kernels leave every counter of `res` at zero when a call completes: cleared only after a failure
    if (!c->kde_result_clean) SS_CUDA_CHECK(c, cudaMemsetAsync(res, 0, sizeof(KdeResult), c->stream));
    c->kde_result_clean = false;
    if (running_sums)
        // device mirror: the sums of the buffer rows are maintained incrementally; add the newest s2 (the last
        // data row) and fit -- no pass over the data
        kde_fit_from_sums_kernel<<<1, 32, 0, c->stream>>>(running_sums, data_dev + (size_t)(n - 1) * d, n, d,
                                                          c->kde_moments.as<double>(), fit);
    else if (d <= 8)
        kde_moments_kernel<8><<<mom_blocks, 256, 0, c->stream>>>(data_dev, n, d, c->kde_moments.as<double>(),
                                                                 &res->moments_ticket, fit, nullptr);
    else
        kde_moments_kernel<SS_MAX_D><<<mom_blocks, 256, 0, c->stream>>>(data_dev, n, d, c->kde_moments.as<double>(),
                                                                        &res->moments_ticket, fit, nullptr);
    c->launches += 1;
    SS_CUDA_CHECK(c, cudaGetLastError());

    int variant = KDE_EXPANDED;
    if (d <= kdetc::MAX_D && !getenv("SS_KDE_NO_TC")) variant = KDE_TC;
    if (getenv("SS_KDE_DIFFERENCE")) variant = KDE_DIFFERENCE;

    for (int attempt = 0; attempt < 2; ++attempt) {
        long long m_pad = 0;
        int n_slices = 0;
        if (variant == KDE_TC) {
            using namespace kdetc;
            const long long n_tiles = (n + NP - 1) / NP, n_pad = n_tiles * NP;
            const long long q_tiles = (m + QT - 1) / QT;
            m_pad = q_tiles * QT;
            // work items (query tile x slice of point tiles) for the persistent CTAs: a whole number
            // of waves of items with ~8 or more point tiles each (slices are balanced in the kernel)
            long long gcd_a = q_tiles, gcd_b = c->sm_count;
            while (gcd_b) { const long long r = gcd_a % gcd_b; gcd_a = gcd_b; gcd_b = r; }
            const long long step = c->sm_count / gcd_a;          // slices % step == 0 -> items % SMs == 0
            long long slices = n_tiles / 8 / step * step;
            if (slices < step) slices = step;
            if (slices * q_tiles > 32LL * c->sm_count) {
                slices = 32LL * c->sm_count / q_tiles / step * step;
                if (slices < step) slices = step;
            }
            if (slices > n_tiles) slices = n_tiles;
            if (slices < 1) slices = 1;
            n_slices = (int)slices * (EPI_WARPS / 4);            // one partial row per (slice, column group)
            const int ks = ks_for(d);
            SS_CUDA_CHECK(c, c->kde_pts.ensure((size_t)n_tiles * b_bytes(ks)));
            SS_CUDA_CHECK(c, c->kde_qw.ensure((size_t)q_tiles * a_bytes(ks)));
            SS_CUDA_CHECK(c, c->kde_partial.ensure((size_t)n_slices * m_pad * 4));
            const unsigned pblocks = (unsigned)((n_pad + 255) / 256), qblocks = (unsigned)((m_pad + 255) / 256);
            const long long items = q_tiles * slices;
            const unsigned grid = (unsigned)(items < c->sm_count ? items : c->sm_count);
            cudaError_t e = cudaSuccess;
#define KDE_TC_CASE(KS_)                                                                                          \
    do {                                                                                                          \
        e = launch_dependent(kde_whiten_tc_kernel<KS_>, dim3(pblocks + qblocks), dim3(256), 0, c->stream, data_dev, n,  \
                             n_pad, c->kde_pts.as<__nv_bfloat16>(), queries_dev, m, m_pad,                         \
                             c->kde_qw.as<__nv_bfloat16>(), d, fit, pblocks);                                      \
        timer_mark(c, "kde_fit_whiten");                                                                         \
        if (e == cudaSuccess)                                                                                     \
            e = cudaFuncSetAttribute(kde_pairs_tc_kernel<KS_>, cudaFuncAttributeMaxDynamicSharedMemorySize,       \
                                     (int)smem_bytes(KS_));                                                       \
        if (e == cudaSuccess)                                                                                     \
            e = launch_dependent(kde_pairs_tc_kernel<KS_>, dim3(grid), dim3(THREADS), smem_bytes(KS_), c->stream,  \
                                 c->kde_qw.as<__nv_bfloat16>(), c->kde_pts.as<__nv_bfloat16>(), n_tiles,           \
                                 (int)q_tiles, (int)slices, m_pad, fit, c->kde_partial.as<float>());               \
    } while (0)
            if (ks == 32) KDE_TC_CASE(32);
            else if (ks == 64) KDE_TC_CASE(64);
            else KDE_TC_CASE(128);
#undef KDE_TC_CASE
            c->launches += 2;
            SS_CUDA_CHECK(c, e);
            SS_CUDA_CHECK(c, cudaGetLastError());
            timer_mark(c, "kde_pairs");
        } else {
            const int Q = kde_queries_per_thread(D);
            const int PS = kde_point_stride(D);
            const int tile_pts = kde_tile_pts(D);
            const long long n_tiles = (n + tile_pts - 1) / tile_pts;
            const long long n_pad = n_tiles * tile_pts;
            const long long qtile = (long long)KDE_THREADS * Q;
            m_pad = (m + qtile - 1) / qtile * qtile;
            const long long q_tiles = m_pad / qtile;
            // fill the GPU: many small CTAs (up to 7 resident per SM; more warps hide the MUFU
            // latency and small work items balance the SMs)
            int per_sm = 24;
            if (const char* e = getenv("SS_KDE_CTAS_PER_SM")) per_sm = atoi(e) > 0 ? atoi(e) : per_sm;
            long long want = (long long)c->sm_count * per_sm;
            long long slices = (want + q_tiles - 1) / q_tiles;
            if (slices > n_tiles) slices = n_tiles;
            if (slices < 1) slices = 1;
            {
                long long per = (n_tiles + slices - 1) / slices;      // drop empty trailing slices
                slices = (n_tiles + per - 1) / per;
            }
            n_slices = (int)slices;
            SS_CUDA_CHECK(c, c->kde_pts.ensure((size_t)n_pad * PS * 4));
            SS_CUDA_CHECK(c, c->kde_qw.ensure((size_t)m_pad * (D + 1) * 4));
            SS_CUDA_CHECK(c, c->kde_partial.ensure((size_t)slices * m_pad * 4));
            kde_whiten_kernel<true><<<(unsigned)((n_pad + 255) / 256), 256, 0, c->stream>>>(
                data_dev, n, n_pad, d, D, fit, c->kde_pts.as<float>());
            kde_whiten_kernel<false><<<(unsigned)((m_pad + 255) / 256), 256, 0, c->stream>>>(
                queries_dev, m, m_pad, d, D, fit, c->kde_qw.as<float>());
            c->launches += 2;
            SS_CUDA_CHECK(c, cudaGetLastError());
            timer_mark(c, "kde_fit_whiten");
            cudaError_t e = cudaSuccess;
            const float* pts = c->kde_pts.as<float>();
            const float* qw = c->kde_qw.as<float>();
            float* partial = c->kde_partial.as<float>();
            const bool expanded = variant == KDE_EXPANDED;
            switch (D) {
#define KDE_CASE(DD) \
    case DD: e = launch_pairs<DD>(c, expanded, pts, n_tiles, qw, m_pad, (int)slices, fit, partial); break;
                KDE_CASE(1) KDE_CASE(2) KDE_CASE(3) KDE_CASE(4) KDE_CASE(6) KDE_CASE(8)
                KDE_CASE(12) KDE_CASE(16) KDE_CASE(24) KDE_CASE(32)
#undef KDE_CASE
            }
            SS_CUDA_CHECK(c, e);
            timer_mark(c, "kde_pairs");
        }

        double* bv = c->kde_block_best.as<double>();
        long long* bi = reinterpret_cast<long long*>(bv + fin_blocks);
        if (!c->host_kde) {
            SS_CUDA_CHECK(c, cudaHostAlloc(&c->host_kde, 4096, cudaHostAllocMapped));
            std::memset(c->host_kde, 0, 4096);
            SS_CUDA_CHECK(c, cudaHostGetDevicePointer(&c->host_kde_dev, c->host_kde, 0));
        }
        const unsigned long long seq = ++c->host_kde_seq;
        SS_CUDA_CHECK(c, launch_dependent(kde_finish_kernel, dim3(fin_blocks), dim3(256), 0, c->stream,
                                          c->kde_partial.as<float>(), n_slices, m, m_pad, data_dev, n, d, queries_dev,
                                          values_dev, fit, (double)n_transitions, volume, alpha, beta, density_dev,
                                          ucb_dev, bv, bi, res, reinterpret_cast<unsigned long long*>(c->host_kde_dev), seq));
        c->launches++;
        SS_CUDA_CHECK(c, cudaGetLastError());
        timer_mark(c, "kde_finish");

        // the result arrives in mapped host memory as tagged slots
        double slots[KDE_HOST_SLOTS];
        const int rc_wait = host_slots_wait(c, c->host_kde, KDE_HOST_SLOTS, host_slot_tag(seq), slots, "kde");
        if (rc_wait) return rc_wait;
        KdeResult hres;
        hres.best_ucb = slots[0];
        std::memcpy(&hres.best_j, &slots[1], 8);
        int hstat[2];                                     // status (low word), max_norm2_bits (high word)
        std::memcpy(hstat, &slots[2], 8);
        if (hstat[0] != 0)
            SS_FAIL(c, SS_ESINGULAR, "kde: data covariance is not positive definite (singular matrix)");
        float max_norm2;
        std::memcpy(&max_norm2, &hstat[1], 4);
        if (variant != KDE_DIFFERENCE && !(max_norm2 <= (variant == KDE_TC ? KDE_TC_LIMIT : KDE_EXPAND_LIMIT))) {
            // the expanded exponent would cancel too much for this data: redo the pair stage with
            // exact differences (rare: some |y|^2 above KDE_EXPAND_LIMIT, e.g. a far outlier query)
            variant = KDE_DIFFERENCE;
            continue;
        }
        *out_best_j = hres.best_j;
        *out_best_ucb = hres.best_ucb;
        c->kde_result_clean = true;
        return SS_OK;
    }
    SS_FAIL(c, SS_ECUDA, "kde: pair stage did not settle");
}
