// dyn_train.cu -- device-resident training of the dynamics MLP (SURVEY section 8f, row f1).
//
// Replaces Dyn_Model.train (dynamics_model.py:52-171): nEpoch passes of mini-batch Adam on the MSE
// between the network output and the normalised state deltas, every batch = rows of the shuffled
// "old" (initial random-policy) data followed by rows drawn from the "new" (replay-buffer) data.
// The reference builds a float64 TF1 graph (feedforward_network.py:3-23: Linear+ReLU hidden layers,
// linear output; tf.train.AdamOptimizer defaults beta1 .9, beta2 .999, eps 1e-8; loss =
// reduce_mean(square(z - f(x))) over batch x outputs) and feeds numpy batches through sess.run.
//
// Here everything stays on the GPU: both data sets, the master parameters, the Adam moments and the
// step counter live in the context; a training epoch uploads only the batch row
// indices (drawn on the host with the reference's numpy calls, so the batches are the reference's)
// and queues, per Adam step, a fixed sequence of kernels:
//
//   first layer  gather the batch rows + Linear(din -> h) + ReLU              (K = din is tiny)
//   hidden       H_{l+1} = relu(H_l W_l + b_l)                 tiled FP32 GEMM (NN)
//   output+loss  out = H_L W_L + b_L; dOut = 2 (out - z) / (B dout); loss; dH_L = dOut W_L^T (.) [H_L > 0]
//   backward     per hidden layer: dH_l = dY_{l+1} W_l^T (.) [H_l > 0]  (NT GEMM, old W_l),
//                                  dW_l = H_l^T dY_{l+1} + Adam           (TN GEMM, update fused)
//   thin updates dW_L, dW_0 and all bias gradients (column sums) + Adam in one launch
// (6 launches per step for the 2-hidden-layer network)
//
// No host synchronisation inside an epoch; the per-step losses come back in one copy.  After
// training, ss_dyn_commit re-packs the parameters for the rollout kernels ON THE DEVICE (FP32
// padded matrices for the SIMT kernel, BF16 UMMA operand images for the tcgen05 kernel): the weights
// never visit the host unless ss_dyn_get_params asks for them.
//
// Arithmetic: FP32 FFMA with FP32 accumulation (the reference is float64).  Why not the tensor
// pipe: one step is 0.8 GFLOP (three 512 x 500 x 500 GEMMs) -- launch/latency-bound, not
// throughput-bound -- and Adam divides by sqrt(v) + 1e-8, so weights whose gradient hovers near
// zero amplify operand noise: already FP32 drifts from the float64 oracle by 7e-4 of the movement
// (Frobenius) after 40 steps, exactly as a float32 numpy run of the oracle does; BF16/TF32 operands
// would put 1e-3 relative noise on every gradient (tests/test_gpu_dyn_train.py states the bounds).
//
// SS_PRECISION_FP64 (ss_dyn_set_precision): the same kernels instantiated for double -- data sets
// stored without float32 rounding, float64 masters, moments and activations in the same buffers, DFMA
// GEMMs (not DMMA: 37.0 vs 36.0 TFLOP/s measured, profiles/r03_fp64_time.json, too close to pay for
// fragment shuffling), and Adam in the oracle's operation order with every product and sum rounded on
// its own.  A step then differs from oracle/dyn_train_oracle.py only in the summation order of the GEMMs
// and of the batch reductions (tests/test_gpu_dyn_train_fp64.py).  ss_dyn_commit hands the float64
// masters unchanged to the float64 rollout and packs the FP32 / tcgen05 images from them rounded once
// to float.
#include <cstring>

#include "mpc_kernels.cuh"

namespace {

constexpr int DYN_MAX_LAYERS = SS_MAX_LAYERS + 1;

// Every training kernel is a template on the scalar type T: float (the FP32 trainer) or double
// (SS_PRECISION_FP64: masters, moments, data and activations in float64, DFMA).  The helpers below map
// to fmaf / fmaxf for float, so the FP32 trainer's instructions do not depend on the templating.
__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float relu_t(float a) { return fmaxf(a, 0.f); }
__device__ __forceinline__ double relu_t(double a) { return fmax(a, 0.0); }

template <typename T>
struct AdamArgs {
    T lr_t;            // lr * sqrt(1 - beta2^t) / (1 - beta1^t)   (tf.train.AdamOptimizer)
    T beta1, beta2, eps;
    T omb1, omb2;      // 1 - beta, rounded once from float64 (1.f - 0.999f is off by 1e-5 relative)
};

__device__ __forceinline__ void adam_update(float g, float& w, float& m, float& v, const AdamArgs<float>& a) {
    m = a.beta1 * m + a.omb1 * g;
    v = a.beta2 * v + a.omb2 * g * g;
    w -= a.lr_t * m / (sqrtf(v) + a.eps);
}
// float64: oracle/dyn_train_oracle.adam_step operation for operation (m *= b1; m += (1 - b1) g;
// v *= b2; v += (1 - b2) g g; w -= lr_t m / (sqrt(v) + eps)), every product and sum rounded on its own
// (no FMA contraction), so a step differs from the oracle only through the gradient's summation order
__device__ __forceinline__ void adam_update(double g, double& w, double& m, double& v, const AdamArgs<double>& a) {
    m = __dadd_rn(__dmul_rn(a.beta1, m), __dmul_rn(a.omb1, g));
    v = __dadd_rn(__dmul_rn(a.beta2, v), __dmul_rn(__dmul_rn(a.omb2, g), g));
    w = __dsub_rn(w, __ddiv_rn(__dmul_rn(a.lr_t, m), __dadd_rn(__dsqrt_rn(v), a.eps)));
}

// dynamic shared memory of the first-layer kernel, typed per instantiation
template <typename T> __device__ __forceinline__ T* dyn_smem();
template <> __device__ __forceinline__ float* dyn_smem<float>() {
    extern __shared__ float s_x[];
    return s_x;
}
template <> __device__ __forceinline__ double* dyn_smem<double>() {
    extern __shared__ double s_x64[];
    return s_x64;
}

// ---- forward, first layer: gather + Linear + ReLU ---------------------------------------------
// batch row b < n_old: old data row idx_old[b]; else new data row idx_new[b - n_old]
template <typename T>
__global__ void __launch_bounds__(256)
dyn_first_layer_kernel(const T* __restrict__ x_old, const T* __restrict__ z_old,
                       const T* __restrict__ x_new, const T* __restrict__ z_new,
                       const int* __restrict__ idx_old, const int* __restrict__ idx_new, int n_old, int B, int din,
                       int dout, const T* __restrict__ W0, const T* __restrict__ b0, int h, int relu,
                       T* __restrict__ X, T* __restrict__ Z, T* __restrict__ H1) {
    T* s_x = dyn_smem<T>();                 // [rows_per_block][din]
    const int rows = blockDim.x / 32;       // one warp per batch row
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * rows + warp;
    if (b >= B) return;
    const bool is_old = b < n_old;
    const long long r = is_old ? idx_old[b] : idx_new[b - n_old];
    const T* xs = (is_old ? x_old : x_new) + (size_t)r * din;
    const T* zs = (is_old ? z_old : z_new) + (size_t)r * dout;
    T* sx = s_x + warp * din;
    for (int j = lane; j < din; j += 32) {
        const T v = xs[j];
        sx[j] = v;
        X[(size_t)b * din + j] = v;
    }
    for (int j = lane; j < dout; j += 32) Z[(size_t)b * dout + j] = zs[j];
    __syncwarp();
    for (int n = lane; n < h; n += 32) {
        T acc = b0[n];
        for (int j = 0; j < din; ++j) acc = fma_t(sx[j], W0[(size_t)j * h + n], acc);
        H1[(size_t)b * h + n] = relu ? relu_t(acc) : acc;
    }
}

// ---- tiled GEMM: C[i][j] = sum_p A(i, p) * B(p, j) -----------------------------------------------
//   TA = 0: A stored [i][p] (lda = row length)        TA = 1: A stored [p][i]
//   TB = 0: B stored [p][j]                           TB = 1: B stored [j][p]
// EPI 0: C = relu(acc + bias[j])                      (forward hidden layer)
// EPI 1: C = acc * (mask[i][j] > 0)                   (dH = dY W^T (.) relu')
// EPI 2: Adam on W[i][j] with gradient acc            (dW = H^T dY; C unused)
#ifndef SS_DYN_GT_N
#define SS_DYN_GT_N 32
#endif
constexpr int GT_M = 64, GT_N = SS_DYN_GT_N, GT_P = 16, GT_THREADS = 256;
constexpr int GT_CN = GT_N / 16;           // output columns per thread (4 rows x GT_CN columns)
constexpr int GT_BL = GT_P * GT_N / GT_THREADS;   // B-tile elements staged per thread
template <typename T>
struct GemmEpi {
    const T* bias;
    const T* mask;
    T* w;
    T* m;
    T* v;
    AdamArgs<T> adam;
};

// 64 x GT_N output tile, 16-deep reduction steps, 256 threads with 4 x GT_CN register micro-tiles; both
// operand tiles are stored reduction-major in shared memory ([p][i], [p][j]) so the inner loop reads
// one float4 of A and one of B per 16 FFMA; the next step's global loads are issued into registers
// before the current step's FMAs (software double buffering).  T = double: the same tiling with DFMA
// (27 KB of static shared memory).
template <typename T, int TA, int TB, int EPI>
__global__ void __launch_bounds__(GT_THREADS)
dyn_gemm_kernel(int M, int N, int P, const T* __restrict__ A, int lda, const T* __restrict__ Bm, int ldb,
                T* __restrict__ C, int ldc, GemmEpi<T> e) {
    __shared__ __align__(16) T As[2][GT_P][GT_M + 4];
    __shared__ __align__(16) T Bs[2][GT_P][GT_N + 4];
    const int tid = threadIdx.x;
    const int i0 = blockIdx.y * GT_M, j0 = blockIdx.x * GT_N;
    const int ti = tid / 16, tj = tid % 16;          // rows ti*4.., columns tj*GT_CN..
    // global -> register staging: 4 elements of A and GT_BL of B per thread and step
    int a_i[4], a_p[4], b_j[GT_BL], b_p[GT_BL];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int o = tid + r * GT_THREADS;
        if (TA == 0) { a_i[r] = o / GT_P; a_p[r] = o % GT_P; } else { a_p[r] = o / GT_M; a_i[r] = o % GT_M; }
    }
#pragma unroll
    for (int r = 0; r < GT_BL; ++r) {
        const int o = tid + r * GT_THREADS;
        if (TB == 0) { b_p[r] = o / GT_N; b_j[r] = o % GT_N; } else { b_j[r] = o / GT_P; b_p[r] = o % GT_P; }
    }
    T ra[4], rb[GT_BL];
    auto fetch = [&](int p0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int gi = i0 + a_i[r], gp = p0 + a_p[r];
            ra[r] = (gi < M && gp < P) ? (TA == 0 ? __ldg(A + (size_t)gi * lda + gp) : __ldg(A + (size_t)gp * lda + gi)) : T(0);
        }
#pragma unroll
        for (int r = 0; r < GT_BL; ++r) {
            const int gj = j0 + b_j[r], gq = p0 + b_p[r];
            rb[r] = (gj < N && gq < P) ? (TB == 0 ? __ldg(Bm + (size_t)gq * ldb + gj) : __ldg(Bm + (size_t)gj * ldb + gq)) : T(0);
        }
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int r = 0; r < 4; ++r) As[buf][a_p[r]][a_i[r]] = ra[r];
#pragma unroll
        for (int r = 0; r < GT_BL; ++r) Bs[buf][b_p[r]][b_j[r]] = rb[r];
    };
    T acc[4][GT_CN] = {};
    fetch(0);
    stash(0);
    __syncthreads();
    int buf = 0;
    for (int p0 = 0; p0 < P; p0 += GT_P) {
        const bool more = p0 + GT_P < P;
        if (more) fetch(p0 + GT_P);
#pragma unroll
        for (int pp = 0; pp < GT_P; ++pp) {
            T a4[4];
            if constexpr (sizeof(T) == 4) {
                const float4 av = *reinterpret_cast<const float4*>(&As[buf][pp][ti * 4]);
                a4[0] = av.x; a4[1] = av.y; a4[2] = av.z; a4[3] = av.w;
            } else {
                const double2 a01 = *reinterpret_cast<const double2*>(&As[buf][pp][ti * 4]);
                const double2 a23 = *reinterpret_cast<const double2*>(&As[buf][pp][ti * 4 + 2]);
                a4[0] = a01.x; a4[1] = a01.y; a4[2] = a23.x; a4[3] = a23.y;
            }
            T b4[GT_CN];
#pragma unroll
            for (int cidx = 0; cidx < GT_CN; ++cidx) b4[cidx] = Bs[buf][pp][tj * GT_CN + cidx];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int cidx = 0; cidx < GT_CN; ++cidx) acc[r][cidx] = fma_t(a4[r], b4[cidx], acc[r][cidx]);
        }
        if (more) {
            stash(buf ^ 1);
            __syncthreads();
            buf ^= 1;
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int gi = i0 + ti * 4 + r;
        if (gi >= M) continue;
#pragma unroll
        for (int cidx = 0; cidx < GT_CN; ++cidx) {
            const int gj = j0 + tj * GT_CN + cidx;
            if (gj >= N) continue;
            const T a = acc[r][cidx];
            if (EPI == 0) {
                C[(size_t)gi * ldc + gj] = relu_t(a + e.bias[gj]);
            } else if (EPI == 1) {
                C[(size_t)gi * ldc + gj] = e.mask[(size_t)gi * ldc + gj] > T(0) ? a : T(0);
            } else {
                const size_t o = (size_t)gi * ldc + gj;
                T w = e.w[o], m = e.m[o], v = e.v[o];
                adam_update(a, w, m, v, e.adam);
                e.w[o] = w; e.m[o] = m; e.v[o] = v;
            }
        }
    }
}

// ---- output layer + loss (+ the first backward product) -----------------------------------------
// out[b][j] = H[b] . W[:, j] + bias[j]; dOut = 2 (out - z) / (B dout); loss = mean (out - z)^2;
// when training also dH[b][k] = (sum_j dOut[b][j] W[k][j]) * [H[b][k] > 0] (N = dout is tiny).
// one warp per batch row; per-block partial loss -> last block (ticket) sums them in fixed order
template <typename T>
__global__ void __launch_bounds__(256)
dyn_out_loss_kernel(const T* __restrict__ H, int h, const T* __restrict__ W, const T* __restrict__ bias,
                    const T* __restrict__ Z, int B, int dout, T* __restrict__ dOut, T* __restrict__ dH,
                    double* __restrict__ partial, unsigned int* __restrict__ ticket, double* __restrict__ loss_out,
                    int train) {
    __shared__ double s_part[8];
    __shared__ T s_dout[8][SS_MAX_D];
    __shared__ bool s_last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + warp;
    double sq = 0.0;
    if (b < B) {
        const T* hb = H + (size_t)b * h;
        for (int j = 0; j < dout; ++j) {
            T acc = T(0);
            for (int k = lane; k < h; k += 32) acc = fma_t(hb[k], W[(size_t)k * dout + j], acc);
            for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
            const T out = acc + bias[j];
            const T diff = out - Z[(size_t)b * dout + j];
            if (lane == 0) {
                const T g = T(2) * diff / (T)(B * dout);
                if (train) dOut[(size_t)b * dout + j] = g;
                s_dout[warp][j] = g;
                sq += (double)diff * (double)diff;
            }
        }
        if (train) {
            __syncwarp();
            for (int k = lane; k < h; k += 32) {
                T acc = T(0);
                for (int j = 0; j < dout; ++j) acc = fma_t(s_dout[warp][j], W[(size_t)k * dout + j], acc);
                dH[(size_t)b * h + k] = hb[k] > T(0) ? acc : T(0);
            }
        }
    }
    if (lane == 0) s_part[warp] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_part[w];
        partial[blockIdx.x] = t;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        double t = 0.0;
        for (int i = 0; i < (int)gridDim.x; ++i) t += __ldcg(partial + i);
        *loss_out = t / ((double)B * dout);
        *ticket = 0;
    }
}

// every "thin" parameter update of a step in ONE launch: the first and the last layer's matrices
// (dW[k][j] = sum_b A[b][k] dY[b][j] with a tiny K or N) and all bias vectors (column sums of dY),
// each followed by its Adam update.  One warp per parameter: lanes stride over the batch, shuffle
// tree (fixed order).
template <typename T>
struct SmallSeg {
    const T* A;          // [B][lda] activations, or null for a bias (A = 1)
    const T* dY;         // [B][ldy]
    T* w;
    T* m;
    T* v;
    int lda, ldy, N;     // parameter o of the segment: k = o / N, j = o % N
    int start;           // first warp of the segment
};
template <typename T>
struct SmallJob {
    SmallSeg<T> seg[DYN_MAX_LAYERS + 3];
    int n_seg, total;
};
template <typename T>
__global__ void __launch_bounds__(256)
dyn_small_updates_kernel(SmallJob<T> job, int B, AdamArgs<T> adam) {
    const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (wid >= job.total) return;
    int si = 0;
    while (si + 1 < job.n_seg && wid >= job.seg[si + 1].start) ++si;
    const SmallSeg<T>& g = job.seg[si];
    const int o = wid - g.start, k = o / g.N, j = o % g.N;
    T acc = T(0);
    if (g.A) {
        for (int b = lane; b < B; b += 32) acc = fma_t(g.A[(size_t)b * g.lda + k], g.dY[(size_t)b * g.ldy + j], acc);
    } else {
        for (int b = lane; b < B; b += 32) acc += g.dY[(size_t)b * g.ldy + j];
    }
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) {
        T w = g.w[o], m = g.m[o], v = g.v[o];
        adam_update(acc, w, m, v, adam);
        g.w[o] = w; g.m[o] = m; g.v[o] = v;
    }
}

// ---- re-packing of the trained parameters for the rollout kernels (device -> device) -----------
__global__ void dyn_pack_fp32_kernel(const float* __restrict__ W, const float* __restrict__ b, int in, int out,
                                     int out_pad, float* __restrict__ Wp, float* __restrict__ bp) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o < in * out) Wp[(size_t)(o / out) * out_pad + (o % out)] = W[o];
    if (o < out) bp[o] = b[o];
}

// float64 masters rounded once to float: the source of the FP32 and tcgen05 images after FP64 training
__global__ void dyn_round_kernel(const double* __restrict__ src, float* __restrict__ dst, size_t n) {
    const size_t o = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (o < n) dst[o] = (float)src[o];
}

__device__ __forceinline__ unsigned short bf16_bits_dev(float f) {
    unsigned int u = __float_as_uint(f);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (unsigned short)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (unsigned short)(u >> 16);
}
__device__ __forceinline__ float bf16_val_dev(unsigned short b) { return __uint_as_float((unsigned int)b << 16); }

// the images of mpc_tc.cu (mpc_tc_prepare), same index maps, built from the FP32 master weights.
// geometry constants are passed in so this file does not depend on the kernel's namespace.
struct TcGeom {
    int h, d, din, dz, k1, hp, nch, nslab;
    int NC, NH, KSLAB, CLUSTER, w1_chunk_halfs, stage_halfs, dzp;
};
__global__ void dyn_pack_tc_kernel(TcGeom g, const float* __restrict__ W1, const float* __restrict__ B1,
                                   const float* __restrict__ W2, const float* __restrict__ B2,
                                   const float* __restrict__ W3, const float* __restrict__ B3,
                                   unsigned short* __restrict__ w1img, unsigned short* __restrict__ w2img,
                                   float* __restrict__ w3p, float* __restrict__ b3_out) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    auto w1_at = [&](int slot, int u) -> size_t {
        const int cidx = u / g.NC, r = (u % g.NC) / g.NH, nn = u % g.NH;
        return ((size_t)r * g.nch + cidx) * g.w1_chunk_halfs + (size_t)(slot / 8) * (g.NH * 8) + nn * 8 + (slot % 8);
    };
    auto w2_at = [&](int k, int u) -> size_t {
        const int n = u / g.NC, r = (u % g.NC) / g.NH, nn = u % g.NH, ksl = k / g.KSLAB, kk = k % g.KSLAB;
        return (((size_t)n * g.nslab + ksl) * g.CLUSTER + r) * g.stage_halfs + (size_t)(kk / 8) * (g.NH * 8) + nn * 8 +
               (kk % 8);
    };
    // layer-2 image: one thread per (k, u) incl. the two bias rows k = h, h + 1
    if (t < (long long)(g.h + 2) * g.h) {
        const int k = (int)(t / g.h), u = (int)(t % g.h);
        unsigned short val;
        if (k < g.h) val = bf16_bits_dev(W2[(size_t)k * g.h + u]);
        else {
            const float b = B2[u];
            const unsigned short hi = bf16_bits_dev(b);
            val = k == g.h ? hi : bf16_bits_dev(b - bf16_val_dev(hi));
        }
        w2img[w2_at(k, u)] = val;
    }
    // layer-1 image: one thread per unit
    if (t < g.h) {
        const int u = (int)t;
        for (int j = 0; j < g.din; ++j) {
            const float w = W1[(size_t)j * g.h + u];
            const unsigned short hi = bf16_bits_dev(w), lo = bf16_bits_dev(w - bf16_val_dev(hi));
            const int in = j < g.d ? j : g.dz + (j - g.d);
            w1img[w1_at(3 * in, u)] = hi;
            w1img[w1_at(3 * in + 1, u)] = lo;
            w1img[w1_at(3 * in + 2, u)] = hi;
        }
        const float b = B1[u];
        const unsigned short hi = bf16_bits_dev(b), lo = bf16_bits_dev(b - bf16_val_dev(hi));
        w1img[w1_at(g.k1 - 2, u)] = hi;
        w1img[w1_at(g.k1 - 1, u)] = lo;
        for (int j = 0; j < g.d; ++j) w3p[((size_t)(u / 2) * g.dzp + j) * 2 + (u & 1)] = W3[(size_t)u * g.d + j];
    }
    if (t == 0) {
        w1img[w1_at(g.k1 - 2, g.h)] = 0x3f80;          // constant-one hidden units h, h + 1 (bf16 1.0)
        w1img[w1_at(g.k1 - 2, g.h + 1)] = 0x3f80;
    }
    if (t < g.d) b3_out[t] = B3[t];
}

}  // namespace

// geometry of the tcgen05 images (mpc_tc.cu)
void mpc_tc_geometry(const ss_ctx* c, int* k1, int* dz, int* hp, int* NC, int* NH, int* KSLAB, int* CLUSTER, int* dzp);

struct DynLayout {
    int L, din, dout, h;
    size_t w_off[DYN_MAX_LAYERS], b_off[DYN_MAX_LAYERS], total;
    int in[DYN_MAX_LAYERS], out[DYN_MAX_LAYERS];
};

static DynLayout dyn_layout(const ss_ctx* c) {
    DynLayout y;
    y.L = c->L; y.din = c->d + c->da; y.dout = c->d; y.h = c->h;
    size_t off = 0;
    for (int l = 0; l <= y.L; ++l) {
        y.in[l] = l == 0 ? y.din : y.h;
        y.out[l] = l == y.L ? y.dout : y.h;
        y.w_off[l] = off; off += (size_t)y.in[l] * y.out[l];
        y.b_off[l] = off; off += (size_t)y.out[l];
        off = (off + 3) / 4 * 4;
    }
    y.total = off;
    return y;
}

// (re)create the master copy (T = float: FP32 trainer, double: SS_PRECISION_FP64) + zeroed Adam state
// from the float64 host parameters of ss_mpc_set_model; called lazily by the first training call after
// a host-side set_model
template <typename T>
static int dyn_sync_from_host(ss_ctx* c) {
    const DynLayout y = dyn_layout(c);
    const size_t bytes = y.total * sizeof(T);
    std::vector<T> host(y.total, T(0));
    for (int l = 0; l <= y.L; ++l) {
        for (size_t i = 0; i < (size_t)y.in[l] * y.out[l]; ++i) host[y.w_off[l] + i] = (T)c->hw[l][i];
        for (int i = 0; i < y.out[l]; ++i) host[y.b_off[l] + i] = (T)c->hb[l][i];
    }
    SS_CUDA_CHECK(c, c->dyn_params.ensure(bytes));
    SS_CUDA_CHECK(c, c->dyn_m.ensure(bytes));
    SS_CUDA_CHECK(c, c->dyn_v.ensure(bytes));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->dyn_params.p, host.data(), bytes, cudaMemcpyHostToDevice, c->stream));
    if (!c->dyn_adam_valid) {
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->dyn_m.p, 0, bytes, c->stream));
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->dyn_v.p, 0, bytes, c->stream));
        c->dyn_t = 0;
        c->dyn_adam_valid = true;
    }
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    c->dyn_params_valid = true;
    return SS_OK;
}

template <typename T>
static int dyn_upload_data(ss_ctx* c, int which, const double* X, const double* Z, int64_t n_rows) {
    const int din = c->d + c->da, dout = c->d;
    std::vector<T> x((size_t)n_rows * din), z((size_t)n_rows * dout);
    for (size_t i = 0; i < x.size(); ++i) x[i] = (T)X[i];
    for (size_t i = 0; i < z.size(); ++i) z[i] = (T)Z[i];
    SS_CUDA_CHECK(c, c->dyn_x[which].ensure(x.size() * sizeof(T) + 16));
    SS_CUDA_CHECK(c, c->dyn_z[which].ensure(z.size() * sizeof(T) + 16));
    if (n_rows > 0) {
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->dyn_x[which].p, x.data(), x.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->dyn_z[which].p, z.data(), z.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    }
    c->dyn_rows[which] = n_rows;
    return SS_OK;
}

extern "C" int ss_dyn_set_data(ss_ctx* c, int which, const double* X, const double* Z, int64_t n_rows) {
    if (!c) return SS_EINVAL;
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "dyn: set the model first (ss_mpc_set_model)");
    if ((which != 0 && which != 1) || n_rows < 0 || (n_rows > 0 && (!X || !Z))) SS_FAIL(c, SS_EINVAL, "dyn: bad data arguments");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    return c->dyn_fp64 ? dyn_upload_data<double>(c, which, X, Z, n_rows) : dyn_upload_data<float>(c, which, X, Z, n_rows);
}

extern "C" int ss_dyn_reset_optimizer(ss_ctx* c) {
    if (!c) return SS_EINVAL;
    c->dyn_adam_valid = false;
    c->dyn_params_valid = false;     // the next training call re-reads the host parameters
    return SS_OK;
}

extern "C" int ss_dyn_set_precision(ss_ctx* c, int precision) {
    if (!c) return SS_EINVAL;
    if (precision != SS_PRECISION_FP32 && precision != SS_PRECISION_FP64)
        SS_FAIL(c, SS_EINVAL, "dyn: the trainer's precision is SS_PRECISION_FP32 or SS_PRECISION_FP64");
    const bool fp64 = precision == SS_PRECISION_FP64;
    if (fp64 == c->dyn_fp64) return SS_OK;
    // the buffers change their element type: nothing in them survives
    c->dyn_fp64 = fp64;
    c->dyn_adam_valid = false;
    c->dyn_params_valid = false;
    c->dyn_dirty = false;
    c->dyn_rows[0] = c->dyn_rows[1] = 0;
    return SS_OK;
}

template <typename T, int TA, int TB, int EPI>
static void launch_gemm(ss_ctx* c, int M, int N, int P, const T* A, int lda, const T* B, int ldb, T* C, int ldc,
                        const GemmEpi<T>& e) {
    dim3 grid((N + GT_N - 1) / GT_N, (M + GT_M - 1) / GT_M);
    dyn_gemm_kernel<T, TA, TB, EPI><<<grid, GT_THREADS, 0, c->stream>>>(M, N, P, A, lda, B, ldb, C, ldc, e);
    c->launches++;
}

// one batch through the network: forward (+ loss) and, when train != 0, backward + Adam
template <typename T>
static int dyn_step(ss_ctx* c, const DynLayout& y, const int* idx_old, const int* idx_new, int n_old, int B,
                    double* loss_out, int train, T lr, int src_old, int src_new) {
    T* P = c->dyn_params.as<T>();
    T* Mo = c->dyn_m.as<T>();
    T* Vo = c->dyn_v.as<T>();
    const int h = y.h, din = y.din, dout = y.dout, L = y.L;
    // activations: X [B][din], Z [B][dout], H_1..H_L [B][h]; gradients dOut [B][dout], dH_1..dH_L [B][h]
    T* X = c->dyn_act.as<T>();
    T* Z = X + (size_t)B * din;
    T* H = Z + (size_t)B * dout;                              // H_l at H + (l - 1) * B * h
    T* dOut = H + (size_t)L * B * h;
    T* dH = dOut + (size_t)B * dout;                          // dH_l at dH + (l - 1) * B * h
    double* partial = c->dyn_scratch.as<double>();
    unsigned int* ticket = reinterpret_cast<unsigned int*>(partial + 256);
    AdamArgs<T> adam;
    adam.beta1 = (T)0.9; adam.beta2 = (T)0.999; adam.eps = (T)1e-8;
    adam.omb1 = (T)(1.0 - 0.9); adam.omb2 = (T)(1.0 - 0.999);
    if (train) {
        c->dyn_t += 1;
        const double t = (double)c->dyn_t;
        adam.lr_t = (T)((double)lr * std::sqrt(1.0 - std::pow(0.999, t)) / (1.0 - std::pow(0.9, t)));
    } else {
        adam.lr_t = T(0);
    }
    const int rows_pb = 8;
    dyn_first_layer_kernel<T><<<(B + rows_pb - 1) / rows_pb, rows_pb * 32, (size_t)rows_pb * din * sizeof(T), c->stream>>>(
        c->dyn_x[src_old].as<T>(), c->dyn_z[src_old].as<T>(), c->dyn_x[src_new].as<T>(),
        c->dyn_z[src_new].as<T>(), idx_old, idx_new, n_old, B, din, dout, P + y.w_off[0], P + y.b_off[0], h, 1, X, Z, H);
    c->launches++;
    GemmEpi<T> e;
    std::memset(&e, 0, sizeof(e));
    for (int l = 1; l < L; ++l) {
        e.bias = P + y.b_off[l];
        launch_gemm<T, 0, 0, 0>(c, B, h, h, H + (size_t)(l - 1) * B * h, h, P + y.w_off[l], h, H + (size_t)l * B * h, h, e);
    }
    const T* HL = H + (size_t)(L - 1) * B * h;
    T* dHL = dH + (size_t)(L - 1) * B * h;
    dyn_out_loss_kernel<T><<<(B + 7) / 8, 256, 0, c->stream>>>(HL, h, P + y.w_off[L], P + y.b_off[L], Z, B, dout, dOut,
                                                               dHL, partial, ticket, loss_out, train);
    c->launches++;
    if (!train) {
        SS_CUDA_CHECK(c, cudaGetLastError());
        return SS_OK;
    }
    // ---- backward.  Every dH uses the weights of the forward pass: it is computed BEFORE the Adam
    // update of the same layer's matrix (dH_L came out of the loss kernel; W_L is updated last).
    for (int l = L - 1; l >= 1; --l) {
        // dH_l [B][h] = dH_{l+1} [B][h] W_l^T (W_l stored [in = h][out = h]) (.) [H_l > 0]
        e.mask = H + (size_t)(l - 1) * B * h;
        launch_gemm<T, 0, 1, 1>(c, B, h, h, dH + (size_t)l * B * h, h, P + y.w_off[l], h, dH + (size_t)(l - 1) * B * h, h, e);
        // dW_l [h][h] = H_l^T [h][B] dH_{l+1} [B][h], Adam fused
        e.w = P + y.w_off[l]; e.m = Mo + y.w_off[l]; e.v = Vo + y.w_off[l]; e.adam = adam;
        launch_gemm<T, 1, 0, 2>(c, h, h, B, H + (size_t)(l - 1) * B * h, h, dH + (size_t)l * B * h, h, nullptr, h, e);
    }
    // first / last layer matrices and every bias vector: one launch
    SmallJob<T> job;
    std::memset(&job, 0, sizeof(job));
    int ns = 0, start = 0;
    auto add_seg = [&](const T* A, int lda, const T* dY, int ldy, int K, int N, size_t off) {
        SmallSeg<T>& g = job.seg[ns++];
        g.A = A; g.lda = lda; g.dY = dY; g.ldy = ldy; g.N = N;
        g.w = P + off; g.m = Mo + off; g.v = Vo + off;
        g.start = start;
        start += K * N;
    };
    add_seg(HL, h, dOut, dout, h, dout, y.w_off[L]);                 // dW_L = H_L^T dOut
    add_seg(X, din, dH, h, din, h, y.w_off[0]);                      // dW_0 = X^T dH_1
    for (int l = 0; l <= L; ++l)                                     // db_l = column sums of dY_l
        add_seg(nullptr, 0, l == L ? dOut : dH + (size_t)l * B * h, y.out[l], 1, y.out[l], y.b_off[l]);
    job.n_seg = ns;
    job.total = start;
    dyn_small_updates_kernel<T><<<(start + 7) / 8, 256, 0, c->stream>>>(job, B, adam);
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}

static int dyn_prepare(ss_ctx* c, int B) {
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "dyn: set the model first (ss_mpc_set_model)");
    if (B < 1) SS_FAIL(c, SS_EINVAL, "dyn: empty batch");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    if (!c->dyn_params_valid) {
        int rc = c->dyn_fp64 ? dyn_sync_from_host<double>(c) : dyn_sync_from_host<float>(c);
        if (rc) return rc;
    }
    const DynLayout y = dyn_layout(c);
    const size_t act = ((size_t)B * (y.din + 2 * y.dout) + 2 * (size_t)y.L * B * y.h) * (c->dyn_fp64 ? 8 : 4);
    SS_CUDA_CHECK(c, c->dyn_act.ensure(act));
    if (!c->dyn_scratch.p) {
        SS_CUDA_CHECK(c, c->dyn_scratch.ensure(256 * 8 + 64));
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->dyn_scratch.p, 0, 256 * 8 + 64, c->stream));
    }
    if ((B + 7) / 8 > 256) SS_FAIL(c, SS_EUNSUPPORTED, "dyn: batch size above 2048");
    return SS_OK;
}

// n_batches Adam steps: batch i = old rows idx_old[i*n_old .. ) followed by new rows idx_new[i*n_new .. )
extern "C" int ss_dyn_train_batches(ss_ctx* c, const int32_t* idx_old, const int32_t* idx_new, int n_batches, int n_old,
                                    int n_new, double lr, double* out_losses) {
    if (!c) return SS_EINVAL;
    if (n_batches < 1 || n_old < 0 || n_new < 0 || n_old + n_new < 1 || (n_old > 0 && !idx_old) || (n_new > 0 && !idx_new))
        SS_FAIL(c, SS_EINVAL, "dyn: bad batch arguments");
    const int B = n_old + n_new;
    int rc = dyn_prepare(c, B);
    if (rc) return rc;
    for (long long i = 0; i < (long long)n_batches * n_old; ++i)
        if (idx_old[i] < 0 || idx_old[i] >= c->dyn_rows[0]) SS_FAIL(c, SS_EINVAL, "dyn: old-data row index out of range");
    for (long long i = 0; i < (long long)n_batches * n_new; ++i)
        if (idx_new[i] < 0 || idx_new[i] >= c->dyn_rows[1]) SS_FAIL(c, SS_EINVAL, "dyn: new-data row index out of range");
    const DynLayout y = dyn_layout(c);
    const size_t n_idx = (size_t)n_batches * B;
    SS_CUDA_CHECK(c, c->dyn_idx.ensure(n_idx * 4 + 16));
    SS_CUDA_CHECK(c, c->dyn_losses.ensure((size_t)n_batches * 8));
    int* d_old = c->dyn_idx.as<int>();
    int* d_new = d_old + (size_t)n_batches * n_old;
    if (n_old) SS_CUDA_CHECK(c, cudaMemcpyAsync(d_old, idx_old, (size_t)n_batches * n_old * 4, cudaMemcpyHostToDevice, c->stream));
    if (n_new) SS_CUDA_CHECK(c, cudaMemcpyAsync(d_new, idx_new, (size_t)n_batches * n_new * 4, cudaMemcpyHostToDevice, c->stream));
    timer_begin(c);
    for (int i = 0; i < n_batches; ++i) {
        int* io = d_old + (size_t)i * n_old;
        int* inw = d_new + (size_t)i * n_new;
        double* li = c->dyn_losses.as<double>() + i;
        rc = c->dyn_fp64 ? dyn_step<double>(c, y, io, inw, n_old, B, li, 1, lr, 0, 1)
                         : dyn_step<float>(c, y, io, inw, n_old, B, li, 1, (float)lr, 0, 1);
        if (rc) return rc;
    }
    timer_mark(c, "dyn_train");
    c->dyn_dirty = true;             // the rollout kernels still hold the previous parameters
    if (out_losses) {
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_losses, c->dyn_losses.p, (size_t)n_batches * 8, cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    }
    return SS_OK;
}

// mean over consecutive full batches of `batchsize` rows of data set `which` of the batch MSE
// (the old_loss / new_loss of dynamics_model.py:139-166 and run_validation :174-197)
extern "C" int ss_dyn_eval_loss(ss_ctx* c, int which, int batchsize, double* out_mean_loss, int* out_batches) {
    if (!c) return SS_EINVAL;
    if ((which != 0 && which != 1) || batchsize < 1 || !out_mean_loss) SS_FAIL(c, SS_EINVAL, "dyn: bad eval arguments");
    int rc = dyn_prepare(c, batchsize);
    if (rc) return rc;
    const DynLayout y = dyn_layout(c);
    const int nb = (int)(c->dyn_rows[which] / batchsize);
    if (out_batches) *out_batches = nb;
    *out_mean_loss = 0.0;
    if (nb == 0) return SS_OK;
    std::vector<int> idx((size_t)nb * batchsize);
    for (size_t i = 0; i < idx.size(); ++i) idx[i] = (int)i;
    SS_CUDA_CHECK(c, c->dyn_idx.ensure(idx.size() * 4 + 16));
    SS_CUDA_CHECK(c, c->dyn_losses.ensure((size_t)nb * 8));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->dyn_idx.p, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice, c->stream));
    for (int i = 0; i < nb; ++i) {
        int* io = c->dyn_idx.as<int>() + (size_t)i * batchsize;
        double* li = c->dyn_losses.as<double>() + i;
        rc = c->dyn_fp64 ? dyn_step<double>(c, y, io, nullptr, batchsize, batchsize, li, 0, 0.0, which, which)
                         : dyn_step<float>(c, y, io, nullptr, batchsize, batchsize, li, 0, 0.f, which, which);
        if (rc) return rc;
    }
    std::vector<double> l(nb);
    SS_CUDA_CHECK(c, cudaMemcpyAsync(l.data(), c->dyn_losses.p, (size_t)nb * 8, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    double s = 0.0;
    for (double v : l) s += v;
    *out_mean_loss = s / nb;
    return SS_OK;
}

// the trained parameters as float64 [in][out] matrices / [out] vectors (export, checkpoints, tests)
extern "C" int ss_dyn_get_params(ss_ctx* c, double* const* out_weights, double* const* out_biases) {
    if (!c) return SS_EINVAL;
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "dyn: no model");
    if (!out_weights || !out_biases) SS_FAIL(c, SS_EINVAL, "dyn: null output");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const DynLayout y = dyn_layout(c);
    if (!c->dyn_params_valid) {
        for (int l = 0; l <= y.L; ++l) {
            std::memcpy(out_weights[l], c->hw[l].data(), c->hw[l].size() * 8);
            std::memcpy(out_biases[l], c->hb[l].data(), c->hb[l].size() * 8);
        }
        return SS_OK;
    }
    if (c->dyn_fp64) {                // the float64 masters as they are
        std::vector<double> host(y.total);
        SS_CUDA_CHECK(c, cudaMemcpyAsync(host.data(), c->dyn_params.p, y.total * 8, cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        for (int l = 0; l <= y.L; ++l) {
            std::memcpy(out_weights[l], host.data() + y.w_off[l], (size_t)y.in[l] * y.out[l] * 8);
            std::memcpy(out_biases[l], host.data() + y.b_off[l], (size_t)y.out[l] * 8);
        }
        return SS_OK;
    }
    std::vector<float> host(y.total);
    SS_CUDA_CHECK(c, cudaMemcpyAsync(host.data(), c->dyn_params.p, y.total * 4, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    for (int l = 0; l <= y.L; ++l) {
        for (size_t i = 0; i < (size_t)y.in[l] * y.out[l]; ++i) out_weights[l][i] = (double)host[y.w_off[l] + i];
        for (int i = 0; i < y.out[l]; ++i) out_biases[l][i] = (double)host[y.b_off[l] + i];
    }
    return SS_OK;
}

// hand the trained parameters to the rollout kernels without leaving the device
extern "C" int ss_dyn_commit(ss_ctx* c) {
    if (!c) return SS_EINVAL;
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "dyn: no model");
    if (!c->dyn_params_valid || !c->dyn_dirty) return SS_OK;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const DynLayout y = dyn_layout(c);
    // the FP32 and tcgen05 images come from FP32 parameters: after FP64 training, the masters rounded once
    const float* P = c->dyn_params.as<float>();
    if (c->dyn_fp64) {
        SS_CUDA_CHECK(c, c->dyn_round.ensure(y.total * 4));
        dyn_round_kernel<<<(unsigned)((y.total + 255) / 256), 256, 0, c->stream>>>(c->dyn_params.as<double>(),
                                                                                  c->dyn_round.as<float>(), y.total);
        c->launches++;
        P = c->dyn_round.as<float>();
    }
    for (int l = 0; l <= y.L; ++l) {
        const int out_pad = l == y.L ? (c->d + 7) / 8 * 8 : c->h_pad;
        const int n = std::max(y.in[l] * y.out[l], y.out[l]);
        dyn_pack_fp32_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(P + y.w_off[l], P + y.b_off[l], y.in[l], y.out[l],
                                                                    out_pad, c->w32[l].as<float>(), c->b32[l].as<float>());
        c->launches++;
    }
    // the float64 copies of SS_PRECISION_FP64 roll out the same parameters Dyn_Model.export() returns: the
    // float64 masters unchanged, or the FP32 masters widened
    for (int l = 0; l <= y.L; ++l) {
        const int out_pad = l == y.L ? (c->d + 7) / 8 * 8 : c->h_pad;
        if (c->dyn_fp64) {
            const double* P64 = c->dyn_params.as<double>();
            SS_CUDA_CHECK(c, cudaMemcpy2DAsync(c->w64[l].p, (size_t)out_pad * 8, P64 + y.w_off[l], (size_t)y.out[l] * 8,
                                               (size_t)y.out[l] * 8, y.in[l], cudaMemcpyDeviceToDevice, c->stream));
            SS_CUDA_CHECK(c, cudaMemcpyAsync(c->b64[l].p, P64 + y.b_off[l], (size_t)y.out[l] * 8, cudaMemcpyDeviceToDevice,
                                             c->stream));
            continue;
        }
        int rc = mpc_fp64_widen(c, P + y.w_off[l], P + y.b_off[l], y.in[l], y.out[l], out_pad, c->w64[l].as<double>(),
                                c->b64[l].as<double>());
        if (rc) return rc;
    }
    if (c->tc_ready) {
        TcGeom g;
        std::memset(&g, 0, sizeof(g));
        g.h = c->h; g.d = c->d; g.din = c->d + c->da;
        mpc_tc_geometry(c, &g.k1, &g.dz, &g.hp, &g.NC, &g.NH, &g.KSLAB, &g.CLUSTER, &g.dzp);
        g.nch = g.hp / g.NC; g.nslab = g.hp / g.KSLAB;
        g.w1_chunk_halfs = g.NH * g.k1; g.stage_halfs = g.NH * g.KSLAB;
        SS_CUDA_CHECK(c, c->tc_b3.ensure(SS_MAX_D * 4));
        const long long threads = (long long)(g.h + 2) * g.h;
        dyn_pack_tc_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(
            g, P + y.w_off[0], P + y.b_off[0], P + y.w_off[1], P + y.b_off[1], P + y.w_off[2], P + y.b_off[2],
            c->tc_w1.as<unsigned short>(), c->tc_w2.as<unsigned short>(), c->tc_w3.as<float>(), c->tc_b3.as<float>());
        c->launches++;
    }
    SS_CUDA_CHECK(c, cudaGetLastError());
    c->dyn_dirty = false;
    c->host_params_stale = true;      // hw / hb (float64 host copies) no longer match the device
    c->run.valid = false;
    return SS_OK;
}
