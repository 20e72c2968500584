// mpc_fp64.cu -- float64 rollout of the dynamics MLP (SS_PRECISION_FP64).
//
// The reference plans in float64 (NND_MB_agent.tf_datatype; Dyn_Model.do_forward_sim and the numpy of
// generate_scores_add_delta).  This kernel does the same arithmetic in the same precision: normalisation,
// MLP, state update and the scoring of every point in float64, the element-wise parts in the reference's
// operation order (score.cuh, float64 twin), so a decision returns the reference's decision up to the
// summation order of the matrix products and of the projection sums.
//
// Layout follows the FP32 CTA kernel (mpc_simt.cu): one CTA = 32 sequences for all H steps, activations in
// shared memory, weights streamed from L2 through a double-buffered cp.async stage.  In doubles two activation
// buffers of h_pad x 32 rows would be 256 KB at h = 500, so the CTA runs the MLP of a step in two passes of 16
// rows; the scoring still sees 32 sequences, and one CTA is one column of the projection-sum table, the layout
// mpc_fold_partials / mpc_reduce_sums / the peer all-reduce expect.
//
// Matrix products are DFMA on the CUDA cores (DESIGN.md 3.6: DMMA measured at the same peak on B200).
#include "mpc_kernels.cuh"

namespace {

constexpr int SEQ = 32;    // sequences per CTA (one projection-sum column)
constexpr int R = 16;      // rows of one MLP pass
constexpr int NT = 256;    // threads per CTA
constexpr int KT = 8;      // k-tile of a weight stage
constexpr int UT = 256;    // units per pass (32 unit groups x 8)

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N));
}

// out[u][r] = act(sum_k in[k][r] * Wg[k][u] + bias[u])   in: [K_pad][R], out: [N_pad][R]
__device__ void dense_layer64(const double* __restrict__ in, int K_pad, const double* __restrict__ Wg,
                              const double* __restrict__ bias, int N_pad, double* __restrict__ out, bool relu,
                              double* __restrict__ Ws) {
    const int tid = threadIdx.x;
    const int rg = tid & 7;       // rows 2*rg, 2*rg+1
    const int ug = tid >> 3;      // units ug*8 .. ug*8+7 of the pass
    const int ntile = K_pad / KT;
    for (int u_pass = 0; u_pass < N_pad; u_pass += UT) {
        const int cols = N_pad - u_pass < UT ? N_pad - u_pass : UT;   // multiple of 8
        const int vec_per_row = cols >> 1;                              // 16-byte pieces
        const int nvec = KT * vec_per_row;
        double acc[2][8];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.0;

        auto stage_load = [&](int kt, int stage) {
            double* dst = Ws + stage * (KT * UT);
            const double* src = Wg + (size_t)kt * KT * N_pad + u_pass;
            for (int v = tid; v < nvec; v += NT) {
                int kk = v / vec_per_row, c2 = v - kk * vec_per_row;
                cp_async16(dst + kk * UT + 2 * c2, src + (size_t)kk * N_pad + 2 * c2);
            }
            cp_async_commit();
        };
        stage_load(0, 0);
        for (int kt = 0; kt < ntile; ++kt) {
            if (kt + 1 < ntile) {
                stage_load(kt + 1, (kt + 1) & 1);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            if (ug * 8 < cols) {
                const double* wt = Ws + (kt & 1) * (KT * UT) + ug * 8;
                const double* it = in + (size_t)kt * KT * R + 2 * rg;
#pragma unroll
                for (int kk = 0; kk < KT; ++kk) {
                    const double2 av = *reinterpret_cast<const double2*>(it + kk * R);
                    double wv[8];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const double2 w = *reinterpret_cast<const double2*>(wt + kk * UT + 2 * q);
                        wv[2 * q] = w.x;
                        wv[2 * q + 1] = w.y;
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        acc[0][j] = fma(av.x, wv[j], acc[0][j]);
                        acc[1][j] = fma(av.y, wv[j], acc[1][j]);
                    }
                }
            }
            __syncthreads();
        }
        if (ug * 8 < cols) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int u = u_pass + ug * 8 + j;
                const double bj = bias[u];
                double2 o;
                o.x = acc[0][j] + bj;
                o.y = acc[1][j] + bj;
                if (relu) {            // np.maximum(h, 0): NaN stays NaN
                    o.x = o.x < 0.0 ? 0.0 : o.x;
                    o.y = o.y < 0.0 ? 0.0 : o.y;
                }
                *reinterpret_cast<double2*>(out + (size_t)u * R + 2 * rg) = o;
            }
        }
    }
    __syncthreads();
}

// z[j][r] = sum_k in[k][r] * Wg[k][j] + b[j],  j < d; K split over 16 slices, eight outputs at a time
__device__ void output_layer64(const double* __restrict__ in, int K_pad, const double* __restrict__ Wg,
                               const double* __restrict__ bias, int N_pad, int d, double* __restrict__ z,
                               double* __restrict__ red /* [16][8][R] */) {
    const int r = threadIdx.x & (R - 1), ks = threadIdx.x >> 4;
    const int per = (K_pad + 15) / 16;
    const int k0 = ks * per, k1 = k0 + per < K_pad ? k0 + per : K_pad;
    for (int j0 = 0; j0 < d; j0 += 8) {
        double acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.0;
        for (int k = k0; k < k1; ++k) {
            const double a = in[(size_t)k * R + r];
            const double2* wr = reinterpret_cast<const double2*>(Wg + (size_t)k * N_pad + j0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double2 w = __ldg(wr + q);
                acc[2 * q] = fma(a, w.x, acc[2 * q]);
                acc[2 * q + 1] = fma(a, w.y, acc[2 * q + 1]);
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) red[(ks * 8 + j) * R + r] = acc[j];
        __syncthreads();
        for (int o = threadIdx.x; o < 8 * R; o += NT) {
            const int j = o / R, rr = o - j * R;
            if (j0 + j < d) {
                double s = red[j * R + rr];
#pragma unroll
                for (int q = 1; q < 16; ++q) s += red[(q * 8 + j) * R + rr];
                z[(size_t)(j0 + j) * R + rr] = s + bias[j0 + j];
            }
        }
        __syncthreads();
    }
}

template <int DT, bool ROWS>            // ROWS: per-sequence start rows (load_start)
__global__ void __launch_bounds__(NT, 1) mpc_rollout_fp64_kernel(const Rollout64Args a) {
    pdl_trigger();      // the reduce / tail kernels behind this launch may be scheduled (they wait for its completion)
    extern __shared__ __align__(16) double sm64[];
    const int act_elems = (a.h_pad > a.din_pad ? a.h_pad : a.din_pad) * R;
    double* actA = sm64;
    double* actB = actA + act_elems;
    double* Ws = actB + act_elems;                // 2 * KT * UT (the output layer's partial sums reuse it)
    double* st = Ws + 2 * KT * UT;                // state [SS_MAX_D][SEQ]
    double* z = st + SS_MAX_D * SEQ;              // [SS_MAX_D][R]

    const int tid = threadIdx.x;
    const long long k_local = (long long)blockIdx.x * SEQ + tid;   // sequence owners: tid < SEQ
    const bool owner = tid < SEQ;
    const bool live = owner && k_local < a.K_local;
    const int T = a.H + 1;
    const int d = a.d, rs = d + 1;
    const MpcNorm64& nm = a.norm;

    ScoreAcc64 sc;
    if (owner) {
        double x[DT];
        load_start<ROWS, DT>(a, live, k_local, x);
        if constexpr (ROWS) {
#pragma unroll
            for (int j = 0; j < DT; ++j)
                if (j < d) st[j * SEQ + tid] = x[j];
        } else {
            for (int j = 0; j < d; ++j) st[j * SEQ + tid] = a.state0[j];
        }
        score_init64<DT>(a.plan, a.wp_index, x, sc);
    }
    for (int o = tid; o < a.din_pad * R; o += NT) actA[o] = 0.0;
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        // ---- score the current point (sequence owners, warp 0; the state is read back from shared memory so
        // that it holds no registers during the MLP) ----------------------------------------------------------
        if (owner) {
            double x[DT];
#pragma unroll
            for (int j = 0; j < DT; ++j) x[j] = j < d ? st[j * SEQ + tid] : 0.0;
            if (a.per_sample) score_point64_per_sample<DT>(a.plan, t, x, sc);
            else progress64<DT>(a.plan, t, x, sc);      // (reference mode: the tail scores the rows)
            if (live && a.rows_out) {
                double* row = a.rows_out + ((size_t)t * a.K_local + k_local) * rs;
#pragma unroll
                for (int j = 0; j < DT; ++j)
                    if (j < d) row[j] = x[j];
                row[d] = (double)sc.idx;
            }
            if (a.qsums) {
                double ab = 0.0, bb = 0.0;
                if (live) proj_terms64<DT>(a.plan, sc.idx, x, ab, bb);
                for (int off = 16; off > 0; off >>= 1) {
                    ab += __shfl_down_sync(0xffffffffu, ab, off);
                    bb += __shfl_down_sync(0xffffffffu, bb, off);
                }
                if (tid == 0) {
                    a.qsums[((size_t)t * 2) * gridDim.x + blockIdx.x] = ab;
                    a.qsums[((size_t)t * 2 + 1) * gridDim.x + blockIdx.x] = bb;
                }
            }
        }
        if (t == a.H) break;
        for (int half = 0; half < SEQ / R; ++half) {
            // ---- network input: (x - mean) / std of state and action (dynamics_model.py:228-230) ----------
            if (tid < R) {
                const int s = half * R + tid;
                const long long kl = (long long)blockIdx.x * SEQ + s;
                for (int j = 0; j < d; ++j)
                    actA[j * R + tid] = nm.std_x[j] != 0.0 ? (st[j * SEQ + s] - nm.mean_x[j]) / nm.std_x[j] : 0.0;
                for (int j = 0; j < a.da; ++j) {
                    const double act = kl < a.K_local ? fetch_action_f64(a.act, kl, a.k_offset + kl, t, j) : 0.0;
                    actA[(d + j) * R + tid] = nm.std_y[j] != 0.0 ? (act - nm.mean_y[j]) / nm.std_y[j] : 0.0;
                }
            }
            __syncthreads();
            // ---- MLP: L hidden layers (Linear + ReLU) and a linear output layer ------------------------------
            double* cur = actA;
            double* nxt = actB;
            int K_pad = a.din_pad;
            for (int l = 0; l < a.L; ++l) {
                dense_layer64(cur, K_pad, a.w[l], a.b[l], a.h_pad, nxt, true, Ws);
                double* tmp = cur; cur = nxt; nxt = tmp;
                K_pad = a.h_pad;
            }
            output_layer64(cur, K_pad, a.w[a.L], a.b[a.L], a.dout_pad, d, z, Ws);
            // ---- state update s + (z * std_z + mean_z) (dynamics_model.py:234-237) ---------------------------
            if (tid < R) {
                const int s = half * R + tid;
                for (int j = 0; j < d; ++j)
                    st[j * SEQ + s] = st[j * SEQ + s] + (__dmul_rn(z[j * R + tid], nm.std_z[j]) + nm.mean_z[j]);
            }
            // hidden layers 1, 3, .. write into actA: its padded input rows must be zero again
            if (a.L >= 2) {
                __syncthreads();
                for (int o = tid + (d + a.da) * R; o < a.din_pad * R; o += NT) actA[o] = 0.0;
            }
            __syncthreads();
        }
    }
    if (live && a.scores_out) a.scores_out[k_local] = sc.score;
}

__global__ void widen_kernel(const float* __restrict__ W, const float* __restrict__ b, int in, int out, int out_pad,
                             double* __restrict__ Wp, double* __restrict__ bp) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o < in * out) Wp[(size_t)(o / out) * out_pad + (o % out)] = (double)W[o];
    if (o < out) bp[o] = (double)b[o];
}

template <int DT>
cudaError_t launch_fp64(ss_ctx* c, const Rollout64Args& a, int grid, size_t smem) {
    auto kern = a.state0_rows ? mpc_rollout_fp64_kernel<DT, true> : mpc_rollout_fp64_kernel<DT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) kern<<<grid, NT, smem, c->stream>>>(a);
    return e;
}

}  // namespace

int mpc_fp64_grid(long long K_local) { return (int)((K_local + SEQ - 1) / SEQ); }

size_t mpc_fp64_smem_bytes(int din_pad, int h_pad) {
    const size_t act_elems = (size_t)(h_pad > din_pad ? h_pad : din_pad) * R;
    return sizeof(double) * (2 * act_elems + 2 * KT * UT + SS_MAX_D * SEQ + SS_MAX_D * R);
}

int mpc_fp64_launch(ss_ctx* c, const Rollout64Args& a) {
    const size_t smem = mpc_fp64_smem_bytes(a.din_pad, a.h_pad);
    if (smem > 227 * 1024)
        SS_FAIL(c, SS_EUNSUPPORTED, "mpc: depth_fc_layers too large for the FP64 kernel's shared memory");
    const int grid = mpc_fp64_grid(a.K_local);
    cudaError_t e = a.d <= 4 ? launch_fp64<4>(c, a, grid, smem)
                  : a.d <= 8 ? launch_fp64<8>(c, a, grid, smem)
                             : launch_fp64<SS_MAX_D>(c, a, grid, smem);
    if (e == cudaSuccess) e = cudaGetLastError();
    c->launches++;
    SS_CUDA_CHECK(c, e);
    return SS_OK;
}

// FP32 [in][out] / [out] parameters -> the padded float64 copies (ss_dyn_commit)
int mpc_fp64_widen(ss_ctx* c, const float* W, const float* b, int in, int out, int out_pad, double* Wp, double* bp) {
    const int n = std::max(in * out, out);
    widen_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(W, b, in, out, out_pad, Wp, bp);
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}
