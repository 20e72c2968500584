// mpc_simt.cu -- FP32 (FFMA) rollout of the dynamics MLP for random-shooting MPC.
//
// Replaces Dyn_Model.do_forward_sim (dynamics_model.py:204-240; one sess.run per horizon
// step, float64 TF GEMMs) fused with the trajectory scoring of
// NND_MB_agent.generate_scores_add_delta (NND_MB_agent.py:566-628).  This is the
// SS_PRECISION_FP32 path: every layer in FP32 on the CUDA cores, any (d, da, L, h) within
// SS_MAX_*.  The tcgen05 kernel (mpc_tc.cu) is the fast path for the hidden x hidden layers.
//
// One CTA = 32 sequences ("rows") for all H steps; activations never leave shared memory:
//   act[k][row] (unit-major) ping/pong buffers, weights streamed from L2 through a
//   double-buffered cp.async stage, 4 rows x 8 units register tile per thread.
#include "mpc_kernels.cuh"
#include "tc_score_row.cuh"

namespace {

constexpr int SR = 32;     // sequences per CTA
constexpr int ST = 256;    // threads per CTA
constexpr int KT = 16;     // k-tile of a weight stage
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

// out[u][r] = act(bias[u] + sum_k in[k][r] * Wg[k][u])   in: [K_pad][SR], out: [N_pad][SR]
__device__ void dense_layer(const float* __restrict__ in, int K_pad, const float* __restrict__ Wg,
                            const float* __restrict__ bias, int N_pad, float* __restrict__ out,
                            bool relu, float* __restrict__ Ws) {
    const int tid = threadIdx.x;
    const int rg = tid & 7;       // rows 4*rg .. 4*rg+3
    const int ug = tid >> 3;      // units ug*8 .. ug*8+7 of the pass
    const int ntile = K_pad / KT;
    for (int u_pass = 0; u_pass < N_pad; u_pass += UT) {
        const int cols = N_pad - u_pass < UT ? N_pad - u_pass : UT;   // multiple of 8
        const int vec_per_row = cols >> 2;
        const int nvec = KT * vec_per_row;
        float acc[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

        auto stage_load = [&](int kt, int stage) {
            float* dst = Ws + stage * (KT * UT);
            const float* src = Wg + (size_t)kt * KT * N_pad + u_pass;
            for (int v = tid; v < nvec; v += ST) {
                int kk = v / vec_per_row, c4 = v - kk * vec_per_row;
                cp_async16(dst + kk * UT + 4 * c4, src + (size_t)kk * N_pad + 4 * c4);
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
                const float* wt = Ws + (kt & 1) * (KT * UT) + ug * 8;
                const float* it = in + (size_t)kt * KT * SR + 4 * rg;
#pragma unroll
                for (int kk = 0; kk < KT; ++kk) {
                    const float4 a = *reinterpret_cast<const float4*>(it + kk * SR);
                    const float4 w0 = *reinterpret_cast<const float4*>(wt + kk * UT);
                    const float4 w1 = *reinterpret_cast<const float4*>(wt + kk * UT + 4);
                    const float av[4] = {a.x, a.y, a.z, a.w};
                    const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
                }
            }
            __syncthreads();
        }
        if (ug * 8 < cols) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int u = u_pass + ug * 8 + j;
                const float bj = bias[u];
                float4 o;
                o.x = acc[0][j] + bj; o.y = acc[1][j] + bj; o.z = acc[2][j] + bj; o.w = acc[3][j] + bj;
                if (relu) {
                    o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f);
                    o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                }
                *reinterpret_cast<float4*>(out + (size_t)u * SR + 4 * rg) = o;
            }
        }
    }
    __syncthreads();
}

// z[j][r] = b[j] + sum_k in[k][r] * Wg[k][j],  j < d  (N_pad columns in Wg); K split over 8 warps
__device__ void output_layer(const float* __restrict__ in, int K_pad, const float* __restrict__ Wg,
                             const float* __restrict__ bias, int N_pad, int d, float* __restrict__ z,
                             float* __restrict__ red /* [8][SS_MAX_D][SR] */) {
    const int r = threadIdx.x & 31, ks = threadIdx.x >> 5;
    const int per = (K_pad + 7) / 8;
    const int k0 = ks * per, k1 = k0 + per < K_pad ? k0 + per : K_pad;
    for (int j0 = 0; j0 < d; j0 += 8) {
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        for (int k = k0; k < k1; ++k) {
            const float a = in[(size_t)k * SR + r];
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(Wg + (size_t)k * N_pad + j0));
            const float4 w1 = __ldg(reinterpret_cast<const float4*>(Wg + (size_t)k * N_pad + j0 + 4));
            acc[0] = fmaf(a, w0.x, acc[0]); acc[1] = fmaf(a, w0.y, acc[1]);
            acc[2] = fmaf(a, w0.z, acc[2]); acc[3] = fmaf(a, w0.w, acc[3]);
            acc[4] = fmaf(a, w1.x, acc[4]); acc[5] = fmaf(a, w1.y, acc[5]);
            acc[6] = fmaf(a, w1.z, acc[6]); acc[7] = fmaf(a, w1.w, acc[7]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (j0 + j < d) red[((size_t)ks * SS_MAX_D + j0 + j) * SR + r] = acc[j];
    }
    __syncthreads();
    for (int o = threadIdx.x; o < d * SR; o += ST) {
        const int j = o / SR, rr = o - j * SR;
        float s = bias[j];
#pragma unroll
        for (int q = 0; q < 8; ++q) s += red[((size_t)q * SS_MAX_D + j) * SR + rr];
        z[(size_t)j * SR + rr] = s;
    }
    __syncthreads();
}

// ROWS: per-sequence start rows (load_start).  <4, ROWS> gets a minimum of one CTA per SM: left to its occupancy
// heuristic, ptxas fits it into 80 registers and spills the scoring state inside the step loop.
template <int DT, bool ROWS>
__global__ void __launch_bounds__(ST, ROWS && DT == 4 ? 1 : 0) mpc_rollout_simt_kernel(const RolloutArgs a) {
    pdl_trigger();      // the reduce / tail kernels behind this launch may be scheduled (they wait for its completion)
    extern __shared__ __align__(16) float sm[];
    const int act_elems = (a.h_pad > a.din_pad ? a.h_pad : a.din_pad) * SR;
    float* actA = sm;
    float* actB = actA + act_elems;
    float* Ws = actB + act_elems;                 // 2 * KT * UT
    float* st = Ws + 2 * KT * UT;                 // state [SS_MAX_D][SR]
    float* z = st + SS_MAX_D * SR;                // [SS_MAX_D][SR]
    float* red = z + SS_MAX_D * SR;               // [8][SS_MAX_D][SR]

    const int tid = threadIdx.x;
    const long long k_local = (long long)blockIdx.x * SR + tid;   // row owners: tid < SR
    const bool owner = tid < SR;
    const bool live = owner && k_local < a.K_local;
    const int T = a.H + 1;

    ScoreAcc sc;
    float x[DT];
    if (owner) {
        load_start<ROWS, DT>(a, live, k_local, x);
        if constexpr (ROWS) {
#pragma unroll
            for (int j = 0; j < DT; ++j)
                if (j < a.d) st[j * SR + tid] = x[j];
        } else {
            for (int j = 0; j < a.d; ++j) st[j * SR + tid] = a.state0[j];
        }
        score_init<DT>(a.plan, a.wp_index, x, sc);
    }
    // zero the padded input rows once (rows d+da .. din_pad)
    for (int o = tid; o < a.din_pad * SR; o += ST) actA[o] = 0.f;
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        // ---- score the current point (row owners) -------------------------------------
        // (reference penalty: the step's projection terms summed over the CTA's 32 sequences, one column
        // of a.qsums per CTA -- the same scheme as the tcgen05 kernels, no pass over the spilled rows)
        if (owner) tc::score_row<DT>(a, t, x, sc, live, k_local, (long long)blockIdx.x, (long long)gridDim.x, tid);
        if (t == a.H) break;
        // ---- network input: normalised state and action (dynamics_model.py:228-230) ------
        if (owner) {
            for (int j = 0; j < a.d; ++j)
                actA[j * SR + tid] = (st[j * SR + tid] - a.norm.mean_x[j]) * a.norm.inv_std_x[j];
            for (int j = 0; j < a.da; ++j) {
                float act = live ? fetch_action(a.act, k_local, a.k_offset + k_local, t, j) : 0.f;
                actA[(a.d + j) * SR + tid] = (act - a.norm.mean_y[j]) * a.norm.inv_std_y[j];
            }
        }
        __syncthreads();
        // ---- MLP: L hidden layers (Linear + ReLU) and a linear output layer ---------------
        float* cur = actA;
        float* nxt = actB;
        int K_pad = a.din_pad;
        for (int l = 0; l < a.L; ++l) {
            dense_layer(cur, K_pad, a.w[l], a.b[l], a.h_pad, nxt, true, Ws);
            float* tmp = cur; cur = nxt; nxt = tmp;
            K_pad = a.h_pad;
        }
        output_layer(cur, K_pad, a.w[a.L], a.b[a.L], a.dout_pad, a.d, z, red);
        // ---- state update (dynamics_model.py:234-237) -------------------------------------
        if (owner) {
#pragma unroll
            for (int j = 0; j < DT; ++j)
                if (j < a.d) {
                    float s = st[j * SR + tid] + fmaf(z[j * SR + tid], a.norm.std_z[j], a.norm.mean_z[j]);
                    st[j * SR + tid] = s;
                    x[j] = s;
                }
        }
        // hidden layers 1, 3, .. write into actA: its padded input rows must be zero again
        if (a.L >= 2) {
            __syncthreads();
            for (int o = tid + (a.d + a.da) * SR; o < a.din_pad * SR; o += ST) actA[o] = 0.f;
        }
        __syncthreads();
    }
    if (live && a.scores_out) a.scores_out[k_local] = sc.score;
}

// ---- small single-hidden-layer networks (the reference's default NND_MB model: 1 x 32) -----------------
// The CTA kernel above gives 32 sequences to 256 threads and runs the MLP as tiled GEMMs between block barriers;
// for a 160-MAC network that is all barrier and the owner warp's serial chain (score -> sample -> normalise ->
// update): ncu on config 1 (K = 5000, H = 4) shows 8 warps stalled on the barrier per issued instruction and 22 us
// for 20 000 rollout steps.  Here a THREAD rolls its own sequence: weights in shared memory (broadcast reads), one
// layer of activations in registers, no barrier after the staging; a warp is still one column of the
// projection-sum table (32 consecutive sequences), so the tail and the multi-GPU exchange see the same layout.
constexpr int TT = 128;                    // threads = sequences per CTA (4 warps = 4 table columns)

template <int DT, int HP, bool ROWS>       // d <= DT, h_pad <= HP; ROWS: per-sequence start rows (load_start)
__global__ void __launch_bounds__(TT) mpc_rollout_thread_kernel(const RolloutArgs a) {
    pdl_trigger();
    extern __shared__ __align__(16) float sm[];
    float* W0 = sm;                                // [din_pad][h_pad]
    float* W1 = W0 + a.din_pad * a.h_pad;          // [h_pad][dout_pad]
    float* B0 = W1 + a.h_pad * a.dout_pad;         // [h_pad]
    float* B1 = B0 + a.h_pad;                      // [dout_pad]
    const int tid = threadIdx.x;
    for (int v = tid; v < a.din_pad * a.h_pad / 4; v += TT)
        reinterpret_cast<float4*>(W0)[v] = __ldg(reinterpret_cast<const float4*>(a.w[0]) + v);
    for (int v = tid; v < a.h_pad * a.dout_pad / 4; v += TT)
        reinterpret_cast<float4*>(W1)[v] = __ldg(reinterpret_cast<const float4*>(a.w[1]) + v);
    for (int v = tid; v < a.h_pad; v += TT) B0[v] = __ldg(a.b[0] + v);
    for (int v = tid; v < a.dout_pad; v += TT) B1[v] = v < a.d ? __ldg(a.b[1] + v) : 0.f;
    __syncthreads();

    const int lane = tid & 31;
    const long long n_qcols = (a.K_local + 31) / 32;
    const long long qcol = (long long)blockIdx.x * (TT / 32) + (tid >> 5);
    if (qcol >= n_qcols) return;                   // (no barrier below)
    const long long k_local = (long long)blockIdx.x * TT + tid;
    const bool live = k_local < a.K_local;
    const int T = a.H + 1;
    const int nq = a.h_pad >> 2;                   // float4 pieces of a hidden row

    ScoreAcc sc;
    float x[DT];
    load_start<ROWS, DT>(a, live, k_local, x);
    score_init<DT>(a.plan, a.wp_index, x, sc);

    for (int t = 0; t < T; ++t) {
        tc::score_row<DT>(a, t, x, sc, live, k_local, qcol, n_qcols, lane);
        if (t == a.H) break;
        // ---- hidden layer: h[u] = relu(b0[u] + sum_k in[k] W0[k][u]), inputs = normalised state, then action
        float h[HP];
#pragma unroll
        for (int q = 0; q < HP / 4; ++q) {
            float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
            if (q < nq) b = reinterpret_cast<const float4*>(B0)[q];
            h[4 * q] = b.x; h[4 * q + 1] = b.y; h[4 * q + 2] = b.z; h[4 * q + 3] = b.w;
        }
#pragma unroll
        for (int k = 0; k < DT + SS_MAX_DA; ++k) {
            if (k < a.d + a.da) {
                float in;
                if (k < a.d) in = (x[k < DT ? k : 0] - a.norm.mean_x[k]) * a.norm.inv_std_x[k];
                else {
                    const int j = k - a.d;
                    const float act = live ? fetch_action(a.act, k_local, a.k_offset + k_local, t, j) : 0.f;
                    in = (act - a.norm.mean_y[j]) * a.norm.inv_std_y[j];
                }
                const float4* wr = reinterpret_cast<const float4*>(W0 + k * a.h_pad);
#pragma unroll
                for (int q = 0; q < HP / 4; ++q) {
                    if (q < nq) {
                        const float4 w = wr[q];
                        h[4 * q] = fmaf(in, w.x, h[4 * q]); h[4 * q + 1] = fmaf(in, w.y, h[4 * q + 1]);
                        h[4 * q + 2] = fmaf(in, w.z, h[4 * q + 2]); h[4 * q + 3] = fmaf(in, w.w, h[4 * q + 3]);
                    }
                }
            }
        }
        // ---- output layer: z[j] = b1[j] + sum_u relu(h[u]) W1[u][j]
        float z[DT];
#pragma unroll
        for (int j = 0; j < DT; ++j) z[j] = B1[j < 8 ? j : 0];
#pragma unroll
        for (int u = 0; u < HP; ++u) {
            if (u < a.h_pad) {
                const float hu = fmaxf(h[u], 0.f);
                const float4* wr = reinterpret_cast<const float4*>(W1 + u * a.dout_pad);
                const float4 w0 = wr[0];
                z[0] = fmaf(hu, w0.x, z[0]);
                if (DT > 1) z[1] = fmaf(hu, w0.y, z[1]);
                if (DT > 2) z[2] = fmaf(hu, w0.z, z[2]);
                if (DT > 3) z[3] = fmaf(hu, w0.w, z[3]);
                if (DT > 4) {
                    const float4 w1 = wr[1];
                    z[4 % DT] = fmaf(hu, w1.x, z[4 % DT]);
                    z[5 % DT] = fmaf(hu, w1.y, z[5 % DT]);
                    z[6 % DT] = fmaf(hu, w1.z, z[6 % DT]);
                    z[7 % DT] = fmaf(hu, w1.w, z[7 % DT]);
                }
            }
        }
        // ---- state update (dynamics_model.py:234-237)
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < a.d) x[j] = x[j] + fmaf(z[j], a.norm.std_z[j], a.norm.mean_z[j]);
    }
    if (live && a.scores_out) a.scores_out[k_local] = sc.score;
}

bool simt_thread_variant(const RolloutArgs& a) {
    return a.L == 1 && a.h_pad <= 64 && a.d <= 8 && a.dout_pad == 8 && !getenv("SS_SIMT_GENERAL");
}

size_t simt_smem_bytes(const RolloutArgs& a) {
    const int act_elems = (a.h_pad > a.din_pad ? a.h_pad : a.din_pad) * SR;
    return sizeof(float) * ((size_t)2 * act_elems + 2 * KT * UT + 2 * SS_MAX_D * SR + 8 * SS_MAX_D * SR);
}

}  // namespace

int mpc_simt_grid(const RolloutArgs& a) { return (int)((a.K_local + SR - 1) / SR); }

bool mpc_simt_is_thread_kernel(const RolloutArgs& a) { return simt_thread_variant(a); }

template <int DT>
static cudaError_t launch_simt_kernel(ss_ctx* c, const RolloutArgs& a, int grid, size_t smem) {
    auto kern = a.state0_rows ? mpc_rollout_simt_kernel<DT, true> : mpc_rollout_simt_kernel<DT, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) kern<<<grid, ST, smem, c->stream>>>(a);
    return e;
}

template <int DT, int HP>
static cudaError_t launch_thread_kernel(ss_ctx* c, const RolloutArgs& a, int grid, size_t smem) {
    if (a.state0_rows) mpc_rollout_thread_kernel<DT, HP, true><<<grid, TT, smem, c->stream>>>(a);
    else mpc_rollout_thread_kernel<DT, HP, false><<<grid, TT, smem, c->stream>>>(a);
    return cudaGetLastError();
}

int mpc_simt_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out) {
    if (simt_thread_variant(a)) {
        const int grid = (int)((a.K_local + TT - 1) / TT);
        if (grid_blocks_out) *grid_blocks_out = grid;
        const size_t smem = sizeof(float) * ((size_t)a.din_pad * a.h_pad + (size_t)a.h_pad * a.dout_pad + a.h_pad + a.dout_pad);
        cudaError_t e;
        if (a.d <= 4) e = a.h_pad <= 32 ? launch_thread_kernel<4, 32>(c, a, grid, smem) : launch_thread_kernel<4, 64>(c, a, grid, smem);
        else e = a.h_pad <= 32 ? launch_thread_kernel<8, 32>(c, a, grid, smem) : launch_thread_kernel<8, 64>(c, a, grid, smem);
        c->launches++;
        SS_CUDA_CHECK(c, e);
        return SS_OK;
    }
    const size_t smem = simt_smem_bytes(a);
    if (smem > 227 * 1024)
        SS_FAIL(c, SS_EUNSUPPORTED, "mpc: depth_fc_layers too large for the FP32 kernel's shared memory");
    const int grid = mpc_simt_grid(a);
    if (grid_blocks_out) *grid_blocks_out = grid;
    cudaError_t e = a.d <= 4 ? launch_simt_kernel<4>(c, a, grid, smem)
                  : a.d <= 8 ? launch_simt_kernel<8>(c, a, grid, smem)
                             : launch_simt_kernel<SS_MAX_D>(c, a, grid, smem);
    if (e == cudaSuccess) e = cudaGetLastError();
    c->launches++;
    SS_CUDA_CHECK(c, e);
    return SS_OK;
}
