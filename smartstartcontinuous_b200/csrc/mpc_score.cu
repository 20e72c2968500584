// mpc_score.cu -- the scoring tail of the MPC planner.
//
//   mpc_fold_partials    the rollout kernels leave the projection terms a'.b' and b'.b' of every time step
//   mpc_reduce_sums      (numerical.py:89-93) as one float64 table column per (tile, row warp) / 32-sequence
//                        CTA: deterministic fold + reduction to the 2 (H + 1) sums of the batch
//   mpc_tail             ONE launch for the whole tail of a decision: projection-sum columns -> global
//                        coefficients, penalty pass, arg-max, and the winner's package (score, k, action
//                        sequence, predicted path; NND_MB_agent.py:516-518) written to device memory and
//                        to mapped pinned host memory with a completion flag -- the call ends without
//                        a device->host copy
#include "mpc_kernels.cuh"

namespace {

// sums[2t + w] = sum over the blocks' partials, one warp per output, fixed order (lanes stride over
// the blocks, then a shuffle tree): deterministic for a given K_local
__global__ void __launch_bounds__(256)
mpc_reduce_sums_kernel(const double* __restrict__ partial, int blocks, int T, double* __restrict__ sums) {
    pdl_trigger();
    pdl_wait();
    const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (o >= 2 * T) return;
    const int t = o >> 1, w = o & 1, lane = threadIdx.x & 31;
    double s = 0.0;
    for (int b = lane; b < blocks; b += 32) s += partial[(size_t)o * blocks + b];      // [t][2][blocks]
    for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    if (lane == 0) sums[o] = s;
}

// many partial columns (one per tile and row warp from the tcgen05 kernel) -> FOLD columns per
// output, fixed order: column segment f of output o is summed by one warp (lanes stride, shuffle tree)
constexpr int SUMS_FOLD = 16;
__global__ void __launch_bounds__(256)
mpc_fold_partials_kernel(const double* __restrict__ partial, int blocks, int n_out, double* __restrict__ folded) {
    pdl_trigger();
    pdl_wait();
    const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wid >= n_out * SUMS_FOLD) return;
    const int o = wid / SUMS_FOLD, f = wid % SUMS_FOLD, lane = threadIdx.x & 31;
    const int seg = (blocks + SUMS_FOLD - 1) / SUMS_FOLD;
    const int b0 = f * seg, b1 = min(blocks, b0 + seg);
    double s = 0.0;
    for (int b = b0 + lane; b < b1; b += 32) s += partial[(size_t)o * blocks + b];
    for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    if (lane == 0) folded[(size_t)o * SUMS_FOLD + f] = s;
}

// ---- the fused tail -------------------------------------------------------------------------
// grid = ceil(K / 256) blocks of 256 threads, one sequence per thread.
//   sum_cols != null (reference penalty): the final per-step sums of a'.b' / b'.b' [2T]; every block
//     takes lambda_t = sum a'.b' / sum b'.b' and subtracts the penalties of its sequences from the
//     progress term (a per-block reduction of the partial columns was measured: 4-13 us of dependent
//     loads in front of every block, more than the extra 3 us launch of mpc_reduce_sums);
//   then the np.argmax-ordered block arg-max, and in the last block to finish (atomic ticket) the final
//   arg-max and the winner's package.
struct TailOut {
    double* pkg;                    // device package [2 + H*da + T*d]
    double* host_pkg;               // mapped pinned host copy as tagged slots (common.cuh host_slot_put), or null
    unsigned long long seq;         // the call's sequence number (-> tag of the slots)
    double* sums_out;               // [2T] reduced sums (block 0 writes them), or null
    float* scores_final;            // where the final scores go (== scores in place)
};

// the winner's package: [score, k (global), sequence (H*da), path (T*d)]; rows of d + 1 values (state, waypoint index)
template <typename Row>
__device__ __forceinline__ void write_package(double best_v, long long kl, long long k_offset, const Row* rows,
                                              long long K, int T, int d, const ActionSource* actp, int want_path,
                                              TailOut out) {
    const ActionSource& act = *actp;
    const int tid = threadIdx.x;
    const long long kg = kl < 0 ? -1 : kl + k_offset;
    const int n_seq = act.H * act.da, n_path = T * d;
    unsigned long long* hp = reinterpret_cast<unsigned long long*>(out.host_pkg);
    const unsigned int tag = (unsigned int)out.seq | 0x80000000u;          // host_slot_tag
    for (int o = tid; o < 2 + n_seq + n_path; o += blockDim.x) {
        double val = 0.0;
        if (o == 0) val = best_v;
        else if (o == 1) val = (double)kg;
        else if (want_path && kl >= 0) {
            const int q = o - 2;
            if (q < n_seq) val = fetch_action_f64(act, kl, kg, q / act.da, q % act.da);
            else {
                const int r = q - n_seq;
                val = (double)__ldcg(rows + ((size_t)(r / d) * K + kl) * (d + 1) + (r % d));
            }
        }
        out.pkg[o] = val;
        if (hp) host_slot_put(hp, o, val, tag);      // self-validating: no fence, barrier or flag behind it
    }
}

// kept out of line so that its Philox / float64 code does not inflate the register count of the
// bandwidth-bound penalty loop
__device__ __noinline__ void tail_write_package(double best_v, long long kl, long long k_offset, const float* rows,
                                                long long K, int T, int d, const ActionSource* actp, int want_path,
                                                TailOut out) {
    write_package<float>(best_v, kl, k_offset, rows, K, T, d, actp, want_path, out);
}
__device__ __noinline__ void tail_write_package(double best_v, long long kl, long long k_offset, const double* rows,
                                                long long K, int T, int d, const ActionSource* actp, int want_path,
                                                TailOut out) {
    write_package<double>(best_v, kl, k_offset, rows, K, T, d, actp, want_path, out);
}

template <int DT>
// (128-thread blocks, seven per SM for d <= 4: 896 x 148 = 132 608 resident threads hold the whole bench batch of
// 131 072 sequences in ONE wave; with 256-thread blocks at three per SM 15 % of the blocks ran in a second wave and
// doubled the kernel's time)
__global__ void __launch_bounds__(128, DT <= 4 ? 7 : 4)
mpc_tail_kernel(const PlanView Pg, const float* __restrict__ rows, long long K, int T, int ds_in_smem,
                const double* __restrict__ sum_cols, int n_cols, float* __restrict__ scores, long long k_offset,
                double* __restrict__ block_v, long long* __restrict__ block_i, MpcResult* __restrict__ result,
                ActionSource act, int want_path, TailOut out) {
    extern __shared__ float s_dyn[];             // [T] lambda | [W * d] waypoints (optional)
    pdl_wait();                                  // (launched as a programmatic dependent of the kernel in front)
    __shared__ double s_v[32];
    __shared__ long long s_i[32];
    __shared__ bool s_last;
    float* s_lam = s_dyn;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    PlanView P = Pg;
    const long long k = blockIdx.x * (long long)blockDim.x + tid;
    if (sum_cols) {
        // sum_cols = the final per-step sums [2T] (n_cols == 1; reduced -- and, on a sharded batch,
        // all-reduced -- by the kernel in front of this one)
        for (int t = tid; t < T; t += blockDim.x) s_lam[t] = (float)(sum_cols[2 * t] / sum_cols[2 * t + 1]);
        if (ds_in_smem) {
            float* s_ds = s_dyn + T;
            for (int i = tid; i < Pg.W * Pg.d; i += blockDim.x) s_ds[i] = Pg.ds[i];
            P.ds = s_ds;
        }
        __syncthreads();
    }
    double v = 0.0;
    long long bi = -1;
    if (k < K) {
        float score = scores[k];
        if (sum_cols) {
            // the H + 1 trajectory rows of a sequence are independent loads: issue them eight at a time
            // (a plain loop serialises one L2 / DRAM round trip per step, which is all a small batch does)
            constexpr int TB = 8;
            for (int t0 = 0; t0 < T; t0 += TB) {
                float xs[TB][DT];
                int idxs[TB];
#pragma unroll
                for (int i = 0; i < TB; ++i) {
                    const int t = t0 + i < T ? t0 + i : T - 1;
                    traj_load<DT>(rows, (size_t)t * K + k, P.d, xs[i], idxs[i]);
                }
#pragma unroll
                for (int i = 0; i < TB; ++i)
                    if (t0 + i < T) score -= penalty_with_lambda<DT>(P, idxs[i], xs[i], s_lam[t0 + i]);
            }
            scores[k] = score;
        }
        v = (double)score;
        bi = k;
    }
    block_argmax(v, bi, s_v, s_i);
    if (tid == 0) {
        block_v[blockIdx.x] = v;
        block_i[blockIdx.x] = bi;
        __threadfence();
        s_last = atomicAdd(&result->blocks_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    v = 0.0;
    bi = -1;
    for (int b = tid; b < gridDim.x; b += blockDim.x) {
        const double ov = __ldcg(block_v + b);
        const long long oi = __ldcg(block_i + b);
        if (argmax_better(ov, oi, v, bi)) { v = ov; bi = oi; }
    }
    block_argmax(v, bi, s_v, s_i);
    if (tid == 0) {
        s_v[0] = v;
        s_i[0] = bi;
        result->best_score = v;
        result->best_k = bi < 0 ? -1 : bi + k_offset;
        result->blocks_done = 0;
    }
    __syncthreads();
    tail_write_package(s_v[0], s_i[0], k_offset, rows, K, T, Pg.d, &act, want_path, out);
}

// float64 tail (SS_PRECISION_FP64), one sequence per thread.  Reference penalty (sums != null): the score is
// recomputed from the rows in the reference's order -- per step the progress term, then the penalty with the
// step's global coefficient lambda_t = sum a'.b' / sum b'.b' (float64) -- so it is the reference's sum, not the
// progress sum minus the penalty sum.  Per-sample penalty: the rollout kernel's scores are final.
template <int DT>
__global__ void __launch_bounds__(128)
mpc_tail64_kernel(const Plan64 P, int wp_index, const double* __restrict__ rows, long long K, int T,
                  const double* __restrict__ sums, double* __restrict__ scores, long long k_offset,
                  double* __restrict__ block_v, long long* __restrict__ block_i, MpcResult* __restrict__ result,
                  ActionSource act, int want_path, TailOut out) {
    extern __shared__ double s_lam64[];          // [T]
    pdl_wait();
    __shared__ double s_v[32];
    __shared__ long long s_i[32];
    __shared__ bool s_last;
    const int tid = threadIdx.x;
    const long long k = blockIdx.x * (long long)blockDim.x + tid;
    if (sums) {
        for (int t = tid; t < T; t += blockDim.x) s_lam64[t] = sums[2 * t] / sums[2 * t + 1];
        __syncthreads();
    }
    double v = 0.0;
    long long bi = -1;
    if (k < K) {
        double score;
        if (sums) {
            const int d = P.d;
            double x[DT];
            ScoreAcc64 sc;
            for (int t = 0; t < T; ++t) {
                const double* row = rows + ((size_t)t * K + k) * (d + 1);
#pragma unroll
                for (int j = 0; j < DT; ++j) x[j] = j < d ? __ldg(row + j) : 0.0;
                const int idx = (int)__ldg(row + d);
                if (t == 0) score_init64<DT>(P, wp_index, x, sc);
                // to_end = distances_left[idx] + dist(desired_states[idx], x) with idx after the move (dc after
                // :605 is dn exactly when the sample moved)
                const double to_end = P.dl[idx] + ell_dist64<DT>(P, P.ds + (size_t)idx * d, x);
                sc.score = sc.score + __dmul_rn(sc.prev - to_end, P.gpow[t]);
                sc.prev = to_end;
                sc.score = sc.score - penalty64<DT>(P, idx, x, s_lam64[t]);
            }
            score = sc.score;
            scores[k] = score;
        } else {
            score = scores[k];
        }
        v = score;
        bi = k;
    }
    // (the arg-max / package part of mpc_tail_kernel; kept as a copy so that the FP32 tail's code stays as it was)
    block_argmax(v, bi, s_v, s_i);
    if (tid == 0) {
        block_v[blockIdx.x] = v;
        block_i[blockIdx.x] = bi;
        __threadfence();
        s_last = atomicAdd(&result->blocks_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    v = 0.0;
    bi = -1;
    for (int b = tid; b < gridDim.x; b += blockDim.x) {
        const double ov = __ldcg(block_v + b);
        const long long oi = __ldcg(block_i + b);
        if (argmax_better(ov, oi, v, bi)) { v = ov; bi = oi; }
    }
    block_argmax(v, bi, s_v, s_i);
    if (tid == 0) {
        s_v[0] = v;
        s_i[0] = bi;
        result->best_score = v;
        result->best_k = bi < 0 ? -1 : bi + k_offset;
        result->blocks_done = 0;
    }
    __syncthreads();
    tail_write_package(s_v[0], s_i[0], k_offset, rows, K, T, P.d, &act, want_path, out);
}

}  // namespace

int mpc_reduce_sums(ss_ctx* c, const double* partial, int blocks, int T, double* sums) {
    SS_CUDA_CHECK(c, launch_dependent(mpc_reduce_sums_kernel, dim3((2 * T + 7) / 8), dim3(256), 0, c->stream, partial, blocks, T, sums));
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}

// folds [2T][blocks] partial columns in place-compatible layout into [2T][SUMS_FOLD] at `folded`
// (blocks > SUMS_FOLD); returns the new column count through *blocks_out
int mpc_fold_partials(ss_ctx* c, const double* partial, int blocks, int T, double* folded, int* blocks_out) {
    const int warps = 2 * T * SUMS_FOLD;
    SS_CUDA_CHECK(c, launch_dependent(mpc_fold_partials_kernel, dim3((warps + 7) / 8), dim3(256), 0, c->stream, partial, blocks, 2 * T, folded));
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    *blocks_out = SUMS_FOLD;
    return SS_OK;
}

// small batches: 64-thread blocks, four times as many of them (the pass is latency-bound there)
static int mpc_tail_threads(long long K_local) { return K_local <= 16384 ? 64 : 128; }
int mpc_tail_blocks(long long K_local) {
    const int t = mpc_tail_threads(K_local);
    return (int)((K_local + t - 1) / t);
}

// sum_cols may be null (per-sample penalty: the scores are final already); out_pkg / host_pkg as TailOut
int mpc_tail(ss_ctx* c, const PlanView& plan, const float* rows, long long K_local, int T, const double* sum_cols,
             int n_cols, float* scores, long long k_offset, double* block_v, long long* block_i, void* result_dev,
             const ActionSource& act, int want_path, double* pkg, double* host_pkg, unsigned long long seq,
             double* sums_out) {
    const unsigned grid = (unsigned)mpc_tail_blocks(K_local);
    const unsigned threads = (unsigned)mpc_tail_threads(K_local);
    const size_t ds_bytes = (size_t)plan.W * plan.d * 4;
    const int in_smem = sum_cols && ds_bytes + (size_t)T * 4 <= 40 * 1024;
    const size_t smem = (size_t)T * sizeof(float) + (in_smem ? ds_bytes : 0);
    TailOut out;
    out.pkg = pkg; out.host_pkg = host_pkg; out.seq = seq; out.sums_out = sums_out; out.scores_final = scores;
    MpcResult* res = reinterpret_cast<MpcResult*>(result_dev);
    // after a peer-memory exchange kernel (sharded batch) the tail is an ordinary launch: those kernels do not
    // release their dependents early; after the reduce kernel of an unsharded batch it is a programmatic one
    cudaError_t e;
    const dim3 g(grid), b(threads);
#define TAIL_LAUNCH(DT_)                                                                                            \
    e = launch_dependent(mpc_tail_kernel<DT_>, g, b, smem, c->stream, plan, rows, K_local, T, in_smem, sum_cols, n_cols, \
                         scores, k_offset, block_v, block_i, res, act, want_path, out)
    if (plan.d <= 4) TAIL_LAUNCH(4);
    else if (plan.d <= 8) TAIL_LAUNCH(8);
    else TAIL_LAUNCH(SS_MAX_D);
#undef TAIL_LAUNCH
    SS_CUDA_CHECK(c, e);
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}

int mpc_tail64(ss_ctx* c, const Plan64& plan, int wp_index, const double* rows, long long K_local, int T,
               const double* sums, double* scores, long long k_offset, double* block_v, long long* block_i,
               void* result_dev, const ActionSource& act, int want_path, double* pkg, double* host_pkg,
               unsigned long long seq) {
    const dim3 g((unsigned)mpc_tail_blocks(K_local)), b((unsigned)mpc_tail_threads(K_local));
    const size_t smem = (size_t)T * sizeof(double);
    TailOut out;
    out.pkg = pkg; out.host_pkg = host_pkg; out.seq = seq; out.sums_out = nullptr; out.scores_final = nullptr;
    MpcResult* res = reinterpret_cast<MpcResult*>(result_dev);
    cudaError_t e;
#define TAIL64_LAUNCH(DT_)                                                                                         \
    e = launch_dependent(mpc_tail64_kernel<DT_>, g, b, smem, c->stream, plan, wp_index, rows, K_local, T, sums,   \
                         scores, k_offset, block_v, block_i, res, act, want_path, out)
    if (plan.d <= 4) TAIL64_LAUNCH(4);
    else if (plan.d <= 8) TAIL64_LAUNCH(8);
    else TAIL64_LAUNCH(SS_MAX_D);
#undef TAIL64_LAUNCH
    SS_CUDA_CHECK(c, e);
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    return SS_OK;
}
