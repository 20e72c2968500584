// mpc_kernels.cuh -- declarations shared between the MPC host code and the kernel files.
#pragma once

#include "common.cuh"
#include "score.cuh"

// everything a rollout kernel needs, passed by value
struct RolloutArgs {
    // model (fp32, zero padded): w[l] is [in_pad_l][out_pad_l] row-major
    const float* w[SS_MAX_LAYERS + 1];
    const float* b[SS_MAX_LAYERS + 1];
    int d, da, L, h;
    int din_pad, h_pad, dout_pad;
    MpcNorm norm;
    ActionSource act;
    PlanView plan;
    float state0[SS_MAX_D];
    int wp_index, H;
    long long K_local, k_offset;
    int per_sample;          // 1: full score in the rollout kernel (per-sample penalty);
                             // 0: reference mode -- the kernel accumulates the progress term and
                             //    spills (state, waypoint index) rows; the penalty passes
                             //    (mpc_score.cu) run over them afterwards
    float* states_out;       // [H+1][K_local][d + 1] trajectory rows (score.cuh) or null
    float* scores_out;       // [K_local] (per-sample mode: final; reference mode: progress term)
    double* qsums;           // tcgen05 kernel, reference mode: [H+1][2][4 * tiles] a'.b' and b'.b' summed over the
                             // 32 rows of every (tile, row warp), or null (per-sample penalty)
    const float* state0_rows;   // [K_local][d] per-sequence start states (forward simulation) or null: every
                                // sequence starts at state0 (set: the launchers pick the kernels' ROWS = true)
};

// float64 rollout (mpc_fp64.cu): every operand and every operation in float64, the reference's element-wise
// operation order (score.cuh, float64 twin)
struct Rollout64Args {
    const double* w[SS_MAX_LAYERS + 1];     // [in_pad_l][out_pad_l], zero padded like RolloutArgs
    const double* b[SS_MAX_LAYERS + 1];
    int d, da, L, h;
    int din_pad, h_pad, dout_pad;
    MpcNorm64 norm;
    ActionSource act;
    Plan64 plan;
    double state0[SS_MAX_D];
    int wp_index, H;
    long long K_local, k_offset;
    int per_sample;          // 1: final scores (per-sample penalty); 0: reference mode, the tail scores the rows
    double* rows_out;        // [H+1][K_local][d + 1] (state, waypoint index after the move)
    double* scores_out;      // [K_local] (per-sample mode) or null
    double* qsums;           // reference mode: [H+1][2][ceil(K_local / 32)] a'.b' and b'.b' per 32 sequences, or null
    const double* state0_rows;  // [K_local][d] per-sequence start states or null, as RolloutArgs::state0_rows
};

// Start state of sequence k_local, loaded once per sequence.  ROWS (a rollout kernel's template flag, set by the
// launchers when state0_rows is given): a live sequence loads its own row, indexed by its batch-local k_local
// (never a chunk-relative row), and a row that is not live (past K_local, a ragged last tile, a padding tile)
// keeps zeros without reading the buffer, which has exactly K_local rows.  Otherwise every sequence starts at
// state0.  Every thread that keeps a copy of a sequence's state calls this with the same (live, k_local).
template <bool ROWS, int DT, typename T, typename A>
__device__ __forceinline__ void load_start(const A& a, bool live, long long k_local, T (&x)[DT]) {
    if constexpr (ROWS) {
        const T* s = a.state0_rows + (size_t)k_local * a.d;
#pragma unroll
        for (int j = 0; j < DT; ++j) x[j] = live && j < a.d ? __ldg(s + j) : T(0);
    } else {
#pragma unroll
        for (int j = 0; j < DT; ++j) x[j] = j < a.d ? a.state0[j] : T(0);
    }
}

int mpc_fp64_launch(ss_ctx* c, const Rollout64Args& a);
int mpc_fp64_grid(long long K_local);      // = projection-sum columns
size_t mpc_fp64_smem_bytes(int din_pad, int h_pad);
int mpc_fp64_widen(ss_ctx* c, const float* W, const float* b, int in, int out, int out_pad, double* Wp, double* bp);
// float64 tail: penalties (reference mode: every score recomputed from the rows in the reference's order),
// arg-max and package, like mpc_tail
int mpc_tail64(ss_ctx* c, const Plan64& plan, int wp_index, const double* rows, long long K_local, int T,
               const double* sums, double* scores, long long k_offset, double* block_v, long long* block_i,
               void* result_dev, const ActionSource& act, int want_path, double* pkg, double* host_pkg,
               unsigned long long seq);

// fp32 SIMT rollout (mpc_simt.cu)
int mpc_simt_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out);
int mpc_simt_grid(const RolloutArgs& a);
bool mpc_simt_is_thread_kernel(const RolloutArgs& a);   // small single-hidden-layer nets: one thread per sequence

// tcgen05 rollout (mpc_tc.cu)
bool mpc_tc_shape_supported(const ss_ctx* c);
int mpc_tc_prepare(ss_ctx* c);      // builds the BF16 operand images after ss_mpc_set_model
// rolls the tiles [tile_begin, tile_begin + tile_count) of the local batch (tile = mpc_tc_tile_rows()
// consecutive sequences); tile_count < 0 = all of them
int mpc_tc_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out, long long tile_begin = 0,
                  long long tile_count = -1);
int mpc_tc_grid(const ss_ctx* c, long long tiles);
int mpc_tc_tile_rows();
// small batches (mpc_tc_quad.cu): one tile per 4-CTA cluster, the hidden layer split over the cluster
bool mpc_tc_quad_supported(const ss_ctx* c);
int mpc_tc_quad_clusters(ss_ctx* c);
int mpc_tc_quad_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out);

// scoring tail (mpc_score.cu)
int mpc_reduce_sums(ss_ctx* c, const double* partial, int blocks, int T, double* sums);
int mpc_fold_partials(ss_ctx* c, const double* partial, int blocks, int T, double* folded, int* blocks_out);
// the fused tail: [2T][n_cols] partial sum columns (or null) -> coefficients, penalties, arg-max, package
// (device copy at pkg; host_pkg = mapped pinned memory [flag, -, package...] or null; flag := seq when done)
int mpc_tail_blocks(long long K_local);
int mpc_tail(ss_ctx* c, const PlanView& plan, const float* rows, long long K_local, int T, const double* sum_cols,
             int n_cols, float* scores, long long k_offset, double* block_v, long long* block_i, void* result_dev,
             const ActionSource& act, int want_path, double* pkg, double* host_pkg, unsigned long long seq,
             double* sums_out);

// peer-memory exchange (peer.cu): fused reduce + all-reduce of the projection sums, and the
// all-gather + pick of the winner packages
int peer_allreduce_sums(ss_ctx* c, const double* partial, int blocks, int T, double* sums);
int peer_package_exchange(ss_ctx* c, const double* pkg_local, int n, double* pkg_out);

struct MpcResult {
    double best_score;
    long long best_k;
    unsigned int blocks_done;
    int pad;
};
