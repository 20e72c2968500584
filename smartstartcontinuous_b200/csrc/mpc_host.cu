// mpc_host.cu -- host side of the MPC planner: model / plan upload, phase orchestration.
//
//   ss_mpc_set_model  <- Dyn_Model weights + NND_MB_agent.py:302-315 statistics
//   ss_mpc_set_plan   <- NND_MB_agent.start_new_episode_plan (NND_MB_agent.py:375-418)
//   ss_mpc_rollout    phase A: sample/fetch actions, roll the MLP for H steps, score
//   ss_mpc_finish     phase B (reference penalty) + arg-max
//   ss_mpc_replay     re-roll the winner for best_sequence / best_path (NND_MB_agent.py:516-518)
// SS_PRECISION_FP64 keeps its own float64 copies of the model and the plan and its own rows / scores buffers
// (mpc_fp64.cu, the float64 tail of mpc_score.cu); the projection sums and the package are shared.
#include <atomic>
#include <cstdlib>
#include <cstring>

#include "mpc_kernels.cuh"

namespace {

int round_up(int v, int m) { return (v + m - 1) / m * m; }

__global__ void sample_actions_kernel(ActionSource src, long long K, long long k_offset,
                                      double* __restrict__ out) {
    const long long n = K * src.H * src.da;
    for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n;
         o += (long long)gridDim.x * blockDim.x) {
        const long long k = o / (src.H * src.da);
        const int rem = (int)(o - k * (src.H * src.da));
        const int t = rem / src.da, j = rem - t * src.da;
        out[o] = fetch_action_f64(src, k, k_offset + k, t, j);
    }
}

// rows: [T][K][d + 1] (state, waypoint index) -> out [T][d]
__global__ void gather_path_kernel(const float* __restrict__ rows, long long K, long long k, int T,
                                   int d, float* __restrict__ out) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o < T * d) out[o] = rows[((size_t)(o / d) * K + k) * (d + 1) + (o % d)];
}

int fill_action_source(ss_ctx* c, ActionSource& s, int H, int da, uint64_t seed, const double* low,
                       const double* high) {
    s.host_actions = nullptr;
    s.seed = seed;
    s.da = da;
    s.H = H;
    for (int j = 0; j < SS_MAX_DA; ++j) { s.low[j] = 0.0; s.range[j] = 0.0; }
    if (low && high)
        for (int j = 0; j < da; ++j) { s.low[j] = low[j]; s.range[j] = high[j] - low[j]; }
    else if (!low != !high)
        SS_FAIL(c, SS_EINVAL, "mpc: act_low and act_high must both be given");
    // FP32 fast path of fetch_action_seq: both constants exact in FP32 and the float64 sum
    // low + u * range exact (u has 24 bits, range 24: the product needs 48; adding low must not
    // push the span past 53 bits)
    s.fp32_exact = 1;
    for (int j = 0; j < SS_MAX_DA; ++j) {
        s.low_f[j] = (float)s.low[j];
        s.range_f[j] = (float)s.range[j];
        if ((double)s.low_f[j] != s.low[j] || (double)s.range_f[j] != s.range[j]) s.fp32_exact = 0;
        if (s.low[j] != 0.0 && s.range[j] != 0.0) {
            int el = 0, er = 0;
            std::frexp(s.low[j], &el);
            std::frexp(s.range[j], &er);
            if (el - er > 4 || !std::isfinite(s.low[j]) || !std::isfinite(s.range[j])) s.fp32_exact = 0;
        }
    }
    return SS_OK;
}

PlanView make_plan_view(ss_ctx* c, const float* gpow, double gamma, double hpf) {
    PlanView p;
    p.ds = c->plan_ds.as<float>();
    p.dl = c->plan_dl.as<float>();
    p.gpow = gpow;
    p.W = c->W;
    p.d = c->d;
    for (int j = 0; j < SS_MAX_D; ++j) p.inv_r[j] = c->inv_radii[j];
    p.pen_scale = (float)(hpf * gamma);
    return p;
}

Plan64 make_plan64(ss_ctx* c, double gamma, double hpf) {
    Plan64 p;
    p.ds = c->plan_ds64.as<double>();
    p.dl = c->plan_dl64.as<double>();
    p.gpow = c->mpc_misc64.as<double>();
    p.W = c->W;
    p.d = c->d;
    for (int j = 0; j < SS_MAX_D; ++j) p.r[j] = c->radii64[j];
    p.hpf = hpf;
    p.gamma = gamma;
    return p;
}

// Forward simulation: a two-waypoint plan of the context's own (waypoints 0 and 1, unit radii, gamma^t = 1, no
// penalty) for the scoring code every rollout kernel runs.  Its scores are discarded; it only keeps the kernels
// away from the caller's plan, which may not exist.
constexpr int FSIM_GPOW = 2 * SS_MAX_D + 2;     // offset of gamma^t after [ds 2 x d | dl 2]

template <typename T>
int upload_fsim_plan(ss_ctx* c, DevBuf& buf, int T_steps) {
    std::vector<T> v(FSIM_GPOW + T_steps, T(1));
    for (int i = 0; i < 2 * SS_MAX_D; ++i) v[i] = i < c->d ? T(0) : T(1);     // ds rows 0 and 1 at stride d
    v[2 * SS_MAX_D] = T(1);
    v[2 * SS_MAX_D + 1] = T(0);
    SS_CUDA_CHECK(c, buf.ensure(v.size() * sizeof(T)));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(buf.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

PlanView fsim_plan_view(ss_ctx* c) {
    PlanView p;
    p.ds = c->fsim_plan.as<float>();
    p.dl = p.ds + 2 * SS_MAX_D;
    p.gpow = p.ds + FSIM_GPOW;
    p.W = 2;
    p.d = c->d;
    for (int j = 0; j < SS_MAX_D; ++j) p.inv_r[j] = j < c->d ? 1.f : 0.f;
    p.pen_scale = 0.f;
    return p;
}

Plan64 fsim_plan64(ss_ctx* c) {
    Plan64 p;
    p.ds = c->fsim_plan64.as<double>();
    p.dl = p.ds + 2 * SS_MAX_D;
    p.gpow = p.ds + FSIM_GPOW;
    p.W = 2;
    p.d = c->d;
    for (int j = 0; j < SS_MAX_D; ++j) p.r[j] = 1.0;
    p.hpf = 0.0;
    p.gamma = 0.0;
    return p;
}

// float64 rows of the fp64 replay (after the gamma^t table)
double* misc64_rows(ss_ctx* c) { return c->mpc_misc64.as<double>() + (c->run.H + 2) / 2 * 2; }

void fill_model64_args(ss_ctx* c, Rollout64Args& a) {
    for (int l = 0; l <= c->L; ++l) {
        a.w[l] = c->w64[l].as<double>();
        a.b[l] = c->b64[l].as<double>();
    }
    a.d = c->d; a.da = c->da; a.L = c->L; a.h = c->h;
    a.din_pad = c->din_pad; a.h_pad = c->h_pad; a.dout_pad = round_up(c->d, 8);
    a.norm = c->norm64;
}

void fill_model_args(ss_ctx* c, RolloutArgs& a) {
    for (int l = 0; l <= c->L; ++l) {
        a.w[l] = c->w32[l].as<float>();
        a.b[l] = c->b32[l].as<float>();
    }
    a.d = c->d; a.da = c->da; a.L = c->L; a.h = c->h;
    a.din_pad = c->din_pad; a.h_pad = c->h_pad; a.dout_pad = round_up(c->d, 8);
    a.norm = c->norm;
}

}  // namespace

extern "C" int ss_mpc_set_model(ss_ctx* c, int d, int da, int num_fc_layers, int depth,
                                const double* const* weights, const double* const* biases,
                                const double* mean_x, const double* std_x, const double* mean_y,
                                const double* std_y, const double* mean_z, const double* std_z) {
    if (!c) return SS_EINVAL;
    if (d < 1 || d > SS_MAX_D || da < 1 || da > SS_MAX_DA)
        SS_FAIL(c, SS_EUNSUPPORTED, "mpc: need 1 <= d <= 32 and 1 <= da <= 8");
    if (num_fc_layers < 1 || num_fc_layers > SS_MAX_LAYERS || depth < 1)
        SS_FAIL(c, SS_EUNSUPPORTED, "mpc: need 1 <= num_fc_layers <= 8 and depth_fc_layers >= 1");
    if (!weights || !biases || !mean_x || !std_x || !mean_y || !std_y || !mean_z || !std_z)
        SS_FAIL(c, SS_EINVAL, "mpc: null model pointer");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    if (d != c->d) c->plan_set = false;   // a plan refers to the state dimension
    // the trainer's master copy follows the host parameters again; the Adam moments outlive a weight
    // assignment of the same shape (like the optimizer slots of the reference's TF graph)
    if (d != c->d || da != c->da || num_fc_layers != c->L || depth != c->h) c->dyn_adam_valid = false;
    c->dyn_params_valid = false;
    c->dyn_dirty = false;
    c->host_params_stale = false;
    c->d = d; c->da = da; c->L = num_fc_layers; c->h = depth;
    c->din_pad = round_up(d + da, 16);
    c->h_pad = round_up(depth, 16);
    c->w32.resize(num_fc_layers + 1);
    c->b32.resize(num_fc_layers + 1);
    c->w64.resize(num_fc_layers + 1);
    c->b64.resize(num_fc_layers + 1);
    c->hw.assign(num_fc_layers + 1, {});
    c->hb.assign(num_fc_layers + 1, {});
    for (int l = 0; l <= num_fc_layers; ++l) {
        const int in = l == 0 ? d + da : depth, out = l == num_fc_layers ? d : depth;
        c->hw[l].assign(weights[l], weights[l] + (size_t)in * out);
        c->hb[l].assign(biases[l], biases[l] + out);
        const int in_pad = l == 0 ? c->din_pad : c->h_pad;
        const int out_pad = l == num_fc_layers ? round_up(d, 8) : c->h_pad;
        std::vector<float> w((size_t)in_pad * out_pad, 0.f), b(out_pad, 0.f);
        for (int i = 0; i < in; ++i)
            for (int o = 0; o < out; ++o) w[(size_t)i * out_pad + o] = (float)weights[l][(size_t)i * out + o];
        for (int o = 0; o < out; ++o) b[o] = (float)biases[l][o];
        SS_CUDA_CHECK(c, c->w32[l].ensure(w.size() * 4));
        SS_CUDA_CHECK(c, c->b32[l].ensure(b.size() * 4));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->w32[l].p, w.data(), w.size() * 4, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->b32[l].p, b.data(), b.size() * 4, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));   // w, b are stack-local staging
        // the caller's doubles as they are for SS_PRECISION_FP64
        std::vector<double> w64((size_t)in_pad * out_pad, 0.0), b64(out_pad, 0.0);
        for (int i = 0; i < in; ++i)
            for (int o = 0; o < out; ++o) w64[(size_t)i * out_pad + o] = weights[l][(size_t)i * out + o];
        for (int o = 0; o < out; ++o) b64[o] = biases[l][o];
        SS_CUDA_CHECK(c, c->w64[l].ensure(w64.size() * 8));
        SS_CUDA_CHECK(c, c->b64[l].ensure(b64.size() * 8));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->w64[l].p, w64.data(), w64.size() * 8, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->b64[l].p, b64.data(), b64.size() * 8, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    }
    // Q4 (SURVEY 8a): the reference evaluates nan_to_num((x - mean) / std); for std == 0 that is 0
    // when x == mean and +-1.8e308 otherwise.  A zero-variance feature carries no information, so
    // the kernels use 0 for it (documented deviation, DESIGN.md).
    std::memset(&c->norm, 0, sizeof(c->norm));
    for (int j = 0; j < d; ++j) {
        c->norm.mean_x[j] = (float)mean_x[j];
        c->norm.inv_std_x[j] = std_x[j] != 0.0 ? (float)(1.0 / std_x[j]) : 0.f;
        c->norm.mean_z[j] = (float)mean_z[j];
        c->norm.std_z[j] = (float)std_z[j];
    }
    for (int j = 0; j < da; ++j) {
        c->norm.mean_y[j] = (float)mean_y[j];
        c->norm.inv_std_y[j] = std_y[j] != 0.0 ? (float)(1.0 / std_y[j]) : 0.f;
    }
    std::memset(&c->norm64, 0, sizeof(c->norm64));
    for (int j = 0; j < d; ++j) {
        c->norm64.mean_x[j] = mean_x[j];
        c->norm64.std_x[j] = std_x[j];
        c->norm64.mean_z[j] = mean_z[j];
        c->norm64.std_z[j] = std_z[j];
    }
    for (int j = 0; j < da; ++j) {
        c->norm64.mean_y[j] = mean_y[j];
        c->norm64.std_y[j] = std_y[j];
    }
    c->model_set = true;
    c->run.valid = false;
    c->fsim_plan_T = 0;                   // the forward-simulation plan's layout follows d
    c->tc_ready = false;
    if (mpc_tc_shape_supported(c)) {
        int rc = mpc_tc_prepare(c);
        if (rc != SS_OK) return rc;
    }
    return SS_OK;
}

extern "C" int ss_mpc_tc_supported(ss_ctx* c) { return c && c->model_set && c->tc_ready ? 1 : 0; }
extern "C" int ss_mpc_last_kernel(ss_ctx* c) { return c && c->run.valid ? c->run.kernel : -1; }

extern "C" int ss_mpc_set_plan(ss_ctx* c, const double* desired_states, int W,
                               const double* distances_left, const double* radii, int d) {
    if (!c) return SS_EINVAL;
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "mpc: set the model before the plan");
    if (d != c->d) SS_FAIL(c, SS_EINVAL, "mpc: plan state dimension differs from the model's");
    if (W < 2) SS_FAIL(c, SS_EINVAL, "mpc: a plan needs at least two desired states");
    if (!desired_states || !distances_left || !radii) SS_FAIL(c, SS_EINVAL, "mpc: null plan pointer");
    for (int j = 0; j < d; ++j)
        if (!(radii[j] > 0.0)) SS_FAIL(c, SS_EINVAL, "mpc: radii must be > 0 (AssertionError in the reference)");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    std::vector<float> ds((size_t)W * d), dl(W);
    for (size_t i = 0; i < ds.size(); ++i) ds[i] = (float)desired_states[i];
    for (int i = 0; i < W; ++i) dl[i] = (float)distances_left[i];
    SS_CUDA_CHECK(c, c->plan_ds.ensure(ds.size() * 4));
    SS_CUDA_CHECK(c, c->plan_dl.ensure(dl.size() * 4));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->plan_ds.p, ds.data(), ds.size() * 4, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->plan_dl.p, dl.data(), dl.size() * 4, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    for (int j = 0; j < SS_MAX_D; ++j) c->inv_radii[j] = j < d ? (float)(1.0 / radii[j]) : 0.f;
    SS_CUDA_CHECK(c, c->plan_ds64.ensure((size_t)W * d * 8));
    SS_CUDA_CHECK(c, c->plan_dl64.ensure((size_t)W * 8));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->plan_ds64.p, desired_states, (size_t)W * d * 8, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->plan_dl64.p, distances_left, (size_t)W * 8, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    for (int j = 0; j < SS_MAX_D; ++j) c->radii64[j] = j < d ? radii[j] : 1.0;
    c->W = W;
    c->plan_set = true;
    c->run.valid = false;
    return SS_OK;
}

extern "C" int ss_mpc_sample_actions(ss_ctx* c, int64_t K_local, int64_t k_offset, int H, int da,
                                     uint64_t seed, const double* act_low, const double* act_high,
                                     double* out_actions) {
    if (!c) return SS_EINVAL;
    if (K_local < 1 || H < 1 || da < 1 || da > SS_MAX_DA || !act_low || !act_high || !out_actions)
        SS_FAIL(c, SS_EINVAL, "mpc: bad sample_actions arguments");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    ActionSource src;
    int rc = fill_action_source(c, src, H, da, seed, act_low, act_high);
    if (rc) return rc;
    const size_t n = (size_t)K_local * H * da;
    SS_CUDA_CHECK(c, c->mpc_sampled.ensure(n * 8));
    sample_actions_kernel<<<c->sm_count * 4, 256, 0, c->stream>>>(src, K_local, k_offset,
                                                                   c->mpc_sampled.as<double>());
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    SS_CUDA_CHECK(c, cudaMemcpyAsync(out_actions, c->mpc_sampled.p, n * 8, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

static int reduce_projection_sums(ss_ctx* c, long long n_qcols);
static int rollout_batch(ss_ctx* c, const double* actions, uint64_t seed, const double* act_low,
                         const double* act_high, const float* start_rows, const double* start_rows64);

// SS_PRECISION_AUTO -> the kernel family the model shape allows; errors for an unknown or unavailable precision
static int resolve_precision(ss_ctx* c, int& precision) {
    if (precision == SS_PRECISION_AUTO) precision = c->tc_ready ? SS_PRECISION_BF16_TC : SS_PRECISION_FP32;
    if (precision == SS_PRECISION_BF16_TC && !c->tc_ready)
        SS_FAIL(c, SS_EUNSUPPORTED, "mpc: this model shape has no tcgen05 kernel (use precision FP32 or AUTO)");
    if (precision != SS_PRECISION_FP32 && precision != SS_PRECISION_BF16_TC && precision != SS_PRECISION_FP64)
        SS_FAIL(c, SS_EINVAL, "mpc: unknown precision");
    return SS_OK;
}

// SS_PRECISION_FP64 rollout of the batch described by c->run (its actions already in place); start_rows:
// per-sequence start states [K_local][d] on the device, or null
static int rollout_fp64(ss_ctx* c, bool ref, const double* start_rows) {
    auto& r = c->run;
    const int T = r.H + 1, d = c->d;
    if (!r.forward_sim && (c->gpow64_gamma != r.gamma || c->gpow64_T != T || !c->mpc_misc64.p)) {
        std::vector<double> gp(T);
        for (int t = 0; t < T; ++t) gp[t] = std::pow(r.gamma, (double)t);     // gamma ** t (NND_MB_agent.py:611)
        // [gamma^t (T, padded to even) | replay rows T x (d + 1)]
        SS_CUDA_CHECK(c, c->mpc_misc64.ensure(((size_t)T + 2 + (size_t)T * (SS_MAX_D + 1)) * 8));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mpc_misc64.p, gp.data(), T * 8, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        c->gpow64_gamma = r.gamma;
        c->gpow64_T = T;
    }
    Rollout64Args a;
    std::memset(&a, 0, sizeof(a));
    fill_model64_args(c, a);
    a.act = r.act;
    a.plan = r.forward_sim ? fsim_plan64(c) : make_plan64(c, r.gamma, r.hpf);
    for (int j = 0; j < SS_MAX_D; ++j) a.state0[j] = r.state64[j];
    a.state0_rows = start_rows;
    a.wp_index = r.wp_index; a.H = r.H; a.K_local = r.K_local; a.k_offset = r.k_offset;
    a.per_sample = !ref;
    SS_CUDA_CHECK(c, c->mpc_states64.ensure((size_t)T * r.K_local * (d + 1) * 8));
    SS_CUDA_CHECK(c, c->mpc_scores64.ensure((size_t)r.K_local * 8));
    a.rows_out = c->mpc_states64.as<double>();
    a.scores_out = ref ? nullptr : c->mpc_scores64.as<double>();
    if (ref) {
        const size_t cols = (size_t)mpc_fp64_grid(r.K_local);
        SS_CUDA_CHECK(c, c->mpc_partial_sums.ensure((cols + 64) * T * 2 * 8));
        SS_CUDA_CHECK(c, c->mpc_sums.ensure((size_t)T * 2 * 8));
        a.qsums = c->mpc_partial_sums.as<double>();
    }
    timer_mark(c, "mpc_setup");
    int rc = mpc_fp64_launch(c, a);
    if (rc) return rc;
    r.kernel = 4;
    return SS_OK;
}

extern "C" int ss_mpc_rollout(ss_ctx* c, const double* state, int wp_index, int64_t K_local,
                              int64_t k_offset, int64_t K_global, int H, const double* actions,
                              uint64_t seed, const double* act_low, const double* act_high,
                              double gamma, double hpf, int penalty_mode, int precision) {
    if (!c) return SS_EINVAL;
    if (!c->model_set || !c->plan_set) SS_FAIL(c, SS_ESTATE, "mpc: model and plan must be set before planning");
    if (!state || K_local < 1 || H < 1 || k_offset < 0 || K_global < k_offset + K_local)
        SS_FAIL(c, SS_EINVAL, "mpc: bad K / H / state arguments");
    if (wp_index < 0 || wp_index >= c->W) SS_FAIL(c, SS_EINVAL, "mpc: wp_index outside the plan");
    if (penalty_mode != SS_PENALTY_REFERENCE && penalty_mode != SS_PENALTY_PER_SAMPLE)
        SS_FAIL(c, SS_EINVAL, "mpc: unknown penalty_mode");
    if (!actions && (!act_low || !act_high))
        SS_FAIL(c, SS_EINVAL, "mpc: device sampling needs act_low / act_high");
    int rc = resolve_precision(c, precision);
    if (rc) return rc;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    timer_begin(c);

    auto& r = c->run;
    r.valid = false;
    r.finished = false;
    r.forward_sim = false;
    r.K_local = K_local; r.k_offset = k_offset; r.K_global = K_global; r.H = H;
    r.wp_index = wp_index; r.penalty_mode = penalty_mode; r.precision = precision;
    r.gamma = gamma; r.hpf = hpf;
    for (int j = 0; j < SS_MAX_D; ++j) r.state[j] = j < c->d ? (float)state[j] : 0.f;
    for (int j = 0; j < SS_MAX_D; ++j) r.state64[j] = j < c->d ? state[j] : 0.0;
    return rollout_batch(c, actions, seed, act_low, act_high, nullptr, nullptr);
}

// Sets up and launches the rollout of the batch c->run describes (ss_mpc_rollout and ss_mpc_forward_sim): action
// upload, kernel dispatch, projection sums.  start_rows / start_rows64: per-sequence start states [K_local][d] on
// the device for the precision's kernels, or null (every sequence starts at run.state).  A forward simulation
// (run.forward_sim) scores against the context's own plan view and leaves the gamma^t tables of the decisions alone.
static int rollout_batch(ss_ctx* c, const double* actions, uint64_t seed, const double* act_low,
                         const double* act_high, const float* start_rows, const double* start_rows64) {
    auto& r = c->run;
    const int64_t K_local = r.K_local, k_offset = r.k_offset, K_global = r.K_global;
    const int H = r.H, wp_index = r.wp_index, penalty_mode = r.penalty_mode, precision = r.precision;
    const double gamma = r.gamma, hpf = r.hpf;
    int rc = fill_action_source(c, r.act, H, c->da, seed, act_low, act_high);
    if (rc) return rc;
    const int T = H + 1;
    // Host-provided samples: upload in chunks on a second stream while earlier chunks already roll
    // (tcgen05 path, batches of at least two waves of tiles); chunk boundaries are whole waves so
    // no launch ends on a partial wave except the last one.
    int n_chunks = 0;
    long long chunk_tile[ss_ctx::MAX_COPY_CHUNKS + 1] = {0};
    bool actions_on_device = false;
    if (actions) {
        // samples already in device memory (ss_mt19937_uniform's buffer, or any device allocation of
        // the caller's) are rolled in place
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, actions) == cudaSuccess && pa.type == cudaMemoryTypeDevice)
            actions_on_device = true;
        else
            (void)cudaGetLastError();
    }
    if (actions_on_device) {
        r.act.host_actions = actions;
    } else if (actions) {
        const size_t n = (size_t)K_local * H * c->da;
        SS_CUDA_CHECK(c, c->mpc_actions64.ensure(n * 8));
        r.act.host_actions = c->mpc_actions64.as<double>();
        const long long tiles = (K_local + mpc_tc_tile_rows() - 1) / mpc_tc_tile_rows();
        const long long wave = mpc_tc_grid(c, tiles);
        if (precision == SS_PRECISION_BF16_TC && tiles >= 2 * wave) {
            if (!c->copy_ready) {
                SS_CUDA_CHECK(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
                for (int i = 0; i <= ss_ctx::MAX_COPY_CHUNKS; ++i)
                    SS_CUDA_CHECK(c, cudaEventCreateWithFlags(&c->copy_ev[i], cudaEventDisableTiming));
                c->copy_ready = true;
            }
            // first chunk one wave (start rolling early), then two waves per chunk
            const long long waves = (tiles + wave - 1) / wave;
            long long per = 2;
            while (1 + (waves - 1 + per - 1) / per > ss_ctx::MAX_COPY_CHUNKS) ++per;
            chunk_tile[0] = 0;
            for (long long w = 1; w < waves; w += per) chunk_tile[++n_chunks] = w * wave;
            chunk_tile[++n_chunks] = tiles;
            // the staging buffer may still be read by earlier work on the compute stream
            SS_CUDA_CHECK(c, cudaEventRecord(c->copy_ev[ss_ctx::MAX_COPY_CHUNKS], c->stream));
            SS_CUDA_CHECK(c, cudaStreamWaitEvent(c->copy_stream, c->copy_ev[ss_ctx::MAX_COPY_CHUNKS], 0));
            const size_t row_elems = (size_t)H * c->da;
            for (int i = 0; i < n_chunks; ++i) {
                const size_t r0 = (size_t)chunk_tile[i] * mpc_tc_tile_rows();
                size_t r1 = (size_t)chunk_tile[i + 1] * mpc_tc_tile_rows();
                if (r1 > (size_t)K_local) r1 = (size_t)K_local;
                SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mpc_actions64.as<double>() + r0 * row_elems, actions + r0 * row_elems,
                                                 (r1 - r0) * row_elems * 8, cudaMemcpyHostToDevice, c->copy_stream));
                SS_CUDA_CHECK(c, cudaEventRecord(c->copy_ev[i], c->copy_stream));
            }
        } else {
            SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mpc_actions64.p, actions, n * 8, cudaMemcpyHostToDevice, c->stream));
        }
    }
    // gamma^t table (float64 pow, rounded once); re-uploaded only when gamma or the horizon change
    if (!r.forward_sim && (c->gpow_gamma != gamma || c->gpow_T != T || !c->mpc_replay.p)) {
        std::vector<float> misc(T);
        for (int t = 0; t < T; ++t) misc[t] = (float)std::pow(gamma, (double)t);
        // [gamma^t (T) | pad | replay rows T x (d+1) | replay path T x d]
        SS_CUDA_CHECK(c, c->mpc_replay.ensure((size_t)(T + SS_MAX_D + 4) * 4 + (size_t)T * (2 * SS_MAX_D + 1) * 4));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mpc_replay.p, misc.data(), misc.size() * 4, cudaMemcpyHostToDevice, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        c->gpow_gamma = gamma;
        c->gpow_T = T;
    }
    const float* gpow = c->mpc_replay.as<float>();
    const bool ref = penalty_mode == SS_PENALTY_REFERENCE;
    r.states_stored = true;
    if (precision == SS_PRECISION_FP64) {
        rc = rollout_fp64(c, ref, start_rows64);
        if (rc) return rc;
        return reduce_projection_sums(c, mpc_fp64_grid(K_local));
    }

    RolloutArgs a;
    std::memset(&a, 0, sizeof(a));
    fill_model_args(c, a);
    a.act = r.act;
    a.plan = r.forward_sim ? fsim_plan_view(c) : make_plan_view(c, gpow, gamma, hpf);
    for (int j = 0; j < SS_MAX_D; ++j) a.state0[j] = r.state[j];
    a.state0_rows = start_rows;
    a.wp_index = wp_index; a.H = H; a.K_local = K_local; a.k_offset = k_offset;
    a.per_sample = penalty_mode == SS_PENALTY_PER_SAMPLE;
    SS_CUDA_CHECK(c, c->mpc_scores.ensure((size_t)K_local * 4));
    a.scores_out = c->mpc_scores.as<float>();
    // The trajectory rows (state, waypoint index) are spilled in both penalty modes: the stores
    // hide behind the layer-2 MMAs (no measurable cost), the reference-mode passes need them, and the
    // winner's predicted path (NND_MB_agent.py:517) is then a gather instead of a re-roll.
    SS_CUDA_CHECK(c, c->mpc_states.ensure((size_t)T * K_local * traj_row_stride(c->d) * 4));
    a.states_out = c->mpc_states.as<float>();
    // projection sums come out of the rollout kernel: one table column per (tile, row warp) of the tcgen05
    // kernels, one per 32-sequence CTA of the FP32 kernel
    RolloutArgs probe;
    probe.K_local = K_local;
    const long long tc_qcols = precision == SS_PRECISION_BF16_TC
                                   ? 4 * ((K_local + mpc_tc_tile_rows() - 1) / mpc_tc_tile_rows())
                                   : (long long)mpc_simt_grid(probe);
    if (ref) {
        // reference penalty: the penalties themselves come from the tail's pass over the rows (mpc_score.cu)
        SS_CUDA_CHECK(c, c->mpc_partial_sums.ensure(((size_t)tc_qcols + 64) * T * 2 * 8));     // + room for the folded columns
        SS_CUDA_CHECK(c, c->mpc_sums.ensure((size_t)T * 2 * 8));
        a.qsums = c->mpc_partial_sums.as<double>();
    }
    timer_mark(c, "mpc_setup");
    int grid = 0;
    if (n_chunks > 0) {
        for (int i = 0; i < n_chunks; ++i) {
            SS_CUDA_CHECK(c, cudaStreamWaitEvent(c->stream, c->copy_ev[i], 0));
            rc = mpc_tc_launch(c, a, &grid, chunk_tile[i], chunk_tile[i + 1] - chunk_tile[i]);
            if (rc) return rc;
        }
        r.kernel = 1;
    } else if (precision == SS_PRECISION_BF16_TC) {
        // small batches: one tile per 4-CTA cluster with the hidden layer split over the cluster
        // (mpc_tc_quad.cu).  The choice follows the GLOBAL batch, so every shard of a batch runs the same
        // kernel as the unsharded decision would.  SS_TC_QUAD = 0 / 1 forces the pair / quad kernel.
        bool quad = false;
        if (mpc_tc_quad_supported(c)) {
            const char* env = std::getenv("SS_TC_QUAD");
            const long long global_tiles = (K_global + mpc_tc_tile_rows() - 1) / mpc_tc_tile_rows();
            quad = env ? std::atoi(env) != 0 : global_tiles <= mpc_tc_quad_clusters(c);
        }
        rc = quad ? mpc_tc_quad_launch(c, a, &grid) : mpc_tc_launch(c, a, &grid);
        if (rc) return rc;
        r.kernel = quad ? 2 : 1;
    } else {
        rc = mpc_simt_launch(c, a, &grid);
        if (rc) return rc;
        r.kernel = mpc_simt_is_thread_kernel(a) ? 3 : 0;
    }
    return reduce_projection_sums(c, tc_qcols);
}

// reference penalty: the rollout kernel's [2T][n_qcols] projection-sum columns -> the 2T sums of the batch
static int reduce_projection_sums(ss_ctx* c, long long n_qcols) {
    auto& r = c->run;
    const int T = r.H + 1;
    int rc = SS_OK;
    timer_mark(c, "mpc_rollout");
    r.sum_cols = nullptr;
    r.n_cols = 0;
    r.sums_reduced = false;
    if (r.penalty_mode == SS_PENALTY_REFERENCE) {
        int red_blocks = (int)n_qcols;
        const double* red_src = c->mpc_partial_sums.as<double>();
        if (red_blocks > 256) {
            // thousands of columns (one per tile and row warp): fold them to 16 per output first
            double* folded = c->mpc_partial_sums.as<double>() + (size_t)red_blocks * T * 2;
            rc = mpc_fold_partials(c, red_src, red_blocks, T, folded, &red_blocks);
            if (rc) return rc;
            red_src = folded;
        }
        // On a shard of a larger batch the sums of ALL shards are needed before the penalties: with an
        // open peer exchange the reduction kernel also all-reduces them over NVLink peer memory (no
        // NCCL call, no host round trip); otherwise the caller all-reduces the buffer
        // ss_mpc_projection_sums returns.
        r.peer_sums = c->peer_ready && r.K_global != r.K_local;
        rc = r.peer_sums ? peer_allreduce_sums(c, red_src, red_blocks, T, c->mpc_sums.as<double>())
                         : mpc_reduce_sums(c, red_src, red_blocks, T, c->mpc_sums.as<double>());
        if (rc) return rc;
        r.sum_cols = c->mpc_sums.as<double>();
        r.n_cols = 1;
        r.sums_reduced = true;
        r.sum_blocks = red_blocks;
        timer_mark(c, "mpc_sums_pass1");
    }
    r.valid = true;
    return SS_OK;
}

extern "C" int ss_mpc_projection_sums(ss_ctx* c, double** sums_dev, int* count) {
    if (!c) return SS_EINVAL;
    if (!c->run.valid || c->run.forward_sim) SS_FAIL(c, SS_ESTATE, "mpc: no rollout to take projection sums from");
    if (c->run.penalty_mode != SS_PENALTY_REFERENCE) {
        if (sums_dev) *sums_dev = nullptr;
        if (count) *count = 0;
        return SS_OK;
    }
    if (!c->run.sums_reduced) {
        // unsharded batch: the columns were left for the fused tail; reduce them now for this caller
        SS_CUDA_CHECK(c, cudaSetDevice(c->device));
        int rc = mpc_reduce_sums(c, c->run.sum_cols, c->run.n_cols, c->run.H + 1, c->mpc_sums.as<double>());
        if (rc) return rc;
        c->run.sum_cols = c->mpc_sums.as<double>();
        c->run.n_cols = 1;
        c->run.sums_reduced = true;
    }
    if (sums_dev) *sums_dev = c->mpc_sums.as<double>();
    if (count) *count = 2 * (c->run.H + 1);
    return SS_OK;
}

// phase B on the device, ONE launch (mpc_tail): reference-mode coefficients + penalty pass, arg-max,
// and the local winner's package at pkg_dst (and in mapped host memory when host_pkg is given)
static int finish_device(ss_ctx* c, int want_path, double* pkg_dst, double* host_pkg, unsigned long long seq) {
    auto& r = c->run;
    if (!r.valid || r.forward_sim) SS_FAIL(c, SS_ESTATE, "mpc: ss_mpc_finish without ss_mpc_rollout");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const int T = r.H + 1;
    const float* gpow = c->mpc_replay.as<float>();
    const bool penalties = r.penalty_mode == SS_PENALTY_REFERENCE && !r.finished;
    PlanView p = make_plan_view(c, gpow, r.gamma, r.hpf);
    const int blocks = mpc_tail_blocks(r.K_local);
    SS_CUDA_CHECK(c, c->mpc_block_best.ensure((size_t)blocks * 16 + 64));
    if (!c->mpc_result.p) {
        SS_CUDA_CHECK(c, c->mpc_result.ensure(sizeof(MpcResult)));
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->mpc_result.p, 0, sizeof(MpcResult), c->stream));
    }
    double* bv = c->mpc_block_best.as<double>();
    if (r.precision == SS_PRECISION_FP64) {
        int rc = mpc_tail64(c, make_plan64(c, r.gamma, r.hpf), r.wp_index, c->mpc_states64.as<double>(), r.K_local, T,
                            penalties ? r.sum_cols : nullptr, c->mpc_scores64.as<double>(), r.k_offset, bv,
                            reinterpret_cast<long long*>(bv + blocks), c->mpc_result.p, r.act, want_path, pkg_dst,
                            host_pkg, seq);
        if (rc) return rc;
        r.finished = true;
        timer_mark(c, "mpc_tail");
        return SS_OK;
    }
    int rc = mpc_tail(c, p, c->mpc_states.as<float>(), r.K_local, T, penalties ? r.sum_cols : nullptr, r.n_cols,
                      c->mpc_scores.as<float>(), r.k_offset, bv, reinterpret_cast<long long*>(bv + blocks),
                      c->mpc_result.p, r.act, want_path, pkg_dst, host_pkg, seq,
                      penalties && !r.sums_reduced ? c->mpc_sums.as<double>() : nullptr);
    if (rc) return rc;
    r.finished = true;      // the penalty pass rewrites the scores in place: run it once per rollout
    timer_mark(c, "mpc_tail");
    return SS_OK;
}

static int package_count(ss_ctx* c) { return 2 + c->run.H * c->da + (c->run.H + 1) * c->d; }

// the scores of the last finished decision, queued on the stream; widen_scores() completes them after the
// synchronisation (FP32 buffer widened on the host, float64 buffer copied as it is)
static int queue_scores(ss_ctx* c, std::vector<float>& sc, double* out_scores) {
    auto& r = c->run;
    if (r.precision == SS_PRECISION_FP64) {
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_scores, c->mpc_scores64.p, (size_t)r.K_local * 8, cudaMemcpyDeviceToHost, c->stream));
        return SS_OK;
    }
    sc.resize(r.K_local);
    SS_CUDA_CHECK(c, cudaMemcpyAsync(sc.data(), c->mpc_scores.p, (size_t)r.K_local * 4, cudaMemcpyDeviceToHost, c->stream));
    return SS_OK;
}
static void widen_scores(const std::vector<float>& sc, double* out_scores) {
    for (size_t k = 0; k < sc.size(); ++k) out_scores[k] = (double)sc[k];
}

extern "C" int ss_mpc_finish(ss_ctx* c, int64_t* out_best_k, double* out_best_score, double* out_scores) {
    if (!c) return SS_EINVAL;
    auto& r = c->run;
    if (!r.valid || r.forward_sim) SS_FAIL(c, SS_ESTATE, "mpc: ss_mpc_finish without ss_mpc_rollout");
    SS_CUDA_CHECK(c, c->mpc_package.ensure((size_t)package_count(c) * 8));
    int rc = finish_device(c, 0, c->mpc_package.as<double>(), nullptr, 0);
    if (rc) return rc;
    r.pkg_on_host = false;
    MpcResult h;
    SS_CUDA_CHECK(c, cudaMemcpyAsync(&h, c->mpc_result.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    std::vector<float> sc;
    if (out_scores) {
        rc = queue_scores(c, sc, out_scores);
        if (rc) return rc;
    }
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    if (out_scores) widen_scores(sc, out_scores);
    if (out_best_k) *out_best_k = h.best_k;
    if (out_best_score) *out_best_score = h.best_score;
    return SS_OK;
}

static int reroll_winner(ss_ctx* c, int64_t k_global, float* rows_dev);

extern "C" int ss_mpc_finish_package(ss_ctx* c, int want_path, double** package_dev, int* count) {
    if (!c) return SS_EINVAL;
    auto& r = c->run;
    if (!r.valid || r.forward_sim) SS_FAIL(c, SS_ESTATE, "mpc: ss_mpc_finish_package without ss_mpc_rollout");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const int n = package_count(c);
    SS_CUDA_CHECK(c, c->mpc_package.ensure((size_t)n * 8));
    const bool peer = c->peer_ready && r.K_global != r.K_local;
    double* pkg_dst = c->mpc_package.as<double>();
    double* host_pkg = nullptr;
    r.pkg_on_host = false;
    if (peer) {
        SS_CUDA_CHECK(c, c->mpc_package_local.ensure((size_t)n * 8));
        pkg_dst = c->mpc_package_local.as<double>();
    } else if ((size_t)n * 16 <= ss_ctx::HOST_PKG_BYTES) {
        // the package also lands in mapped pinned host memory as self-validating tagged slots (common.cuh
        // host_slot_put): ss_mpc_read_package then needs no device->host copy and no stream synchronisation
        if (!c->host_pkg) {
            SS_CUDA_CHECK(c, cudaHostAlloc(&c->host_pkg, ss_ctx::HOST_PKG_BYTES, cudaHostAllocMapped));
            std::memset(c->host_pkg, 0, ss_ctx::HOST_PKG_BYTES);
            SS_CUDA_CHECK(c, cudaHostGetDevicePointer(&c->host_pkg_dev, c->host_pkg, 0));
        }
        host_pkg = reinterpret_cast<double*>(c->host_pkg_dev);
        r.pkg_seq = ++c->host_pkg_seq;
        r.pkg_on_host = true;
    }
    int rc = finish_device(c, want_path, pkg_dst, host_pkg, r.pkg_seq);
    if (rc) return rc;
    if (peer) {
        // every rank's package goes to every peer; the same kernel picks the global winner
        rc = peer_package_exchange(c, pkg_dst, n, c->mpc_package.as<double>());
        if (rc) return rc;
        timer_mark(c, "mpc_package");
    }
    if (package_dev) *package_dev = c->mpc_package.as<double>();
    if (count) *count = n;
    return SS_OK;
}

extern "C" int ss_mpc_read_package(ss_ctx* c, double* out_package, int count) {
    if (!c) return SS_EINVAL;
    if (!out_package || count < 2 || (size_t)count * 8 > c->mpc_package.cap)
        SS_FAIL(c, SS_EINVAL, "mpc: bad package buffer");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    auto& r = c->run;
    if (r.pkg_on_host && (size_t)count * 16 <= ss_ctx::HOST_PKG_BYTES)
        return host_slots_wait(c, c->host_pkg, count, host_slot_tag(r.pkg_seq), out_package, "mpc");
    SS_CUDA_CHECK(c, cudaMemcpyAsync(out_package, c->mpc_package.p, (size_t)count * 8, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

extern "C" int ss_mpc_get_states(ss_ctx* c, double* out_states) {
    if (!c) return SS_EINVAL;
    auto& r = c->run;
    if (!r.valid || !r.states_stored)
        SS_FAIL(c, SS_ESTATE, "mpc: no stored trajectories (roll out in reference penalty mode first)");
    if (!out_states) SS_FAIL(c, SS_EINVAL, "mpc: null output");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const size_t rows = (size_t)(r.H + 1) * r.K_local;
    const int d = c->d, rs = traj_row_stride(d);
    if (r.precision == SS_PRECISION_FP64) {
        SS_CUDA_CHECK(c, cudaMemcpy2DAsync(out_states, d * 8, c->mpc_states64.p, rs * 8, d * 8, rows,
                                           cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        return SS_OK;
    }
    std::vector<float> tmp(rows * rs);
    SS_CUDA_CHECK(c, cudaMemcpyAsync(tmp.data(), c->mpc_states.p, tmp.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < rows; ++i)
        for (int j = 0; j < d; ++j) out_states[i * d + j] = (double)tmp[i * rs + j];
    return SS_OK;
}

// re-roll ONE sequence of the last batch (global index) into rows_dev [T][1][d + 1]
static int reroll_winner(ss_ctx* c, int64_t k_global, float* rows_dev) {
    auto& r = c->run;
    const int da = c->da;
    const int64_t k_local = k_global - r.k_offset;
    const bool mine = k_local >= 0 && k_local < r.K_local;
    if (r.act.host_actions && !mine)
        SS_FAIL(c, SS_EINVAL, "mpc: host-provided actions of another shard cannot be replayed here");
    const float* gpow = c->mpc_replay.as<float>();
    RolloutArgs a;
    std::memset(&a, 0, sizeof(a));
    fill_model_args(c, a);
    a.act = r.act;
    if (a.act.host_actions) a.act.host_actions += (size_t)k_local * r.H * da;
    a.plan = make_plan_view(c, gpow, r.gamma, r.hpf);
    for (int j = 0; j < SS_MAX_D; ++j) a.state0[j] = r.state[j];
    a.wp_index = r.wp_index; a.H = r.H; a.K_local = 1; a.k_offset = k_global;
    a.per_sample = 1;
    a.states_out = rows_dev;
    // a 1-row tile on the tcgen05 kernel costs H * ~7 us; the FP32 kernel serves the other shapes
    return r.precision == SS_PRECISION_BF16_TC ? mpc_tc_launch(c, a, nullptr) : mpc_simt_launch(c, a, nullptr);
}

// SS_PRECISION_FP64: the winner's path from the float64 rows (resident, or re-rolled through the fp64 kernel)
static int replay_path_fp64(ss_ctx* c, int64_t k_global, double* out_path) {
    auto& r = c->run;
    const int T = r.H + 1, d = c->d;
    const int64_t k_local = k_global - r.k_offset;
    const bool mine = k_local >= 0 && k_local < r.K_local;
    const double* rows = c->mpc_states64.as<double>() + (size_t)k_local * (d + 1);
    size_t pitch = (size_t)r.K_local * (d + 1) * 8;
    if (!(r.states_stored && mine)) {
        if (r.act.host_actions && !mine)
            SS_FAIL(c, SS_EINVAL, "mpc: host-provided actions of another shard cannot be replayed here");
        Rollout64Args a;
        std::memset(&a, 0, sizeof(a));
        fill_model64_args(c, a);
        a.act = r.act;
        if (a.act.host_actions) a.act.host_actions += (size_t)k_local * r.H * c->da;
        a.plan = make_plan64(c, r.gamma, r.hpf);
        for (int j = 0; j < SS_MAX_D; ++j) a.state0[j] = r.state64[j];
        a.wp_index = r.wp_index; a.H = r.H; a.K_local = 1; a.k_offset = k_global;
        a.per_sample = 1;
        a.rows_out = misc64_rows(c);
        int rc = mpc_fp64_launch(c, a);
        if (rc) return rc;
        rows = a.rows_out;
        pitch = (size_t)(d + 1) * 8;
    }
    if (out_path)
        SS_CUDA_CHECK(c, cudaMemcpy2DAsync(out_path, d * 8, rows, pitch, d * 8, T, cudaMemcpyDeviceToHost, c->stream));
    return SS_OK;
}

extern "C" int ss_mpc_replay(ss_ctx* c, int64_t k_global, double* out_sequence, double* out_path) {
    if (!c) return SS_EINVAL;
    auto& r = c->run;
    if (!r.valid || r.forward_sim) SS_FAIL(c, SS_ESTATE, "mpc: ss_mpc_replay without ss_mpc_rollout");
    if (k_global < 0 || k_global >= r.K_global) SS_FAIL(c, SS_EINVAL, "mpc: replay index outside the batch");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    const int T = r.H + 1, d = c->d, da = c->da;
    const int64_t k_local = k_global - r.k_offset;
    const bool mine = k_local >= 0 && k_local < r.K_local;
    const bool f64 = r.precision == SS_PRECISION_FP64;
    float* rows_dev = c->mpc_replay.as<float>() + (T + SS_MAX_D + 3) / 4 * 4;   // 16-byte aligned rows
    float* path_dev = rows_dev + (size_t)T * (SS_MAX_D + 1);
    int rc = SS_OK;
    if (f64) {
        rc = replay_path_fp64(c, k_global, out_path);
        if (rc) return rc;
    } else if (r.states_stored && mine) {
        // the trajectories of this batch are still resident (reference mode): just gather the row
        gather_path_kernel<<<(T * d + 127) / 128, 128, 0, c->stream>>>(c->mpc_states.as<float>(), r.K_local,
                                                                       k_local, T, d, path_dev);
        c->launches++;
        SS_CUDA_CHECK(c, cudaGetLastError());
    } else {
        rc = reroll_winner(c, k_global, rows_dev);
        if (rc) return rc;
        gather_path_kernel<<<(T * d + 127) / 128, 128, 0, c->stream>>>(rows_dev, 1, 0, T, d, path_dev);
        c->launches++;
        SS_CUDA_CHECK(c, cudaGetLastError());
    }
    std::vector<float> path(f64 ? 0 : (size_t)T * d);
    if (!f64) SS_CUDA_CHECK(c, cudaMemcpyAsync(path.data(), path_dev, path.size() * 4, cudaMemcpyDeviceToHost, c->stream));
    if (out_sequence) {
        const size_t n = (size_t)r.H * da;
        SS_CUDA_CHECK(c, c->mpc_block_best.ensure(1024 * 16 + n * 8));
        double* seq_dev = reinterpret_cast<double*>(c->mpc_block_best.as<char>() + 1024 * 16);
        ActionSource act = r.act;
        if (act.host_actions) act.host_actions += (size_t)k_local * r.H * da;
        sample_actions_kernel<<<1, 128, 0, c->stream>>>(act, 1, k_global, seq_dev);
        c->launches++;
        SS_CUDA_CHECK(c, cudaGetLastError());
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_sequence, seq_dev, n * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    if (out_path && !f64)
        for (size_t i = 0; i < path.size(); ++i) out_path[i] = (double)path[i];
    timer_mark(c, "mpc_replay");
    return SS_OK;
}

extern "C" int ss_mpc_plan(ss_ctx* c, const double* state, int wp_index, int64_t K_local,
                           int64_t k_offset, int64_t K_global, int H, const double* actions,
                           uint64_t seed, const double* act_low, const double* act_high, double gamma,
                           double hpf, int penalty_mode, int precision, int64_t* out_best_k,
                           double* out_best_score, double* out_best_sequence, double* out_best_path,
                           double* out_scores) {
    if (!c) return SS_EINVAL;
    if (penalty_mode == SS_PENALTY_REFERENCE && K_global != K_local)
        SS_FAIL(c, SS_EINVAL,
                "mpc: reference penalty over a sharded batch needs ss_mpc_rollout / all-reduce / ss_mpc_finish");
    int rc = ss_mpc_rollout(c, state, wp_index, K_local, k_offset, K_global, H, actions, seed, act_low,
                            act_high, gamma, hpf, penalty_mode, precision);
    if (rc) return rc;
    const bool want_path = out_best_sequence || out_best_path;
    double* pkg_dev = nullptr;
    int n = 0;
    rc = ss_mpc_finish_package(c, want_path ? 1 : 0, &pkg_dev, &n);
    if (rc) return rc;
    std::vector<double> pkg(n);
    std::vector<float> sc;
    if (out_scores) {
        rc = queue_scores(c, sc, out_scores);
        if (rc) return rc;
    }
    rc = ss_mpc_read_package(c, pkg.data(), n);       // the one host synchronisation of the decision
    if (rc) return rc;
    if (out_scores) {
        // the package may have come through mapped host memory without a stream synchronisation, and the
        // float64 scores were copied straight into the caller's array (which may be pinned)
        if (c->run.precision == SS_PRECISION_FP64) SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        widen_scores(sc, out_scores);
    }
    if (out_best_score) *out_best_score = pkg[0];
    if (out_best_k) *out_best_k = (int64_t)pkg[1];
    const int n_seq = H * c->da;
    if (out_best_sequence) std::memcpy(out_best_sequence, pkg.data() + 2, (size_t)n_seq * 8);
    if (out_best_path) std::memcpy(out_best_path, pkg.data() + 2 + n_seq, (size_t)(H + 1) * c->d * 8);
    return SS_OK;
}

extern "C" int ss_mpc_forward_sim(ss_ctx* c, const double* start_states, int64_t n_starts, int64_t K, int H,
                                  const double* actions, int precision, double* out_states) {
    if (!c) return SS_EINVAL;
    if (!c->model_set) SS_FAIL(c, SS_ESTATE, "mpc: set the model before a forward simulation");
    if (!start_states || !actions || !out_states) SS_FAIL(c, SS_EINVAL, "mpc: null forward-simulation pointer");
    if (K < 1 || H < 1) SS_FAIL(c, SS_EINVAL, "mpc: a forward simulation needs K >= 1 and H >= 1");
    if (n_starts != 1 && n_starts != K) SS_FAIL(c, SS_EINVAL, "mpc: n_starts must be 1 or K");
    const int d = c->d;
    for (size_t i = 0; i < (size_t)n_starts * d; ++i)
        if (!std::isfinite(start_states[i])) SS_FAIL(c, SS_EINVAL, "mpc: a start state is NaN or infinite");
    int rc = resolve_precision(c, precision);
    if (rc) return rc;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    timer_begin(c);

    auto& r = c->run;
    r.valid = false;
    r.finished = false;
    r.forward_sim = true;
    r.K_local = K; r.k_offset = 0; r.K_global = K; r.H = H;
    r.wp_index = 0; r.penalty_mode = SS_PENALTY_PER_SAMPLE; r.precision = precision;
    r.gamma = 0.0; r.hpf = 0.0;
    const bool per_row = n_starts > 1;
    for (int j = 0; j < SS_MAX_D; ++j) r.state[j] = !per_row && j < d ? (float)start_states[j] : 0.f;
    for (int j = 0; j < SS_MAX_D; ++j) r.state64[j] = !per_row && j < d ? start_states[j] : 0.0;
    const bool f64 = precision == SS_PRECISION_FP64;
    if (c->fsim_plan_T < H + 1) {
        rc = f64 ? upload_fsim_plan<double>(c, c->fsim_plan64, H + 1) : upload_fsim_plan<float>(c, c->fsim_plan, H + 1);
        if (rc) return rc;
        rc = f64 ? upload_fsim_plan<float>(c, c->fsim_plan, H + 1) : upload_fsim_plan<double>(c, c->fsim_plan64, H + 1);
        if (rc) return rc;
        c->fsim_plan_T = H + 1;
    }
    // per-sequence starts: float64 rows as they are, or rounded to float as run.state is
    std::vector<float> rows32;
    const float* dev32 = nullptr;
    const double* dev64 = nullptr;
    if (per_row) {
        const size_t n = (size_t)K * d;
        SS_CUDA_CHECK(c, c->fsim_start.ensure(n * 8));
        if (f64) {
            SS_CUDA_CHECK(c, cudaMemcpyAsync(c->fsim_start.p, start_states, n * 8, cudaMemcpyHostToDevice, c->stream));
            dev64 = c->fsim_start.as<double>();
        } else {
            rows32.resize(n);
            for (size_t i = 0; i < n; ++i) rows32[i] = (float)start_states[i];
            SS_CUDA_CHECK(c, cudaMemcpyAsync(c->fsim_start.p, rows32.data(), n * 4, cudaMemcpyHostToDevice, c->stream));
            dev32 = c->fsim_start.as<float>();
        }
    }
    rc = rollout_batch(c, actions, 0, nullptr, nullptr, dev32, dev64);
    if (rc) return rc;
    return ss_mpc_get_states(c, out_states);       // synchronises the stream (rows32 lives until then)
}
