/*
 * ss_b200.h -- C ABI of libss_b200.so: the B200 (sm_100a) implementation of the
 * SmartStartContinuous hot path (start-state selection + MPC navigation).
 *
 * The reference (darren-huang/SmartStartContinuous) is pure Python; the "FFI" a
 * maintainer would bind is ctypes (see INTEGRATION.md for the stub).  Every entry
 * point below names the reference code it replaces (file:line, relative to the
 * reference root).
 *
 * Conventions
 *   - every function returns 0 on success or a negative SS_E* code; a human readable
 *     message for the last failure on a context is returned by ss_last_error().
 *   - all matrices are C-contiguous (row-major); `double` on the host side because the
 *     reference works in float64 numpy end to end.
 *   - the caller owns every buffer it passes; the library copies inputs in during the
 *     call, owns all device memory inside the context, and writes results into the
 *     caller's output buffers before returning (calls are synchronous, exactly like
 *     the scipy / sess.run calls they replace).
 *   - `*_dev` variants take DEVICE pointers for the bulk inputs (zero-copy from torch
 *     tensors); their small outputs are still written to host memory.
 *   - a context is bound to one GPU and is not thread-safe (one agent per process in
 *     the reference; multi-GPU = one process and one context per GPU).
 *   - there is no CPU fallback anywhere behind this interface.
 */
#ifndef SS_B200_H_
#define SS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ss_ctx ss_ctx;

enum {
    SS_OK = 0,
    SS_EINVAL = -1,      /* bad argument (maps to ValueError)                         */
    SS_ECUDA = -2,       /* CUDA runtime failure (maps to RuntimeError)               */
    SS_ESINGULAR = -3,   /* covariance not positive definite (numpy.linalg.LinAlgError,
                            as scipy.stats.gaussian_kde raises)                       */
    SS_ESTATE = -4,      /* call order: model / plan not set                          */
    SS_EUNSUPPORTED = -5 /* shape outside what the kernels were built for             */
};

/* penalty_mode of the MPC scorer (SURVEY.md section 8a, quirk Q1) */
enum {
    SS_PENALTY_REFERENCE = 0,  /* numerical.py:89-93: one projection coefficient per time step,
                                  global over all K samples (reference-exact; two-phase)     */
    SS_PENALTY_PER_SAMPLE = 1  /* per-sample projection; fully fused, no HBM round trip      */
};

/* precision of the dynamics-MLP rollout */
enum {
    SS_PRECISION_FP32 = 0,     /* FP32 FFMA everywhere (SIMT kernel; parity mode)            */
    SS_PRECISION_BF16_TC = 1,  /* hidden x hidden layers on tcgen05 (BF16 in, FP32 accumulate
                                  in TMEM); first/last layer, state and scoring in FP32      */
    SS_PRECISION_AUTO = 2,     /* BF16_TC when the shape is supported, else FP32             */
    SS_PRECISION_FP64 = 3      /* everything in float64 in the reference's element-wise order
                                  (DFMA rollout, float64 scores and arg-max): the reference's
                                  decision up to the summation order of GEMMs and reductions;
                                  AUTO never selects it                                       */
};

/* ---- context --------------------------------------------------------------------- */
int ss_create(ss_ctx** out, int device);
int ss_destroy(ss_ctx* ctx);
const char* ss_last_error(ss_ctx* ctx);          /* ctx may be NULL: last create() error */
/* run all work of this context on an existing CUDA stream (e.g. torch's current one) */
int ss_set_stream(ss_ctx* ctx, void* cuda_stream);
/* sm_count, cc_major, cc_minor, max SM clock (kHz) */
int ss_device_info(ss_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int* sm_clock_khz);
/* device time (ms, CUDA events on the context's stream) of the most recent call, split in
 * up to 8 named phases; returns the number of phases written */
int ss_last_timings(ss_ctx* ctx, float* ms, const char** names, int max_phases);
/* per-phase CUDA events (they feed ss_last_timings) are recorded after ss_set_timing(ctx, 1); off by
 * default -- the events between the kernels cost ~30 us per call, a third of a K = 4096 decision */
int ss_set_timing(ss_ctx* ctx, int enabled);
/* number of kernel launches issued by this context since creation */
int64_t ss_launch_count(ss_ctx* ctx);
/* pinned host memory for end-to-end callers (bench e2e leg) */
void* ss_host_alloc(int64_t bytes);
void ss_host_free(void* p);
void* ss_device_alloc(int64_t bytes);
void ss_device_free(void* p);
int ss_memcpy_h2d(ss_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes);
int ss_memcpy_d2h(ss_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes);

/* ---- stage 1: Gaussian KDE + UCB + argmax --------------------------------------------
 * Replaces smartexplorationcontinuous.py:260 (scipy.stats.gaussian_kde(all_states.T,
 * bw_method='scott')), :275 (kernel(possible_ss_states.T) * one_radii_volume),
 * :276-279 (C_hat, UCB) and :280 (np.argmax).
 *
 *   data     [n_pts, d]   all_states (every s in the buffer + the newest s2)
 *   queries  [m, d]       candidate smart-start states (s2 of the sampled steps)
 *   values   [m]          float32 state values from agent.get_state_value (:274)
 *   n_transitions         len(replay_buffer)  (|D| in the UCB term; n_pts - 1 in the reference)
 *   volume                one-step hyper-ellipsoid volume (:262-268), 1 when radii is None
 *   alpha, beta           exploitation_param, exploration_param
 *   out_density [m] / out_ucb [m]   optional (may be NULL): kernel(q) (before * volume) and ucb
 *   out_best_j            first index of the maximum ucb (np.argmax semantics: NaN wins, first wins)
 * Errors: SS_EINVAL for d > n_pts or empty inputs (scipy raises ValueError),
 *         SS_ESINGULAR when the data covariance is not positive definite.
 */
int ss_kde_ucb_argmax(ss_ctx* ctx, const double* data, int64_t n_pts, int d,
                      const double* queries, int64_t m, const float* values,
                      int64_t n_transitions, double volume, double alpha, double beta,
                      double* out_density, double* out_ucb,
                      int64_t* out_best_j, double* out_best_ucb);
/* same, bulk inputs already resident in device memory (outputs: host; out_density/out_ucb: device) */
int ss_kde_ucb_argmax_dev(ss_ctx* ctx, const double* data_dev, int64_t n_pts, int d,
                          const double* queries_dev, int64_t m, const float* values_dev,
                          int64_t n_transitions, double volume, double alpha, double beta,
                          double* out_density_dev, double* out_ucb_dev,
                          int64_t* out_best_j, double* out_best_ucb);
/* precision of the selection (all three ss_kde_ucb_argmax* entry points; signatures, errors and outputs
 * unchanged): SS_PRECISION_FP32 (default; FP32 / tcgen05 pair stage, densities to ~1e-5) or SS_PRECISION_FP64,
 * which follows scipy.stats.gaussian_kde 1.18 operation for operation in float64 (two-pass weighted
 * covariance, Cholesky times the Scott factor, triangular solves, sum_i w * (exp(-|P_i - Z_j|^2 / 2) * norm))
 * and forms alpha * values in float32 as numpy does with the float32 values: densities agree with scipy to
 * ~1e-13 relative, so the choice is scipy's whenever the top-two UCB gap is larger than that.  The mirror entry
 * point then fits from the mirror's rows, not from its running moments.  A query's density does not depend on
 * the batch it is evaluated in.  Setting the current value is a no-op; any other value: SS_EINVAL. */
int ss_kde_set_precision(ss_ctx* ctx, int precision);

/* ---- stage 2: NND_MB random-shooting MPC ---------------------------------------------
 * ss_mpc_set_model: the weights Dyn_Model holds (dynamics_model.py:36-37,
 * feedforward_network.py:3-23) and the normalisation statistics of NND_MB_agent.py:302-315.
 * Call after construction and after every train_dynamics_model (NND_MB_agent.py:437-480).
 *   weights[l] [in_l, out_l] (y = x W + b), l = 0..num_fc_layers (hidden layers use ReLU,
 *   the last layer is linear); in_0 = d + da, out_last = d.
 */
int ss_mpc_set_model(ss_ctx* ctx, int d, int da, int num_fc_layers, int depth_fc_layers,
                     const double* const* weights, const double* const* biases,
                     const double* mean_x, const double* std_x,
                     const double* mean_y, const double* std_y,
                     const double* mean_z, const double* std_z);

/* ss_mpc_set_plan: what start_new_episode_plan leaves on the agent (NND_MB_agent.py:375-418):
 * desired_states [W, d], distances_left [W], radii [d] (all > 0, numerical.py:112-113).  W >= 2. */
int ss_mpc_set_plan(ss_ctx* ctx, const double* desired_states, int W,
                    const double* distances_left, const double* radii, int d);

/* ss_mpc_plan: get_best_sim_actions (NND_MB_agent.py:498-520) = sample (:500-501) +
 * Dyn_Model.do_forward_sim (dynamics_model.py:204-240) + generate_scores_add_delta
 * (NND_MB_agent.py:566-628) + argmax/selection (:516-518).
 *
 *   state [d]           current state;  wp_index = current_desired_state_index
 *   K_local sequences are evaluated by this context; they are sequences
 *   [k_offset, k_offset + K_local) of a global batch of K_global (multi-GPU sharding;
 *   single GPU: k_offset = 0, K_global = K_local).
 *   actions             [K_local, H, da] float64 action samples in host memory (uploaded) or in device
 *                       memory (used in place, e.g. ss_mt19937_uniform's buffer), or NULL:
 *                       sampled on the device with Philox4x32-10(seed) indexed by the GLOBAL
 *                       sequence number, uniform in [act_low, act_high) like npr.uniform.
 *   out_best_k          GLOBAL index of the first maximum score on this shard
 *   out_best_sequence   [H, da], out_best_path [H+1, d] (rolled out in FP32; float64 with SS_PRECISION_FP64), out_scores [K_local]
 *                       (nullable)
 * In SS_PENALTY_REFERENCE mode with K_global != K_local use the three-call form below so the
 * per-time-step projection sums can be all-reduced across GPUs.
 */
int ss_mpc_plan(ss_ctx* ctx, const double* state, int wp_index,
                int64_t K_local, int64_t k_offset, int64_t K_global, int H,
                const double* actions, uint64_t seed,
                const double* act_low, const double* act_high,
                double gamma, double horizontal_penalty_factor,
                int penalty_mode, int precision,
                int64_t* out_best_k, double* out_best_score,
                double* out_best_sequence, double* out_best_path, double* out_scores);

/* three-call form: rollout (phase A) -> [all-reduce the 2*(H+1) doubles at *sums_dev] -> finish.
 * ss_mpc_rollout returns while its work (including the host->device copies of `actions`) is still
 * queued on the context's stream: the `actions` buffer must stay untouched until ss_mpc_finish,
 * ss_mpc_read_package or ss_mpc_replay of the same decision has returned (they synchronise the
 * stream).  ss_mpc_plan is synchronous and has no such window. */
int ss_mpc_rollout(ss_ctx* ctx, const double* state, int wp_index,
                   int64_t K_local, int64_t k_offset, int64_t K_global, int H,
                   const double* actions, uint64_t seed,
                   const double* act_low, const double* act_high,
                   double gamma, double horizontal_penalty_factor,
                   int penalty_mode, int precision);
int ss_mpc_projection_sums(ss_ctx* ctx, double** sums_dev, int* count);
int ss_mpc_finish(ss_ctx* ctx, int64_t* out_best_k, double* out_best_score, double* out_scores);
/* ss_mpc_finish_package: ss_mpc_finish + the local winner's action sequence and predicted path
 * (NND_MB_agent.py:516-518), all left in DEVICE memory as one float64 package
 *   [best_score, best_k (global, as double), best_sequence (H*da), best_path ((H+1)*d)]
 * without a host synchronisation (the trajectory rows of the batch are kept on the device in both
 * penalty modes, the winner's path is a gather).  Multi-GPU callers all-gather the packages and pick with
 * np.argmax ordering -- one collective and one device->host copy per decision.  want_path = 0
 * leaves the sequence / path part zero.  Phase B is ONE kernel launch (coefficients, penalties, arg-max
 * and package); on an unsharded batch the same kernel also writes the package to mapped pinned host
 * memory (self-validating tagged slots, no fence or flag), so ss_mpc_read_package returns it without a
 * device->host copy or a stream synchronisation. */
int ss_mpc_finish_package(ss_ctx* ctx, int want_path, double** package_dev, int* count);
int ss_mpc_read_package(ss_ctx* ctx, double* out_package, int count);
/* ---- NVLink peer-memory exchange for sharded batches (one process per GPU, one node) -------
 * ss_peer_init allocates this rank's exchange buffer and returns its 64-byte CUDA IPC handle; the
 * caller all-gathers the handles (any transport) and passes all of them, in rank order, to
 * ss_peer_open.  From then on a sharded ss_mpc_rollout (K_global != K_local) in reference penalty
 * mode leaves the GLOBAL projection sums in place (the reduction kernel stores its sums into every
 * peer's slot and adds the peers' in rank order), and ss_mpc_finish_package leaves the GLOBAL
 * winner's package on every rank (np.argmax ordering over the ranks' winners) -- no NCCL call and no
 * host synchronisation between the phases.  Every rank must make the same sequence of sharded
 * calls.  world <= 8. */
int ss_peer_init(ss_ctx* ctx, int rank, int world, void* out_ipc_handle_64_bytes);
int ss_peer_open(ss_ctx* ctx, const void* all_handles_world_x_64_bytes, int world);
int ss_peer_close(ss_ctx* ctx);
int ss_peer_ready(ss_ctx* ctx);
/* merge of per-rank (value, global index) pairs over the same exchange: every rank gets the
 * np.argmax-ordered winner (NaN first, then the larger value, then the lower index; index < 0 = this
 * rank has nothing).  Used for the KDE query shards: (ucb, j) of smartexplorationcontinuous.py:280. */
int ss_peer_argmax_merge(ss_ctx* ctx, double value, int64_t index, double* out_value, int64_t* out_index);
/* roll out ONE sequence of the last ss_mpc_rollout batch again (the global winner) in FP32 and
 * return its actions [H, da] and predicted path [H+1, d] (NND_MB_agent.py:516-518) */
int ss_mpc_replay(ss_ctx* ctx, int64_t k_global, double* out_sequence, double* out_path);
/* trajectories of the last ss_mpc_rollout (kept on the device for the reference-mode passes and
 * for the winner's path): out_states [H+1, K_local, d], as do_forward_sim returns them
 * (dynamics_model.py:199-240). */
int ss_mpc_get_states(ss_ctx* ctx, double* out_states);
/* ss_mpc_forward_sim: Dyn_Model.do_forward_sim(many_in_parallel=True) (dynamics_model.py:204-240), no scoring.
 * Needs ss_mpc_set_model only: no plan, and the caller's plan is left as it was.
 *   start_states [n_starts, d] float64, host memory; n_starts = 1 (every sequence starts there: the reference's
 *                [state, 0] form) or K (sequence k starts at row k).  A NaN or infinite start is SS_EINVAL (the
 *                reference would carry it through every later state of that sequence).
 *   actions      [K, H, da] float64, host or device memory (as ss_mpc_rollout)
 *   precision    SS_PRECISION_AUTO / FP32 / BF16_TC / FP64, dispatched exactly as ss_mpc_rollout dispatches a
 *                decision of the same K (pair vs quad kernel by the batch's tiles, thread vs CTA FP32 kernel)
 *   out_states   [H+1, K, d] float64 (FP32 / BF16_TC: the FP32 rows widened, t = 0 is the start rounded to
 *                float; FP64: the start rows exactly)
 * Afterwards the context's last run is this simulation: ss_mpc_last_kernel reports its kernel and
 * ss_mpc_get_states returns its states, while ss_mpc_finish, ss_mpc_finish_package, ss_mpc_replay and
 * ss_mpc_projection_sums return SS_ESTATE until the next ss_mpc_rollout / ss_mpc_plan.  A decision after a
 * forward simulation is bit-identical to the same decision without one.  SS_EINVAL: n_starts not 1 or K, K < 1,
 * H < 1, a null pointer; SS_ESTATE: no model. */
int ss_mpc_forward_sim(ss_ctx* ctx, const double* start_states, int64_t n_starts, int64_t K, int H,
                       const double* actions, int precision, double* out_states);
/* the device sampler alone: actions [K_local, H, da] for sequences k_offset.. (tests / oracle) */
int ss_mpc_sample_actions(ss_ctx* ctx, int64_t K_local, int64_t k_offset, int H, int da,
                          uint64_t seed, const double* act_low, const double* act_high,
                          double* out_actions);
/* ---- numpy's legacy RandomState stream on the device ---------------------------------------
 * The reference draws the action samples of every decision from numpy's global Mersenne Twister:
 *     all_samples = npr.uniform(self.low, self.high, (self.N, self.horizon, da))   NND_MB_agent.py:500-501
 * (element i = low[i % da] + (high - low)[i % da] * random_sample(), in C order).  ss_mt19937_uniform
 * produces elements [first, first + count) of that draw of n_total doubles bit for bit on the GPU
 * (MT19937 with polynomial jump-ahead, csrc/mt19937.cu) from the generator state
 * np.random.get_state() returns -- key[624], pos (0..624) -- and leaves them in device memory:
 * *out_dev is valid until the next ss_mt19937_uniform / host-sample ss_mpc_rollout on this context and
 * can be passed as `actions` to ss_mpc_rollout / ss_mpc_plan (device pointers are rolled in place).
 * A rank of a sharded batch passes its own [first, first + count) and gets the same numbers the
 * single-process draw would have put there.  ss_mt19937_state returns the generator state AFTER the
 * whole n_total draw (what np.random.set_state needs so that the host stream continues exactly as if
 * the host had drawn); it waits for the kernel.  period = da. */
int ss_mt19937_uniform(ss_ctx* ctx, const uint32_t* key, int pos, int64_t n_total, int64_t first,
                       int64_t count, int period, const double* low, const double* high,
                       double** out_dev);
int ss_mt19937_state(ss_ctx* ctx, uint32_t* out_key, int* out_pos);
/* get_best_sim_actions (NND_MB_agent.py:498-520) INCLUDING its draw (:500-501), in one call: the samples come
 * from the generator state (mt_key[624], *mt_pos) as ss_mt19937_uniform produces them, the decision is ss_mpc_plan's,
 * and the state after the draw is written back through the same two pointers -- which may be the address of numpy's
 * own state struct {uint32 key[624]; int pos} (BitGenerator.ctypes.state_address): the host generator then continues
 * exactly as if npr.uniform had run, without a get_state / set_state round trip. */
int ss_mpc_plan_mt19937(ss_ctx* ctx, const double* state, int wp_index,
                        int64_t K_local, int64_t k_offset, int64_t K_global, int H,
                        uint32_t* mt_key, int* mt_pos,
                        const double* act_low, const double* act_high,
                        double gamma, double horizontal_penalty_factor,
                        int penalty_mode, int precision,
                        int64_t* out_best_k, double* out_best_score,
                        double* out_best_sequence, double* out_best_path, double* out_scores);
/* host-only helpers behind the jump-ahead (no GPU work; used by the CPU tests): the coefficient words
 * of x^J mod phi (624 x uint32, bit i of word w = x^(32 w + i)), and the exponents of phi, MT19937's
 * characteristic polynomial (returns their number, 135). */
int ss_mt19937_jump_poly(uint64_t J, uint32_t* out_words);
int ss_mt19937_phi_exponents(int* out, int cap);

/* CPython's random.sample(range(first, first + n), k) in C++ on the generator state random.getstate()
 * exposes (mt_state[624], *mt_index = the 625th entry): replaces the candidate draw of
 * ReplayBuffer.get_possible_smart_start_indices (replay_buffer.py:145-152), ~0.6 us per index in the
 * interpreter, with the same indices in the same order; state and index are advanced in place.
 * Host only (csrc/py_random.cu); n < 2^31. */
int ss_py_random_sample(uint32_t* mt_state, int* mt_index, int64_t first, int64_t n, int64_t k, int64_t* out);

/* 1 when ss_mpc_set_model's shape can run on the tcgen05 kernel */
int ss_mpc_tc_supported(ss_ctx* ctx);
/* rollout kernel of the last ss_mpc_rollout: 0 = FP32 SIMT, 1 = tcgen05 CTA pairs (mpc_tc.cu), 2 = tcgen05
 * 4-CTA clusters with the hidden layer split over the cluster (small batches, mpc_tc_quad.cu), 3 = FP32 thread per
 * sequence (one hidden layer of <= 64 units, the reference's default 1 x 32 model), 4 = float64 (SS_PRECISION_FP64,
 * mpc_fp64.cu); -1 = none */
int ss_mpc_last_kernel(ss_ctx* ctx);
/* schedule of the last ss_mpc_rollout on the tcgen05 CTA-pair kernel: 0 = one tile per CTA at a time, 1 = two tiles
 * per CTA offset by half a step (layouts with K1 = 16 and a padded hidden width of 512, at least two tiles per CTA;
 * an odd last tile of a CTA still runs alone); -1 = the last rollout did not run that kernel */
int ss_mpc_last_tc_schedule(ss_ctx* ctx);

/* ---- dynamics-model training on the device (SURVEY 8f, row f1) ------------------------------
 * Replaces Dyn_Model.train (dynamics_model.py:52-171) as NND_MB_agent.train_dynamics_model calls it
 * (NND_MB_agent.py:437-480): mini-batch Adam (tf.train.AdamOptimizer defaults) on
 * reduce_mean(square(z - f(x))) for the network set with ss_mpc_set_model.  Data sets, master
 * parameters and Adam moments stay on the device across calls, in FP32 (default) or, after
 * ss_dyn_set_precision(ctx, SS_PRECISION_FP64), in float64 like the reference's graph.
 *   ss_dyn_set_data       which = 0: the initial ("old") data set, 1: the aggregated ("new") one;
 *                         X [n, d + da] normalised inputs, Z [n, d] normalised state deltas
 *   ss_dyn_train_batches  n_batches Adam steps; batch i = old rows idx_old[i*n_old ..] followed by
 *                         new rows idx_new[i*n_new ..] (the reference's batching rule: the caller draws
 *                         the indices with the reference's numpy calls); out_losses [n_batches] = the
 *                         batch MSE before each update (what sess.run returns), nullable
 *   ss_dyn_eval_loss      mean batch MSE over the consecutive full batches of a data set
 *                         (old_loss / new_loss :139-166, run_validation :174-197)
 *   ss_dyn_commit         re-pack the trained parameters for the rollout kernels on the device (no
 *                         host round trip); ss_mpc_plan uses them from then on
 *   ss_dyn_get_params     export as float64 [in, out] / [out] (checkpoints, tests)
 *   ss_dyn_reset_optimizer  forget the Adam moments and step count
 * With SS_PRECISION_FP64 the data sets are stored without float32 rounding, every step runs in float64
 * (DFMA; Adam in the oracle's operation order), ss_dyn_get_params returns the float64 masters exactly
 * and ss_dyn_commit hands them unchanged to SS_PRECISION_FP64 rollouts (the FP32 and tcgen05 images
 * are packed from the masters rounded once to float). */
int ss_dyn_set_data(ss_ctx* ctx, int which, const double* X, const double* Z, int64_t n_rows);
int ss_dyn_train_batches(ss_ctx* ctx, const int32_t* idx_old, const int32_t* idx_new, int n_batches, int n_old,
                         int n_new, double lr, double* out_losses);
int ss_dyn_eval_loss(ss_ctx* ctx, int which, int batchsize, double* out_mean_loss, int* out_batches);
int ss_dyn_commit(ss_ctx* ctx);
int ss_dyn_get_params(ss_ctx* ctx, double* const* out_weights, double* const* out_biases);
int ss_dyn_reset_optimizer(ss_ctx* ctx);
/* precision of the device trainer: SS_PRECISION_FP32 (default, today's trainer) or SS_PRECISION_FP64.
 * Changing it discards the trainer state -- master parameters, Adam moments, step count and both data
 * sets -- so the next training call starts from the parameters of the last ss_mpc_set_model, as after
 * ss_dyn_reset_optimizer; the data sets must be uploaded again.  Setting the current value is a no-op.
 * Any other value: SS_EINVAL. */
int ss_dyn_set_precision(ss_ctx* ctx, int precision);

/* ---- critic value batch in front of the UCB (SURVEY 8f, row f4) --------------------------
 * V_j = critic(q_j, actor(q_j)) of the DDPG base agent (agent.get_state_value,
 * smartexplorationcontinuous.py:274 -> ddpg_editted.py:274-279; graph :106-131; networks
 * models_editted.py:22-100), FP32 like the TF graph.  Weights [in, out] (tf.layers.dense kernels);
 * critic W2 is [(h1c + da), h2c] (the action is concatenated after the first hidden layer).
 * gamma / beta pointers are only read with layer_norm; obs_mean / obs_std NULL = no observation
 * normalisation (normalize_observations=False); has_ret_norm = 0 = no return normalisation.
 * Once set, ss_kde_ucb_argmax / _mirror accept values = NULL and compute them on the device. */
typedef struct {
    int d, da, h1a, h2a, h1c, h2c, layer_norm, last_layer_tanh;
    const float *aW1, *ab1, *ag1, *abe1, *aW2, *ab2, *ag2, *abe2, *aW3, *ab3;
    const float *cW1, *cb1, *cg1, *cbe1, *cW2, *cb2, *cg2, *cbe2, *cW3, *cb3;
    const double *obs_mean, *obs_std;
    double obs_clip_lo, obs_clip_hi;
    int has_ret_norm;
    double ret_mean, ret_std, ret_clip_lo, ret_clip_hi;
} ss_value_net;
int ss_value_net_set(ss_ctx* ctx, const ss_value_net* net);      /* net = NULL clears it */
int ss_value_net_eval(ss_ctx* ctx, const double* queries, int64_t m, int d, float* out_values);

/* ---- device-resident replay-state mirror (SURVEY 8f, row f2) ------------------------------
 * The KDE data set is every `s` in the buffer plus the newest `s2` (ReplayBuffer.get_all_states,
 * replay_buffer.py:102) and the candidate queries are `s2` rows of sampled steps (:136-152, :205).
 * Instead of shipping both from the host at every selection, the caller mirrors its ring of
 * (s, s2) rows on the device incrementally -- ss_mirror_write(which = 0 for s / 1 for s2, ring
 * capacity, d, first physical row, row count, rows) after the adds since the last selection --
 * and ss_kde_ucb_argmax_mirror selects from the mirror: only m row indices and m values cross
 * PCIe.  count = rows in use, last_row = physical row of the newest step, query_rows = physical
 * rows of the candidates.  Everything else as ss_kde_ucb_argmax. */
int ss_mirror_write(ss_ctx* ctx, int which, int64_t capacity, int d, int64_t row0, int64_t n_rows,
                    const double* rows);
/* forget the mirror's contents (a new ring object on the host side); the next writes start from row 0 */
int ss_mirror_reset(ss_ctx* ctx);
int ss_kde_ucb_argmax_mirror(ss_ctx* ctx, int64_t count, int64_t last_row, const int64_t* query_rows, int64_t m,
                             const float* values, int64_t n_transitions, double volume, double alpha, double beta,
                             double* out_density, double* out_ucb, int64_t* out_best_j, double* out_best_ucb);

/* ---- plan set-up geometry (SURVEY 8f, row f3) ------------------------------------------
 * ss_path_close_pairs: the pair-extraction half of path_shortcutter (numerical.py:226-246,
 * called from start_new_episode_plan, NND_MB_agent.py:398-401): all (s, e) with e >= s + 2 whose
 * elliptical distance sqrt(sum(((path[s] - path[e]) / radii)^2)) (numerical.py:116-124) is <= theta,
 * in np.argwhere(np.triu(mask, k=2)) order.  float64 with the reference's operation order, so the
 * threshold decisions are the ones numpy makes.  out_pairs [max_pairs][2] int32 receives the first
 * min(*out_count, max_pairs) pairs; *out_count is the total (call again with a larger buffer if it
 * exceeds max_pairs).  The interval-scheduling DP (numerical.py:189-222) stays on the host. */
int ss_path_close_pairs(ss_ctx* ctx, const double* path, int P, int d, const double* radii, double theta,
                        int32_t* out_pairs, int64_t max_pairs, int64_t* out_count);
/* ss_path_shortcut: all of path_shortcutter (numerical.py:226-246) on the device -- the pair mask
 * above plus the weighted-interval-scheduling DP of length_weighted_activities_solver
 * (numerical.py:189-222, weight = end - start - 1, ties resolved as the reference does, including
 * its first-interval quirk at :202).  out_keep [P] receives the indices of the states that remain
 * (ascending), *out_count how many. */
int ss_path_shortcut(ss_ctx* ctx, const double* path, int P, int d, const double* radii, double theta,
                     int32_t* out_keep, int* out_count);

#ifdef __cplusplus
}
#endif
#endif /* SS_B200_H_ */
