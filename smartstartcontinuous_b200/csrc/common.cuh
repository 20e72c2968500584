// common.cuh -- context, device buffers and small device helpers shared by the kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/ss_b200.h"

#define SS_CUDA_CHECK(ctx, expr)                                                        \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) {                                                        \
            (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);            \
            return SS_ECUDA;                                                            \
        }                                                                               \
    } while (0)

#define SS_FAIL(ctx, code, msg)                                                         \
    do {                                                                                \
        (ctx)->err = (msg);                                                             \
        return (code);                                                                  \
    } while (0)

// grow-only device buffer
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int SS_MAX_D = 32;    // state dimension the MPC kernels accept
constexpr int SS_MAX_DA = 8;    // action dimension
constexpr int SS_MAX_LAYERS = 8;
constexpr int SS_MAX_PHASES = 8;

// normalisation statistics + action bounds, passed to kernels by value
struct MpcNorm {
    float mean_x[SS_MAX_D], inv_std_x[SS_MAX_D];
    float mean_y[SS_MAX_DA], inv_std_y[SS_MAX_DA];
    float mean_z[SS_MAX_D], std_z[SS_MAX_D];
};

// the caller's float64 statistics as they are (SS_PRECISION_FP64 divides by the standard deviations)
struct MpcNorm64 {
    double mean_x[SS_MAX_D], std_x[SS_MAX_D];
    double mean_y[SS_MAX_DA], std_y[SS_MAX_DA];
    double mean_z[SS_MAX_D], std_z[SS_MAX_D];
};

struct ActionSource {
    const double* host_actions;  // device copy of host-provided [K_local, H, da] doubles, or null
    uint64_t seed;
    double low[SS_MAX_DA], range[SS_MAX_DA];
    int da, H;
    // 1 when low/range are FP32-representable and low + u * range (u a 24-bit fraction) is exact in
    // float64: then fmaf(u, range, low) in FP32 rounds the same exact value once and gives the same
    // bits as the float64 expression (set by the host, see fill_action_source)
    int fp32_exact;
    float low_f[SS_MAX_DA], range_f[SS_MAX_DA];
};

// NVLink peer-memory exchange (peer.cu)
constexpr int SS_PEER_MAX_WORLD = 8;
constexpr int SS_PEER_SLOT_DOUBLES = 8192;     // 64 KB per (channel, parity, source rank)
struct PeerView {
    double* base[SS_PEER_MAX_WORLD];           // exchange buffer of every rank (own: local pointer)
    int rank, world;
};

struct PhaseTimer {
    cudaEvent_t ev[SS_MAX_PHASES + 1];
    const char* names[SS_MAX_PHASES];
    int n = 0;
    bool created = false;
};

struct ss_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0, cc_major = 0, cc_minor = 0, clock_khz = 0;
    std::string err;
    int64_t launches = 0;
    PhaseTimer timer;
    // second stream + events: host action samples are uploaded in chunks while earlier chunks
    // are already rolling (ss_mpc_rollout)
    cudaStream_t copy_stream = nullptr;
    static constexpr int MAX_COPY_CHUNKS = 8;
    cudaEvent_t copy_ev[MAX_COPY_CHUNKS + 1] = {};
    bool copy_ready = false;

    // ---- KDE scratch
    DevBuf kde_data64, kde_q64, kde_vals, kde_pts, kde_qw, kde_partial, kde_fit, kde_moments;
    DevBuf kde_density, kde_ucb, kde_block_best, kde_result;
    bool kde_tc_attr_set = false;
    bool kde_result_clean = false;     // the counters in kde_result are zero (left so by the last completed call)
    bool kde_fp64 = false;             // selections follow scipy's float64 evaluation (ss_kde_set_precision, kde_fp64.cu)
    // mapped pinned host memory the finish kernel writes the selection result to (+ completion flag)
    void* host_kde = nullptr;
    void* host_kde_dev = nullptr;
    unsigned long long host_kde_seq = 0;
    // ---- plan set-up geometry scratch (plan_geom.cu)
    DevBuf geom_in, geom_rows, geom_pairs;
    // ---- peer-memory exchange of the sharded planner (peer.cu)
    void* peer_buf = nullptr;
    void* peer_opened[SS_PEER_MAX_WORLD] = {};
    PeerView peer_view = {};
    unsigned long long peer_epoch[2] = {0, 0};
    bool peer_ready = false;
    DevBuf mpc_package_local;
    // ---- critic value net in front of the UCB (value_net.cu)
    DevBuf value_net_params;
    std::vector<char> value_net_desc;
    bool value_net_set = false;
    // ---- device mirror of the replay buffer's state ring (capi.cu)
    DevBuf mirror_s, mirror_s2, mirror_idx;
    int64_t mirror_capacity = 0;
    int mirror_d = 0;
    // running first / second moments of the `s` rows in the mirror (shifted by mirror_mom[nm .. nm + d) = x0), kept
    // up to date by ss_mirror_write (new rows added, overwritten rows subtracted): a selection from the mirror
    // fits the estimator from them instead of re-reducing the whole buffer
    DevBuf mirror_mom, mirror_stage;
    void* host_rows = nullptr;         // pinned staging of a selection's candidate rows (+ values)
    size_t host_rows_cap = 0;
    int64_t mirror_filled = 0;         // rows [0, mirror_filled) of mirror_s are valid and included in the sums
    int64_t mirror_mom_age = 0;        // rows added / replaced since the sums were last computed exactly
    bool mirror_mom_valid = false;

    // ---- MPC model
    bool model_set = false;
    int d = 0, da = 0, L = 0, h = 0;
    int din_pad = 0, h_pad = 0;
    std::vector<DevBuf> w32, b32;      // padded fp32 weights [in_pad][out_pad], biases [out_pad]
    MpcNorm norm;
    // tcgen05 images (built lazily by mpc_tc.cu)
    DevBuf tc_w1, tc_w2, tc_w3, tc_misc, tc_b3;
    bool tc_ready = false;
    int tc_hp = 0;
    // layer-1 layout the images were packed with (mpc_tc_prepare): state slots dz (action j -> input dz + j)
    // and K slots k1.  The launchers and the device re-pack of ss_dyn_commit read it from here.
    int tc_dz = 0, tc_k1 = 0;
    int tc_quad_clusters = -1;         // co-resident 4-CTA clusters of the small-batch kernel (-1: not probed)
    std::vector<std::vector<double>> hw, hb;   // host copies of the float64 parameters
    std::vector<DevBuf> w64, b64;      // padded float64 weights / biases (SS_PRECISION_FP64), same layout as w32 / b32
    MpcNorm64 norm64;
    // ---- dynamics-model training on the device (dyn_train.cu): master parameters, Adam moments, both
    // training sets, per-batch activations -- float, or double when dyn_fp64 (ss_dyn_set_precision)
    DevBuf dyn_params, dyn_m, dyn_v, dyn_x[2], dyn_z[2], dyn_act, dyn_scratch, dyn_idx, dyn_losses;
    DevBuf dyn_round;                  // float64 masters rounded to float (ss_dyn_commit after FP64 training)
    bool dyn_fp64 = false;             // the trainer runs in float64 (SS_PRECISION_FP64)
    int64_t dyn_rows[2] = {0, 0};
    long long dyn_t = 0;               // Adam step counter (persists across training calls like TF's slots)
    bool dyn_adam_valid = false;       // moments / counter belong to the current model shape
    bool dyn_params_valid = false;     // dyn_params mirrors (or is ahead of) the model
    bool dyn_dirty = false;            // trained since the last ss_dyn_commit
    bool host_params_stale = false;    // hw / hb are older than the device parameters
    // ---- MPC plan
    bool plan_set = false;
    int W = 0;
    DevBuf plan_ds, plan_dl;           // fp32 [W][d], [W]
    float inv_radii[SS_MAX_D];
    DevBuf plan_ds64, plan_dl64;       // float64 copies for SS_PRECISION_FP64
    double radii64[SS_MAX_D];
    // ---- MPC run state
    DevBuf mpc_actions64, mpc_states, mpc_scores, mpc_partial_sums, mpc_sums, mpc_block_best,
        mpc_result, mpc_replay, mpc_sampled, mpc_package;
    double gpow_gamma = -1.0;          // gamma^t table currently resident in mpc_replay
    int gpow_T = 0;
    // SS_PRECISION_FP64: trajectory rows [T][K][d + 1], scores, and [gamma^t (T) | replay rows T x (d + 1)]
    DevBuf mpc_states64, mpc_scores64, mpc_misc64;
    double gpow64_gamma = -1.0;
    int gpow64_T = 0;
    // ss_mpc_forward_sim: the plan view its kernels score against (the caller's plan is neither needed nor
    // touched), fp32 [ds 2 x SS_MAX_D | dl 2 | gamma^t fsim_plan_T] and the float64 twin, and the per-sequence
    // start rows (fp32 [K][d] rounded from the caller's doubles, then float64 [K][d])
    DevBuf fsim_plan, fsim_plan64, fsim_start;
    int fsim_plan_T = 0;
    struct {
        bool valid = false;
        bool forward_sim = false;      // the last run is a forward simulation: no decision to finish or replay
        int64_t K_local = 0, k_offset = 0, K_global = 0;
        int H = 0, wp_index = 0, penalty_mode = 0, precision = 0;
        double gamma = 0, hpf = 0;
        float state[SS_MAX_D];
        double state64[SS_MAX_D];
        ActionSource act;
        bool states_stored = false;
        int kernel = 0;                // rollout kernel of this decision (ss_mpc_last_kernel)
        bool finished = false;         // the reference-mode penalty pass has rewritten the scores
        bool peer_sums = false;        // the projection sums were all-reduced over peer memory
        int sum_blocks = 0;
        // reference penalty: [2T][n_cols] partial columns of the projection sums the fused tail kernel
        // reduces (n_cols == 1 and sums_reduced: they are final, in mpc_sums)
        const double* sum_cols = nullptr;
        int n_cols = 0;
        bool sums_reduced = false;
        bool pkg_on_host = false;      // the winner package of this decision lands in host_pkg
        unsigned long long pkg_seq = 0;
    } run;
    // mapped pinned host memory the tail kernel writes the winner package to: [0] completion flag
    // (= run.pkg_seq when done), [2..] the package
    static constexpr size_t HOST_PKG_BYTES = 64 * 1024;
    void* host_pkg = nullptr;
    void* host_pkg_dev = nullptr;
    unsigned long long host_pkg_seq = 0;
    void* mt_cache = nullptr;          // MT19937 jump-ahead plans + state read-back buffer (mt19937.cu)
    bool timing = false;               // per-phase CUDA events (ss_last_timings) on request (ss_set_timing(1)): they
                                       // cost ~30 us per decision, a third of a small one
};

// ---- phase timing helpers (CUDA events on the context stream) -------------------------
static inline void timer_begin(ss_ctx* c) {
    PhaseTimer& t = c->timer;
    if (!c->timing) { t.n = 0; return; }
    if (!t.created) {
        for (int i = 0; i <= SS_MAX_PHASES; ++i) cudaEventCreate(&t.ev[i]);
        t.created = true;
    }
    t.n = 0;
    cudaEventRecord(t.ev[0], c->stream);
}
static inline void timer_mark(ss_ctx* c, const char* name) {
    PhaseTimer& t = c->timer;
    if (!c->timing || !t.created || t.n >= SS_MAX_PHASES) return;
    t.names[t.n] = name;
    t.n++;
    cudaEventRecord(t.ev[t.n], c->stream);
}

// ---- programmatic dependent launch (the small kernels behind a rollout) -------------------------
// A kernel launched with launch_dependent() may be scheduled while its predecessor in the stream still runs
// (once every CTA of the predecessor has executed pdl_trigger() or exited); it must execute pdl_wait() before it
// touches anything the predecessor writes -- the wait returns when the predecessor has completed and its
// memory operations are visible.  This takes the launch latency of the reduce / tail kernels (2-3 us each) off
// a small decision's critical path.  Both instructions are no-ops in a normally launched kernel.  (Not for long
// launch trains: the attributed launch costs the host more than a plain one -- the trainer's 960 launches per
// epoch became host-bound with it, 174 instead of 104 us per Adam step.)
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_dependent(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                           cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- small results through mapped pinned host memory, without a fence -------------------------------
// A result double travels as two 8-byte units {32 payload bits | 32-bit tag of the call}, written with ONE
// 16-byte store; the host accepts a slot once both of its tags equal the call's tag.  Every unit validates itself
// (an aligned 8-byte write is atomic on the way to host memory, the granularity NCCL's LL protocol relies on), so
// the payload needs no __threadfence_system() + barrier + release-store of a flag behind it.  Measured on B200
// (scripts/dev/micro/host_flag_latency.cu): the host sees a fence-free store 8.0 us after the launch call, a
// payload + fence + flag 11.5-13.0 us after it.
__device__ __forceinline__ void host_slot_put(unsigned long long* slots, int slot, double v, unsigned int tag) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    const unsigned long long t = (unsigned long long)tag << 32;
    const unsigned long long u0 = t | (bits & 0xffffffffull), u1 = t | (bits >> 32);
    asm volatile("st.global.v2.b64 [%0], {%1, %2};" ::"l"(slots + 2 * slot), "l"(u0), "l"(u1) : "memory");
}
inline unsigned int host_slot_tag(unsigned long long seq) { return (unsigned int)seq | 0x80000000u; }   // never 0
// waits until slots [0, count) carry `tag` and copies their doubles out; the stream is queried now and then so that
// a failed launch cannot hang the caller
inline int host_slots_wait(ss_ctx* c, const void* mapped, int count, unsigned int tag, double* out, const char* what) {
    const volatile unsigned long long* u = static_cast<const volatile unsigned long long*>(mapped);
    unsigned spins = 0;
    bool drained = false;
    for (int o = 0; o < count;) {
        const unsigned long long u0 = u[2 * o], u1 = u[2 * o + 1];
        if ((unsigned int)(u0 >> 32) == tag && (unsigned int)(u1 >> 32) == tag) {
            const unsigned long long bits = (u0 & 0xffffffffull) | (u1 << 32);
            std::memcpy(out + o, &bits, 8);
            ++o;
            continue;
        }
        if ((++spins & 0x3fff) == 0) {
            if (drained) {
                c->err = std::string(what) + ": the kernel ended without delivering its result";
                return SS_ECUDA;
            }
            cudaError_t e = cudaStreamQuery(c->stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) SS_CUDA_CHECK(c, e);
            if (e == cudaSuccess) {
                SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
                drained = true;                       // one more pass over the slot, then give up
                spins = 0x3fff - 64;
            }
        }
    }
    return SS_OK;
}

// ---- device helpers --------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// np.argmax ordering on (value, index): NaN beats everything, then larger value, then lower index
__device__ __forceinline__ bool argmax_better(double va, long long ia, double vb, long long ib) {
    if (ia < 0) return false;
    if (ib < 0) return true;
    bool na = va != va, nb = vb != vb;
    if (na || nb) {
        if (na && nb) return ia < ib;
        return na;
    }
    if (va > vb) return true;
    if (va < vb) return false;
    return ia < ib;
}

// block-wide argmax (blockDim.x <= 1024); result valid in thread 0
__device__ __forceinline__ void block_argmax(double& v, long long& i, double* s_v, long long* s_i) {
    for (int off = 16; off > 0; off >>= 1) {
        double ov = __shfl_down_sync(0xffffffffu, v, off);
        long long oi = __shfl_down_sync(0xffffffffu, i, off);
        if (argmax_better(ov, oi, v, i)) { v = ov; i = oi; }
    }
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_v[warp] = v; s_i[warp] = i; }
    __syncthreads();
    if (warp == 0) {
        int nw = (blockDim.x + 31) >> 5;
        v = lane < nw ? s_v[lane] : 0.0;
        i = lane < nw ? s_i[lane] : -1;
        for (int off = 16; off > 0; off >>= 1) {
            double ov = __shfl_down_sync(0xffffffffu, v, off);
            long long oi = __shfl_down_sync(0xffffffffu, i, off);
            if (argmax_better(ov, oi, v, i)) { v = ov; i = oi; }
        }
    }
    __syncthreads();
}

// Philox4x32-10 (Salmon et al., SC'11); counter-based so the sample of sequence k at step t
// does not depend on how sequences are sharded over GPUs.
__device__ __host__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                       uint32_t c3, uint32_t k0, uint32_t k1,
                                                       uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// action a[k_global][t][j]: host-provided double or Philox uniform in [low, high)
__device__ __forceinline__ float fetch_action(const ActionSource& src, long long k_local,
                                              long long k_global, int t, int j) {
    if (src.host_actions) {
        return (float)src.host_actions[((size_t)k_local * src.H + t) * src.da + j];
    }
    uint32_t e = (uint32_t)(t * src.da + j);
    uint32_t r[4];
    philox4x32_10((uint32_t)k_global, (uint32_t)((uint64_t)k_global >> 32), e >> 2, 0u,
                  (uint32_t)src.seed, (uint32_t)(src.seed >> 32), r);
    const uint32_t sel = e & 3;     // select without indexing (keeps r[] in registers)
    const uint32_t w = sel == 0 ? r[0] : (sel == 1 ? r[1] : (sel == 2 ? r[2] : r[3]));
    double u = (double)(w >> 8) * (1.0 / 16777216.0);
    return (float)(src.low[j] + u * src.range[j]);
}

// The sample as the caller gets it back (best_sequence, NND_MB_agent.py:516-518): host-provided / MT19937
// samples are float64 and are returned bit for bit (the rollout itself consumes them rounded to FP32); the
// Philox sampler is defined in FP32 (oracle/philox.py).
__device__ __forceinline__ double fetch_action_f64(const ActionSource& src, long long k_local, long long k_global,
                                                   int t, int j) {
    if (src.host_actions) return src.host_actions[((size_t)k_local * src.H + t) * src.da + j];
    return (double)fetch_action(src, k_local, k_global, t, j);
}

// Same values as fetch_action() for a thread that walks t = 0, 1, 2, ... of ONE sequence: the
// Philox block of four samples is kept in registers and recomputed only when (t * da + j) / 4
// changes; the affine map runs in FP32 when that is bit-identical (ActionSource::fp32_exact).
struct ActionCursor {
    uint32_t r[4];
    uint32_t blk;
};
__device__ __forceinline__ void action_cursor_init(ActionCursor& c) { c.blk = 0xffffffffu; }
__device__ __forceinline__ float fetch_action_seq(const ActionSource& src, ActionCursor& c, long long k_local,
                                                  long long k_global, int t, int j) {
    if (src.host_actions) return (float)src.host_actions[((size_t)k_local * src.H + t) * src.da + j];
    const uint32_t e = (uint32_t)(t * src.da + j);
    if ((e >> 2) != c.blk) {
        c.blk = e >> 2;
        philox4x32_10((uint32_t)k_global, (uint32_t)((uint64_t)k_global >> 32), c.blk, 0u, (uint32_t)src.seed,
                      (uint32_t)(src.seed >> 32), c.r);
    }
    const uint32_t sel = e & 3;
    const uint32_t w = sel == 0 ? c.r[0] : (sel == 1 ? c.r[1] : (sel == 2 ? c.r[2] : c.r[3]));
    if (src.fp32_exact) return fmaf((float)(w >> 8) * (1.0f / 16777216.0f), src.range_f[j], src.low_f[j]);
    const double u = (double)(w >> 8) * (1.0 / 16777216.0);
    return (float)(src.low[j] + u * src.range[j]);
}
