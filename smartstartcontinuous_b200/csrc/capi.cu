// capi.cu -- context management and the stage-1 entry points of the C ABI (include/ss_b200.h).
#include <cstdlib>
#include <cstring>

#include "common.cuh"

int kde_run(ss_ctx* c, const double* data_dev, long long n, int d, const double* queries_dev,
            long long m, const float* values_dev, long long n_transitions, double volume,
            double alpha, double beta, double* density_dev, double* ucb_dev, int64_t* out_best_j,
            double* out_best_ucb, const double* running_sums = nullptr);
int kde_exact_sums(ss_ctx* c, const double* data_dev, long long n, int d, double* sums_dev);

int value_net_eval_dev(ss_ctx* c, const double* queries_dev, long long m, float* values_dev);
void mt19937_release(ss_ctx* c);

static std::string g_create_error;

extern "C" int ss_create(ss_ctx** out, int device) {
    if (!out) return SS_EINVAL;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return SS_ECUDA;
    }
    if (device < 0 || device >= count) {
        g_create_error = "device index out of range";
        return SS_EINVAL;
    }
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess ||
        (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        return SS_ECUDA;
    }
    if (prop.major != 10) {
        g_create_error = "libss_b200 is built for sm_100a (B200) only; found compute capability " +
                         std::to_string(prop.major) + "." + std::to_string(prop.minor);
        return SS_EUNSUPPORTED;
    }
    ss_ctx* c = new ss_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->clock_khz = prop.clockRate;
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete c;
        return SS_ECUDA;
    }
    c->own_stream = true;
    *out = c;
    return SS_OK;
}

extern "C" int ss_destroy(ss_ctx* c) {
    if (!c) return SS_EINVAL;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    DevBuf* bufs[] = {&c->kde_data64, &c->kde_q64, &c->kde_vals, &c->kde_pts, &c->kde_qw,
                      &c->kde_partial, &c->kde_fit, &c->kde_moments, &c->kde_density, &c->kde_ucb,
                      &c->kde_block_best, &c->kde_result, &c->tc_w1, &c->tc_w2, &c->tc_w3,
                      &c->tc_misc, &c->plan_ds, &c->plan_dl, &c->mpc_actions64, &c->mpc_states,
                      &c->mpc_scores, &c->mpc_partial_sums, &c->mpc_sums, &c->mpc_block_best,
                      &c->mpc_result, &c->mpc_replay, &c->mpc_sampled, &c->mpc_package,
                      &c->geom_in, &c->geom_rows, &c->geom_pairs, &c->mirror_s, &c->mirror_s2, &c->mirror_idx, &c->mirror_mom,
                      &c->mirror_stage, &c->value_net_params,
                      &c->tc_b3, &c->dyn_params, &c->dyn_m, &c->dyn_v, &c->dyn_x[0], &c->dyn_x[1], &c->dyn_z[0], &c->dyn_z[1],
                      &c->dyn_act, &c->dyn_scratch, &c->dyn_idx, &c->dyn_losses, &c->dyn_round,
                      &c->plan_ds64, &c->plan_dl64, &c->mpc_states64, &c->mpc_scores64, &c->mpc_misc64,
                      &c->fsim_plan, &c->fsim_plan64, &c->fsim_start};
    for (DevBuf* b : bufs) b->release();
    for (auto& b : c->w32) b.release();
    for (auto& b : c->b32) b.release();
    for (auto& b : c->w64) b.release();
    for (auto& b : c->b64) b.release();
    if (c->timer.created)
        for (int i = 0; i <= SS_MAX_PHASES; ++i) cudaEventDestroy(c->timer.ev[i]);
    ss_peer_close(c);
    c->mpc_package_local.release();
    mt19937_release(c);
    if (c->host_pkg) cudaFreeHost(c->host_pkg);
    if (c->host_kde) cudaFreeHost(c->host_kde);
    if (c->host_rows) cudaFreeHost(c->host_rows);
    if (c->copy_ready) {
        for (int i = 0; i <= ss_ctx::MAX_COPY_CHUNKS; ++i) cudaEventDestroy(c->copy_ev[i]);
        cudaStreamDestroy(c->copy_stream);
    }
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return SS_OK;
}

extern "C" const char* ss_last_error(ss_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

extern "C" int ss_set_stream(ss_ctx* c, void* stream) {
    if (!c) return SS_EINVAL;
    if (c->own_stream) {
        cudaStreamSynchronize(c->stream);
        cudaStreamDestroy(c->stream);
        c->own_stream = false;
    }
    c->stream = reinterpret_cast<cudaStream_t>(stream);
    return SS_OK;
}

extern "C" int ss_device_info(ss_ctx* c, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz) {
    if (!c) return SS_EINVAL;
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (clock_khz) *clock_khz = c->clock_khz;
    return SS_OK;
}

extern "C" int ss_last_timings(ss_ctx* c, float* ms, const char** names, int max_phases) {
    if (!c || !c->timer.created || !c->timing) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    int n = c->timer.n < max_phases ? c->timer.n : max_phases;
    for (int i = 0; i < n; ++i) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, c->timer.ev[i], c->timer.ev[i + 1]) != cudaSuccess) t = -1.f;
        if (ms) ms[i] = t;
        if (names) names[i] = c->timer.names[i];
    }
    return n;
}

extern "C" int64_t ss_launch_count(ss_ctx* c) { return c ? c->launches : 0; }

extern "C" int ss_set_timing(ss_ctx* c, int enabled) {
    if (!c) return SS_EINVAL;
    c->timing = enabled != 0;
    c->timer.n = 0;
    return SS_OK;
}

extern "C" void* ss_host_alloc(int64_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void ss_host_free(void* p) {
    if (p) cudaFreeHost(p);
}
extern "C" void* ss_device_alloc(int64_t bytes) {
    void* p = nullptr;
    if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void ss_device_free(void* p) {
    if (p) cudaFree(p);
}
extern "C" int ss_memcpy_h2d(ss_ctx* c, void* dst, const void* src, int64_t bytes) {
    if (!c) return SS_EINVAL;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

extern "C" int ss_memcpy_d2h(ss_ctx* c, void* dst, const void* src, int64_t bytes) {
    if (!c) return SS_EINVAL;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

static int kde_check(ss_ctx* c, const void* data, int64_t n_pts, int d, const void* queries, int64_t m,
                     const void* values, int64_t n_transitions, int64_t* out_best_j, double* out_best_ucb) {
    if (!data || !queries || !out_best_j || !out_best_ucb) SS_FAIL(c, SS_EINVAL, "kde: null pointer");
    if (!values && !c->value_net_set)
        SS_FAIL(c, SS_EINVAL, "kde: values is NULL and no value net is set (ss_value_net_set)");
    if (d < 1 || d > SS_MAX_D) SS_FAIL(c, SS_EUNSUPPORTED, "kde: need 1 <= d <= 32");
    if (m < 1) SS_FAIL(c, SS_EINVAL, "kde: no candidate queries");
    if (n_transitions < 1) SS_FAIL(c, SS_EINVAL, "kde: empty replay buffer");
    // scipy: "data appears to lie in a lower-dimensional subspace" / needs n > d
    if (n_pts <= d)
        SS_FAIL(c, SS_EINVAL, "kde: number of data points must exceed the state dimension (scipy ValueError)");
    return SS_OK;
}

extern "C" int ss_kde_ucb_argmax_dev(ss_ctx* c, const double* data_dev, int64_t n_pts, int d,
                                     const double* queries_dev, int64_t m, const float* values_dev,
                                     int64_t n_transitions, double volume, double alpha, double beta,
                                     double* out_density_dev, double* out_ucb_dev, int64_t* out_best_j,
                                     double* out_best_ucb) {
    if (!c) return SS_EINVAL;
    int rc = kde_check(c, data_dev, n_pts, d, queries_dev, m, values_dev, n_transitions, out_best_j, out_best_ucb);
    if (rc) return rc;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    timer_begin(c);
    if (!values_dev) {
        SS_CUDA_CHECK(c, c->kde_vals.ensure((size_t)m * 4));
        rc = value_net_eval_dev(c, queries_dev, m, c->kde_vals.as<float>());
        if (rc) return rc;
        values_dev = c->kde_vals.as<float>();
    }
    return kde_run(c, data_dev, n_pts, d, queries_dev, m, values_dev, n_transitions, volume, alpha, beta,
                   out_density_dev, out_ucb_dev, out_best_j, out_best_ucb);
}

extern "C" int ss_kde_ucb_argmax(ss_ctx* c, const double* data, int64_t n_pts, int d,
                                 const double* queries, int64_t m, const float* values,
                                 int64_t n_transitions, double volume, double alpha, double beta,
                                 double* out_density, double* out_ucb, int64_t* out_best_j,
                                 double* out_best_ucb) {
    if (!c) return SS_EINVAL;
    int rc = kde_check(c, data, n_pts, d, queries, m, values, n_transitions, out_best_j, out_best_ucb);
    if (rc) return rc;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    timer_begin(c);
    const size_t nd = (size_t)n_pts * d * 8, nq = (size_t)m * d * 8;
    SS_CUDA_CHECK(c, c->kde_data64.ensure(nd));
    SS_CUDA_CHECK(c, c->kde_q64.ensure(nq));
    SS_CUDA_CHECK(c, c->kde_vals.ensure((size_t)m * 4));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->kde_data64.p, data, nd, cudaMemcpyHostToDevice, c->stream));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->kde_q64.p, queries, nq, cudaMemcpyHostToDevice, c->stream));
    if (values) {
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->kde_vals.p, values, (size_t)m * 4, cudaMemcpyHostToDevice, c->stream));
    } else {
        rc = value_net_eval_dev(c, c->kde_q64.as<double>(), m, c->kde_vals.as<float>());
        if (rc) return rc;
    }
    double* dens_dev = nullptr;
    double* ucb_dev = nullptr;
    if (out_density) {
        SS_CUDA_CHECK(c, c->kde_density.ensure((size_t)m * 8));
        dens_dev = c->kde_density.as<double>();
    }
    if (out_ucb) {
        SS_CUDA_CHECK(c, c->kde_ucb.ensure((size_t)m * 8));
        ucb_dev = c->kde_ucb.as<double>();
    }
    timer_mark(c, "kde_h2d");
    rc = kde_run(c, c->kde_data64.as<double>(), n_pts, d, c->kde_q64.as<double>(), m,
                 c->kde_vals.as<float>(), n_transitions, volume, alpha, beta, dens_dev, ucb_dev,
                 out_best_j, out_best_ucb);
    if (rc) return rc;
    if (out_density)
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_density, dens_dev, (size_t)m * 8, cudaMemcpyDeviceToHost, c->stream));
    if (out_ucb)
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_ucb, ucb_dev, (size_t)m * 8, cudaMemcpyDeviceToHost, c->stream));
    SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}

// ---- device-resident mirror of the replay buffer's state ring (SURVEY 8f, row f2) --------------
// rows: [capacity + 1][d] float64 for `s` (the extra row receives the newest s2 at selection time,
// replay_buffer.py:102) and [capacity][d] for `s2`; row index = physical ring row.
constexpr int64_t MIRROR_INCREMENTAL_MAX = 8192;     // rows per write handled incrementally (one block)

// mirror[row0 + i] <- stage[i]; sums += f(stage[i]) - (row0 + i < filled ? f(old row) : 0), f = shifted first and
// second moments (shift x0 = sums[nm .. nm + d)); one block, fixed reduction order
__global__ void __launch_bounds__(256)
mirror_update_kernel(double* __restrict__ mirror, const double* __restrict__ stage, int d, long long row0,
                     long long n_rows, long long filled, double* __restrict__ sums) {
    __shared__ double red[8];
    const int nm = d + d * (d + 1) / 2;
    const double* x0 = sums + nm;
    for (int q0 = 0; q0 < nm; q0 += 8) {
        // eight moments per pass over the rows (registers), so any d <= 32 works with a fixed footprint
        double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (long long i = threadIdx.x; i < n_rows; i += blockDim.x) {
            const double* nw = stage + i * d;
            const double* od = mirror + (row0 + i) * d;
            const bool had = row0 + i < filled;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int q = q0 + u;
                if (q >= nm) break;
                int j, k = -1;
                if (q < d) j = q;
                else {
                    int r = q - d;
                    j = 0;
                    while (r > j) { r -= j + 1; ++j; }
                    k = r;
                }
                double vn = nw[j] - x0[j], vo = had ? od[j] - x0[j] : 0.0;
                if (k >= 0) { vn *= nw[k] - x0[k]; if (had) vo *= od[k] - x0[k]; }
                acc[u] += vn - vo;
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            double v = acc[u];
            for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
            __syncthreads();
            if (threadIdx.x == 0 && q0 + u < nm) {
                double t = 0.0;
                for (int w = 0; w < 8; ++w) t += red[w];
                sums[q0 + u] += t;
            }
            __syncthreads();
        }
    }
    // only now overwrite the rows (every pass above read the old ones)
    for (long long i = threadIdx.x; i < n_rows * d; i += blockDim.x) mirror[row0 * d + i] = stage[i];
}

extern "C" int ss_mirror_write(ss_ctx* c, int which, int64_t capacity, int d, int64_t row0, int64_t n_rows,
                               const double* rows) {
    if (!c) return SS_EINVAL;
    if ((which != 0 && which != 1) || capacity < 1 || d < 1 || d > SS_MAX_D || row0 < 0 || n_rows < 0 ||
        row0 + n_rows > capacity || (n_rows > 0 && !rows))
        SS_FAIL(c, SS_EINVAL, "mirror: bad arguments");
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    if (c->mirror_capacity != capacity || c->mirror_d != d) {
        // a new ring (other capacity / dimension): both mirrors start empty
        c->mirror_s.release();
        c->mirror_s2.release();
        c->mirror_capacity = capacity;
        c->mirror_d = d;
        c->mirror_filled = 0;
        c->mirror_mom_valid = false;
    }
    // allocate geometrically up to capacity + 1 rows, keeping what is there
    DevBuf& buf = which == 0 ? c->mirror_s : c->mirror_s2;
    const size_t need = (size_t)(row0 + n_rows + 1) * d * 8;
    if (need > buf.cap) {
        size_t want = buf.cap ? buf.cap * 2 : (size_t)4096 * d * 8;
        const size_t full = (size_t)(capacity + 1) * d * 8;
        if (want < need) want = need;
        if (want > full) want = full;
        void* np_ = nullptr;
        SS_CUDA_CHECK(c, cudaMalloc(&np_, want));
        if (buf.p) {
            SS_CUDA_CHECK(c, cudaMemcpyAsync(np_, buf.p, buf.cap, cudaMemcpyDeviceToDevice, c->stream));
            SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
            cudaFree(buf.p);
        }
        buf.p = np_;
        buf.cap = want;
    }
    if (n_rows > 0 && which == 0 && c->mirror_mom_valid && n_rows <= MIRROR_INCREMENTAL_MAX && row0 <= c->mirror_filled) {
        // keep the running moments of the `s` rows current: the new rows go through a staging buffer and one
        // block adds them to the sums, subtracts the rows they overwrite (ring wrap) and stores them
        SS_CUDA_CHECK(c, c->mirror_stage.ensure((size_t)n_rows * d * 8));
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mirror_stage.p, rows, (size_t)n_rows * d * 8, cudaMemcpyHostToDevice, c->stream));
        mirror_update_kernel<<<1, 256, 0, c->stream>>>(buf.as<double>(), c->mirror_stage.as<double>(), d, row0, n_rows,
                                                       c->mirror_filled, c->mirror_mom.as<double>());
        c->launches++;
        SS_CUDA_CHECK(c, cudaGetLastError());
        c->mirror_mom_age += n_rows;
        if (c->mirror_mom_age > capacity) c->mirror_mom_valid = false;      // exact recompute once per buffer turnover
    } else if (n_rows > 0) {
        SS_CUDA_CHECK(c, cudaMemcpyAsync(buf.as<double>() + (size_t)row0 * d, rows, (size_t)n_rows * d * 8,
                                         cudaMemcpyHostToDevice, c->stream));
        if (which == 0) c->mirror_mom_valid = false;                         // bulk upload: recomputed at the next selection
    }
    if (which == 0 && n_rows > 0) {
        if (row0 > c->mirror_filled) c->mirror_mom_valid = false;            // a gap: not a ring any more
        c->mirror_filled = std::max<int64_t>(c->mirror_filled, row0 + n_rows);
    }
    return SS_OK;
}

extern "C" int ss_mirror_reset(ss_ctx* c) {
    if (!c) return SS_EINVAL;
    c->mirror_filled = 0;
    c->mirror_mom_valid = false;
    c->mirror_mom_age = 0;
    return SS_OK;
}

__global__ void mirror_gather_kernel(const double* __restrict__ s2_rows, double* __restrict__ s_rows, int d,
                                     long long count, long long last_row, const long long* __restrict__ query_rows,
                                     long long m, double* __restrict__ queries) {
    const long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (o < m * d) queries[o] = s2_rows[query_rows[o / d] * d + (o % d)];
    if (o < d) s_rows[count * d + o] = s2_rows[last_row * d + o];       // data set = every s + the newest s2
}

extern "C" int ss_kde_ucb_argmax_mirror(ss_ctx* c, int64_t count, int64_t last_row, const int64_t* query_rows,
                                        int64_t m, const float* values, int64_t n_transitions, double volume,
                                        double alpha, double beta, double* out_density, double* out_ucb,
                                        int64_t* out_best_j, double* out_best_ucb) {
    if (!c) return SS_EINVAL;
    const int d = c->mirror_d;
    if (!c->mirror_s.p || !c->mirror_s2.p) SS_FAIL(c, SS_ESTATE, "mirror: nothing uploaded yet (ss_mirror_write)");
    if (count < 1 || count > c->mirror_capacity || last_row < 0 || last_row >= count ||
        (size_t)(count + 1) * d * 8 > c->mirror_s.cap || (size_t)count * d * 8 > c->mirror_s2.cap)
        SS_FAIL(c, SS_EINVAL, "mirror: count / last_row outside the uploaded rows");
    int rc = kde_check(c, c->mirror_s.p, count + 1, d, query_rows, m, values, n_transitions, out_best_j, out_best_ucb);
    if (rc) return rc;
    SS_CUDA_CHECK(c, cudaSetDevice(c->device));
    timer_begin(c);
    // rows (checked on the way) and values go through one pinned staging buffer: a copy from the caller's pageable
    // arrays is staged by the driver and costs ~25 us more per call at m = 16 384
    const size_t stage_bytes = (size_t)m * 8 + (values ? (size_t)m * 4 : 0);
    if (stage_bytes > c->host_rows_cap) {
        if (c->host_rows) cudaFreeHost(c->host_rows);
        c->host_rows = nullptr;
        c->host_rows_cap = 0;
        SS_CUDA_CHECK(c, cudaHostAlloc(&c->host_rows, stage_bytes * 2, cudaHostAllocDefault));
        c->host_rows_cap = stage_bytes * 2;
    }
    int64_t* rows_pinned = static_cast<int64_t*>(c->host_rows);
    int64_t bad = 0;
    for (int64_t j = 0; j < m; ++j) {
        const int64_t r = query_rows[j];
        bad |= (r < 0) | (r >= count);
        rows_pinned[j] = r;
    }
    if (bad) SS_FAIL(c, SS_EINVAL, "mirror: query row outside the buffer");
    SS_CUDA_CHECK(c, c->kde_q64.ensure((size_t)m * d * 8));
    SS_CUDA_CHECK(c, c->kde_vals.ensure((size_t)m * 4));
    SS_CUDA_CHECK(c, c->mirror_idx.ensure((size_t)m * 8));
    SS_CUDA_CHECK(c, cudaMemcpyAsync(c->mirror_idx.p, rows_pinned, (size_t)m * 8, cudaMemcpyHostToDevice, c->stream));
    if (values) {
        float* vals_pinned = reinterpret_cast<float*>(rows_pinned + m);
        std::memcpy(vals_pinned, values, (size_t)m * 4);
        SS_CUDA_CHECK(c, cudaMemcpyAsync(c->kde_vals.p, vals_pinned, (size_t)m * 4, cudaMemcpyHostToDevice, c->stream));
    }
    mirror_gather_kernel<<<(unsigned)((m * d + 255) / 256), 256, 0, c->stream>>>(
        c->mirror_s2.as<double>(), c->mirror_s.as<double>(), d, count, last_row, c->mirror_idx.as<long long>(), m,
        c->kde_q64.as<double>());
    c->launches++;
    SS_CUDA_CHECK(c, cudaGetLastError());
    if (!values) {
        rc = value_net_eval_dev(c, c->kde_q64.as<double>(), m, c->kde_vals.as<float>());
        if (rc) return rc;
    }
    double* dens_dev = nullptr;
    double* ucb_dev = nullptr;
    if (out_density) {
        SS_CUDA_CHECK(c, c->kde_density.ensure((size_t)m * 8));
        dens_dev = c->kde_density.as<double>();
    }
    if (out_ucb) {
        SS_CUDA_CHECK(c, c->kde_ucb.ensure((size_t)m * 8));
        ucb_dev = c->kde_ucb.as<double>();
    }
    // the estimator is fitted from the running moments of the buffer rows; they are recomputed exactly after a
    // bulk upload and once per buffer turnover (SS_PRECISION_FP64 fits from the rows themselves, in two passes)
    const double* sums = nullptr;
    if (c->mirror_filled == count && !c->kde_fp64 && !getenv("SS_MIRROR_NO_RUNNING_MOMENTS")) {
        const int nm = d + d * (d + 1) / 2;
        if (!c->mirror_mom_valid) {
            SS_CUDA_CHECK(c, c->mirror_mom.ensure((size_t)(nm + d) * 8));
            rc = kde_exact_sums(c, c->mirror_s.as<double>(), count, d, c->mirror_mom.as<double>());
            if (rc) return rc;
            c->mirror_mom_valid = true;
            c->mirror_mom_age = 0;
        }
        sums = c->mirror_mom.as<double>();
    }
    timer_mark(c, "kde_h2d");
    rc = kde_run(c, c->mirror_s.as<double>(), count + 1, d, c->kde_q64.as<double>(), m, c->kde_vals.as<float>(),
                 n_transitions, volume, alpha, beta, dens_dev, ucb_dev, out_best_j, out_best_ucb, sums);
    if (rc) return rc;
    if (out_density)
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_density, dens_dev, (size_t)m * 8, cudaMemcpyDeviceToHost, c->stream));
    if (out_ucb)
        SS_CUDA_CHECK(c, cudaMemcpyAsync(out_ucb, ucb_dev, (size_t)m * 8, cudaMemcpyDeviceToHost, c->stream));
    if (out_density || out_ucb) SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
    return SS_OK;
}
