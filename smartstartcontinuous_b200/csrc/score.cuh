// score.cuh -- per-(sequence, time-step) trajectory scoring shared by every rollout kernel.
//
// Restates NND_MB_agent.generate_scores_add_delta (NND_MB_agent.py:566-628) with
// move_to_next (:491-496), the elliptical distance (numerical.py:116-124) and
// dist_line_seg_to_point / projection_of_a_onto_b (numerical.py:74-98) for ONE sample.
// The reference's projection coefficient is global over the K samples of a time step
// (np.sum without axis, numerical.py:89-93): in SS_PENALTY_REFERENCE mode score_point()
// only returns the two dot products a'.b' and b'.b' (to be summed over all samples and
// GPUs, from the spilled rows) and the penalty is applied afterwards by penalty_with_lambda(); in
// SS_PENALTY_PER_SAMPLE mode the coefficient is local and everything fuses.
#pragma once

#include "common.cuh"

struct PlanView {
    const float* ds;        // desired_states [W][d]
    const float* dl;        // distances_left [W]
    const float* gpow;      // gamma^t, t = 0..H   (rounded from float64 on the host)
    int W, d;
    float inv_r[SS_MAX_D];  // 1 / radii
    float pen_scale;        // horizontal_penalty_factor * gamma   (NND_MB_agent.py:622)
};

struct ScoreAcc {
    int idx;       // samples_desired_state_indices[k]
    float prev;    // prev_distances_to_end[k]
    float score;   // scores[k]
};

template <int DT>
__device__ __forceinline__ float ell_dist(const PlanView& P, const float* __restrict__ w,
                                          const float (&x)[DT]) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < DT; ++j)
        if (j < P.d) {
            float df = (w[j] - x[j]) * P.inv_r[j];
            s = fmaf(df, df, s);
        }
    return sqrtf(s);
}

// NND_MB_agent.py:571-577
template <int DT>
__device__ __forceinline__ void score_init(const PlanView& P, int wp_index, const float (&x0)[DT],
                                           ScoreAcc& a) {
    a.idx = wp_index;
    a.prev = P.dl[wp_index] + ell_dist<DT>(P, P.ds + (size_t)wp_index * P.d, x0);
    a.score = 0.f;
}

// Spilled trajectories (reference penalty mode): row (t, k) = d state floats followed by the
// sample's waypoint index after the move of that step, so the projection sums and the penalties
// can be recomputed for every (t, k) independently (no serial waypoint scan in the tail passes).
__host__ __device__ __forceinline__ int traj_row_stride(int d) { return d + 1; }

template <int DT>
__device__ __forceinline__ void traj_store(float* __restrict__ rows, size_t row, int d, const float (&x)[DT],
                                           int idx) {
    if (DT >= 3 && d == 3) {
        *reinterpret_cast<float4*>(rows + row * 4) = make_float4(x[0], x[1], x[2], __int_as_float(idx));
    } else {
        float* o = rows + row * (size_t)(d + 1);
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < d) o[j] = x[j];
        o[d] = __int_as_float(idx);
    }
}
template <int DT>
__device__ __forceinline__ void traj_load(const float* __restrict__ rows, size_t row, int d, float (&x)[DT],
                                          int& idx) {
    if (DT >= 3 && d == 3) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(rows + row * 4));
        x[0] = v.x; x[1] = v.y; x[2] = v.z;
        idx = __float_as_int(v.w);
    } else {
        const float* o = rows + row * (size_t)(d + 1);
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < d) x[j] = __ldg(o + j);
        idx = __float_as_int(__ldg(o + d));
    }
}

// a'.b' and b'.b' of the line-segment projection (NND_MB_agent.py:616-621, numerical.py:89-93)
// for a point whose waypoint index after the move is idx
template <int DT>
__device__ __forceinline__ void proj_terms(const PlanView& P, int idx, const float (&x)[DT], float& ab, float& bb) {
    const int b0 = idx - 1 > 0 ? idx - 1 : 0;
    const float* w0 = P.ds + (size_t)b0 * P.d;
    const float* w1 = w0 + P.d;
    ab = 0.f;
    bb = 0.f;
#pragma unroll
    for (int j = 0; j < DT; ++j)
        if (j < P.d) {
            const float av = (x[j] - w0[j]) * P.inv_r[j];
            const float bv = (w1[j] - w0[j]) * P.inv_r[j];
            ab = fmaf(av, bv, ab);
            bb = fmaf(bv, bv, bb);
        }
}

// One trajectory point (NND_MB_agent.py:582-622): waypoint move + progress term; when per_sample
// is true the penalty (per-sample projection coefficient) is applied here as well, otherwise it
// is left to the reference-mode passes (which recompute a'.b', b'.b' from the spilled row).
template <int DT>
__device__ __forceinline__ void score_point(const PlanView& P, int t, const float (&x)[DT],
                                            ScoreAcc& a, bool per_sample) {
    const int last = P.W - 1;
    const int nxt = a.idx + 1 < last ? a.idx + 1 : last;
    float dc = ell_dist<DT>(P, P.ds + (size_t)a.idx * P.d, x);
    const float dn = ell_dist<DT>(P, P.ds + (size_t)nxt * P.d, x);
    const bool mv = ((dc <= 1.0f) || (dn <= dc)) && (a.idx != last);     // theta == 1
    if (mv) { a.idx += 1; dc = dn; }
    const float to_end = P.dl[a.idx] + dc;
    a.score = fmaf(a.prev - to_end, P.gpow[t], a.score);
    a.prev = to_end;
    if (per_sample) {
        const int b0 = a.idx - 1 > 0 ? a.idx - 1 : 0;
        const float* w0 = P.ds + (size_t)b0 * P.d;
        const float* w1 = w0 + P.d;
        float av[DT], bv[DT];
        float ab = 0.f, bb = 0.f;
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < P.d) {
                av[j] = (x[j] - w0[j]) * P.inv_r[j];
                bv[j] = (w1[j] - w0[j]) * P.inv_r[j];
                ab = fmaf(av[j], bv[j], ab);
                bb = fmaf(bv[j], bv[j], bb);
            }
        const float lam = ab / bb;
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < P.d) {
                float df = fmaf(lam, bv[j], -av[j]);
                s = fmaf(df, df, s);
            }
        a.score -= sqrtf(s) * P.pen_scale;
    }
}

// reference mode, second pass: penalty of one point given the global coefficient of its step
template <int DT>
__device__ __forceinline__ float penalty_with_lambda(const PlanView& P, int idx_after_move,
                                                     const float (&x)[DT], float lam) {
    const int b0 = idx_after_move - 1 > 0 ? idx_after_move - 1 : 0;
    const float* w0 = P.ds + (size_t)b0 * P.d;
    const float* w1 = w0 + P.d;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < DT; ++j)
        if (j < P.d) {
            float av = (x[j] - w0[j]) * P.inv_r[j];
            float bv = (w1[j] - w0[j]) * P.inv_r[j];
            float df = fmaf(lam, bv, -av);
            s = fmaf(df, df, s);
        }
    return sqrtf(s) * P.pen_scale;
}

// ---- float64 twin (SS_PRECISION_FP64, mpc_fp64.cu / the float64 tail of mpc_score.cu) ---------------------------
// The reference's own operation order, element by element: the products are __dmul_rn so that the compiler
// cannot contract them into an FMA with the following add, divisions divide, and the sums over the state
// dimension run in numpy's order (pairwise_sum of numpy/core/src/umath/loops_utils.h: plain left-to-right
// below 8 terms, eight interleaved accumulators above).
struct Plan64 {
    const double* ds;        // desired_states [W][d]
    const double* dl;        // distances_left [W]
    const double* gpow;      // gamma ** t, t = 0..H  (host pow in float64)
    int W, d;
    double r[SS_MAX_D];      // radii
    double hpf, gamma;
};

struct ScoreAcc64 {
    int idx;
    double prev, score;
};

template <int DT>
__device__ __forceinline__ double np_sum(const double (&v)[DT], int n) {
    if (n < 8) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < DT; ++j)
            if (j < n) s = __dadd_rn(s, v[j]);
        return s;
    }
    double r[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) r[q] = v[q < DT ? q : 0];
    const int n8 = n - n % 8;
#pragma unroll
    for (int j = 8; j < DT; ++j)
        if (j < n8) r[j % 8] = __dadd_rn(r[j % 8], v[j]);
    double s = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
#pragma unroll
    for (int j = 8; j < DT; ++j)
        if (j >= n8 && j < n) s = __dadd_rn(s, v[j]);
    return s;
}

// numerical.py:116-124: sqrt(sum(((a - b) / r) ** 2))
template <int DT>
__device__ __forceinline__ double ell_dist64(const Plan64& P, const double* __restrict__ w, const double (&x)[DT]) {
    double q[DT];
#pragma unroll
    for (int j = 0; j < DT; ++j) {
        q[j] = 0.0;
        if (j < P.d) {
            const double df = (w[j] - x[j]) / P.r[j];
            q[j] = __dmul_rn(df, df);
        }
    }
    return sqrt(np_sum<DT>(q, P.d));
}

template <int DT>
__device__ __forceinline__ void score_init64(const Plan64& P, int wp_index, const double (&x0)[DT], ScoreAcc64& a) {
    a.idx = wp_index;
    a.prev = P.dl[wp_index] + ell_dist64<DT>(P, P.ds + (size_t)wp_index * P.d, x0);
    a.score = 0.0;
}

// a' = (x - w0) / r, b' = (w1 - w0) / r of the segment the point projects on (numerical.py:76-88)
template <int DT>
__device__ __forceinline__ void proj_vectors64(const Plan64& P, int idx, const double (&x)[DT], double (&av)[DT],
                                               double (&bv)[DT]) {
    const int b0 = idx - 1 > 0 ? idx - 1 : 0;
    const double* w0 = P.ds + (size_t)b0 * P.d;
    const double* w1 = w0 + P.d;
#pragma unroll
    for (int j = 0; j < DT; ++j) {
        av[j] = 0.0;
        bv[j] = 0.0;
        if (j < P.d) {
            av[j] = (x[j] - w0[j]) / P.r[j];
            bv[j] = (w1[j] - w0[j]) / P.r[j];
        }
    }
}

// sum(a' * b') and sum(b' * b') (numerical.py:89-93, per point)
template <int DT>
__device__ __forceinline__ void proj_terms64(const Plan64& P, int idx, const double (&x)[DT], double& ab, double& bb) {
    double av[DT], bv[DT];
    proj_vectors64<DT>(P, idx, x, av, bv);
#pragma unroll
    for (int j = 0; j < DT; ++j) { av[j] = __dmul_rn(av[j], bv[j]); bv[j] = __dmul_rn(bv[j], bv[j]); }
    ab = np_sum<DT>(av, P.d);
    bb = np_sum<DT>(bv, P.d);
}

// pen * hpf * gamma of numerical.py:80-81 / NND_MB_agent.py:622 for a given coefficient lam
template <int DT>
__device__ __forceinline__ double penalty64(const Plan64& P, int idx, const double (&x)[DT], double lam) {
    double av[DT], bv[DT];
    proj_vectors64<DT>(P, idx, x, av, bv);
#pragma unroll
    for (int j = 0; j < DT; ++j) {
        const double df = __dmul_rn(lam, bv[j]) - av[j];
        av[j] = __dmul_rn(df, df);
    }
    return __dmul_rn(__dmul_rn(sqrt(np_sum<DT>(av, P.d)), P.hpf), P.gamma);
}

// waypoint move + progress term of one point (NND_MB_agent.py:582-611); returns to_end
template <int DT>
__device__ __forceinline__ void progress64(const Plan64& P, int t, const double (&x)[DT], ScoreAcc64& a) {
    const int last = P.W - 1;
    const int nxt = a.idx + 1 < last ? a.idx + 1 : last;
    double dc = ell_dist64<DT>(P, P.ds + (size_t)a.idx * P.d, x);
    const double dn = ell_dist64<DT>(P, P.ds + (size_t)nxt * P.d, x);
    const bool mv = ((dc <= 1.0) || (dn <= dc)) && (a.idx != last);
    if (mv) { a.idx += 1; dc = dn; }
    const double to_end = P.dl[a.idx] + dc;
    a.score = a.score + __dmul_rn(a.prev - to_end, P.gpow[t]);
    a.prev = to_end;
}

// the whole step with the per-sample coefficient (SS_PENALTY_PER_SAMPLE)
template <int DT>
__device__ __forceinline__ void score_point64_per_sample(const Plan64& P, int t, const double (&x)[DT], ScoreAcc64& a) {
    progress64<DT>(P, t, x, a);
    double ab, bb;
    proj_terms64<DT>(P, a.idx, x, ab, bb);
    a.score = a.score - penalty64<DT>(P, a.idx, x, ab / bb);
}
