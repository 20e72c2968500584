// mpc_tc_quad.cu -- tcgen05 rollout for SMALL batches: one tile of 128 sequences per 4-CTA cluster.
//
// The pair kernel (mpc_tc.cu) gives every CTA pair two whole tiles, so a batch of K = 4096 (BASELINE
// config 3: 32 tiles) occupies 32 of 148 SMs and every step costs the full 8192 tensor clocks of layer 2
// plus ~2800 exposed clocks of prologue / epilogue.  Here the HIDDEN LAYER is split instead: the four CTAs
// of a cluster keep identical copies of the tile's state, each computes layer 1 completely (K = 16 or 32:
// negligible) and ONE 128-unit chunk of layer 2 -- its 128 KB slice of W2 stays resident in shared memory for
// the whole kernel, nothing is streamed -- followed by its share of layer 3; the partial state deltas
// (128 rows x d floats per CTA) are exchanged through distributed shared memory (one 16-byte st.async per
// row and destination, completing transaction bytes on the destination's mbarrier; buffers and barriers
// double-buffered by step parity) and summed in a fixed order, so the four copies of the state stay
// bit-identical.  Layer 2 drops to 2048 tensor clocks per step; 32 tiles use 128 SMs.
//
// Same operand images in global memory as the pair kernel; the loader warp interleaves the two 64-unit halves
// of every block into one 128-row K-major tile in shared memory (1 KB bulk copies), so one N = 128 MMA per K step,
// same layer-1 split-bf16 scheme, same TMEM map ([0,256) H1 as bf16 A operand, [256,512) accumulators),
// same scoring (tc_score_row.cuh; quarter q of the rows is scored by CTA q of the cluster).  Model shapes:
// padded hidden width 512 (four chunks), d <= 4.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "mpc_kernels.cuh"
#include "tc_ptx.cuh"
#include "tc_score_row.cuh"

namespace tcq {

using namespace tc;

constexpr int TM = 128;                 // rows per tile
constexpr int NC = 128;                 // hidden units per chunk
constexpr int NH = 64;                  // units per image half (one N = 64 MMA)
constexpr int KSLAB = 256;              // K elements per W2 image block
constexpr int BLOCK_BYTES = NH * KSLAB * 2;          // 32 KB
constexpr int HP = 512, NCH = HP / NC, NSLAB = HP / KSLAB;
constexpr int QUAD = 4;
constexpr int K1_MAX = 32;
constexpr int W1_CHUNK_BYTES_MAX = NH * K1_MAX * 2;
constexpr int A1_BYTES_MAX = TM * K1_MAX * 2;
constexpr int ROW_WARPS = 8, TPR = 2, CPT = NC / TPR;
constexpr int THREADS = ROW_WARPS * 32 + 64;
constexpr int DZ_MAX = 4;
constexpr uint32_t TMEM_COLS = 512, COL_H1 = 0, COL_ACC = 256;
// D f32, A/B bf16, K-major, N = 128, M = 128 (cta_group::1)
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NC >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

__host__ __device__ constexpr int w3_pair_floats(int dz) { return dz <= 2 ? 4 : 8; }

struct Params {
    const __nv_bfloat16* w1_img;        // [2 (half)][4 (chunk)][K1/8][64][8]
    const __nv_bfloat16* w2_img;        // [4 (chunk)][2 (k-slab)][2 (half)][32][64][8]
    const float* w3;                    // [256 (unit pairs)][DZP][2]
    const float* b3;
    long long tile_begin, tile_end;
    int iters;                          // tile iterations per cluster
    unsigned long long* prof;           // SS_TC_TRACE: clock stamps of cluster 0 / CTA 0, steps 10..12
};

struct Smem {
    static constexpr size_t W2 = 0;                                                  // this CTA's chunk: 128 KB
    static constexpr size_t W1 = W2 + (size_t)NSLAB * 2 * BLOCK_BYTES;               // all chunks, both halves
    static constexpr size_t A1 = W1 + (size_t)2 * NCH * W1_CHUNK_BYTES_MAX;
    static constexpr size_t W3 = A1 + (size_t)A1_BYTES_MAX;
    static constexpr size_t ZX = W3 + (size_t)(HP / 2) * 8 * 4;                       // [DZ_MAX][2 halves][128] local partials
    static constexpr size_t ZQ = ZX + (size_t)DZ_MAX * TPR * TM * 4;                  // [2 parity][4 src][128 rows][4] exchanged
    static constexpr size_t BARS = ZQ + (size_t)2 * QUAD * TM * 16;
    static constexpr int N_BARS = 2 + 2 + NCH + 2 + 1 + 2 + 2;
    static constexpr size_t TMEM_PTR = BARS + (size_t)N_BARS * 8;
    static constexpr size_t END = TMEM_PTR + 16;
};

#define TQ_TRACE(ev)                                                                             \
    do {                                                                                         \
        if (p.prof && blockIdx.x == 0 && lane == 0 && trace_on && trace_t >= 10 && trace_t < 13)  \
            p.prof[(trace_t - 10) * 64 + (ev)] = (unsigned long long)clock64();                   \
    } while (0)

// ROWS: every sequence starts at its own row of a.state0_rows (load_start, forward simulation)
template <int DT, int DZ, int K1T, bool ROWS = false>
__global__ void __launch_bounds__(THREADS, 1) mpc_rollout_tc_quad_kernel(const RolloutArgs a, const Params p) {
    pdl_trigger();      // the reduce / tail kernels behind this launch may be scheduled (they wait for its completion)
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int MAXIN = (K1T - 2) / 3;
    constexpr int W1_CHUNK_BYTES = NH * K1T * 2;
    constexpr int DZP = w3_pair_floats(DZ) / 2;
    unsigned char* w2s = smem + Smem::W2;
    unsigned char* w1s = smem + Smem::W1;
    unsigned char* a1s = smem + Smem::A1;
    float* w3s = reinterpret_cast<float*>(smem + Smem::W3);
    float* zx = reinterpret_cast<float*>(smem + Smem::ZX);
    float4* zq = reinterpret_cast<float4*>(smem + Smem::ZQ);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::BARS);
    uint64_t* acc_full = bars;            // [1] layer-2 chunk complete (commit)            (+1 spare)
    uint64_t* acc_free = acc_full + 2;    // [2] accumulator slot drained by the row warps
    uint64_t* h1_ready = acc_free + 2;    // [NCH] layer-1 chunk converted (an A operand now)
    uint64_t* l1_full = h1_ready + NCH;   // [2] layer-1 chunk 0 / all chunks complete (commit)
    uint64_t* x_ready = l1_full + 2;      // the layer-1 A tile is in shared memory
    uint64_t* w_full = x_ready + 1;       // [2] W1 / this CTA's W2 chunk have landed (once)
    uint64_t* z_full = w_full + 2;        // [2 parity] the four CTAs' partial state deltas of the step have landed (tx bytes)
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + Smem::TMEM_PTR);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();         // = the layer-2 chunk this CTA computes
    const long long cluster_id = blockIdx.x / QUAD, n_clusters = gridDim.x / QUAD;
    if (p.prof && blockIdx.x == 0 && tid == 0) p.prof[192] = (unsigned long long)clock64();

    if (tid == 0) {
        mbar_init(&acc_full[0], 1);
        mbar_init(&acc_full[1], 1);
        for (int s = 0; s < 2; ++s) mbar_init(&acc_free[s], ROW_WARPS);
        for (int c = 0; c < NCH; ++c) mbar_init(&h1_ready[c], ROW_WARPS);
        mbar_init(&l1_full[0], 1);
        mbar_init(&l1_full[1], 1);
        mbar_init(x_ready, 4);
        mbar_init(&w_full[0], 1);
        mbar_init(&w_full[1], 1);
        mbar_init(&z_full[0], 1);
        mbar_init(&z_full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (p.prof && blockIdx.x == 0) p.prof[196] = (unsigned long long)clock64();
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)),
                     "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        if (p.prof && blockIdx.x == 0 && tid == 0) p.prof[197] = (unsigned long long)clock64();
    }
    __syncthreads();
    if (p.prof && blockIdx.x == 0 && tid == 0) p.prof[198] = (unsigned long long)clock64();
    if (warp == ROW_WARPS + 1) {
        // resident operands, each as 128-row K-major tiles [k/8][128 units][8]: the two 64-unit halves of the
        // global images are interleaved k-group by k-group (1 KB bulk copies spread over the lanes).  W1 of
        // every chunk first (the first MMAs need it), then this CTA's chunk of W2 (needed ~1000 clocks later).
        constexpr int KG1 = K1T / 8, KG2 = KSLAB / 8;
        if (lane == 0) {
            // (layer-3 weights ride on the first barrier: a 320-thread global-load loop here cost ~4000 clocks of
            // every launch)
            mbar_expect_tx(&w_full[0], (uint32_t)(NCH * 2 * W1_CHUNK_BYTES) + (uint32_t)((HP / 2) * (2 * DZP) * 4));
            bulk_g2s(w3s, p.w3, (uint32_t)((HP / 2) * (2 * DZP) * 4), &w_full[0]);
            mbar_expect_tx(&w_full[1], (uint32_t)(NSLAB * 2 * BLOCK_BYTES));
        }
        __syncwarp();
        const unsigned char* g1 = reinterpret_cast<const unsigned char*>(p.w1_img);
        for (int i = lane; i < NCH * KG1 * 2; i += 32) {
            const int r = i & 1, kg = (i >> 1) % KG1, c = (i >> 1) / KG1;
            bulk_g2s(w1s + (size_t)c * (2 * W1_CHUNK_BYTES) + (size_t)kg * (NC * 16) + (size_t)r * (NH * 16),
                     g1 + ((size_t)r * NCH + c) * W1_CHUNK_BYTES + (size_t)kg * (NH * 16), NH * 16, &w_full[0]);
        }
        const unsigned char* g2 = reinterpret_cast<const unsigned char*>(p.w2_img) + (size_t)rank * NSLAB * 2 * BLOCK_BYTES;
        for (int i = lane; i < NSLAB * KG2 * 2; i += 32) {
            const int r = i & 1, kg = (i >> 1) % KG2, ksl = (i >> 1) / KG2;
            bulk_g2s(w2s + (size_t)ksl * (2 * BLOCK_BYTES) + (size_t)kg * (NC * 16) + (size_t)r * (NH * 16),
                     g2 + ((size_t)ksl * 2 + r) * BLOCK_BYTES + (size_t)kg * (NH * 16), NH * 16, &w_full[1]);
        }
    }
    tc_fence_before();
    __syncthreads();
    // every CTA's barriers must exist before anybody arrives on them remotely -- but the first remote operation is
    // the exchange at the END of step 0, ~4000 clocks of purely local work away.  The four CTAs of a cluster start
    // up to ~10 000 clocks apart (launch skew), so: arrive here, wait in front of the first exchange (row warps) /
    // in the teardown (the others), and the early CTAs spend the skew on step 0 instead of in a barrier.
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    bool joined = false;                 // this warp has completed the wait of the start-up barrier
    tc_fence_after();
    const uint32_t tmem = *tmem_ptr;
    if (p.prof && blockIdx.x == 0 && tid == 0) p.prof[193] = (unsigned long long)clock64();

    if (warp < ROW_WARPS) {
        // =============================== ROW WARPS ========================================
        const int q = warp & 3, ch = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
        const bool scorer = ch == 1 && (uint32_t)q == rank;       // quarter q of the rows is scored by CTA q
        uint32_t step_it = 0;
        float upd_s[DZ], upd_c[DZ];
#pragma unroll
        for (int j = 0; j < DZ; ++j) {
            upd_s[j] = j < a.d ? a.norm.std_z[j] : 0.f;
            upd_c[j] = j < a.d ? fmaf(__ldg(p.b3 + j), a.norm.std_z[j], a.norm.mean_z[j]) : 0.f;
            asm volatile("" : "+f"(upd_s[j]), "+f"(upd_c[j]));
        }
        mbar_wait<false>(&w_full[0], 0);             // W3 (read by these warps) has landed
        for (int it = 0; it < p.iters; ++it) {
            const long long tile = p.tile_begin + (long long)it * n_clusters + cluster_id;   // >= tile_end: padding
            const long long k_local = tile * TM + row;
            const bool live = tile < p.tile_end && k_local < a.K_local;
            const long long n_qcols = 4 * ((a.K_local + TM - 1) / TM);
            const long long qcol = tile < p.tile_end ? tile * 4 + q : -1;
            float x[DT];
            ScoreAcc sc;
            load_start<ROWS, DT>(a, live, k_local, x);     // every CTA of the cluster holds this tile's rows
            if (scorer) score_init<DT>(a.plan, a.wp_index, x, sc);
            float act[SS_MAX_DA];
#pragma unroll
            for (int j = 0; j < SS_MAX_DA; ++j) act[j] = 0.f;
            ActionCursor cur;
            action_cursor_init(cur);
            if (ch == 0 && live) {
#pragma unroll
                for (int j = 0; j < SS_MAX_DA; ++j)
                    if (j < a.da) act[j] = fetch_action_seq(a.act, cur, k_local, a.k_offset + k_local, 0, j);
            }
            for (int t = 0; t < a.H; ++t, ++step_it) {
                const uint32_t ph = step_it & 1;
                const bool trace_on = it == 0 && warp == 0;
                const int trace_t = t;
                TQ_TRACE(0);
                // this step's exchange: 4 sources x 128 rows x 16 bytes land on z_full[ph] (its previous phase,
                // two steps ago, completed before this thread left that step)
                if (tid == 0) mbar_expect_tx(&z_full[ph], QUAD * TM * 16);
                // ---- layer-1 A operand: hi/lo split of the normalised (state, action) (as in mpc_tc.cu)
                if (ch == 0) {
                    float xin[MAXIN];
#pragma unroll
                    for (int j = 0; j < MAXIN; ++j) xin[j] = 0.f;
#pragma unroll
                    for (int j = 0; j < DZ; ++j)
                        if (j < MAXIN) xin[j] = (x[j] - a.norm.mean_x[j]) * a.norm.inv_std_x[j];
#pragma unroll
                    for (int j = 0; j < SS_MAX_DA; ++j)
                        if (DZ + j < MAXIN) xin[DZ + j] = (act[j] - a.norm.mean_y[j]) * a.norm.inv_std_y[j];
                    float slot[K1T];
#pragma unroll
                    for (int s = 0; s < K1T; ++s) slot[s] = 0.f;
#pragma unroll
                    for (int j = 0; j < MAXIN; ++j) {
                        const float hi = bf16_hi(xin[j]);
                        const float lo = xin[j] - hi;
                        slot[3 * j] = hi;
                        slot[3 * j + 1] = hi;
                        slot[3 * j + 2] = lo;
                    }
                    slot[K1T - 2] = 1.f;
                    slot[K1T - 1] = 1.f;
#pragma unroll
                    for (int kc = 0; kc < K1T / 8; ++kc) {
                        uint4 v;
                        v.x = pack_bf16(slot[8 * kc], slot[8 * kc + 1]);
                        v.y = pack_bf16(slot[8 * kc + 2], slot[8 * kc + 3]);
                        v.z = pack_bf16(slot[8 * kc + 4], slot[8 * kc + 5]);
                        v.w = pack_bf16(slot[8 * kc + 6], slot[8 * kc + 7]);
                        *reinterpret_cast<uint4*>(a1s + kc * (TM * 16) + row * 16) = v;
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(x_ready);
                }
                TQ_TRACE(1);
                // ---- layer-1 epilogue: relu, bf16, becomes the layer-2 A operand (as in mpc_tc.cu: even
                // chunks sit in the dead H1 columns and are converted in place, odd chunks in the two
                // accumulator slots)
                for (int c0 = 0; c0 < NCH; c0 += 2) {
                    const uint32_t slot_i = (uint32_t)(c0 >> 1);
                    uint32_t v0[32], v1[32], pk0[16], pk1[16];
                    if (c0 == 0) mbar_wait<false>(&l1_full[0], ph);
                    TQ_TRACE(2 + c0);
                    tc_fence_after();
                    tmem_ld32(lane_addr + COL_H1 + slot_i * NC + ch * CPT, v0);
                    tmem_ld32(lane_addr + COL_H1 + slot_i * NC + ch * CPT + 32, v1);
                    tmem_wait_ld();
                    asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");   // both threads of the row have loaded
#pragma unroll
                    for (int c2 = 0; c2 < 16; ++c2) {
                        pk0[c2] = pack_bf16_relu(__uint_as_float(v0[2 * c2]), __uint_as_float(v0[2 * c2 + 1]));
                        pk1[c2] = pack_bf16_relu(__uint_as_float(v1[2 * c2]), __uint_as_float(v1[2 * c2 + 1]));
                    }
                    tmem_st16(lane_addr + COL_H1 + c0 * (NC / 2) + ch * (CPT / 2), pk0);
                    tmem_st16(lane_addr + COL_H1 + c0 * (NC / 2) + ch * (CPT / 2) + 16, pk1);
                    if (c0 == 0) {
                        mbar_wait<false>(&l1_full[1], ph);
                        tc_fence_after();
                    }
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT, v0);
                    tmem_ld32(lane_addr + COL_ACC + slot_i * NC + ch * CPT + 32, v1);
                    tmem_wait_st();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&h1_ready[c0]);
                    tmem_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&acc_free[slot_i]);
#pragma unroll
                    for (int c2 = 0; c2 < 16; ++c2) {
                        pk0[c2] = pack_bf16_relu(__uint_as_float(v0[2 * c2]), __uint_as_float(v0[2 * c2 + 1]));
                        pk1[c2] = pack_bf16_relu(__uint_as_float(v1[2 * c2]), __uint_as_float(v1[2 * c2 + 1]));
                    }
                    tmem_st16(lane_addr + COL_H1 + (c0 + 1) * (NC / 2) + ch * (CPT / 2), pk0);
                    tmem_st16(lane_addr + COL_H1 + (c0 + 1) * (NC / 2) + ch * (CPT / 2) + 16, pk1);
                    tmem_wait_st();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&h1_ready[c0 + 1]);
                    TQ_TRACE(3 + c0);
                }
                // ---- in the shadow of the layer-2 MMAs
                if (scorer) {
                    score_row<DT>(a, t, x, sc, live, k_local, qcol, n_qcols, lane);
                } else if (ch == 0 && live && t + 1 < a.H) {
#pragma unroll
                    for (int j = 0; j < SS_MAX_DA; ++j)
                        if (j < a.da) act[j] = fetch_action_seq(a.act, cur, k_local, a.k_offset + k_local, t + 1, j);
                }
                // ---- layer-2 epilogue of THIS CTA's 128 units, fused with its share of layer 3
                float2 zacc[DZ];
#pragma unroll
                for (int j = 0; j < DZ; ++j) zacc[j] = make_float2(0.f, 0.f);
                {
                    TQ_TRACE(6);
                    mbar_wait<false>(&acc_full[0], ph);
                    TQ_TRACE(7);
                    tc_fence_after();
                    uint32_t v0[32], v1[32];
                    tmem_ld32(lane_addr + COL_ACC + ch * CPT, v0);
                    tmem_ld32(lane_addr + COL_ACC + ch * CPT + 32, v1);
                    tmem_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&acc_free[0]);
                    const float* wrow = w3s + (size_t)(((int)rank * NC + ch * CPT) / 2) * (2 * DZP);
#pragma unroll
                    for (int j2 = 0; j2 < CPT / 2; ++j2) {
                        const uint32_t ua = j2 < 16 ? v0[(2 * j2) & 31] : v1[(2 * j2) & 31];
                        const uint32_t ub = j2 < 16 ? v0[(2 * j2 + 1) & 31] : v1[(2 * j2 + 1) & 31];
                        const float2 hh = make_float2(fmaxf(__uint_as_float(ua), 0.f), fmaxf(__uint_as_float(ub), 0.f));
                        const float* wp = wrow + j2 * (2 * DZP);
#pragma unroll
                        for (int jq = 0; jq < DZP / 2; ++jq) {
                            const float4 w = *reinterpret_cast<const float4*>(wp + 4 * jq);
                            if (2 * jq < DZ) zacc[2 * jq] = __ffma2_rn(hh, make_float2(w.x, w.y), zacc[2 * jq]);
                            if (2 * jq + 1 < DZ)
                                zacc[2 * jq + 1] = __ffma2_rn(hh, make_float2(w.z, w.w), zacc[2 * jq + 1]);
                        }
                    }
                }
                TQ_TRACE(8);
                // ---- all-reduce of the partial deltas over the cluster.  The two column halves of a row meet
                // through local shared memory; the ch-0 thread then sends the row's partial (one 16-byte
                // st.async per destination, completing transaction bytes on the destination's barrier of this
                // step's parity) to all four CTAs, and everybody adds the four partials in rank order.
                {
#pragma unroll
                    for (int j = 0; j < DZ; ++j) zx[(j * TPR + ch) * TM + row] = zacc[j].x + zacc[j].y;
                    asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
                    float4* zbuf = zq + (size_t)ph * (QUAD * TM);
                    if (!joined) {
                        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
                        joined = true;
                    }
                    if (ch == 0) {
                        float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                        for (int j = 0; j < DZ; ++j) part[j] = zx[(j * TPR) * TM + row] + zx[(j * TPR + 1) * TM + row];
                        const uint32_t dst_local = smem_u32(zbuf + rank * TM + row), bar_local = smem_u32(&z_full[ph]);
#pragma unroll
                        for (uint32_t dst = 0; dst < QUAD; ++dst) {
                            uint32_t dst_addr, bar_addr;
                            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst_addr) : "r"(dst_local), "r"(dst));
                            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar_addr) : "r"(bar_local), "r"(dst));
                            asm volatile(
                                "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::
                                    "r"(dst_addr), "f"(part[0]), "f"(part[1]), "f"(part[2]), "f"(part[3]), "r"(bar_addr)
                                : "memory");
                        }
                    }
                    TQ_TRACE(9);
                    mbar_wait_cluster(&z_full[ph], (step_it >> 1) & 1);
                    TQ_TRACE(10);
                    // fixed order (CTA 0, 1, 2, 3): the four copies of the state stay bit-identical
                    const float4 p0 = zbuf[row], p1 = zbuf[TM + row], p2 = zbuf[2 * TM + row], p3 = zbuf[3 * TM + row];
                    const float zz[4] = {((p0.x + p1.x) + p2.x) + p3.x, ((p0.y + p1.y) + p2.y) + p3.y,
                                         ((p0.z + p1.z) + p2.z) + p3.z, ((p0.w + p1.w) + p2.w) + p3.w};
#pragma unroll
                    for (int j = 0; j < DZ; ++j) x[j] += fmaf(zz[j], upd_s[j], upd_c[j]);
                }
                TQ_TRACE(11);
            }
            if (p.prof && blockIdx.x == 0 && tid == 0 && it == 0) p.prof[194] = (unsigned long long)clock64();
            if (scorer) {
                score_row<DT>(a, a.H, x, sc, live, k_local, qcol, n_qcols, lane);
                if (live && a.scores_out) a.scores_out[k_local] = sc.score;
            }
        }
    } else if (warp == ROW_WARPS) {
        // ================================= MMA ISSUER ========================================
        const uint32_t a1_addr = smem_u32(a1s), w1_addr = smem_u32(w1s), w2_addr = smem_u32(w2s);
        uint32_t step_it = 0;
        const long long steps = (long long)p.iters * a.H;
        for (long long s = 0; s < steps; ++s, ++step_it) {
            const uint32_t ph = step_it & 1;
            const bool trace_on = s < a.H;
            const int trace_t = (int)s;
            // layer 1 overwrites both accumulator slots: slot 0 was last used by the previous step's layer-2
            // chunk (second drain of that step), slot 1 by its layer-1 chunk 3
            mbar_wait2(&acc_free[0], 1u, &acc_free[1], ph ^ 1u);
            if (s == 0) mbar_wait<false>(&w_full[0], 0);
            mbar_wait<false>(x_ready, ph);
            TQ_TRACE(20);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const uint32_t d0 = tmem + ((c & 1) ? COL_ACC : COL_H1) + (uint32_t)(c >> 1) * NC;
#pragma unroll
                    for (int ks = 0; ks < K1T / 16; ++ks)
                        umma1_ss(d0, make_desc(a1_addr + ks * 2 * (TM * 16), TM),
                                 make_desc(w1_addr + c * (2 * W1_CHUNK_BYTES) + ks * 2 * (NC * 16), NC), IDESC, ks);
                    if (c == 0) tc_commit_one(&l1_full[0]);
                    else if (c == NCH - 1) tc_commit_one(&l1_full[1]);
                }
            }
            __syncwarp();
            TQ_TRACE(21);
            // layer 2, this CTA's chunk: D = acc slot 0 (its layer-1 occupant, chunk 1, must be drained: the
            // first drain of this step; every row warp arrives there after h1_ready[0], so the wait also
            // covers "H1 chunk 0 is converted"), K streamed in 128-wide halves as their layer-1 chunks finish
            if (s == 0) mbar_wait<false>(&w_full[1], 0);
            mbar_wait<false>(&acc_free[0], 0u);
            TQ_TRACE(22);
            const uint32_t d_tmem = tmem + COL_ACC;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                if (c > 0) mbar_wait<false>(&h1_ready[c], ph);
                TQ_TRACE(23 + c);
                tc_fence_after();
                if (elect_one()) {
                    const int ksl = c >> 1;
#pragma unroll
                    for (int k8 = 0; k8 < NC / 16; ++k8) {
                        const int ks = (c & 1) * (NC / 16) + k8;                 // K step inside the 256-wide block
                        umma1_ts(d_tmem, tmem + COL_H1 + ksl * (KSLAB / 2) + ks * 8,
                                 make_desc(w2_addr + ksl * (2 * BLOCK_BYTES) + ks * 2 * (NC * 16), NC), IDESC, (c | k8) != 0);
                    }
                    if (c == NCH - 1) tc_commit_one(&acc_full[0]);
                }
                __syncwarp();
                TQ_TRACE(27 + c);
            }
        }
    }
    // ---- teardown ---------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if (!joined) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    cluster_sync_all();                  // nobody leaves while a peer may still write into its buffers
    tc_fence_after();
    if (p.prof && blockIdx.x == 0 && tid == 0) p.prof[195] = (unsigned long long)clock64();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
}

}  // namespace tcq

// the quad kernel serves models whose operand images have four 128-unit chunks and d <= 4
bool mpc_tc_quad_supported(const ss_ctx* c) { return c->tc_ready && c->tc_hp == tcq::HP && c->d <= 4; }

// clusters of four CTAs that can be co-resident (0 when the launch configuration is not possible)
int mpc_tc_quad_clusters(ss_ctx* c) {
    using namespace tcq;
    if (c->tc_quad_clusters >= 0) return c->tc_quad_clusters;
    c->tc_quad_clusters = 0;
    const size_t smem = Smem::END + 128;
    auto kern = mpc_rollout_tc_quad_kernel<4, 3, 16>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(QUAD * 64);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = QUAD;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {
        (void)cudaGetLastError();
        n = 0;
    }
    c->tc_quad_clusters = n;
    return n;
}

int mpc_tc_quad_launch(ss_ctx* c, const RolloutArgs& a, int* grid_blocks_out) {
    using namespace tcq;
    if (!mpc_tc_quad_supported(c)) SS_FAIL(c, SS_EUNSUPPORTED, "mpc: the 4-CTA tcgen05 kernel does not serve this model");
    Params p;
    std::memset(&p, 0, sizeof(p));
    p.w1_img = c->tc_w1.as<__nv_bfloat16>();
    p.w2_img = c->tc_w2.as<__nv_bfloat16>();
    p.w3 = c->tc_w3.as<float>();
    p.b3 = c->tc_b3.as<float>();
    const long long tiles = (a.K_local + TM - 1) / TM;
    p.tile_begin = 0;
    p.tile_end = tiles;
    p.prof = nullptr;
    if (getenv("SS_TC_TRACE")) {
        SS_CUDA_CHECK(c, c->tc_misc.ensure((3 * 256 + 2) * 8));
        SS_CUDA_CHECK(c, cudaMemsetAsync(c->tc_misc.p, 0, (3 * 256 + 2) * 8, c->stream));
        p.prof = c->tc_misc.as<unsigned long long>();
    }
    const int max_clusters = mpc_tc_quad_clusters(c);
    if (max_clusters < 1) SS_FAIL(c, SS_EUNSUPPORTED, "mpc: no 4-CTA cluster fits on this device");
    const int clusters = (int)std::min<long long>(tiles, max_clusters);
    p.iters = (int)((tiles + clusters - 1) / clusters);
    if (grid_blocks_out) *grid_blocks_out = clusters * QUAD;
    const size_t smem = Smem::END + 128;
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(clusters * QUAD);
    cfg.blockDim = dim3(THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = QUAD;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    // the layout of the pair kernel's images (mpc_tc_prepare), instantiated for exactly that layout
    const int dz = c->tc_dz, k1 = c->tc_k1;
#define TCQ_LAUNCH(DT_, DZ_, K1_)                                                                                  \
    do {                                                                                                           \
        auto kern = a.state0_rows ? mpc_rollout_tc_quad_kernel<DT_, DZ_, K1_, true>                                \
                                  : mpc_rollout_tc_quad_kernel<DT_, DZ_, K1_, false>;                               \
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                     \
        if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, kern, a, p);                                            \
    } while (0)
    if (dz == 2 && k1 == 16) TCQ_LAUNCH(4, 2, 16);
    else if (dz == 2 && k1 == 32) TCQ_LAUNCH(4, 2, 32);
    else if (dz == 3 && k1 == 16) TCQ_LAUNCH(4, 3, 16);
    else if (dz == 3 && k1 == 32) TCQ_LAUNCH(4, 3, 32);
    else if (dz == 4 && k1 == 32) TCQ_LAUNCH(4, 4, 32);
    else SS_FAIL(c, SS_EUNSUPPORTED, "mpc: no 4-CTA tcgen05 kernel for this layer-1 layout");
#undef TCQ_LAUNCH
    if (e == cudaSuccess) e = cudaGetLastError();
    c->launches++;
    SS_CUDA_CHECK(c, e);
    if (p.prof) {
        std::vector<unsigned long long> h(3 * 64 + 8);
        SS_CUDA_CHECK(c, cudaMemcpyAsync(h.data(), p.prof, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
        SS_CUDA_CHECK(c, cudaStreamSynchronize(c->stream));
        fprintf(stderr, "[quad trace] entry: barriers %llu tmem alloc %llu first sync %llu\n", h[196] - h[192], h[197] - h[192], h[198] - h[192]);
        fprintf(stderr, "[quad trace] entry->setup done %llu clk | setup->last step end %llu | ->teardown done %llu | step 10 starts %llu after entry\n",
                h[193] - h[192], h[194] - h[193], h[195] - h[194], h[0] - h[192]);
        for (int st = 0; st < 3; ++st) {
            const unsigned long long* ev = &h[st * 64];
            const unsigned long long t0 = ev[0];
            fprintf(stderr, "[quad trace step %d, %d clusters] row: xsplit %llu | l1_full0 %llu epi01 %llu | c2 %llu epi23 %llu | wait acc_full %llu got %llu | l3 done %llu | sent %llu z_full %llu | end %llu\n",
                    10 + st, clusters, ev[1] - t0, ev[2] - t0, ev[3] - t0, ev[4] - t0, ev[5] - t0, ev[6] - t0, ev[7] - t0, ev[8] - t0, ev[9] - t0, ev[10] - t0, ev[11] - t0);
            fprintf(stderr, "[quad trace step %d] mma: x_ready %llu | L1 issued %llu | acc_free0 %llu | h1 %llu %llu %llu %llu | L2 issued %llu %llu %llu %llu\n",
                    10 + st, ev[20] - t0, ev[21] - t0, ev[22] - t0, ev[23] - t0, ev[24] - t0, ev[25] - t0, ev[26] - t0, ev[27] - t0, ev[28] - t0, ev[29] - t0, ev[30] - t0);
        }
    }
    return SS_OK;
}
